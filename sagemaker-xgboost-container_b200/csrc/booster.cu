// booster.cu -- DMatrix / Booster implementation: the round loop of `xgb.train` (Booster.update) on the device.
// Reference call sites served: algorithm_mode/train.py:367-376,432-442 (xgb.train), serve_utils.py:244-250
// (Booster.predict), data_utils.py:309-313,361,384 (DMatrix construction).  Upstream behaviour restated:
// src/learner.cc (UpdateOneIter, EvalOneIter, base_score), src/gbm/gbtree.cc (DoBoost, one tree per class).
#include "booster.h"
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstring>
#include <functional>
#include "comm.h"

namespace b200 {

long long g_kernel_launches = 0;

// ---------------------------------------------------------------------------------------------
// process-wide device context
// ---------------------------------------------------------------------------------------------
namespace {
struct DeviceCtx {
  cudaStream_t stream = nullptr; int num_sms = 148; bool ok = false; std::string why;
  DeviceCtx() {
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) { why = std::string("no CUDA device available (") + cudaGetErrorString(e) + ")"; cudaGetLastError(); return; }
    int dev = 0;
    if (const char* lr = getenv("LOCAL_RANK")) { dev = atoi(lr) % count; }
    if (const char* d = getenv("B200XGB_DEVICE")) { dev = atoi(d) % count; }
    if (cudaSetDevice(dev) != cudaSuccess) { why = "cudaSetDevice failed"; return; }
    if (cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking) != cudaSuccess) { why = "cudaStreamCreate failed"; return; }
    cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
    ok = true;
  }
};
DeviceCtx& ctx() { static DeviceCtx c; if (!c.ok) throw Error("b200xgb: " + c.why + "; this library has no CPU fallback"); return c; }
std::atomic<uint64_t> g_uid{1};
}  // namespace

cudaStream_t engine_stream() { return ctx().stream; }
int engine_num_sms() { return ctx().num_sms; }

// ---------------------------------------------------------------------------------------------
// DMatrix
// ---------------------------------------------------------------------------------------------
DMatrix::DMatrix() : uid(g_uid++) {}

void DMatrix::finish_upload(float missing) {
  cudaStream_t s = engine_stream();
  const int64_t count = n * F;
  const bool use_missing = !std::isnan(missing);
  DevBuf<unsigned long long> cnt; cnt.alloc(1); cnt.zero(s);
  launch_count_nan(X.p, count, missing, use_missing ? 1 : 0, cnt.p, s);
  if (use_missing) launch_replace_missing(X.p, count, missing, s);
  unsigned long long c = 0;
  CUDA_OK(cudaMemcpyAsync(&c, cnt.p, 8, cudaMemcpyDeviceToHost, s));
  Comm::get().sync_stream(s);
  has_missing = c > 0;
}

std::unique_ptr<DMatrix> DMatrix::from_dense(const float* data, int64_t nrow, int ncol, float missing) {
  B200_CHECK(nrow >= 0 && ncol >= 0, "DMatrix: negative shape");
  B200_CHECK(nrow < (int64_t)0x7fffffff, "DMatrix: more than 2^31-1 rows per GPU are not supported");
  auto dm = std::make_unique<DMatrix>();
  dm->n = nrow; dm->F = ncol;
  cudaStream_t s = engine_stream();
  dm->X.alloc((size_t)nrow * ncol);
  if (nrow * ncol > 0) {
    CUDA_OK(cudaMemcpyAsync(dm->X.p, data, sizeof(float) * (size_t)nrow * ncol, cudaMemcpyHostToDevice, s));
  }
  dm->finish_upload(missing);
  return dm;
}

std::unique_ptr<DMatrix> DMatrix::from_device(const float* dptr, int64_t nrow, int ncol, float missing) {
  B200_CHECK(nrow >= 0 && ncol >= 0 && nrow < (int64_t)0x7fffffff, "DMatrix: bad shape");
  auto dm = std::make_unique<DMatrix>();
  dm->n = nrow; dm->F = ncol;
  cudaStream_t s = engine_stream();
  dm->X.alloc((size_t)nrow * ncol);
  CUDA_OK(cudaDeviceSynchronize());       // the producer (e.g. a torch stream) must be done before we read its buffer
  if (nrow * ncol > 0) CUDA_OK(cudaMemcpyAsync(dm->X.p, dptr, sizeof(float) * (size_t)nrow * ncol, cudaMemcpyDeviceToDevice, s));
  dm->finish_upload(missing);
  return dm;
}

// DMatrix::from_csr / from_columns: ingest.cu (device-side densify / column transpose, no dense host copy)

__global__ void gather_rows_kernel(const float* X, int F, const int* idx, int64_t len, float* out) {
  const int64_t total = len * F;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = i / F; int f = (int)(i % F);
    out[i] = X[(int64_t)idx[r] * F + f];
  }
}

std::unique_ptr<DMatrix> DMatrix::slice(const int* idx, int64_t len) const {
  for (int64_t i = 0; i < len; ++i) B200_CHECK(idx[i] >= 0 && idx[i] < n, "DMatrix.slice: row index out of range");
  auto dm = std::make_unique<DMatrix>();
  dm->n = len; dm->F = F; dm->has_missing = has_missing;
  dm->feature_names = feature_names; dm->feature_types = feature_types;
  cudaStream_t s = engine_stream();
  dm->X.alloc((size_t)len * F);
  if (len * F > 0) {
    DevBuf<int> didx; didx.alloc(len);
    CUDA_OK(cudaMemcpyAsync(didx.p, idx, sizeof(int) * len, cudaMemcpyHostToDevice, s));
    int grid = (int)std::min<int64_t>((len * F + 255) / 256, 148 * 16);
    gather_rows_kernel<<<grid, 256, 0, s>>>(X.p, F, didx.p, len, dm->X.p); ++g_kernel_launches;
    CUDA_OK(cudaGetLastError());
    Comm::get().sync_stream(s);
  }
  auto take = [&](const std::vector<float>& src, size_t per_row) { std::vector<float> o; if (src.empty()) return o; o.resize(len * per_row);
    for (int64_t i = 0; i < len; ++i) for (size_t k = 0; k < per_row; ++k) o[i * per_row + k] = src[(size_t)idx[i] * per_row + k]; return o; };
  if (!labels.empty()) { auto v = take(labels, 1); dm->set_float_info("label", v.data(), v.size()); }
  if (!weights.empty()) { auto v = take(weights, 1); dm->set_float_info("weight", v.data(), v.size()); }
  if (!base_margin.empty() && n > 0) { size_t per = base_margin.size() / n; auto v = take(base_margin, per); dm->set_float_info("base_margin", v.data(), v.size()); }
  return dm;
}

void DMatrix::set_float_info(const std::string& field, const float* v, size_t len) {
  cudaStream_t s = engine_stream();
  auto put = [&](std::vector<float>& h, DevBuf<float>& d) {
    h.assign(v, v + len); d.alloc(len);
    if (len) { CUDA_OK(cudaMemcpyAsync(d.p, h.data(), sizeof(float) * len, cudaMemcpyHostToDevice, s)); Comm::get().sync_stream(s); }
  };
  if (field == "label") put(labels, d_labels);
  else if (field == "weight") {
    for (size_t i = 0; i < len; ++i) B200_CHECK(v[i] >= 0 && !std::isnan(v[i]), "Weights must be positive values.");
    put(weights, d_weights);
    binned = false;      // weighted quantiles depend on the weights
  }
  else if (field == "base_margin") put(base_margin, d_base_margin);
  else throw Error("Unknown float field name: " + field);
}

const std::vector<float>& DMatrix::get_float_info(const std::string& field) const {
  if (field == "label") return labels;
  if (field == "weight") return weights;
  if (field == "base_margin") return base_margin;
  throw Error("Unknown float field name: " + field);
}

void DMatrix::bin_with_cuts() {
  cudaStream_t s = engine_stream();
  feature_layout(F, &ngroups, &tw, &ntail);
  ++binned_version;
  d_cut_ptrs.alloc(cuts.ptrs.size()); d_cut_vals.alloc(cuts.vals.size()); d_min_vals.alloc(cuts.mins.size());
  CUDA_OK(cudaMemcpyAsync(d_cut_ptrs.p, cuts.ptrs.data(), sizeof(int) * cuts.ptrs.size(), cudaMemcpyHostToDevice, s));
  if (!cuts.vals.empty()) CUDA_OK(cudaMemcpyAsync(d_cut_vals.p, cuts.vals.data(), sizeof(float) * cuts.vals.size(), cudaMemcpyHostToDevice, s));
  if (!cuts.mins.empty()) CUDA_OK(cudaMemcpyAsync(d_min_vals.p, cuts.mins.data(), sizeof(float) * cuts.mins.size(), cudaMemcpyHostToDevice, s));
  // 512 pad rows: the root kernel's bulk copies always move whole tiles (rows past n are masked in the kernel)
  const size_t n_alloc = (size_t)n + 512;
  bins.alloc(n_alloc * ngroups * kSlots); bins_tail.alloc(tw ? n_alloc * tw : 0);
  CUDA_OK(cudaMemsetAsync(bins.p + (size_t)n * ngroups * kSlots, 0, (size_t)512 * ngroups * kSlots, s));
  if (tw) CUDA_OK(cudaMemsetAsync(bins_tail.p + (size_t)n * tw, 0, (size_t)512 * tw, s));
  launch_bin(X.p, n, F, ngroups, tw, d_cut_ptrs.p, d_cut_vals.p, bins.p, bins_tail.p, s);
  gather_stride = ngroups * kSlots;
  bins_gather.release();
  static const bool no_aligned = getenv("B200XGB_NO_ALIGNED_ROWS") != nullptr;
  if (ngroups * kSlots == 96 && !no_aligned) {           // 96 B rows straddle 128 B DRAM lines half of the time: the gathered levels read an aligned copy
    gather_stride = 128;
    bins_gather.alloc((size_t)n * 128 + 128);
    launch_pad_rows(bins.p, n, 96, bins_gather.p, 128, s);
  }
  bins_col.alloc((size_t)std::max(F, 1) * n);
  launch_transpose_bins(bins.p, bins_tail.p, n, F, ngroups, tw, bins_col.p, s);
  Comm::get().sync_stream(s);
  binned = true;
}

void DMatrix::set_cuts(const HostCuts& c) {
  B200_CHECK((int)c.ptrs.size() == F + 1 && (int)c.mins.size() == F, "SetCuts: cut_ptrs/min_vals do not match the number of features");
  for (int f = 0; f < F; ++f) B200_CHECK(c.ptrs[f + 1] - c.ptrs[f] >= 1 && c.ptrs[f + 1] - c.ptrs[f] <= (has_missing ? 255 : 256), "SetCuts: 1..256 cuts per feature (255 with missing values)");
  cuts = c; binned_max_bin = -1;
  bin_with_cuts();
}

void DMatrix::ensure_binned(int max_bin) {
  if (binned && (binned_max_bin == max_bin || binned_max_bin == -1)) return;
  B200_CHECK(max_bin >= 2, "max_bin must be >= 2");
  cudaStream_t s = engine_stream();
  Comm& comm = Comm::get();
  if (!comm.distributed()) {
    compute_cuts_device(X.p, n, F, weights.empty() ? nullptr : d_weights.p, max_bin, has_missing, &cuts, s);
  } else {
    // every rank summarises its shard (exact when a feature has <= cap distinct values), the summaries are
    // all-gathered and merged, and every rank derives the same cuts.
    const int cap = 2048;
    int hm = has_missing ? 1 : 0;
    {   // has_missing must agree across ranks (bin code 255 reservation)
      DevBuf<unsigned> flag; flag.alloc(1); unsigned v = (unsigned)hm;
      CUDA_OK(cudaMemcpyAsync(flag.p, &v, 4, cudaMemcpyHostToDevice, s));
      comm.allreduce_max_u32(flag.p, 1, s);
      CUDA_OK(cudaMemcpyAsync(&v, flag.p, 4, cudaMemcpyDeviceToHost, s)); Comm::get().sync_stream(s);
      has_missing = v != 0;
    }
    std::vector<FeatureSummary> local;
    compute_summaries_device(X.p, n, F, weights.empty() ? nullptr : d_weights.p, cap, &local, s);
    const size_t per_feat = (size_t)(cap + 2);
    const size_t rec = per_feat * (sizeof(float) + sizeof(double)) + sizeof(double);   // vals, weights, count
    std::vector<unsigned char> sendbuf((size_t)F * rec, 0);
    for (int f = 0; f < F; ++f) {
      unsigned char* p = sendbuf.data() + (size_t)f * rec;
      double cntd = (double)local[f].vals.size(); memcpy(p, &cntd, 8);
      memcpy(p + 8, local[f].vals.data(), sizeof(float) * local[f].vals.size());
      memcpy(p + 8 + per_feat * sizeof(float), local[f].weights.data(), sizeof(double) * local[f].weights.size());
    }
    const int W = comm.world();
    DevBuf<unsigned char> dsend, drecv; dsend.alloc(sendbuf.size()); drecv.alloc(sendbuf.size() * W);
    CUDA_OK(cudaMemcpyAsync(dsend.p, sendbuf.data(), sendbuf.size(), cudaMemcpyHostToDevice, s));
    comm.allgather_bytes(dsend.p, drecv.p, sendbuf.size(), s);
    std::vector<unsigned char> all(sendbuf.size() * W);
    CUDA_OK(cudaMemcpyAsync(all.data(), drecv.p, all.size(), cudaMemcpyDeviceToHost, s));
    Comm::get().sync_stream(s);
    std::vector<FeatureSummary> merged(F);
    for (int f = 0; f < F; ++f) {
      std::vector<std::pair<float, double>> pts;
      for (int r = 0; r < W; ++r) {
        const unsigned char* p = all.data() + (size_t)r * sendbuf.size() + (size_t)f * rec;
        double cntd; memcpy(&cntd, p, 8); size_t c = (size_t)cntd;
        const float* v = reinterpret_cast<const float*>(p + 8);
        std::vector<double> w(c); memcpy(w.data(), p + 8 + per_feat * sizeof(float), sizeof(double) * c);
        for (size_t i = 0; i < c; ++i) pts.emplace_back(v[i], w[i]);
      }
      std::stable_sort(pts.begin(), pts.end(), [](const std::pair<float, double>& a, const std::pair<float, double>& b) { return a.first < b.first; });
      for (auto& pw : pts) {
        if (!merged[f].vals.empty() && merged[f].vals.back() == pw.first) merged[f].weights.back() += pw.second;
        else { merged[f].vals.push_back(pw.first); merged[f].weights.push_back(pw.second); }
      }
    }
    cuts_from_summaries(merged, max_bin, has_missing, &cuts);
  }
  binned_max_bin = max_bin;
  bin_with_cuts();
}

// ---------------------------------------------------------------------------------------------
// tree builder: device buffers + the per-tree launch sequence
// ---------------------------------------------------------------------------------------------
__global__ void pack_tree_kernel(TreeArrays t, const int* n_nodes, DevNode* out, int cap) {
  const int nn = *n_nodes;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < cap; i += gridDim.x * blockDim.x) {
    DevNode d;
    if (i < nn) { d.cond = t.split_cond[i]; d.left = t.left[i]; d.right = t.right[i]; d.fidx_dl = (unsigned)t.split_index[i] | ((unsigned)t.default_left[i] << 31); }
    else { d.cond = 0.f; d.left = -1; d.right = -1; d.fidx_dl = 0; }
    out[i] = d;
  }
}

// Constant-hessian root pass (reg:squarederror without weights / subsampling): the H plane of the root histogram is the
// same every round, so it is snapshotted once and later rounds start the root slot from it and accumulate G only.
__global__ void snapshot_h_kernel(const GH64* slot, long long* cache, size_t entries) {
  for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < entries; e += (size_t)gridDim.x * blockDim.x) cache[e] = slot[e].h;
}
__global__ void slot_from_cache_kernel(GH64* slot, const long long* cache, size_t entries) {
  for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < entries; e += (size_t)gridDim.x * blockDim.x) { GH64 v; v.g = 0; v.h = cache[e]; slot[e] = v; }
}

struct PinnedPool {
  std::vector<std::pair<char*, size_t>> chunks; size_t cur = 0, off = 0;
  ~PinnedPool() { for (auto& c : chunks) cudaFreeHost(c.first); }
  void* take(size_t bytes) {
    bytes = (bytes + 255) & ~(size_t)255;
    while (cur < chunks.size() && off + bytes > chunks[cur].second) { ++cur; off = 0; }
    if (cur >= chunks.size()) { size_t sz = std::max<size_t>(bytes, 4u << 20); char* p = nullptr; CUDA_OK(cudaMallocHost(&p, sz)); chunks.emplace_back(p, sz); off = 0; }
    void* r = chunks[cur].first + off; off += bytes; return r;
  }
  void reset() { cur = 0; off = 0; }
};

struct TreeGraphKey { uint64_t uid, binned_version; const void *margin, *mask, *packed, *bins, *bins_col, *cuts, *mono, *ic_sets, *ic_allowed; int n_ic; int max_depth, max_leaves, lg_iters; float eta, lambda, alpha, gamma, mcw, mds, bynode; unsigned seed; int world, root_mode; int64_t n; };
// The per-tree launch sequence as CUDA graphs.  On one GPU it is a single graph; with NCCL it is cut into SEGMENTS at every
// collective (root + one per level): the segments are replayed as graphs and the all-reduces are issued between them as
// ordinary stream operations, so no NCCL call is ever captured (a capture with lazily connecting NCCL channels hung an
// 8-rank run in round 1) while a tree still costs ~2 host operations per level instead of ~13.
struct TreeGraph {
  std::vector<cudaGraphExec_t> segs; std::vector<std::function<void()>> colls;      // colls[i] runs after segs[i]
  TreeGraphKey key; long long launches = 0;
  TreeGraph() { memset(&key, 0, sizeof key); }
  void destroy() { for (auto e : segs) if (e) cudaGraphExecDestroy(e); segs.clear(); colls.clear(); }
};

struct GrowerImpl {
  int64_t n = 0; int ngroups = 0, tw = 0, max_depth = 0, max_nodes = 0, cap_nodes = 0, max_level_nodes = 0, region = 0;
  int lg_iters = 0;                        // grow_policy=lossguide: expansions per tree (0 = depthwise)
  size_t slot_stride = 0;                  // GH64 entries per histogram slot
  int64_t gp_stride = 0;                   // rows reserved per class in gpair
  int64_t global_n = 0;                    // rows of the whole job (sum over ranks)
  DevBuf<long long> root_h_cache; uint64_t root_h_uid = 0, root_h_version = 0; bool root_h_valid = false;
  GrowState gs{}; TreeArrays ta{};
  DevBuf<unsigned char> state_block;       // all GrowState arrays
  DevBuf<unsigned char> tree_block;        // header + TreeArrays, copied to the host in one piece
  size_t tree_block_bytes = 0;
  DevBuf<GH64> hist_pool; DevBuf<unsigned> ridx0, ridx1, scratch;
  DevBuf<float2> gpair, gp0, gp1; DevBuf<unsigned> tl0, tl1; DevBuf<int> err, tree_index_dev, monotone_dev; DevBuf<unsigned char> feat_mask, ic_path, ic_allowed, ic_sets;
  std::vector<unsigned char> ic_sets_host; // what ic_sets holds
  std::vector<int> monotone_host;          // what monotone_dev holds (re-uploaded when the constraints or the feature count change)
  DevBuf<double> dsum;
  PinnedPool pinned; std::vector<cudaEvent_t> free_events;
  DevBuf<DevNode> packed; std::vector<TreeGraph> graphs; std::vector<char> eager_done;
  TreeGraph* capturing = nullptr;          // set while enqueue_tree runs under stream capture: collectives cut the capture

  void ensure(int64_t n_, int ngroups_, int tw_, int max_depth_, int K, int lg_iters_ = 0) {
    const int64_t stride_ = (n_ + 63) & ~(int64_t)63;
    if (n == n_ && ngroups == ngroups_ && tw == tw_ && max_depth == max_depth_ && lg_iters == lg_iters_ && gpair.n >= (size_t)stride_ * K + 512) return;
    if (lg_iters_ == 0) B200_CHECK(max_depth_ >= 1 && max_depth_ <= kMaxDepth, "max_depth must be in [1, 16] for the B200 depth-wise hist builder");
    n = n_; ngroups = ngroups_; tw = tw_; max_depth = max_depth_; lg_iters = lg_iters_; gp_stride = stride_; root_h_valid = false;
    if (peer_reduce_active()) {                     // peers still map the buffers that are about to be freed: unmap everywhere first
      peer_reduce_close();
      DevBuf<unsigned> bar; bar.alloc(1); bar.zero(engine_stream());
      Comm::get().allreduce_max_u32(bar.p, 1, engine_stream());
      Comm::get().sync_stream(engine_stream());
    }
    for (auto& tg : graphs) tg.destroy();
    size_t pool_slots;
    if (lg_iters > 0) {            // lossguide: two children per expansion; "levels" 0 / 1 hold the split node and its children
      max_nodes = 2 * lg_iters + 1; max_level_nodes = 2; region = 0;
      pool_slots = (size_t)lg_iters + kLgFirstFreeSlot;         // root, staging, one fresh slot per expansion
    } else {
      max_nodes = (1 << (max_depth + 1)) - 1; max_level_nodes = 1 << (max_depth - 1); region = max_level_nodes;
      pool_slots = 2 * (size_t)region;
    }
    cap_nodes = (max_nodes + 15) & ~15;
    slot_stride = hist_slot_entries(ngroups, tw);
    const size_t pool_bytes = pool_slots * slot_stride * sizeof(GH64);
    size_t free_b = 0, total_b = 0; cudaMemGetInfo(&free_b, &total_b);
    B200_CHECK(pool_bytes < free_b / 2 + hist_pool.n * sizeof(GH64), "histogram pool for this max_depth / max_leaves / feature count does not fit in device memory");
    hist_pool.alloc(pool_slots * slot_stride);
    ridx0.alloc(n); ridx1.alloc(n);
    gpair.alloc((size_t)gp_stride * K + 512); gpair.zero(engine_stream()); gp0.alloc(n); gp1.alloc(n); err.alloc(1); dsum.alloc(4);
    root_h_cache.alloc(slot_stride);
    tl0.alloc(tw == 4 ? n : 0); tl1.alloc(tw == 4 ? n : 0);
    const unsigned max_tiles = (unsigned)((n + kPartTile - 1) / kPartTile) + max_level_nodes + 1;
    scratch.alloc(3 * (size_t)max_level_nodes + 8);
    // ---- GrowState block
    size_t off = 0; auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; };
    const size_t N = cap_nodes, L = max_level_nodes;
    size_t o_seg_begin = take(4 * N), o_seg_count = take(4 * N), o_slot = take(4 * N), o_sum = take(16 * N), o_rg = take(4 * N), o_w = take(4 * N);
    size_t o_best = take(sizeof(SplitCand) * N), o_bestg = take(sizeof(SplitCand) * N * (ngroups + (tw > 0 ? 1 : 0)));
    size_t o_lnodes = take(4 * (size_t)(kMaxDepth + 1) * L), o_lcount = take(4 * (kMaxDepth + 2));
    size_t o_bnid = take(4 * L), o_bsub = take(4 * L), o_bps = take(4 * L), o_bcount = take(4), o_bprefix = take(4 * (L + 1));
    size_t o_action = take(4 * L), o_tprefix = take(4 * (L + 1)), o_tleft = take(4 * (size_t)max_tiles), o_toff = take(4 * (size_t)max_tiles);
    size_t o_flags = take((size_t)n + 16), o_nleaves = take(4), o_scales = take(16), o_absmax = take(8);
    size_t o_depth = take(4 * N), o_open = take(N), o_nslots = take(4), o_lgdone = take(4), o_lower = take(4 * N), o_upper = take(4 * N);
    state_block.alloc(off); state_block.zero(engine_stream());
    unsigned char* b = state_block.p;
    gs.seg_begin = (unsigned*)(b + o_seg_begin); gs.seg_count = (unsigned*)(b + o_seg_count); gs.hist_slot = (int*)(b + o_slot);
    gs.node_sum = (GH64*)(b + o_sum); gs.root_gain = (float*)(b + o_rg); gs.weight = (float*)(b + o_w);
    gs.best = (SplitCand*)(b + o_best); gs.best_group = (SplitCand*)(b + o_bestg);
    gs.level_nodes = (int*)(b + o_lnodes); gs.level_count = (int*)(b + o_lcount);
    gs.build_nid = (int*)(b + o_bnid); gs.build_sub_nid = (int*)(b + o_bsub); gs.build_parent_slot = (int*)(b + o_bps);
    gs.build_count = (int*)(b + o_bcount); gs.build_prefix = (unsigned*)(b + o_bprefix);
    gs.part_action = (int*)(b + o_action); gs.tile_prefix = (unsigned*)(b + o_tprefix); gs.tile_left = (unsigned*)(b + o_tleft); gs.tile_off = (unsigned*)(b + o_toff);
    gs.lower = (float*)(b + o_lower); gs.upper = (float*)(b + o_upper);
    gs.depth = (int*)(b + o_depth); gs.open = b + o_open; gs.n_slots = (int*)(b + o_nslots); gs.lg_done = (int*)(b + o_lgdone);
    gs.flags = b + o_flags; gs.n_leaves = (int*)(b + o_nleaves); gs.scales = (float*)(b + o_scales); gs.absmax = (unsigned*)(b + o_absmax);
    // ---- tree block: [n_nodes + pad to 64][5 int arrays][4 float arrays][u8 array]
    tree_block_bytes = 64 + 9 * 4 * N + N;
    tree_block.alloc(tree_block_bytes);
    unsigned char* t = tree_block.p;
    gs.n_nodes = (int*)t;
    int* ip = (int*)(t + 64);
    ta.left = ip; ta.right = ip + N; ta.parent = ip + 2 * N; ta.split_index = ip + 3 * N; ta.split_bin = ip + 4 * N;
    float* fp = (float*)(ip + 5 * N);
    ta.split_cond = fp; ta.base_weight = fp + N; ta.loss_chg = fp + 2 * N; ta.sum_hess = fp + 3 * N;
    ta.default_left = (unsigned char*)(fp + 4 * N);
    hist_configure();
    // multi-rank: map the peers' histogram pools / grow-state blocks over NVLink (collective; every rank gets here in its first update)
    global_n = n;
    if (Comm::get().distributed()) {
      peer_reduce_setup({{hist_pool.p, hist_pool.n * sizeof(GH64)}, {state_block.p, state_block.n}}, engine_stream());
      double v = (double)n;
      CUDA_OK(cudaMemcpyAsync(dsum.p, &v, sizeof v, cudaMemcpyHostToDevice, engine_stream()));
      Comm::get().allreduce_sum_f64(dsum.p, 1, engine_stream());
      CUDA_OK(cudaMemcpyAsync(&v, dsum.p, sizeof v, cudaMemcpyDeviceToHost, engine_stream()));
      Comm::get().sync_stream(engine_stream());
      global_n = (int64_t)v;
    }
  }
};

// ranks must agree on the fixed-point grid: it follows the GLOBAL row count of the job (GrowerImpl::global_n, all-reduced
// once), so that N ranks and one GPU train bit-identical models on the same data
static int job_grad_bits(int64_t global_n) { return grad_bits_for(global_n); }
static int job_window_rows(int64_t global_n) { return window_rows_for(global_n); }

// grow_policy=lossguide: expansions per tree = leaves - 1, bounded by max_leaves or by a full tree of max_depth
static int lossguide_iters(const TrainParam& p) {
  if (!p.lossguide) return 0;
  if (p.max_leaves > 0) return std::max(1, p.max_leaves - 1);
  return (1 << p.max_depth) - 1;
}

static TrainParamDev to_dev(const TrainParam& p) {
  TrainParamDev d; d.eta = p.eta; d.lambda = p.lambda; d.alpha = p.alpha; d.gamma = p.gamma; d.min_child_weight = p.min_child_weight;
  d.max_delta_step = p.max_delta_step; d.max_depth = p.max_depth; d.max_leaves = p.max_leaves; return d;
}

// counter-based RNG shared with the oracle (splitmix64 on (seed, stream, index))
static inline uint64_t splitmix64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ULL; x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ULL; x = (x ^ (x >> 27)) * 0x94D049BB133111EBULL; return x ^ (x >> 31);
}
static inline float rng_uniform(uint32_t seed, uint64_t stream, uint64_t idx) {
  uint64_t h = splitmix64(splitmix64(((uint64_t)seed << 32) ^ stream) ^ idx);
  return (float)(h >> 40) * (1.0f / 16777216.0f);
}
// Column sampling (upstream src/common/random.h ColumnSampler: bytree, then bylevel inside it, then bynode inside that; a
// subset keeps max(1, floor(frac * |parent|)) features).  Upstream shuffles with a mt19937; product and oracle share a
// counter-based rule instead: feature f of the parent set is kept iff fewer than `keep` parent features have a smaller
// hash u(stream, f) (ties: lower index first).  Streams: tree 0x1000 + t, level 0x300000 + 64 t + depth, node (eval kernel)
// 0x80000000 + 2^20 t + nid.
std::string subset_mask(const std::string& parent, float frac, unsigned seed, uint64_t stream) {
  if (frac >= 1.0f) return parent;
  const int F = (int)parent.size();
  int cnt = 0; for (int f = 0; f < F; ++f) cnt += parent[f] ? 1 : 0;
  const int keep = std::max(1, (int)std::floor(frac * (float)cnt));
  std::vector<float> u(F);
  for (int f = 0; f < F; ++f) u[f] = rng_uniform(seed, stream, (uint64_t)f);
  std::string m((size_t)F, (char)0);
  for (int f = 0; f < F; ++f) {
    if (!parent[f]) continue;
    int rank = 0;
    for (int g = 0; g < F; ++g) if (parent[g] && (u[g] < u[f] || (u[g] == u[f] && g < f))) ++rank;
    m[f] = rank < keep ? 1 : 0;
  }
  return m;
}
std::string colsample_mask(unsigned seed, int tree_index, int F, float frac) {
  return subset_mask(std::string((size_t)F, (char)1), frac, seed, 0x1000 + (uint64_t)tree_index);
}

// ---------------------------------------------------------------------------------------------
// Booster
// ---------------------------------------------------------------------------------------------
Booster::Booster() {}
Booster::~Booster() {
  if (grower_) { for (auto e : grower_->free_events) cudaEventDestroy(e); delete grower_; }
  for (auto& p : pending_) if (p.ready) cudaEventDestroy(p.ready);
}

static const std::map<std::string, int>& objective_table() {
  static const std::map<std::string, int> t = {{"reg:squarederror", kSquaredError}, {"reg:linear", kSquaredError}, {"binary:logistic", kBinaryLogistic},
    {"reg:logistic", kRegLogistic}, {"binary:logitraw", kLogitRaw}, {"multi:softprob", kSoftprob}, {"multi:softmax", kSoftmax},
    {"reg:squaredlogerror", kSquaredLogError}, {"reg:pseudohubererror", kPseudoHuber}, {"count:poisson", kPoisson}, {"reg:gamma", kGamma},
    {"reg:tweedie", kTweedie}, {"binary:hinge", kHinge}};
  return t;
}

void Booster::set_param(const std::string& k, const std::string& v) {
  if (k == "eval_metric") { if (std::find(eval_metrics_.begin(), eval_metrics_.end(), v) == eval_metrics_.end()) eval_metrics_.push_back(v); }
  else raw_params_[k] = v;
  configured_ = false;
}

void Booster::configure() {
  if (configured_) return;
  auto getf = [&](const char* a, const char* b, float def) { auto it = raw_params_.find(a); if (it == raw_params_.end() && b) it = raw_params_.find(b);
    if (it == raw_params_.end()) return def; try { return std::stof(it->second); } catch (...) { throw Error(std::string("Invalid value for parameter ") + a + ": " + it->second); } };
  auto geti = [&](const char* a, int def) { auto it = raw_params_.find(a); if (it == raw_params_.end()) return def;
    try { return (int)std::stod(it->second); } catch (...) { throw Error(std::string("Invalid value for parameter ") + a + ": " + it->second); } };
  TrainParam p;
  auto ito = raw_params_.find("objective");
  if (ito != raw_params_.end()) objective_name_ = ito->second;
  auto ot = objective_table().find(objective_name_);
  B200_CHECK(ot != objective_table().end(), "Unknown objective function: `" + objective_name_ + "` (supported on the B200 hist path: reg:squarederror, reg:linear, reg:logistic, reg:squaredlogerror, reg:pseudohubererror, reg:gamma, reg:tweedie, count:poisson, binary:logistic, binary:logitraw, binary:hinge, multi:softprob, multi:softmax)");
  p.objective = ot->second;
  if (objective_name_ == "reg:linear") objective_name_ = "reg:squarederror";
  p.num_class = (p.objective == kSoftprob || p.objective == kSoftmax) ? geti("num_class", 0) : 1;
  if (p.objective == kSoftprob || p.objective == kSoftmax) B200_CHECK(p.num_class >= 1, "num_class must be set (>= 1) for multi:softprob / multi:softmax");
  p.max_depth = geti("max_depth", 6); p.max_leaves = geti("max_leaves", 0); p.max_bin = geti("max_bin", 256);
  p.eta = getf("eta", "learning_rate", 0.3f); p.lambda = getf("lambda", "reg_lambda", 1.0f); p.alpha = getf("alpha", "reg_alpha", 0.0f);
  p.gamma = getf("gamma", "min_split_loss", 0.0f); p.min_child_weight = getf("min_child_weight", nullptr, 1.0f);
  p.max_delta_step = getf("max_delta_step", nullptr, 0.0f); p.scale_pos_weight = getf("scale_pos_weight", nullptr, 1.0f);
  p.subsample = getf("subsample", nullptr, 1.0f); p.colsample_bytree = getf("colsample_bytree", nullptr, 1.0f);
  p.colsample_bylevel = getf("colsample_bylevel", nullptr, 1.0f); p.colsample_bynode = getf("colsample_bynode", nullptr, 1.0f);
  p.seed = (unsigned)geti("seed", 0);
  p.huber_slope = getf("huber_slope", nullptr, 1.0f); p.tweedie_variance_power = getf("tweedie_variance_power", nullptr, 1.5f);
  B200_CHECK(p.huber_slope != 0.0f, "Check failed: slope != 0.0 (huber_slope)");
  B200_CHECK(p.tweedie_variance_power >= 1.0f && p.tweedie_variance_power < 2.0f, "tweedie_variance_power must be in interval [1, 2)");
  // count:poisson: max_delta_step defaults to 0.7 for the objective's hessian AND the tree's leaf clipping (upstream learner.cc sets
  // the shared parameter when the user did not)
  if (p.objective == kPoisson) {
    if (raw_params_.find("max_delta_step") == raw_params_.end()) p.max_delta_step = 0.7f;
    p.poisson_max_delta_step = p.max_delta_step;
    B200_CHECK(p.poisson_max_delta_step >= 0.0f, "max_delta_step must be non-negative for count:poisson");
  }
  B200_CHECK(p.lambda >= 0.0f, "Parameter reg_lambda should be greater equal to 0");
  B200_CHECK(p.subsample > 0.0f && p.subsample <= 1.0f, "Parameter subsample should be in (0, 1]");
  auto tm = raw_params_.find("tree_method");
  if (tm != raw_params_.end()) {
    const std::string& t = tm->second;
    B200_CHECK(t == "hist" || t == "auto" || t == "gpu_hist" || t == "approx" || t == "exact",
               "Unknown tree_method: " + t);
    // every method maps onto the device hist builder; exact/approx are accepted for hyperparameter compatibility
  }
  auto bo = raw_params_.find("booster");
  if (bo != raw_params_.end()) B200_CHECK(bo->second == "gbtree", "Only booster=gbtree is implemented on the B200 hist path (got " + bo->second + ")");
  auto gp = raw_params_.find("grow_policy");
  if (gp != raw_params_.end()) {
    B200_CHECK(gp->second == "depthwise" || gp->second == "lossguide", "Invalid grow_policy: " + gp->second + " (depthwise, lossguide)");
    p.lossguide = gp->second == "lossguide" ? 1 : 0;
  }
  interaction_.clear();
  auto ic = raw_params_.find("interaction_constraints");
  if (ic != raw_params_.end()) {                 // "[[0, 1], [2, 3, 4]]": nested lists of feature indices
    int depth = 0; std::string tok; std::vector<int> cur;
    auto flush = [&]() { if (tok.empty()) return; int v = 0; try { v = std::stoi(tok); } catch (...) { throw Error("Invalid interaction_constraints entry: " + tok); }
      B200_CHECK(v >= 0, "interaction_constraints entries must be feature indices (feature names are not supported)"); cur.push_back(v); tok.clear(); };
    for (char ch : ic->second) {
      if (ch == '[' || ch == '(') { ++depth; }
      else if (ch == ']' || ch == ')') { flush(); if (depth == 2 && !cur.empty()) { interaction_.push_back(cur); cur.clear(); } --depth; }
      else if (ch >= '0' && ch <= '9') tok.push_back(ch);
      else { B200_CHECK(ch == ',' || ch == ' ' || ch == '\t' || ch == '\n' || ch == '"' || ch == '\'', std::string("Invalid character in interaction_constraints: ") + ch); flush(); }
    }
    B200_CHECK(depth == 0, "Unbalanced brackets in interaction_constraints");
  }
  monotone_.clear();
  auto mc = raw_params_.find("monotone_constraints");
  if (mc != raw_params_.end()) {                 // "(1,0,-1)" / "1,0,-1" / "[1, 0, -1]": one entry per feature, missing ones are 0
    std::string tok;
    auto flush = [&]() { if (tok.empty()) return; int v = 0; try { v = std::stoi(tok); } catch (...) { throw Error("Invalid monotone_constraints entry: " + tok); }
      B200_CHECK(v >= -1 && v <= 1, "monotone_constraints entries must be -1, 0 or 1"); monotone_.push_back(v); tok.clear(); };
    for (char ch : mc->second) { if (ch == '-' || ch == '+' || (ch >= '0' && ch <= '9')) tok.push_back(ch); else flush(); }
    flush();
    bool any = false; for (int v : monotone_) any |= v != 0;
    if (!any) monotone_.clear();
  }
  if (p.lossguide) {
    B200_CHECK(p.max_depth >= 0 && p.max_depth <= kMaxDepth, "max_depth must be in [0, 16]");
    B200_CHECK(p.max_leaves > 0 || p.max_depth > 0, "grow_policy=lossguide needs max_leaves > 0 or max_depth > 0");
    B200_CHECK(p.max_leaves <= 4096, "max_leaves above 4096 is not supported by the B200 lossguide builder");
    B200_CHECK(p.colsample_bytree >= 1.0f && p.colsample_bylevel >= 1.0f && p.colsample_bynode >= 1.0f, "column sampling (colsample_*) with grow_policy=lossguide is not implemented by the B200 hist builder");
  }
  auto bs = raw_params_.find("base_score");
  if (bs != raw_params_.end() && !bs->second.empty()) {
    base_score_ = std::stof(bs->second); base_score_set_ = true;
    if (p.objective == kBinaryLogistic || p.objective == kRegLogistic || p.objective == kLogitRaw)
      B200_CHECK(base_score_ > 0.0f && base_score_ < 1.0f, "Check failed: base_score > 0.0f && base_score < 1.0f base_score must be in (0,1) for logistic loss");
  }
  if (!p.lossguide) B200_CHECK(p.max_depth >= 1, "max_depth=" + std::to_string(p.max_depth) + " (no depth limit) needs grow_policy=lossguide with max_leaves; the depth-wise builder takes max_depth in [1, 16]");
  if (p.max_bin > 256) p.max_bin = 256;            // uint8 bin codes (the Python layer warns)
  param_ = p;
  configured_ = true;
}

float Booster::base_margin() const {
  if (objective_is_logistic(param_.objective)) return -std::log(1.0f / base_score_ - 1.0f);
  if (objective_is_log_link(param_.objective)) return std::log(base_score_);          // ProbToMargin of the log-link objectives
  return base_score_;
}

static float objective_aux(const TrainParam& p) {
  switch (p.objective) { case kPseudoHuber: return p.huber_slope; case kTweedie: return p.tweedie_variance_power; case kPoisson: return p.poisson_max_delta_step; default: return 0.0f; }
}

// One Newton stump at margin 0, then PredTransform (upstream src/objective/init_estimation.cc, src/tree/fit_stump.cc)
void Booster::estimate_base_score(DMatrix* dtrain) {
  if (base_score_set_ || base_score_estimated_ || !trees_.empty()) { base_score_estimated_ = true; return; }
  base_score_estimated_ = true;
  if (param_.objective == kSoftprob || param_.objective == kSoftmax) { base_score_ = 0.5f; return; }
  // 3.0.x fits the intercept for the RegLossObj family only; the log-link objectives and binary:hinge keep the 0.5 default
  // [UPSTREAM-RECALL: src/objective/init_estimation.cc; later releases changed the GLM objectives]
  if (objective_is_log_link(param_.objective) || param_.objective == kHinge) { base_score_ = 0.5f; return; }
  cudaStream_t s = engine_stream();
  GrowerImpl& g = *grower_;
  GradArgs ga{}; ga.margin = nullptr; ga.label = dtrain->d_labels.p; ga.weight = dtrain->weights.empty() ? nullptr : dtrain->d_weights.p;
  ga.gpair = g.gpair.p; ga.gp_stride = g.gp_stride; ga.absmax = nullptr; ga.err = g.err.p; ga.n = dtrain->n; ga.row_offset = 0; ga.K = 1; ga.objective = param_.objective;
  ga.scale_pos_weight = param_.scale_pos_weight; ga.subsample = 1.0f; ga.seed = 0; ga.iter = 0; ga.aux = objective_aux(param_);
  CUDA_OK(cudaMemsetAsync(g.dsum.p, 0, 4 * sizeof(double), s));
  launch_gradient(ga, s);
  launch_sum_gpair(g.gpair.p, dtrain->n, g.dsum.p, s);
  Comm::get().allreduce_sum_f64(g.dsum.p, 2, s);
  double h[2];
  CUDA_OK(cudaMemcpyAsync(h, g.dsum.p, 2 * sizeof(double), cudaMemcpyDeviceToHost, s));
  Comm::get().sync_stream(s);
  float w = h[1] <= 0.0 ? 0.0f : (float)(-h[0] / h[1]);
  // binary:logitraw keeps base_score in probability space like the other logistic objectives (the estimated stump weight
  // w is a margin; storing it raw and taking its logit again gives NaN whenever w <= 0, i.e. whenever mean(y) < 0.5)
  if (param_.objective == kBinaryLogistic || param_.objective == kRegLogistic || param_.objective == kLogitRaw) {
    float x = std::min(-w, 88.7f); base_score_ = 1.0f / (std::exp(x) + 1.0f + 1e-16f);
  } else base_score_ = w;
}

void Booster::append_device_tree(int class_id, size_t device_offset, int max_nodes, PendingTree pt) {
  trees_.emplace_back(); tree_info_.push_back(class_id); pending_.push_back(pt); on_device_.push_back(1);
  h_tree_offset.resize(trees_.size() + 1);
  h_tree_offset[trees_.size() - 1] = (int64_t)device_offset;
  h_tree_offset[trees_.size()] = (int64_t)device_offset + max_nodes;
  ++model_version_;
}

void Booster::sync_model() {
  bool any = false;
  for (auto& p : pending_) if (p.staging) { any = true; break; }
  if (!any) return;
  for (size_t t = 0; t < pending_.size(); ++t) {
    PendingTree& p = pending_[t];
    if (!p.staging) continue;
    CUDA_OK(cudaEventSynchronize(p.ready));
    const unsigned char* b = (const unsigned char*)p.staging;
    const int nn = *(const int*)b; const size_t N = p.cap_nodes;
    const int* ip = (const int*)(b + 64); const float* fp = (const float*)(ip + 5 * N); const unsigned char* up = (const unsigned char*)(fp + 4 * N);
    HostTree& h = trees_[t];
    h.left.assign(ip, ip + nn); h.right.assign(ip + N, ip + N + nn); h.parent.assign(ip + 2 * N, ip + 2 * N + nn);
    h.split_index.assign(ip + 3 * N, ip + 3 * N + nn); h.split_bin.assign(ip + 4 * N, ip + 4 * N + nn);
    h.split_cond.assign(fp, fp + nn); h.base_weight.assign(fp + N, fp + N + nn); h.loss_chg.assign(fp + 2 * N, fp + 2 * N + nn); h.sum_hess.assign(fp + 3 * N, fp + 3 * N + nn);
    h.default_left.assign(up, up + nn);
    if (grower_) grower_->free_events.push_back(p.ready); else cudaEventDestroy(p.ready);
    p.ready = nullptr; p.staging = nullptr;
  }
  if (grower_) grower_->pinned.reset();
}

// make sure every tree is present in the device model (trees loaded from a file are uploaded here)
void Booster::upload_model() {
  cudaStream_t s = engine_stream();
  const int nt = (int)trees_.size();
  if ((int)h_tree_offset.size() != nt + 1) h_tree_offset.resize(nt + 1, 0);
  pending_.resize(nt); on_device_.resize(nt, 0);
  for (int t = 0; t < nt; ++t) {
    if (on_device_[t]) continue;
    const HostTree& h = trees_[t];
    const int nn = h.num_nodes();
    std::vector<DevNode> nodes(nn);
    for (int i = 0; i < nn; ++i) { nodes[i].cond = h.split_cond[i]; nodes[i].left = h.left[i]; nodes[i].right = h.right[i]; nodes[i].fidx_dl = (unsigned)h.split_index[i] | ((unsigned)h.default_left[i] << 31);
      if (h.left[i] >= 0 && h.right[i] != h.left[i] + 1) children_adjacent_ = false; }     // foreign model: the tiled predictor assumes sibling pairs
    if (d_nodes_used + nn > d_nodes.n) {
      size_t cap = std::max<size_t>(d_nodes.n * 2, d_nodes_used + nn + 4096);
      DevBuf<DevNode> nb; nb.alloc(cap);
      if (d_nodes_used) CUDA_OK(cudaMemcpyAsync(nb.p, d_nodes.p, sizeof(DevNode) * d_nodes_used, cudaMemcpyDeviceToDevice, s));
      Comm::get().sync_stream(s);
      std::swap(nb.p, d_nodes.p); std::swap(nb.n, d_nodes.n);
    }
    CUDA_OK(cudaMemcpyAsync(d_nodes.p + d_nodes_used, nodes.data(), sizeof(DevNode) * nn, cudaMemcpyHostToDevice, s));
    Comm::get().sync_stream(s);
    h_tree_offset[t] = (int64_t)d_nodes_used; h_tree_offset[t + 1] = (int64_t)d_nodes_used + nn;
    d_nodes_used += nn; on_device_[t] = 1; d_trees_uploaded = 0;
  }
  if (d_trees_uploaded != nt || d_tree_offset.n < (size_t)nt + 1) {
    d_tree_offset.ensure(std::max<size_t>(nt + 1, 64)); d_tree_info.ensure(std::max<size_t>(nt, 64));
    // offsets are per-tree starts (trees trained on the device have fixed-capacity slots, so starts are not cumulative)
    CUDA_OK(cudaMemcpyAsync(d_tree_offset.p, h_tree_offset.data(), sizeof(int64_t) * (nt + 1), cudaMemcpyHostToDevice, s));
    if (nt) CUDA_OK(cudaMemcpyAsync(d_tree_info.p, tree_info_.data(), sizeof(int) * nt, cudaMemcpyHostToDevice, s));
    Comm::get().sync_stream(s);
    d_trees_uploaded = nt;
  }
}

PredictArgs Booster::predict_args(const DMatrix* dm, int tree_begin, int tree_end) const {
  PredictArgs pa{}; pa.X = dm->X.p; pa.n = dm->n; pa.F = dm->F; pa.F_model = num_feature_;
  pa.nodes = d_nodes.p; pa.tree_offset = d_tree_offset.p; pa.tree_info = d_tree_info.p;
  pa.tree_begin = tree_begin; pa.tree_end = tree_end; pa.K = param_.num_class; pa.margin = nullptr; pa.leaf = nullptr;
  pa.h_tree_offset = h_tree_offset.data(); pa.has_nan = dm->has_missing ? 1 : 0; pa.children_adjacent = children_adjacent_ ? 1 : 0;
  return pa;
}

PredCache& Booster::cache_for(DMatrix* dm) {
  PredCache& c = caches_[dm->uid];
  const int K = param_.num_class;
  if (c.n != dm->n || c.margin.n != (size_t)dm->n * K) {
    c.n = dm->n; c.margin.alloc((size_t)dm->n * K); c.trees_applied = -1;
  }
  return c;
}

void Booster::bring_cache_up_to_date(DMatrix* dm, PredCache& c) {
  cudaStream_t s = engine_stream();
  const int K = param_.num_class;
  const int nt = (int)trees_.size();
  if (c.trees_applied < 0) {
    if (!dm->base_margin.empty()) {
      B200_CHECK(dm->base_margin.size() == (size_t)dm->n * K, "base_margin size does not match rows x groups");
      CUDA_OK(cudaMemcpyAsync(c.margin.p, dm->d_base_margin.p, sizeof(float) * dm->n * K, cudaMemcpyDeviceToDevice, s));
    } else launch_fill(c.margin.p, dm->n * K, base_margin(), s);
    c.trees_applied = 0;
  }
  if (c.trees_applied < nt) {
    upload_model();
    PredictArgs pa = predict_args(dm, c.trees_applied, nt); pa.margin = c.margin.p;
    launch_predict(pa, s);
    c.trees_applied = nt;
  }
}

static void check_labels(const DMatrix* dm) {
  B200_CHECK(dm->labels.size() == (size_t)dm->n, "Check failed: preds.size() == info.labels_.size() (" + std::to_string(dm->n) + " vs. " +
             std::to_string(dm->labels.size()) + ") : labels are not correctly provided");
}

void Booster::update_one_iter(int iter, DMatrix* dtrain) {
  configure();
  (void)iter;
  cudaStream_t s = engine_stream();
  check_labels(dtrain);
  if (num_feature_ == 0) num_feature_ = dtrain->F;
  B200_CHECK(num_feature_ == dtrain->F, "Check failed: learner_model_param_.num_feature == p_fmat->Info().num_col_ (" + std::to_string(num_feature_) +
             " vs. " + std::to_string(dtrain->F) + ") : Number of columns does not match number of features in booster.");
  B200_CHECK(dtrain->n > 0 || Comm::get().distributed(), "Empty dataset at worker: 0");
  dtrain->ensure_binned(param_.max_bin);
  const int K = param_.num_class;
  if (!grower_) grower_ = new GrowerImpl();
  GrowerImpl& g = *grower_;
  g.ensure(dtrain->n, dtrain->ngroups, dtrain->tw, param_.max_depth, K, lossguide_iters(param_));
  if (!labels_checked_) {
    // label-range errors must surface from update() (the container maps them to UserError, train.py:461-467)
    const std::vector<float>& y = dtrain->labels;
    if (param_.objective == kBinaryLogistic || param_.objective == kRegLogistic || param_.objective == kLogitRaw)
      for (float v : y) B200_CHECK(v >= 0.0f && v <= 1.0f, "Check failed: label must be in [0,1] for logistic regression");
    if (param_.objective == kSoftprob || param_.objective == kSoftmax)
      for (float v : y) B200_CHECK(v >= 0.0f && (int)v < K, "SoftmaxMultiClassObj: label must be in [0, num_class).");
    if (param_.objective == kSquaredLogError) for (float v : y) B200_CHECK(v > -1.0f, "Check failed: label must be greater than -1 for rmsle so that log(label + 1) can be valid.");
    if (param_.objective == kPoisson) for (float v : y) B200_CHECK(v >= 0.0f, "PoissonRegression: label must be nonnegative");
    if (param_.objective == kGamma) for (float v : y) B200_CHECK(v > 0.0f, "GammaRegression: label must be positive.");
    if (param_.objective == kTweedie) for (float v : y) B200_CHECK(v >= 0.0f, "TweedieRegression: label must be nonnegative");
    labels_checked_ = true;
  }
  estimate_base_score(dtrain);
  PredCache& cache = cache_for(dtrain);
  bring_cache_up_to_date(dtrain, cache);

  const int round = (int)trees_.size() / K;
  // ---- gradients + fixed-point scales
  CUDA_OK(cudaMemsetAsync(g.gs.absmax, 0, 8, s));
  GradArgs ga{}; ga.margin = cache.margin.p; ga.label = dtrain->d_labels.p; ga.weight = dtrain->weights.empty() ? nullptr : dtrain->d_weights.p;
  ga.gpair = g.gpair.p; ga.gp_stride = g.gp_stride; ga.absmax = g.gs.absmax; ga.err = g.err.p; ga.n = dtrain->n; ga.row_offset = 0; ga.K = K; ga.objective = param_.objective;
  ga.scale_pos_weight = param_.scale_pos_weight; ga.subsample = param_.subsample; ga.seed = param_.seed; ga.iter = (unsigned long long)round;
  ga.row_offset = (int64_t)Comm::get().rank() << 40; ga.aux = objective_aux(param_);
  launch_gradient(ga, s);
  Comm::get().allreduce_max_u32(g.gs.absmax, 2, s);
  launch_scales(g.gs, job_grad_bits(g.global_n), s);

  for (int k = 0; k < K; ++k) grow_one_tree(dtrain, cache, k, round * K + k);
}


// The fixed launch sequence of one tree (everything data dependent lives in device memory), capturable in a CUDA graph.
void Booster::enqueue_tree(DMatrix* dtrain, float* margin, int k, const unsigned char* mask, DevNode* packed_out, int root_mode) {
  cudaStream_t s = engine_stream();
  GrowerImpl& g = *grower_;
  Comm& comm = Comm::get();
  const int K = param_.num_class;
  const int D = param_.max_depth;
  const TrainParamDev pd = to_dev(param_);
  const BinnedMatrix bm = dtrain->binned_view();
  const int num_sms = engine_num_sms();
  const unsigned max_tiles = (unsigned)((dtrain->n + kPartTile - 1) / kPartTile) + g.max_level_nodes + 1;

  launch_init_tree(g.gs, g.ta, (unsigned)dtrain->n, 0, g.max_level_nodes, s);
  if (root_mode == 2) { slot_from_cache_kernel<<<148, 256, 0, s>>>(g.hist_pool.p, g.root_h_cache.p, g.slot_stride); ++g_kernel_launches; CUDA_OK(cudaGetLastError()); }
  else CUDA_OK(cudaMemsetAsync(g.hist_pool.p, 0, g.slot_stride * sizeof(GH64), s));

  HistArgs ha{}; ha.bins = bm.bins; ha.bins_tail = bm.bins_tail; ha.n = bm.n; ha.row_stride = bm.ngroups * kSlots; ha.tw = bm.tw;
  ha.bins_gather = bm.bins_gather; ha.gather_stride = bm.gather_stride;
  ha.gpair = g.gpair.p + (size_t)k * g.gp_stride; ha.ridx = nullptr;
  ha.build_count = g.gs.build_count; ha.build_nid = g.gs.build_nid; ha.build_prefix = g.gs.build_prefix; ha.seg_begin = g.gs.seg_begin;
  ha.hist_slot = g.gs.hist_slot; ha.scales = g.gs.scales; ha.hist_pool = g.hist_pool.p; ha.node_sum = g.gs.node_sum; ha.ngroups = bm.ngroups;
  ha.accumulate_sum = 1; ha.g_only = root_mode == 2 ? 1 : 0; ha.window_rows = job_window_rows(g.global_n);
  ha.rows_counter = profile_ ? prof_rows_.p : nullptr;
  prof_begin(0);
  launch_hist_build(ha, num_sms, s);
  prof_end();
  if (root_mode == 1) { snapshot_h_kernel<<<148, 256, 0, s>>>(g.hist_pool.p, g.root_h_cache.p, g.slot_stride); ++g_kernel_launches; CUDA_OK(cudaGetLastError()); }
  ha.g_only = 0;
  // a collective: issued directly, or (under capture) closes the current graph segment and is remembered for the replay
  auto collective = [&](std::function<void()> f) {
    if (!comm.distributed()) return;
    if (!g.capturing) { f(); return; }
    cudaGraph_t graph = nullptr;
    CUDA_OK(cudaStreamEndCapture(s, &graph));
    cudaGraphExec_t exec = nullptr;
    cudaError_t e = cudaGraphInstantiate(&exec, graph, 0);
    cudaGraphDestroy(graph);
    CUDA_OK(e);
    g.capturing->segs.push_back(exec); g.capturing->colls.push_back(f);
    CUDA_OK(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
  };
  // the per-level histogram all-reduce: one NVLink peer-memory kernel inside the graph when the peers are mapped, else NCCL
  auto allreduce_hist = [&](GH64* p, size_t cnt) {
    if (!comm.distributed()) return;
    if (peer_allreduce_i64(reinterpret_cast<long long*>(p), cnt, s)) return;
    collective([p, cnt, s]() { Comm::get().allreduce_sum_i64(p, cnt, s); });
  };
  allreduce_hist(g.hist_pool.p, g.slot_stride * 2);
  allreduce_hist(g.gs.node_sum, 2);
  const int* mono_dev = nullptr;
  if (!monotone_.empty()) {                       // uploaded outside the captured sequence by grow_one_tree
    B200_CHECK((int)monotone_.size() <= bm.F, "monotone_constraints has more entries than the data has features");
    mono_dev = g.monotone_dev.p;
  }
  const bool ic_on = !interaction_.empty();
  if (ic_on) {                                    // root: empty path, every feature allowed (buffers sized / sets uploaded by grow_one_tree)
    CUDA_OK(cudaMemsetAsync(g.ic_path.p, 0, (size_t)bm.F, s));
    CUDA_OK(cudaMemsetAsync(g.ic_allowed.p, 1, (size_t)bm.F, s));
  }
  EvalArgs ea{}; ea.hist_pool = g.hist_pool.p; ea.gs = g.gs; ea.cut_ptrs = dtrain->d_cut_ptrs.p; ea.feat_mask = mask; ea.p = pd; ea.F = bm.F;
  ea.ngroups = bm.ngroups; ea.tw = bm.tw; ea.ntail = bm.ntail; ea.has_missing = bm.has_missing; ea.level = 0; ea.max_level_nodes = g.max_level_nodes;
  ea.colsample_bynode = mask ? param_.colsample_bynode : 1.0f; ea.seed = param_.seed; ea.tree_index = g.tree_index_dev.p; ea.monotone = mono_dev; ea.node_allowed = ic_on ? g.ic_allowed.p : nullptr;
  launch_eval(ea, 1, s);

  const int lg_iters = lossguide_iters(param_);
  for (int it = 0; it < lg_iters; ++it) {                 // grow_policy=lossguide: one expansion per iteration (tree.cu apply_lossguide_kernel)
    ApplyArgs aa{}; aa.gs = g.gs; aa.tree = g.ta; aa.cut_ptrs = dtrain->d_cut_ptrs.p; aa.cut_vals = dtrain->d_cut_vals.p; aa.min_vals = dtrain->d_min_vals.p;
    aa.p = pd; aa.scratch = g.scratch.p; aa.ngroups = bm.ngroups + (bm.tw > 0 ? 1 : 0); aa.level = 0; aa.max_level_nodes = g.max_level_nodes; aa.monotone = mono_dev;
    if (ic_on) { aa.node_path = g.ic_path.p; aa.node_allowed = g.ic_allowed.p; aa.ic_sets = g.ic_sets.p; aa.n_ic_sets = (int)interaction_.size(); aa.F = bm.F; }
    launch_apply_lossguide(aa, it, s);
    // live row segments always sit in buffer set 0; the partition writes the children into set 1 and they are copied straight back
    const bool carry_tail = bm.tw == 4;
    PartArgs pa{}; pa.gs = g.gs; pa.tree = g.ta; pa.bins_col = bm.bins_col; pa.n = bm.n;
    pa.ridx_cur = it == 0 ? nullptr : g.ridx0.p; pa.ridx_next = g.ridx1.p;
    pa.gp_cur = it == 0 ? g.gpair.p + (size_t)k * g.gp_stride : g.gp0.p; pa.gp_next = g.gp1.p;
    pa.tl_cur = !carry_tail ? nullptr : (it == 0 ? reinterpret_cast<const unsigned*>(bm.bins_tail) : g.tl0.p); pa.tl_next = !carry_tail ? nullptr : g.tl1.p;
    pa.has_missing = bm.has_missing; pa.level = 0; pa.max_level_nodes = g.max_level_nodes;
    launch_partition(pa, max_tiles, 1, s);
    launch_lg_copy_back(pa, g.ridx0.p, g.gp0.p, g.tl0.p, max_tiles, s);
    launch_zero_build_slots(g.gs, g.hist_pool.p, g.slot_stride, 1, s);
    ha.ridx = g.ridx0.p; ha.gpair = g.gp0.p; ha.tail_pos = carry_tail ? g.tl0.p : nullptr; ha.accumulate_sum = 0;
    ha.rows_counter = profile_ ? prof_rows_.p + 1 : nullptr;
    prof_begin(1);
    launch_hist_build(ha, num_sms, s);
    prof_end();
    if (comm.distributed()) {                              // the collective needs a fixed address: go through the staging slot
      launch_lg_stage(g.gs, g.hist_pool.p, g.slot_stride, 1, s);
      allreduce_hist(g.hist_pool.p + (size_t)kLgStageSlot * g.slot_stride, g.slot_stride * 2);
      launch_lg_stage(g.gs, g.hist_pool.p, g.slot_stride, 0, s);
    }
    launch_subtract(g.gs, g.hist_pool.p, g.slot_stride, 1, s);
    ea.level = 1; ea.feat_mask = nullptr;
    launch_eval(ea, 2, s);
  }

  for (int L = 0; L < D && lg_iters == 0; ++L) {
    const bool final_level = (L == D - 1);
    const int next_base = ((L + 1) & 1) * g.region, next_half = 1 << L;
    ApplyArgs aa{}; aa.gs = g.gs; aa.tree = g.ta; aa.cut_ptrs = dtrain->d_cut_ptrs.p; aa.cut_vals = dtrain->d_cut_vals.p; aa.min_vals = dtrain->d_min_vals.p;
    aa.p = pd; aa.scratch = g.scratch.p; aa.ngroups = bm.ngroups + (bm.tw > 0 ? 1 : 0); aa.level = L; aa.max_level_nodes = g.max_level_nodes; aa.next_base = next_base; aa.next_half = next_half; aa.monotone = mono_dev;
    if (ic_on) { aa.node_path = g.ic_path.p; aa.node_allowed = g.ic_allowed.p; aa.ic_sets = g.ic_sets.p; aa.n_ic_sets = (int)interaction_.size(); aa.F = bm.F; }
    launch_apply(aa, s);
    if (final_level) break;                  // children of the last level are leaves: no partition, no histograms
    PartArgs pa{}; pa.gs = g.gs; pa.tree = g.ta; pa.bins_col = bm.bins_col; pa.n = bm.n;
    pa.ridx_cur = L == 0 ? nullptr : ((L & 1) ? g.ridx0.p : g.ridx1.p);
    pa.ridx_next = (L & 1) ? g.ridx1.p : g.ridx0.p;
    pa.gp_cur = L == 0 ? g.gpair.p + (size_t)k * g.gp_stride : ((L & 1) ? g.gp0.p : g.gp1.p);
    pa.gp_next = (L & 1) ? g.gp1.p : g.gp0.p;
    const bool carry_tail = bm.tw == 4;                     // the 4 tail bytes of a row ride along with its id instead of being gathered
    pa.tl_cur = !carry_tail ? nullptr : (L == 0 ? reinterpret_cast<const unsigned*>(bm.bins_tail) : ((L & 1) ? g.tl0.p : g.tl1.p));
    pa.tl_next = !carry_tail ? nullptr : ((L & 1) ? g.tl1.p : g.tl0.p);
    pa.has_missing = bm.has_missing; pa.level = L; pa.max_level_nodes = g.max_level_nodes;
    launch_partition(pa, max_tiles, 1 << L, s);
    // histograms of the next level: build the smaller children, all-reduce, subtract for the siblings
    CUDA_OK(cudaMemsetAsync(g.hist_pool.p + (size_t)next_base * g.slot_stride, 0, (size_t)next_half * g.slot_stride * sizeof(GH64), s));
    ha.ridx = pa.ridx_next; ha.gpair = pa.gp_next; ha.tail_pos = pa.tl_next; ha.accumulate_sum = 0;
    ha.rows_counter = profile_ ? prof_rows_.p + 1 : nullptr;
    prof_begin(L + 1);
    launch_hist_build(ha, num_sms, s);
    prof_end();
    allreduce_hist(g.hist_pool.p + (size_t)next_base * g.slot_stride, (size_t)next_half * g.slot_stride * 2);
    launch_subtract(g.gs, g.hist_pool.p, g.slot_stride, next_half, s);
    ea.level = L + 1;
    ea.feat_mask = mask ? mask + (size_t)(L + 1) * bm.F : nullptr;
    launch_eval(ea, 1 << (L + 1), s);
  }

  // prediction cache += leaf values of this tree: one row-order pass over the column-major bins
  launch_update_margin(g.ta, g.gs.n_nodes, bm.bins_col, bm.n, bm.has_missing, margin, K, k, s);

  pack_tree_kernel<<<(g.cap_nodes + 255) / 256, 256, 0, s>>>(g.ta, g.gs.n_nodes, packed_out, g.cap_nodes); ++g_kernel_launches;
  CUDA_OK(cudaGetLastError());
}

// One tree of class k.  The sequence is replayed from a CUDA graph (captured once per (matrix, class, parameters)):
// at small per-GPU shards the ~60 launches + 6 NCCL calls per tree are otherwise CPU-launch bound.
void Booster::grow_one_tree(DMatrix* dtrain, PredCache& cache, int k, int tree_index) {
  cudaStream_t s = engine_stream();
  GrowerImpl& g = *grower_;
  const unsigned char* mask = nullptr;
  const bool sampling = param_.colsample_bytree < 1.0f || param_.colsample_bylevel < 1.0f || param_.colsample_bynode < 1.0f;
  if (sampling) {                               // one mask per level [max_depth][F]: bytree -> bylevel; bynode is applied inside eval_kernel
    const std::string tm = colsample_mask(param_.seed, tree_index, dtrain->F, param_.colsample_bytree);
    std::string all;
    for (int d = 0; d < param_.max_depth; ++d) all += subset_mask(tm, param_.colsample_bylevel, param_.seed, 0x300000ull + 64ull * (uint64_t)tree_index + (uint64_t)d);
    g.feat_mask.ensure(all.size()); g.tree_index_dev.ensure(1);
    CUDA_OK(cudaMemcpyAsync(g.feat_mask.p, all.data(), all.size(), cudaMemcpyHostToDevice, s));
    CUDA_OK(cudaMemcpyAsync(g.tree_index_dev.p, &tree_index, sizeof(int), cudaMemcpyHostToDevice, s));
    Comm::get().sync_stream(s);
    mask = g.feat_mask.p;
  }
  if (!monotone_.empty()) {                     // per-feature constraints in device memory (padded with 0 to the feature count)
    std::vector<int> mh(monotone_); mh.resize((size_t)std::max<int>(dtrain->F, (int)mh.size()), 0);
    if (mh != g.monotone_host || g.monotone_dev.n < mh.size()) {
      g.monotone_dev.ensure(mh.size());
      CUDA_OK(cudaMemcpyAsync(g.monotone_dev.p, mh.data(), sizeof(int) * mh.size(), cudaMemcpyHostToDevice, s));
      Comm::get().sync_stream(s);
      g.monotone_host = mh;
    }
  }
  if (!interaction_.empty()) {                  // constraint sets as a membership matrix, per-node path / allowed flags
    const size_t F = (size_t)dtrain->F;
    std::vector<unsigned char> sets(interaction_.size() * F, 0);
    for (size_t si = 0; si < interaction_.size(); ++si)
      for (int f : interaction_[si]) { B200_CHECK((size_t)f < F, "interaction_constraints names feature " + std::to_string(f) + " but the data has " + std::to_string(F) + " features"); sets[si * F + f] = 1; }
    g.ic_path.ensure((size_t)g.cap_nodes * F); g.ic_allowed.ensure((size_t)g.cap_nodes * F);
    if (sets != g.ic_sets_host || g.ic_sets.n < sets.size()) {
      g.ic_sets.ensure(sets.size());
      CUDA_OK(cudaMemcpyAsync(g.ic_sets.p, sets.data(), sets.size(), cudaMemcpyHostToDevice, s));
      Comm::get().sync_stream(s);
      g.ic_sets_host = sets;
    }
  }
  g.packed.ensure((size_t)g.cap_nodes);
  static const bool no_graph = getenv("B200XGB_NO_GRAPH") != nullptr;
  static const bool no_graph_multi = getenv("B200XGB_NO_GRAPH_MULTI") != nullptr;      // multi-rank: issue every launch directly
  const bool dist = Comm::get().distributed();
  if ((int)g.eager_done.size() <= k) g.eager_done.resize(k + 1, 0);
  // the first tree of every class runs eagerly when ranks are connected: NCCL sets up its channels on first use
  const bool eager_first = dist && !g.eager_done[k];
  // constant-hessian root pass: eligible when every row has h == 1 in every round
  static const bool no_consth = getenv("B200XGB_NO_CONSTH") != nullptr;
  const bool consth = !no_consth && param_.objective == kSquaredError && param_.num_class == 1 && dtrain->weights.empty() &&
                      param_.subsample >= 1.0f && param_.scale_pos_weight == 1.0f;
  int root_mode = 0;
  if (consth) {
    if (g.root_h_valid && g.root_h_uid == dtrain->uid && g.root_h_version == dtrain->binned_version) root_mode = 2;
    else root_mode = 1;
  }
  if (profile_ || no_graph || (dist && no_graph_multi) || eager_first || root_mode == 1) {
    g.eager_done[k] = 1;
    enqueue_tree(dtrain, cache.margin.p, k, mask, g.packed.p, root_mode);
    if (root_mode == 1) { g.root_h_valid = true; g.root_h_uid = dtrain->uid; g.root_h_version = dtrain->binned_version; }
  } else {
    if ((int)g.graphs.size() <= k) g.graphs.resize(k + 1);
    TreeGraph& tg = g.graphs[k];
    TreeGraphKey key; memset(&key, 0, sizeof key);
    key.uid = dtrain->uid; key.binned_version = dtrain->binned_version; key.root_mode = root_mode;
    key.margin = cache.margin.p; key.mask = mask; key.packed = g.packed.p; key.max_depth = param_.max_depth;
    key.bins = dtrain->bins.p; key.bins_col = dtrain->bins_col.p; key.cuts = dtrain->d_cut_vals.p;     // re-binning invalidates the capture
    key.max_leaves = param_.max_leaves; key.lg_iters = lossguide_iters(param_); key.eta = param_.eta; key.lambda = param_.lambda; key.alpha = param_.alpha; key.gamma = param_.gamma;
    key.mcw = param_.min_child_weight; key.mds = param_.max_delta_step; key.world = Comm::get().world(); key.n = dtrain->n;
    key.bynode = param_.colsample_bynode; key.seed = param_.seed; key.mono = monotone_.empty() ? nullptr : g.monotone_dev.p;
    key.ic_sets = interaction_.empty() ? nullptr : g.ic_sets.p; key.ic_allowed = interaction_.empty() ? nullptr : g.ic_allowed.p; key.n_ic = (int)interaction_.size();
    if (tg.segs.empty() || memcmp(&tg.key, &key, sizeof key) != 0) {
      tg.destroy();
      const long long launches_before = g_kernel_launches;
      CUDA_OK(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
      g.capturing = &tg;
      cudaGraph_t graph = nullptr;
      try { enqueue_tree(dtrain, cache.margin.p, k, mask, g.packed.p, root_mode); }
      catch (...) { g.capturing = nullptr; cudaStreamEndCapture(s, &graph); if (graph) cudaGraphDestroy(graph); tg.destroy(); throw; }
      g.capturing = nullptr;
      CUDA_OK(cudaStreamEndCapture(s, &graph));
      cudaGraphExec_t exec = nullptr;
      cudaError_t e = cudaGraphInstantiate(&exec, graph, 0);
      cudaGraphDestroy(graph);
      if (e != cudaSuccess) { tg.destroy(); CUDA_OK(e); }
      tg.segs.push_back(exec);
      tg.key = key; tg.launches = g_kernel_launches - launches_before;
      g_kernel_launches = launches_before;               // capture enqueued nothing
    }
    for (size_t i = 0; i < tg.segs.size(); ++i) {
      CUDA_OK(cudaGraphLaunch(tg.segs[i], s));
      if (i < tg.colls.size()) tg.colls[i]();
    }
    g_kernel_launches += tg.launches;
  }

  // ---- hand the finished tree to the model: device copy for prediction, async host copy for model IO
  const size_t need = d_nodes_used + (size_t)g.cap_nodes;
  if (need > d_nodes.n) {
    size_t cap = std::max<size_t>(d_nodes.n * 2, need + 64 * (size_t)g.cap_nodes);
    DevBuf<DevNode> nb; nb.alloc(cap);
    if (d_nodes_used) CUDA_OK(cudaMemcpyAsync(nb.p, d_nodes.p, sizeof(DevNode) * d_nodes_used, cudaMemcpyDeviceToDevice, s));
    Comm::get().sync_stream(s);
    std::swap(nb.p, d_nodes.p); std::swap(nb.n, d_nodes.n);
  }
  CUDA_OK(cudaMemcpyAsync(d_nodes.p + d_nodes_used, g.packed.p, sizeof(DevNode) * (size_t)g.cap_nodes, cudaMemcpyDeviceToDevice, s));
  if (pending_.size() - (size_t)std::count_if(pending_.begin(), pending_.end(), [](const PendingTree& p) { return p.staging == nullptr; }) >= 512) sync_model();
  PendingTree pt; pt.cap_nodes = (size_t)g.cap_nodes;
  pt.staging = g.pinned.take(g.tree_block_bytes);
  if (!g.free_events.empty()) { pt.ready = g.free_events.back(); g.free_events.pop_back(); }
  else CUDA_OK(cudaEventCreateWithFlags(&pt.ready, cudaEventDisableTiming));
  CUDA_OK(cudaMemcpyAsync(pt.staging, g.tree_block.p, g.tree_block_bytes, cudaMemcpyDeviceToHost, s));
  CUDA_OK(cudaEventRecord(pt.ready, s));
  append_device_tree(k, d_nodes_used, g.cap_nodes, pt);
  d_nodes_used += (size_t)g.cap_nodes;
  d_trees_uploaded = 0;                      // offsets/info arrays need a refresh before the next predict
  cache.trees_applied = (int)trees_.size();  // update_margin_kernel already added this tree's leaves to the cache
}

void Booster::boost_one_iter(DMatrix*, const float*, const float*, size_t) {
  throw Error("custom objective (BoostOneIter) is not implemented on the B200 hist path");
}

int Booster::boosted_rounds() { configure(); return (int)trees_.size() / std::max(1, param_.num_class); }

// ---------------------------------------------------------------------------------------------
// evaluation  (upstream src/learner.cc EvalOneIter: "[iter]\t<name>-<metric>:<value>")
// ---------------------------------------------------------------------------------------------
static std::string default_metric(const TrainParam& p) {
  switch (p.objective) {
    case kSquaredError: case kRegLogistic: return "rmse";
    case kBinaryLogistic: case kLogitRaw: return "logloss";
    case kSquaredLogError: return "rmsle";
    case kPseudoHuber: return "mphe";
    case kPoisson: return "poisson-nloglik";
    case kGamma: return "gamma-nloglik";
    case kTweedie: { char buf[64]; snprintf(buf, sizeof buf, "tweedie-nloglik@%g", (double)p.tweedie_variance_power); return buf; }
    case kHinge: return "error";
    default: return "mlogloss";
  }
}

std::string Booster::eval_one_iter(int iter, const std::vector<DMatrix*>& dms, const std::vector<std::string>& names) {
  configure();
  cudaStream_t s = engine_stream();
  std::vector<std::string> metrics = eval_metrics_;
  if (metrics.empty()) metrics.push_back(default_metric(param_));
  if (!grower_) grower_ = new GrowerImpl();
  grower_->dsum.ensure(4);
  std::string out = "[" + std::to_string(iter) + "]";
  for (size_t i = 0; i < dms.size(); ++i) {
    DMatrix* dm = dms[i];
    check_labels(dm);
    PredCache& c = cache_for(dm);
    bring_cache_up_to_date(dm, c);
    for (const std::string& mname : metrics) {
      MetricArgs ma{}; ma.margin = c.margin.p; ma.label = dm->d_labels.p; ma.weight = dm->weights.empty() ? nullptr : dm->d_weights.p;
      ma.out = grower_->dsum.p; ma.n = dm->n; ma.K = param_.num_class; ma.threshold = 0.5f;
      ma.is_logistic = (param_.objective == kBinaryLogistic || param_.objective == kRegLogistic) ? 1 : 0;
      ma.transform = objective_transform(param_.objective); ma.aux = 0.0f;
      std::string base = mname;
      if (mname.rfind("tweedie-nloglik@", 0) == 0) { base = "tweedie-nloglik"; ma.aux = std::stof(mname.substr(16)); B200_CHECK(ma.aux >= 1.0f && ma.aux < 2.0f, "tweedie variance power must be in interval [1, 2)"); }
      if (mname.rfind("error@", 0) == 0) { base = "error"; ma.threshold = std::stof(mname.substr(6)); }
      if (base == "auc") {
        // validated on hardware against sklearn.metrics.roc_auc_score (tests/test_gpu_parity.py::test_auc_matches_sklearn)
        B200_CHECK(param_.num_class <= 1, "auc is implemented for binary / regression-style predictions only");
        const int logistic = (param_.objective == kBinaryLogistic || param_.objective == kRegLogistic) ? 1 : 0;
        compute_auc_device(c.margin.p, dm->d_labels.p, dm->weights.empty() ? nullptr : dm->d_weights.p, dm->n, logistic, grower_->dsum.p, s);
        double h3[3];
        CUDA_OK(cudaMemcpyAsync(h3, grower_->dsum.p, 3 * sizeof(double), cudaMemcpyDeviceToHost, s));
        Comm::get().sync_stream(s);
        double pair[2] = {h3[0], h3[1] * h3[2]};
        if (Comm::get().distributed()) {
          CUDA_OK(cudaMemcpyAsync(grower_->dsum.p, pair, 2 * sizeof(double), cudaMemcpyHostToDevice, s));
          Comm::get().allreduce_sum_f64(grower_->dsum.p, 2, s);
          CUDA_OK(cudaMemcpyAsync(pair, grower_->dsum.p, 2 * sizeof(double), cudaMemcpyDeviceToHost, s));
          Comm::get().sync_stream(s);
        }
        B200_CHECK(pair[1] > 0.0, "Check failed: !auc_error AUC: the dataset only contains pos or neg samples");
        char buf[64]; snprintf(buf, sizeof buf, "%.17g", pair[0] / pair[1]);
        out += "\t" + names[i] + "-" + mname + ":" + buf;
        continue;
      }
      if (base == "rmse") ma.metric = kMetricRmse; else if (base == "mse") ma.metric = kMetricRmse; else if (base == "mae") ma.metric = kMetricMae;
      else if (base == "logloss") ma.metric = kMetricLogloss; else if (base == "error") ma.metric = kMetricError;
      else if (base == "merror") ma.metric = kMetricMerror; else if (base == "mlogloss") ma.metric = kMetricMlogloss;
      else if (base == "rmsle") ma.metric = kMetricRmsle; else if (base == "mape") ma.metric = kMetricMape;
      else if (base == "mphe") { ma.metric = kMetricMphe; ma.aux = param_.huber_slope; }
      else if (base == "poisson-nloglik") ma.metric = kMetricPoissonNll; else if (base == "gamma-nloglik") ma.metric = kMetricGammaNll;
      else if (base == "gamma-deviance") ma.metric = kMetricGammaDeviance;
      else if (base == "tweedie-nloglik") { ma.metric = kMetricTweedieNll; if (ma.aux == 0.0f) throw Error("tweedie-nloglik needs its variance power: tweedie-nloglik@rho"); }
      else throw Error("Unknown metric function " + mname + " (B200 hist path implements rmse, mse, rmsle, mae, mape, mphe, logloss, error, error@t, merror, mlogloss, auc, poisson-nloglik, gamma-nloglik, gamma-deviance, tweedie-nloglik@rho)");
      if (param_.objective == kLogitRaw && (ma.metric == kMetricLogloss || ma.metric == kMetricError)) ma.is_logistic = 1;
      if ((ma.metric == kMetricMerror || ma.metric == kMetricMlogloss)) B200_CHECK(param_.num_class > 1, "Check failed: preds.size() == info.labels_.size() : label and prediction size not match, hint: use merror or mlogloss for multi-class classification");
      CUDA_OK(cudaMemsetAsync(grower_->dsum.p, 0, 2 * sizeof(double), s));
      launch_metric(ma, s);
      Comm::get().allreduce_sum_f64(grower_->dsum.p, 2, s);
      double h[2];
      CUDA_OK(cudaMemcpyAsync(h, grower_->dsum.p, 2 * sizeof(double), cudaMemcpyDeviceToHost, s));
      Comm::get().sync_stream(s);
      double v = h[1] == 0.0 ? h[0] : h[0] / h[1];
      if (mname == "rmse" || mname == "rmsle") v = std::sqrt(v);
      if (mname == "gamma-deviance") v *= 2.0;
      char buf[64]; snprintf(buf, sizeof buf, "%.17g", v);
      out += "\t" + names[i] + "-" + mname + ":" + buf;
    }
  }
  return out;
}

// ---------------------------------------------------------------------------------------------
// prediction (upstream Booster.predict -> XGBoosterPredictFromDMatrix; cpu_predictor.cc semantics)
// type: 0 value, 1 margin, 6 leaf
// ---------------------------------------------------------------------------------------------
void Booster::predict(DMatrix* dm, int type, bool training, int iter_begin, int iter_end, bool strict_shape,
                      std::vector<float>* out, std::vector<uint64_t>* shape) {
  configure();
  (void)training;
  cudaStream_t s = engine_stream();
  const int K = param_.num_class;
  const int rounds = (int)trees_.size() / K;
  if (iter_end == 0) iter_end = rounds;
  B200_CHECK(iter_begin >= 0 && iter_begin <= iter_end && iter_end <= rounds, "Invalid iteration range: [" + std::to_string(iter_begin) + ", " + std::to_string(iter_end) + ") for a model with " + std::to_string(rounds) + " rounds");
  B200_CHECK(type == 0 || type == 1 || type == 2 || type == 6, "predict type " + std::to_string(type) + " (approximate contributions / interactions) is not implemented on the B200 path");
  if (type == 2) { predict_contribs(dm, iter_begin * K, iter_end * K, out, shape); return; }
  upload_model();
  const int tb = iter_begin * K, te = iter_end * K;
  const int64_t n = dm->n;
  PredictArgs pa = predict_args(dm, tb, te);          // a feature the matrix lacks (column >= dm->F) is missing on every route
  if (type == 6) {
    const int nt = te - tb;
    DevBuf<int>& leaf = pred_leaf_; leaf.ensure((size_t)n * std::max(nt, 1));
    pa.margin = nullptr; pa.leaf = leaf.p;
    launch_predict(pa, s);
    std::vector<int> h((size_t)n * nt);
    if (!h.empty()) CUDA_OK(cudaMemcpyAsync(h.data(), leaf.p, sizeof(int) * h.size(), cudaMemcpyDeviceToHost, s));
    Comm::get().sync_stream(s);
    out->resize(h.size());
    for (size_t i = 0; i < h.size(); ++i) (*out)[i] = (float)h[i];
    shape->assign({(uint64_t)n, (uint64_t)nt});
    return;
  }
  DevBuf<float>& margin = pred_margin_; margin.ensure((size_t)n * K);          // scratch kept across calls: no cudaMalloc / cudaFree per request
  if (!dm->base_margin.empty()) {
    B200_CHECK(dm->base_margin.size() == (size_t)n * K, "base_margin size does not match rows x groups");
    CUDA_OK(cudaMemcpyAsync(margin.p, dm->d_base_margin.p, sizeof(float) * n * K, cudaMemcpyDeviceToDevice, s));
  } else launch_fill(margin.p, n * K, base_margin(), s);
  pa.margin = margin.p; pa.leaf = nullptr;
  launch_predict(pa, s);
  int out_cols = K;
  DevBuf<float>& cls = pred_cls_;
  if (type == 0) {
    if (param_.objective == kSoftmax) { cls.ensure(n); launch_transform(margin.p, n, K, param_.objective, cls.p, s); out_cols = 1; }
    else launch_transform(margin.p, n, K, param_.objective, nullptr, s);
  }
  out->resize((size_t)n * out_cols);
  if (!out->empty()) CUDA_OK(cudaMemcpyAsync(out->data(), (type == 0 && param_.objective == kSoftmax) ? cls.p : margin.p, sizeof(float) * out->size(), cudaMemcpyDeviceToHost, s));
  Comm::get().sync_stream(s);
  if (out_cols == 1 && !strict_shape) shape->assign({(uint64_t)n});
  else shape->assign({(uint64_t)n, (uint64_t)out_cols});
}

__global__ void gather_u32_kernel(const unsigned* src, const unsigned* idx, unsigned* dst, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[idx[i]];
}

// Kernel-level entry point for parity tests and the roofline bench: build the histogram of all rows (or of the row
// subset `row_ids`, gradient pairs by position) from host gradient pairs `repeats` times; returns the int64 histogram in
// pool layout ([ngroups][256][32]{g,h} then the tail [256][tw]{g,h}) and the fixed-point scales.
void Booster::debug_build_root_hist(DMatrix* dm, const float* gpair_host, std::vector<long long>* hist_out, float* scales_out,
                                    int repeats, float* ms_out, int mode, const unsigned* row_ids, int64_t n_ids) {
  configure();
  cudaStream_t s = engine_stream();
  dm->ensure_binned(param_.max_bin);
  if (!grower_) grower_ = new GrowerImpl();
  GrowerImpl& g = *grower_;
  g.ensure(dm->n, dm->ngroups, dm->tw, param_.max_depth, param_.num_class, lossguide_iters(param_));
  hist_configure();
  const int64_t rows = row_ids ? n_ids : dm->n;
  B200_CHECK(rows <= dm->n, "debug_build_root_hist: more row ids than rows");
  CUDA_OK(cudaMemcpyAsync(g.gpair.p, gpair_host, sizeof(float2) * rows, cudaMemcpyHostToDevice, s));
  if (row_ids) CUDA_OK(cudaMemcpyAsync(g.ridx0.p, row_ids, sizeof(unsigned) * rows, cudaMemcpyHostToDevice, s));
  // scales from max|g|, max h of the supplied pairs
  float mg = 0.f, mh = 0.f;
  for (int64_t i = 0; i < rows; ++i) { mg = std::max(mg, std::fabs(gpair_host[2 * i])); mh = std::max(mh, gpair_host[2 * i + 1]); }
  unsigned am[2]; memcpy(&am[0], &mg, 4); memcpy(&am[1], &mh, 4);
  CUDA_OK(cudaMemcpyAsync(g.gs.absmax, am, 8, cudaMemcpyHostToDevice, s));
  launch_scales(g.gs, job_grad_bits(g.global_n), s);
  const BinnedMatrix bm = dm->binned_view();
  HistArgs ha{}; ha.bins = bm.bins; ha.bins_tail = bm.bins_tail; ha.n = bm.n; ha.row_stride = bm.ngroups * kSlots; ha.tw = bm.tw; ha.gpair = g.gpair.p;
  ha.bins_gather = bm.bins_gather; ha.gather_stride = bm.gather_stride;
  ha.ridx = row_ids ? g.ridx0.p : nullptr;
  ha.build_count = g.gs.build_count; ha.build_nid = g.gs.build_nid; ha.build_prefix = g.gs.build_prefix; ha.seg_begin = g.gs.seg_begin;
  ha.hist_slot = g.gs.hist_slot; ha.scales = g.gs.scales; ha.hist_pool = g.hist_pool.p; ha.node_sum = g.gs.node_sum; ha.ngroups = bm.ngroups; ha.accumulate_sum = 1;
  ha.force_gather = (mode & 3) == 1 ? 1 : 0; ha.g_only = (mode & 3) == 2 ? 1 : 0; ha.window_rows = job_window_rows(g.global_n);
  if ((mode & 4) && row_ids && bm.tw == 4) {      // the training path's variant: the rows' tail words by POSITION (as after a partition)
    gather_u32_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, s>>>(reinterpret_cast<const unsigned*>(bm.bins_tail), g.ridx0.p, g.tl0.p, rows); ++g_kernel_launches;
    CUDA_OK(cudaGetLastError());
    ha.tail_pos = g.tl0.p;
  }
  g.root_h_valid = false;                       // the debug entry point overwrites gpair and the root slot
  cudaEvent_t e0, e1; CUDA_OK(cudaEventCreate(&e0)); CUDA_OK(cudaEventCreate(&e1));
  float total = 0.f;
  for (int r = 0; r < std::max(1, repeats); ++r) {
    launch_init_tree(g.gs, g.ta, (unsigned)rows, 0, g.max_level_nodes, s);
    CUDA_OK(cudaMemsetAsync(g.hist_pool.p, 0, g.slot_stride * sizeof(GH64), s));
    CUDA_OK(cudaEventRecord(e0, s));
    launch_hist_build(ha, engine_num_sms(), s);
    CUDA_OK(cudaEventRecord(e1, s));
    CUDA_OK(cudaEventSynchronize(e1));
    float ms = 0; CUDA_OK(cudaEventElapsedTime(&ms, e0, e1)); total += ms;
  }
  if (ms_out) *ms_out = total / std::max(1, repeats);
  hist_out->resize(g.slot_stride * 2);
  CUDA_OK(cudaMemcpyAsync(hist_out->data(), g.hist_pool.p, sizeof(GH64) * g.slot_stride, cudaMemcpyDeviceToHost, s));
  CUDA_OK(cudaMemcpyAsync(scales_out, g.gs.scales, 4 * sizeof(float), cudaMemcpyDeviceToHost, s));
  Comm::get().sync_stream(s);
  cudaEventDestroy(e0); cudaEventDestroy(e1);
}

// pred_contribs: path-dependent Tree SHAP on the device (shap.cu); output [n][F + 1], or [n][K][F + 1] for multi-class models
void Booster::predict_contribs(DMatrix* dm, int tb, int te, std::vector<float>* out, std::vector<uint64_t>* shape) {
  cudaStream_t s = engine_stream();
  sync_model();
  const int K = param_.num_class;
  const int64_t n = dm->n;
  const int F = std::max(dm->F, num_feature_);
  B200_CHECK(dm->F == F, "pred_contribs: the data has " + std::to_string(dm->F) + " columns, the model uses " + std::to_string(F));
  std::vector<ShapNode> nodes; std::vector<int64_t> offs; std::vector<int> info;
  int max_depth = 0;
  for (int t = tb; t < te; ++t) {
    const HostTree& h = trees_[t];
    const int nn = h.num_nodes();
    const size_t base = nodes.size();
    offs.push_back((int64_t)base); info.push_back(tree_info_[t]);
    nodes.resize(base + nn);
    std::vector<int> depth(nn, 0);
    for (int i = 0; i < nn; ++i) {
      ShapNode& d = nodes[base + i];
      d.cond = h.split_cond[i]; d.left = h.left[i]; d.right = h.right[i]; d.fidx_dl = (unsigned)h.split_index[i] | ((unsigned)h.default_left[i] << 31);
      d.sum_hess = h.sum_hess[i]; d.mean = 0.0f;
      if (h.left[i] >= 0) { B200_CHECK(h.left[i] > i && h.right[i] > i, "pred_contribs: children must follow their parent in the node array"); depth[h.left[i]] = depth[h.right[i]] = depth[i] + 1; }
      max_depth = std::max(max_depth, depth[i]);
    }
    // cover-weighted mean value per node, children before parents (upstream FillNodeMeanValues, float arithmetic)
    for (int i = nn - 1; i >= 0; --i) {
      ShapNode& d = nodes[base + i];
      if (d.left < 0) d.mean = d.cond;
      else { float r = nodes[base + d.left].mean * nodes[base + d.left].sum_hess; r += nodes[base + d.right].mean * nodes[base + d.right].sum_hess; d.mean = r / d.sum_hess; }
    }
  }
  DevBuf<ShapNode> d_sn; DevBuf<int64_t> d_off; DevBuf<int> d_info; DevBuf<float> d_out;
  d_sn.alloc(std::max<size_t>(nodes.size(), 1)); d_off.alloc(std::max<size_t>(offs.size(), 1)); d_info.alloc(std::max<size_t>(info.size(), 1));
  const size_t total = (size_t)n * K * (F + 1);
  d_out.alloc(std::max<size_t>(total, 1));
  if (!nodes.empty()) {
    CUDA_OK(cudaMemcpyAsync(d_sn.p, nodes.data(), sizeof(ShapNode) * nodes.size(), cudaMemcpyHostToDevice, s));
    CUDA_OK(cudaMemcpyAsync(d_off.p, offs.data(), sizeof(int64_t) * offs.size(), cudaMemcpyHostToDevice, s));
    CUDA_OK(cudaMemcpyAsync(d_info.p, info.data(), sizeof(int) * info.size(), cudaMemcpyHostToDevice, s));
  }
  CUDA_OK(cudaMemsetAsync(d_out.p, 0, sizeof(float) * std::max<size_t>(total, 1), s));
  ShapArgs sa{}; sa.X = dm->X.p; sa.n = n; sa.F = F; sa.nodes = d_sn.p; sa.tree_offset = d_off.p; sa.tree_info = d_info.p; sa.tree_begin = tb; sa.tree_end = te; sa.K = K;
  sa.out = d_out.p; sa.base_margin = base_margin();
  if (!dm->base_margin.empty()) { B200_CHECK(dm->base_margin.size() == (size_t)n * K, "base_margin size does not match rows x groups"); sa.base_margin_rows = dm->d_base_margin.p; }
  launch_shap(sa, max_depth, s);
  out->resize(total);
  if (total) CUDA_OK(cudaMemcpyAsync(out->data(), d_out.p, sizeof(float) * total, cudaMemcpyDeviceToHost, s));
  Comm::get().sync_stream(s);
  if (K > 1) shape->assign({(uint64_t)n, (uint64_t)K, (uint64_t)(F + 1)}); else shape->assign({(uint64_t)n, (uint64_t)(F + 1)});
}

// device time of the predictor kernel alone (margins of all trees into the scratch buffer), for the roofline line of bench.py
float Booster::debug_predict_kernel_ms(DMatrix* dm, int repeats) {
  configure();
  cudaStream_t s = engine_stream();
  upload_model();
  const int K = param_.num_class;
  pred_margin_.ensure((size_t)dm->n * K);
  PredictArgs pa = predict_args(dm, 0, (int)trees_.size()); pa.margin = pred_margin_.p;
  cudaEvent_t e0, e1; CUDA_OK(cudaEventCreate(&e0)); CUDA_OK(cudaEventCreate(&e1));
  float total = 0.f;
  for (int r = 0; r < std::max(1, repeats); ++r) {
    launch_fill(pred_margin_.p, dm->n * K, base_margin(), s);
    CUDA_OK(cudaEventRecord(e0, s));
    launch_predict(pa, s);
    CUDA_OK(cudaEventRecord(e1, s));
    CUDA_OK(cudaEventSynchronize(e1));
    float ms = 0; CUDA_OK(cudaEventElapsedTime(&ms, e0, e1)); total += ms;
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  return total / std::max(1, repeats);
}

std::string Booster::predict_plan(DMatrix* dm, int iter_begin, int iter_end) {
  configure();
  const int K = param_.num_class;
  const int rounds = (int)trees_.size() / K;
  if (iter_end == 0) iter_end = rounds;
  B200_CHECK(iter_begin >= 0 && iter_begin <= iter_end && iter_end <= rounds, "Invalid iteration range: [" + std::to_string(iter_begin) + ", " + std::to_string(iter_end) + ") for a model with " + std::to_string(rounds) + " rounds");
  upload_model();                                  // device slot sizes: trained trees keep their fixed-capacity slots
  const int tb = iter_begin * K, te = iter_end * K;
  std::vector<int64_t> counts(te - tb);
  for (int t = tb; t < te; ++t) counts[t - tb] = h_tree_offset[t + 1] - h_tree_offset[t];
  return predict_plan_json(plan_predict(dm->F, num_feature_, counts.data(), tb, te, children_adjacent_));
}

void Booster::cached_margin(DMatrix* dm, std::vector<float>* out) {
  configure();
  cudaStream_t s = engine_stream();
  PredCache& c = cache_for(dm);
  bring_cache_up_to_date(dm, c);
  out->resize((size_t)dm->n * param_.num_class);
  if (!out->empty()) CUDA_OK(cudaMemcpyAsync(out->data(), c.margin.p, sizeof(float) * out->size(), cudaMemcpyDeviceToHost, s));
  Comm::get().sync_stream(s);
}

void Booster::set_profile(bool on) {
  profile_ = on;
  if (on) { prof_rows_.alloc(2); prof_rows_.zero(engine_stream()); prof_launches_ = 0; }
  for (auto& e : prof_events_) { cudaEventDestroy(e.a); cudaEventDestroy(e.b); }
  prof_events_.clear();
}
void Booster::prof_begin(int level) {
  if (!profile_) return;
  ProfEvent e; e.level = level;
  CUDA_OK(cudaEventCreate(&e.a)); CUDA_OK(cudaEventCreate(&e.b));
  CUDA_OK(cudaEventRecord(e.a, engine_stream()));
  prof_events_.push_back(e);
}
void Booster::prof_end() {
  if (!profile_) return;
  CUDA_OK(cudaEventRecord(prof_events_.back().b, engine_stream()));
}
std::string Booster::get_profile() {
  cudaStream_t s = engine_stream();
  Comm::get().sync_stream(s);
  double root_ms = 0, deep_ms = 0; long long root_n = 0, deep_n = 0;
  for (auto& e : prof_events_) { float ms = 0; CUDA_OK(cudaEventElapsedTime(&ms, e.a, e.b)); if (e.level == 0) { root_ms += ms; ++root_n; } else { deep_ms += ms; ++deep_n; } }
  unsigned long long rows[2] = {0, 0};
  if (prof_rows_.p) CUDA_OK(cudaMemcpy(rows, prof_rows_.p, sizeof rows, cudaMemcpyDeviceToHost));
  char buf[512];
  snprintf(buf, sizeof buf, "{\"root_hist_ms\":%.6f,\"root_hist_launches\":%lld,\"root_hist_rows\":%llu,\"deep_hist_ms\":%.6f,\"deep_hist_launches\":%lld,\"deep_hist_rows\":%llu}",
           root_ms, root_n, rows[0], deep_ms, deep_n, rows[1]);
  return buf;
}

}  // namespace b200
