// misc.cu -- objective gradients, feature binning, tree-traversal predictor and evaluation metrics.
// SURVEY.md section 8a rows A5, A5b, A6 (binning half), A11, A12.  Formulas restate upstream xgboost
// (src/objective/regression_loss.h, multiclass_obj.cu, src/data/gradient_index.cc, src/predictor/cpu_predictor.cc,
// src/metric/elementwise_metric.cu, multiclass_metric.cu) as written down in oracle/gbt_oracle.c.
#include <algorithm>
#include <cstdlib>
#include <utility>
#include "engine.h"
#include "misc.h"

namespace b200 {

__device__ __forceinline__ float sigmoidf_xgb(float x) {
  const float kEps = 1e-16f;
  x = fminf(-x, 88.7f);
  float denom = expf(x) + 1.0f + kEps;
  return 1.0f / denom;
}

__device__ __forceinline__ unsigned long long splitmix64_dev(unsigned long long x) {
  x += 0x9E3779B97F4A7C15ULL; x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ULL;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBULL; return x ^ (x >> 31);
}
__device__ __forceinline__ float rng_uniform_dev(unsigned seed, unsigned long long stream, unsigned long long idx) {
  unsigned long long h = splitmix64_dev(splitmix64_dev(((unsigned long long)seed << 32) ^ stream) ^ idx);
  return (float)(h >> 40) * (1.0f / 16777216.0f);
}

// ---------------------------------------------------------------------------------------------
// gradient pairs: one thread per row, all K classes; also the running max|g|, max h of the round
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gradient_kernel(GradArgs a) {
  float mg = 0.f, mh = 0.f;
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < a.n; r += (int64_t)gridDim.x * blockDim.x) {
    const float y = a.label[r];
    float w = a.weight ? a.weight[r] : 1.0f;
    bool dropped = false;
    if (a.subsample < 1.0f) dropped = !(rng_uniform_dev(a.seed, 0x2000ull + a.iter, (unsigned long long)(r + a.row_offset)) < a.subsample);
    if (a.objective == kSoftprob || a.objective == kSoftmax) {
      const int K = a.K;
      const float* m = a.margin ? a.margin + r * K : nullptr;
      float wmax = m ? m[0] : 0.f;
      for (int k = 1; k < K; ++k) wmax = fmaxf(wmax, m ? m[k] : 0.f);
      float wsum = 0.f;
      for (int k = 0; k < K; ++k) wsum += expf((m ? m[k] : 0.f) - wmax);
      int label = (int)y;
      if (label < 0 || label >= K) { *a.err = 2; label = 0; }
      for (int k = 0; k < K; ++k) {
        float pk = expf((m ? m[k] : 0.f) - wmax) / wsum;
        float h = fmaxf(2.0f * pk * (1.0f - pk) * w, 1e-16f);
        float g = (label == k ? pk - 1.0f : pk) * w;
        if (dropped) { g = 0.f; h = 0.f; }
        a.gpair[(int64_t)k * a.gp_stride + r] = make_float2(g, h);
        mg = fmaxf(mg, fabsf(g)); mh = fmaxf(mh, h);
      }
    } else {
      const bool reg_loss = a.objective <= kLogitRaw || a.objective == kSquaredLogError || a.objective == kPseudoHuber;     // RegLossObj family
      if (reg_loss && y == 1.0f) w *= a.scale_pos_weight;
      float p = a.margin ? a.margin[r] : 0.f, g, h;
      // upstream src/objective/regression_loss.h (RegLossObj family), regression_obj.cu (Poisson / Gamma / Tweedie), hinge.cu
      switch (a.objective) {
        case kSquaredError: g = p - y; h = 1.0f; break;
        case kSquaredLogError: {
          if (!(y > -1.0f)) *a.err = 3;
          p = fmaxf(p, -1.0f + 1e-6f);
          g = (log1pf(p) - log1pf(y)) / (p + 1.0f);
          h = fmaxf((-log1pf(p) + log1pf(y) + 1.0f) / ((p + 1.0f) * (p + 1.0f)), 1e-6f);
          break; }
        case kPseudoHuber: {
          const float z = p - y, s2 = a.aux * a.aux, scale_sqrt = sqrtf(1.0f + z * z / s2);
          g = z / scale_sqrt; h = s2 / ((s2 + z * z) * scale_sqrt);
          break; }
        case kPoisson: {
          if (y < 0.0f) *a.err = 4;
          g = expf(p) - y; h = expf(p + a.aux);
          break; }
        case kGamma: {
          if (!(y > 0.0f)) *a.err = 5;
          const float ep = expf(p);
          g = 1.0f - y / ep; h = y / ep;
          break; }
        case kTweedie: {
          if (y < 0.0f) *a.err = 6;
          const float rho = a.aux, e1 = expf((1.0f - rho) * p), e2 = expf((2.0f - rho) * p);
          g = -y * e1 + e2; h = -y * (1.0f - rho) * e1 + (2.0f - rho) * e2;
          break; }
        case kHinge: {
          const float yy = y * 2.0f - 1.0f;
          if (p * yy < 1.0f) { g = -yy; h = 1.0f; } else { g = 0.0f; h = 1.17549435e-38f; }      // upstream: numeric_limits<float>::min()
          break; }
        default: {
          if (y < 0.0f || y > 1.0f) *a.err = 1;
          p = sigmoidf_xgb(p); g = p - y; h = fmaxf(p * (1.0f - p), 1e-16f);
          break; }
      }
      g *= w; h *= w;
      if (dropped) { g = 0.f; h = 0.f; }
      a.gpair[r] = make_float2(g, h);
      mg = fmaxf(mg, fabsf(g)); mh = fmaxf(mh, h);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { mg = fmaxf(mg, __shfl_xor_sync(0xffffffffu, mg, o)); mh = fmaxf(mh, __shfl_xor_sync(0xffffffffu, mh, o)); }
  __shared__ float sg[8], sh[8];
  if ((threadIdx.x & 31) == 0) { sg[threadIdx.x >> 5] = mg; sh[threadIdx.x >> 5] = mh; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 8; ++w) { mg = fmaxf(mg, sg[w]); mh = fmaxf(mh, sh[w]); }
    if (a.absmax) { atomicMax(a.absmax, __float_as_uint(mg)); atomicMax(a.absmax + 1, __float_as_uint(mh)); }
  }
}

// sum of (g,h) over rows in double (base-score stump)
__global__ void __launch_bounds__(256) sum_gpair_kernel(const float2* gp, int64_t n, double* out) {
  double g = 0, h = 0;
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x) { float2 v = gp[r]; g += v.x; h += v.y; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { g += __shfl_xor_sync(0xffffffffu, g, o); h += __shfl_xor_sync(0xffffffffu, h, o); }
  if ((threadIdx.x & 31) == 0) { atomicAdd(out, g); atomicAdd(out + 1, h); }
}

// ---------------------------------------------------------------------------------------------
// binning: float matrix (row-major, NaN = missing) -> uint8 codes in the layout of engine.h BinnedMatrix:
// main [n][ngroups*32] (byte column c == feature c) and tail [n][tw] (tail slot s == feature ngroups*32 + s)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint8_t bin_of(float v, const float* c, int nc) {
  if (isnan(v)) return (uint8_t)kMissingBin;
  int lo = 0, hi = nc;
  while (lo < hi) { int mid = (lo + hi) >> 1; if (c[mid] > v) hi = mid; else lo = mid + 1; }
  if (lo >= nc) lo = nc - 1;
  return (uint8_t)lo;
}

__global__ void __launch_bounds__(256) bin_kernel(const float* X, int64_t n, int F, int ngroups, int tw, const int* cut_ptrs, const float* cut_vals,
                                                  uint8_t* bins, uint8_t* bins_tail) {
  const int W = ngroups * kSlots + tw;                  // byte columns per row over both blocks
  const int64_t total = n * W;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(idx % W);
    const int64_t r = idx / W;
    uint8_t b = 0;
    if (c < F) b = bin_of(X[r * F + c], cut_vals + cut_ptrs[c], cut_ptrs[c + 1] - cut_ptrs[c]);     // byte column == feature index in both blocks
    if (c < ngroups * kSlots) bins[r * (ngroups * kSlots) + c] = b;
    else bins_tail[r * tw + (c - ngroups * kSlots)] = b;
  }
}

// rows re-laid at `dst_stride` bytes (whole 128 B lines for 96 B rows): 16 B per thread
__global__ void __launch_bounds__(256) pad_rows_kernel(const uint8_t* src, int64_t n, int src_stride, uint8_t* dst, int dst_stride) {
  const int cpr = dst_stride / 16, spr = src_stride / 16;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n * cpr; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / cpr; const int c = (int)(i - r * cpr);
    uint4 v = make_uint4(0, 0, 0, 0);
    if (c < spr) v = reinterpret_cast<const uint4*>(src + r * src_stride)[c];
    reinterpret_cast<uint4*>(dst + r * dst_stride)[c] = v;
  }
}
void launch_pad_rows(const uint8_t* src, int64_t n, int src_stride, uint8_t* dst, int dst_stride, cudaStream_t s) {
  if (n == 0) return;
  pad_rows_kernel<<<148 * 16, 256, 0, s>>>(src, n, src_stride, dst, dst_stride); ++g_kernel_launches; CUDA_OK(cudaGetLastError());
}

// column-major copy [F][n] of the binned matrix (used by the 1-byte-per-row consumers: partition, cache update)
__global__ void __launch_bounds__(256) transpose_bins_kernel(const uint8_t* bins, const uint8_t* bins_tail, int64_t n, int F, int ngroups, int tw, uint8_t* bins_col) {
  __shared__ uint8_t tile[256][kSlots + 1];
  const int g = blockIdx.y;                             // ngroups == the tail block
  const bool is_tail = g == ngroups;
  const int width = is_tail ? tw : kSlots;
  const int64_t r0 = (int64_t)blockIdx.x * 256;
  for (int i = threadIdx.x; i < 256 * width; i += 256) {
    int rr = i / width, s = i % width;
    int64_t r = r0 + rr;
    tile[rr][s] = r < n ? (is_tail ? bins_tail[r * tw + s] : bins[r * (ngroups * kSlots) + g * kSlots + s]) : 0;
  }
  __syncthreads();
  const int64_t r = r0 + threadIdx.x;
  if (r < n) for (int s = 0; s < width; ++s) { int f = g * kSlots + s; if (f < F) bins_col[(int64_t)f * n + r] = tile[threadIdx.x][s]; }
}

__global__ void __launch_bounds__(256) count_nan_kernel(const float* X, int64_t count, float missing, int use_missing, unsigned long long* out) {
  unsigned long long c = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) {
    float v = X[i];
    c += (isnan(v) || (use_missing && v == missing)) ? 1ull : 0ull;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, c);
}

__global__ void __launch_bounds__(256) replace_missing_kernel(float* X, int64_t count, float missing) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x)
    if (X[i] == missing) X[i] = __int_as_float(0x7fc00000);
}

// ---------------------------------------------------------------------------------------------
// predictor: one thread per row, trees in model order, fp32 accumulation
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) predict_kernel(PredictArgs a) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= a.n) return;
  const float* x = a.X + r * a.F;
  const int nt = a.tree_end - a.tree_begin;
  float acc = (a.K == 1 && a.margin) ? a.margin[r] : 0.f;
  for (int t = a.tree_begin; t < a.tree_end; ++t) {
    const DevNode* nodes = a.nodes + a.tree_offset[t];
    int nid = 0;
    DevNode nd = nodes[0];
    while (nd.left != -1) {
      const unsigned f = nd.fidx_dl & 0x7fffffffu;
      const float v = f < (unsigned)a.F ? __ldg(x + f) : __int_as_float(0x7fc00000);
      if (isnan(v)) nid = (nd.fidx_dl >> 31) ? nd.left : nd.right;
      else nid = v < nd.cond ? nd.left : nd.right;
      nd = nodes[nid];
    }
    if (a.margin) { if (a.K == 1) acc += nd.cond; else a.margin[r * a.K + a.tree_info[t]] += nd.cond; }
    if (a.leaf) a.leaf[r * nt + (t - a.tree_begin)] = nid;
  }
  if (a.K == 1 && a.margin) a.margin[r] = acc;
}

// Block-cooperative predictor (BASELINE config 5): a CTA stages a tile of rows into shared memory with coalesced loads
// (the thread-per-row kernel above gathers 4 B at a time from a 4*F-byte row: 1 % of HBM peak in round 1) and keeps the
// trees there too, 8 B per node, so a traversal step is two LDS.  With T trees of depth D a row costs ~8*T*D instructions
// against 4*F bytes: beyond T*D ~ 100 the kernel is issue-bound, not HBM-bound (DESIGN.md "predictor").
struct PNode { float cond; unsigned w; };            // w = left child (16 bit, 0xffff = leaf) | feature << 16 | default_left << 31

template <bool HAS_NAN, bool LEAF_OUT>
__global__ void __launch_bounds__(1024) predict_tiled_kernel(PredictArgs a, int tree_lo, int tree_hi, int pitch, int rows_per_tile, int64_t num_tiles) {
  extern __shared__ __align__(16) unsigned char psm[];
  const int nt_chunk = tree_hi - tree_lo;
  int* s_toff = reinterpret_cast<int*>(psm);                                   // [nt_chunk + 1] node offsets inside s_nodes
  PNode* s_nodes = reinterpret_cast<PNode*>(psm + (((size_t)(nt_chunk + 1) * 4 + 15) & ~(size_t)15));
  __shared__ int s_total;
  if (threadIdx.x == 0) {
    int off = 0;
    for (int t = 0; t < nt_chunk; ++t) { s_toff[t] = off; off += (int)(a.tree_offset[tree_lo + t + 1] - a.tree_offset[tree_lo + t]); }
    s_toff[nt_chunk] = off; s_total = off;
  }
  __syncthreads();
  for (int t = 0; t < nt_chunk; ++t) {
    const DevNode* src = a.nodes + a.tree_offset[tree_lo + t];
    const int cnt = s_toff[t + 1] - s_toff[t];
    for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
      const DevNode d = src[i];
      PNode p; p.cond = d.cond;
      p.w = (d.left < 0 ? 0xffffu : (unsigned)d.left) | ((d.fidx_dl & 0x7fffu) << 16) | (d.fidx_dl & 0x80000000u);
      s_nodes[s_toff[t] + i] = p;
    }
  }
  float* s_x = reinterpret_cast<float*>(s_nodes + s_total);
  const int F = a.F, K = a.K, nt_all = a.tree_end - a.tree_begin;
  if (F < a.F_model) {                                                          // features the matrix lacks are missing; the tile
    const int w = a.F_model - F;                                                // loads below never overwrite these slots
    for (int i = threadIdx.x; i < rows_per_tile * w; i += blockDim.x) { const int r = i / w; s_x[r * pitch + F + (i - r * w)] = __int_as_float(0x7fc00000); }
  }
  for (int64_t tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
    const int64_t r0 = tile * rows_per_tile;
    const int rows = (int)((a.n - r0 < rows_per_tile) ? a.n - r0 : rows_per_tile);
    __syncthreads();                                                            // trees staged / previous tile consumed
    const float* src = a.X + r0 * F;
    const int total = rows * F;
    for (int i = threadIdx.x; i < total; i += blockDim.x) { const int r = i / F, f = i - r * F; s_x[r * pitch + f] = __ldg(src + i); }
    __syncthreads();
    for (int rl = threadIdx.x; rl < rows; rl += blockDim.x) {
      const float* x = s_x + rl * pitch;
      const int64_t r = r0 + rl;
      float acc = (!LEAF_OUT && K == 1) ? a.margin[r] : 0.f;
      auto step = [&](const PNode* tn, int& nid, PNode& nd) {
        const float v = x[(nd.w >> 16) & 0x7fffu];
        const int left = (int)(nd.w & 0xffffu);
        bool go_left = v < nd.cond;
        if (HAS_NAN) { if (isnan(v)) go_left = (nd.w >> 31) != 0; }
        nid = go_left ? left : left + 1;                                        // children are allocated as adjacent pairs
        nd = tn[nid];
      };
      auto emit = [&](int t, int nid, const PNode& nd) {
        if (LEAF_OUT) a.leaf[r * nt_all + (tree_lo - a.tree_begin) + t] = nid;
        else if (K == 1) acc += nd.cond;                                        // fp32, in tree order (== the reference's sequential sum)
        else a.margin[r * K + a.tree_info[tree_lo + t]] += nd.cond;
      };
      int t = 0;
      for (; t + 4 <= nt_chunk; t += 4) {                                       // four independent traversals in flight hide the LDS latency
        const PNode* tn[4]; int nid[4]; PNode nd[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) { tn[j] = s_nodes + s_toff[t + j]; nid[j] = 0; nd[j] = tn[j][0]; }
        bool any = true;
        while (any) {
          any = false;
#pragma unroll
          for (int j = 0; j < 4; ++j) if ((nd[j].w & 0xffffu) != 0xffffu) { step(tn[j], nid[j], nd[j]); any = true; }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) emit(t + j, nid[j], nd[j]);
      }
      for (; t < nt_chunk; ++t) {
        const PNode* tn = s_nodes + s_toff[t];
        int nid = 0; PNode nd = tn[0];
        while ((nd.w & 0xffffu) != 0xffffu) step(tn, nid, nd);
        emit(t, nid, nd);
      }
      if (!LEAF_OUT && K == 1) a.margin[r] = acc;
    }
  }
}

// margins -> predictions (PredTransform), in place
__global__ void __launch_bounds__(256) transform_kernel(float* m, int64_t n, int K, int objective, float* out_class) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  if (objective == kBinaryLogistic || objective == kRegLogistic) m[r] = sigmoidf_xgb(m[r]);
  else if (objective == kPoisson || objective == kGamma || objective == kTweedie) m[r] = expf(m[r]);
  else if (objective == kHinge) m[r] = m[r] > 0.0f ? 1.0f : 0.0f;
  else if (objective == kSoftprob || objective == kSoftmax) {
    float* p = m + r * K;
    float wmax = p[0]; int arg = 0;
    for (int k = 1; k < K; ++k) if (p[k] > wmax) { wmax = p[k]; arg = k; }
    if (objective == kSoftmax) { out_class[r] = (float)arg; return; }
    float wsum = 0.f;
    for (int k = 0; k < K; ++k) { p[k] = expf(p[k] - wmax); wsum += p[k]; }
    for (int k = 0; k < K; ++k) p[k] /= wsum;
  }
}

__global__ void __launch_bounds__(256) fill_kernel(float* p, int64_t n, float v) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) p[i] = v;
}
__global__ void __launch_bounds__(256) add_base_margin_kernel(float* p, const float* bm, int64_t count) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) p[i] = bm[i];
}

// ---------------------------------------------------------------------------------------------
// element-wise evaluation metrics on raw margins: out[0] += sum(w * loss), out[1] += sum(w)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) metric_kernel(MetricArgs a) {
  double s = 0, ws = 0;
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < a.n; r += (int64_t)gridDim.x * blockDim.x) {
    const float y = a.label[r];
    const float w = a.weight ? a.weight[r] : 1.0f;
    float loss = 0.f;
    if (a.metric == kMetricMlogloss || a.metric == kMetricMerror) {
      const float* m = a.margin + r * a.K;
      float wmax = m[0]; int arg = 0;
      for (int k = 1; k < a.K; ++k) if (m[k] > wmax) { wmax = m[k]; arg = k; }
      int label = (int)y;
      if (a.metric == kMetricMerror) loss = (arg != label) ? 1.f : 0.f;
      else {
        float wsum = 0.f;
        for (int k = 0; k < a.K; ++k) wsum += expf(m[k] - wmax);
        float p = (label >= 0 && label < a.K) ? expf(m[label] - wmax) / wsum : 0.f;
        const float eps = 1e-16f;
        loss = p > eps ? -logf(p) : -logf(eps);
      }
    } else {
      float p = a.margin[r];
      if (a.is_logistic || a.transform == kTransformSigmoid) p = sigmoidf_xgb(p);
      else if (a.transform == kTransformExp) p = expf(p);
      else if (a.transform == kTransformHinge) p = p > 0.0f ? 1.0f : 0.0f;
      switch (a.metric) {          // upstream src/metric/elementwise_metric.cu
        case kMetricRmsle: { float d = log1pf(y) - log1pf(p); loss = d * d; break; }
        case kMetricMape: loss = fabsf((y - p) / y); break;
        case kMetricMphe: { const float z = (y - p) / a.aux; loss = a.aux * a.aux * (sqrtf(1.0f + z * z) - 1.0f); break; }
        case kMetricPoissonNll: { const float py = fmaxf(p, 1e-16f); loss = lgammaf(y + 1.0f) + py - logf(py) * y; break; }
        case kMetricGammaNll: { const float py = fmaxf(p, 1e-6f); loss = y / py + logf(py); break; }       // psi = 1: -((y * theta - b) / a + c), theta = -1 / py, b = -log(-theta)
        case kMetricGammaDeviance: { const float py = p + 1e-6f, yy = y + 1e-6f; loss = logf(py / yy) + yy / py - 1.0f; break; }      // x 2 on the host
        case kMetricTweedieNll: { const float rho = a.aux, lp = logf(p); loss = -y * expf((1.0f - rho) * lp) / (1.0f - rho) + expf((2.0f - rho) * lp) / (2.0f - rho); break; }
        case kMetricRmse: { float d = p - y; loss = d * d; break; }
        case kMetricMae: loss = fabsf(p - y); break;
        case kMetricLogloss: {
          const float eps = 1e-16f;
          float pneg = 1.0f - p;
          if (p < eps) loss = -y * logf(eps) - (1.0f - y) * logf(1.0f - eps);
          else if (pneg < eps) loss = -y * logf(1.0f - eps) - (1.0f - y) * logf(eps);
          else loss = -y * logf(p) - (1.0f - y) * logf(pneg);
          break; }
        case kMetricError: loss = (p > a.threshold) ? (1.0f - y) : y; break;
        default: break;
      }
    }
    s += (double)(loss * w); ws += (double)w;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { s += __shfl_xor_sync(0xffffffffu, s, o); ws += __shfl_xor_sync(0xffffffffu, ws, o); }
  if ((threadIdx.x & 31) == 0) { atomicAdd(a.out, s); atomicAdd(a.out + 1, ws); }
}

// ---------------------------------------------------------------------------------------------
static inline int grid_for(int64_t n, int block = 256, int cap = 148 * 16) {
  int64_t g = (n + block - 1) / block; if (g < 1) g = 1; if (g > cap) g = cap; return (int)g;
}
void launch_gradient(const GradArgs& a, cudaStream_t s) {
  if (a.n == 0) return;
  gradient_kernel<<<grid_for(a.n, 256, 148 * 8), 256, 0, s>>>(a); ++g_kernel_launches; CUDA_OK(cudaGetLastError());
}
void launch_sum_gpair(const float2* gp, int64_t n, double* out, cudaStream_t s) {
  sum_gpair_kernel<<<grid_for(n), 256, 0, s>>>(gp, n, out); ++g_kernel_launches; CUDA_OK(cudaGetLastError());
}
void launch_bin(const float* X, int64_t n, int F, int ngroups, int tw, const int* cut_ptrs, const float* cut_vals, uint8_t* bins, uint8_t* bins_tail, cudaStream_t s) {
  if (n == 0) return;
  bin_kernel<<<grid_for(n * (ngroups * kSlots + tw), 256, 148 * 32), 256, 0, s>>>(X, n, F, ngroups, tw, cut_ptrs, cut_vals, bins, bins_tail); ++g_kernel_launches;
  CUDA_OK(cudaGetLastError());
}
void launch_transpose_bins(const uint8_t* bins, const uint8_t* bins_tail, int64_t n, int F, int ngroups, int tw, uint8_t* bins_col, cudaStream_t s) {
  if (n == 0) return;
  dim3 grid((unsigned)((n + 255) / 256), ngroups + (tw > 0 ? 1 : 0));
  transpose_bins_kernel<<<grid, 256, 0, s>>>(bins, bins_tail, n, F, ngroups, tw, bins_col); ++g_kernel_launches; CUDA_OK(cudaGetLastError());
}
void launch_count_nan(const float* X, int64_t count, float missing, int use_missing, unsigned long long* out, cudaStream_t s) {
  if (count == 0) return;
  count_nan_kernel<<<grid_for(count), 256, 0, s>>>(X, count, missing, use_missing, out); ++g_kernel_launches; CUDA_OK(cudaGetLastError());
}
void launch_replace_missing(float* X, int64_t count, float missing, cudaStream_t s) {
  if (count == 0) return;
  replace_missing_kernel<<<grid_for(count), 256, 0, s>>>(X, count, missing); ++g_kernel_launches; CUDA_OK(cudaGetLastError());
}
// Plan of the tiled predictor: trees are cut, in order, into chunks whose packed nodes fit in shared memory next to a tile of
// at least 32 rows.  Anything the tiled kernel cannot hold takes the thread-per-row kernel.
PredictPlan plan_predict(int F, int F_model, const int64_t* node_counts, int tree_begin, int tree_end, bool children_adjacent) {
  PredictPlan p;
  const int width = std::max(F, F_model);                          // a narrower matrix is staged at the model's width, NaN-padded
  p.pitch = width | 1;                                             // odd pitch: threads of a warp (rows) hit different banks for the same feature
  p.absent_features = F < F_model;
  const size_t min_tile = (size_t)p.pitch * 4 * 32;
  if (!(width <= 32767 && children_adjacent) || min_tile + 64 * 1024 > kPredictSmem) return p;   // 15-bit feature field
  p.node_budget = 96 * 1024;                                       // bytes of packed nodes per chunk
  auto offsets = [](int trees) { return ((size_t)(trees + 1) * 4 + 15) & ~(size_t)15; };
  auto fits = [&](int trees, size_t bytes) { return bytes <= p.node_budget && offsets(trees) + bytes + min_tile <= kPredictSmem; };
  int lo = tree_begin;
  while (lo < tree_end) {
    int hi = lo; size_t bytes = 0;
    while (hi < tree_end) {
      const int64_t nn = node_counts[hi - tree_begin];
      if (nn > 65534) { p.chunks.clear(); return p; }              // the packed node keeps a 16-bit child index
      if (!fits(hi - lo + 1, bytes + (size_t)nn * 8)) {
        if (hi == lo) { p.chunks.clear(); return p; }              // a tree too large for any chunk
        break;
      }
      bytes += (size_t)nn * 8; ++hi;
    }
    PredictChunk c;
    c.tree_lo = lo; c.tree_hi = hi;
    c.head = offsets(hi - lo) + bytes;
    int rows = (int)((kPredictSmem - c.head) / ((size_t)p.pitch * 4));
    rows = rows > 1024 ? 1024 : (rows / 32) * 32;
    c.threads = rows >= 1024 ? 1024 : (rows >= 512 ? 512 : 256);
    c.rows = rows > c.threads ? c.threads : rows;                  // one row per thread and tile
    c.smem = c.head + (size_t)c.rows * p.pitch * 4;
    p.chunks.push_back(c);
    lo = hi;
  }
  p.tiled = true;
  return p;
}

std::string predict_plan_json(const PredictPlan& p) {
  std::string s = std::string("{\"route\":\"") + (p.tiled ? "tiled" : "thread_per_row") + "\",\"kernel\":\"" +
                  (p.tiled ? "predict_tiled_kernel" : "predict_kernel") + "\",\"pitch\":" + std::to_string(p.pitch) +
                  ",\"absent_features\":" + (p.absent_features ? "true" : "false") + ",\"node_budget\":" + std::to_string(p.node_budget) +
                  ",\"smem_limit\":" + std::to_string(kPredictSmem) + ",\"chunks\":[";
  for (size_t i = 0; i < p.chunks.size(); ++i) {
    const PredictChunk& c = p.chunks[i];
    s += std::string(i ? "," : "") + "{\"tree_lo\":" + std::to_string(c.tree_lo) + ",\"tree_hi\":" + std::to_string(c.tree_hi) +
         ",\"rows\":" + std::to_string(c.rows) + ",\"threads\":" + std::to_string(c.threads) + ",\"head\":" + std::to_string(c.head) +
         ",\"smem\":" + std::to_string(c.smem) + "}";
  }
  return s + "]}";
}

void launch_predict(const PredictArgs& a, cudaStream_t s) {
  if (a.n == 0 || a.tree_end <= a.tree_begin) return;
  std::vector<int64_t> counts(a.tree_end - a.tree_begin);
  for (int t = a.tree_begin; t < a.tree_end; ++t) counts[t - a.tree_begin] = a.h_tree_offset[t + 1] - a.h_tree_offset[t];
  const PredictPlan p = plan_predict(a.F, a.F_model, counts.data(), a.tree_begin, a.tree_end, a.children_adjacent != 0);
  if (!p.tiled) {
    predict_kernel<<<(unsigned)((a.n + 255) / 256), 256, 0, s>>>(a); ++g_kernel_launches; CUDA_OK(cudaGetLastError());
    return;
  }
  static bool attr = false;
  if (!attr) {
    CUDA_OK(cudaFuncSetAttribute(predict_tiled_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPredictSmem));
    CUDA_OK(cudaFuncSetAttribute(predict_tiled_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPredictSmem));
    CUDA_OK(cudaFuncSetAttribute(predict_tiled_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPredictSmem));
    CUDA_OK(cudaFuncSetAttribute(predict_tiled_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPredictSmem));
    attr = true;
  }
  const bool nan = a.has_nan || p.absent_features;
  for (const PredictChunk& c : p.chunks) {
    const int64_t tiles = (a.n + c.rows - 1) / c.rows;
    const int grid = (int)std::min<int64_t>(tiles, 148 * (c.threads == 1024 ? 1 : 2048 / c.threads));
    if (a.leaf) { if (nan) predict_tiled_kernel<true, true><<<grid, c.threads, c.smem, s>>>(a, c.tree_lo, c.tree_hi, p.pitch, c.rows, tiles);
                  else predict_tiled_kernel<false, true><<<grid, c.threads, c.smem, s>>>(a, c.tree_lo, c.tree_hi, p.pitch, c.rows, tiles); }
    else { if (nan) predict_tiled_kernel<true, false><<<grid, c.threads, c.smem, s>>>(a, c.tree_lo, c.tree_hi, p.pitch, c.rows, tiles);
           else predict_tiled_kernel<false, false><<<grid, c.threads, c.smem, s>>>(a, c.tree_lo, c.tree_hi, p.pitch, c.rows, tiles); }
    ++g_kernel_launches; CUDA_OK(cudaGetLastError());
  }
}
void launch_transform(float* m, int64_t n, int K, int objective, float* out_class, cudaStream_t s) {
  if (n == 0) return;
  transform_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(m, n, K, objective, out_class); ++g_kernel_launches; CUDA_OK(cudaGetLastError());
}
void launch_fill(float* p, int64_t n, float v, cudaStream_t s) {
  if (n == 0) return;
  fill_kernel<<<grid_for(n), 256, 0, s>>>(p, n, v); ++g_kernel_launches; CUDA_OK(cudaGetLastError());
}
void launch_metric(const MetricArgs& a, cudaStream_t s) {
  if (a.n == 0) return;
  metric_kernel<<<grid_for(a.n), 256, 0, s>>>(a); ++g_kernel_launches; CUDA_OK(cudaGetLastError());
}

}  // namespace b200
