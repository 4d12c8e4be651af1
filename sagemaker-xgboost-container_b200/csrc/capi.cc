// capi.cc -- extern "C" surface of libb200xgb.so (declared in include/b200xgb.h).
// Same conventions as libxgboost's c_api.cc: int return code, thread-local last error, handle-owned buffers.
#include "../../include/b200xgb.h"
#include <cmath>
#include <cstdio>
#include <cstring>
#include <algorithm>
#include <dirent.h>
#include <fstream>
#include <map>
#include <memory>
#include <sstream>
#include <sys/stat.h>
#include <string>
#include <vector>
#include "booster.h"
#include "comm.h"

using namespace b200;

namespace {
thread_local std::string g_last_error;
struct DMatrixBox {
  std::unique_ptr<DMatrix> dm;
  std::vector<const char*> str_ptrs; std::vector<std::string> strs;
  std::vector<uint8_t> scratch_u8;
};
struct BoosterBox {
  std::unique_ptr<Booster> bst;
  std::string ret_str; std::vector<float> ret_vec; std::vector<uint64_t> ret_shape;
  std::vector<const char*> str_ptrs; std::vector<std::string> strs;
};
thread_local std::string g_ret_str;

int fail(const std::exception& e) { g_last_error = e.what(); return -1; }
DMatrix* DM(DMatrixHandle h) { if (!h) throw Error("DMatrix handle is NULL"); return static_cast<DMatrixBox*>(h)->dm.get(); }
Booster* BST(BoosterHandle h) { if (!h) throw Error("Booster handle is NULL"); return static_cast<BoosterBox*>(h)->bst.get(); }
#define API_BEGIN() try {
#define API_END() } catch (const std::exception& e) { return fail(e); } return 0;

std::string hex_encode(const std::string& s) { static const char* d = "0123456789abcdef"; std::string o; for (unsigned char c : s) { o.push_back(d[c >> 4]); o.push_back(d[c & 15]); } return o; }
std::string hex_decode(const std::string& s) { std::string o; auto v = [](char c) { return c <= '9' ? c - '0' : (c | 32) - 'a' + 10; };
  for (size_t i = 0; i + 1 < s.size(); i += 2) o.push_back((char)((v(s[i]) << 4) | v(s[i + 1]))); return o; }
}  // namespace

extern "C" {

const char* XGBGetLastError(void) { return g_last_error.c_str(); }
void XGBoostVersion(int* major, int* minor, int* patch) { if (major) *major = 3; if (minor) *minor = 0; if (patch) *patch = 5; }
int XGBuildInfo(const char** out) {
  API_BEGIN();
  g_ret_str = "{\"USE_CUDA\":true,\"USE_NCCL\":true,\"arch\":\"sm_100a\",\"library\":\"b200xgb\",\"CPU_FALLBACK\":false}";
  *out = g_ret_str.c_str();
  API_END();
}

// ------------------------------------------------------------------------------------------- DMatrix
int XGDMatrixCreateFromMat(const float* data, bst_ulong nrow, bst_ulong ncol, float missing, DMatrixHandle* out) {
  API_BEGIN();
  auto box = new DMatrixBox(); std::unique_ptr<DMatrixBox> guard(box);
  box->dm = DMatrix::from_dense(data, (int64_t)nrow, (int)ncol, missing);
  *out = guard.release();
  API_END();
}
int XGDMatrixCreateFromCSREx(const size_t* indptr, const unsigned* indices, const float* data, size_t nindptr, size_t nelem,
                             size_t num_col, DMatrixHandle* out) {
  API_BEGIN();
  auto box = new DMatrixBox(); std::unique_ptr<DMatrixBox> guard(box);
  box->dm = DMatrix::from_csr(indptr, indices, data, nindptr, nelem, num_col);
  *out = guard.release();
  API_END();
}
int XGDMatrixCreateFromCudaArrayInterface(const char* data, const char* config, DMatrixHandle* out) {
  API_BEGIN();
  JPtr a = parse_json(data); JPtr cfg = parse_json(config ? config : "{}");
  const JValue& shape = a->at("shape");
  if (shape.length() != 2) throw Error("cuda array interface: expecting a 2-dimensional array");
  if (a->at("typestr").s != "<f4") throw Error("cuda array interface: only float32 (<f4) is supported, got " + a->at("typestr").s);
  if (a->has("strides") && a->at("strides").type != JValue::kNull) throw Error("cuda array interface: only C-contiguous arrays are supported");
  const float* ptr = reinterpret_cast<const float*>((uintptr_t)a->at("data").arr[0]->as_int());
  float missing = cfg->has("missing") ? (float)cfg->at("missing").as_double() : std::nanf("");
  auto box = new DMatrixBox(); std::unique_ptr<DMatrixBox> guard(box);
  box->dm = DMatrix::from_device(ptr, (int64_t)shape.num_at(0), (int)shape.num_at(1), missing);
  *out = guard.release();
  API_END();
}
// ---- host array interface (numpy `__array_interface__` as JSON): what upstream's Python package passes for ndarray inputs
namespace {
struct HostArray { const void* ptr; int64_t n, m; std::string typestr; };
HostArray parse_array_interface(const char* json) {
  JPtr a = parse_json(json);
  HostArray h{};
  const JValue& shape = a->at("shape");
  if (shape.length() < 1 || shape.length() > 2) throw Error("array interface: expecting a 1- or 2-dimensional array");
  h.n = (int64_t)shape.num_at(0); h.m = shape.length() == 2 ? (int64_t)shape.num_at(1) : 1;
  if (a->has("strides") && a->at("strides").type != JValue::kNull) throw Error("array interface: only C-contiguous arrays are supported");
  h.typestr = a->at("typestr").s;
  h.ptr = reinterpret_cast<const void*>((uintptr_t)a->at("data").arr[0]->as_int());
  return h;
}
std::vector<float> to_float32(const HostArray& h) {
  const size_t cnt = (size_t)h.n * h.m;
  std::vector<float> v(cnt);
  const std::string& t = h.typestr;
#define CONV(T) { const T* p = static_cast<const T*>(h.ptr); for (size_t i = 0; i < cnt; ++i) v[i] = (float)p[i]; }
  if (t == "<f4") memcpy(v.data(), h.ptr, cnt * 4);
  else if (t == "<f8") CONV(double) else if (t == "<i4") CONV(int32_t) else if (t == "<i8") CONV(int64_t) else if (t == "<u4") CONV(uint32_t)
  else if (t == "<u8") CONV(uint64_t) else if (t == "<i2") CONV(int16_t) else if (t == "<u2") CONV(uint16_t) else if (t == "|i1") CONV(int8_t)
  else if (t == "|u1" || t == "|b1") CONV(uint8_t)
  else throw Error("array interface: unsupported typestr " + t);
#undef CONV
  return v;
}
}  // namespace

int XGDMatrixCreateFromDense(const char* data, const char* config, DMatrixHandle* out) {
  API_BEGIN();
  HostArray h = parse_array_interface(data);
  JPtr cfg = parse_json(config ? config : "{}");
  float missing = cfg->has("missing") ? (float)cfg->at("missing").as_double() : std::nanf("");
  auto box = new DMatrixBox(); std::unique_ptr<DMatrixBox> guard(box);
  if (h.typestr == "<f4") box->dm = DMatrix::from_dense(static_cast<const float*>(h.ptr), h.n, (int)h.m, missing);
  else { std::vector<float> v = to_float32(h); box->dm = DMatrix::from_dense(v.data(), h.n, (int)h.m, missing); }
  *out = guard.release();
  API_END();
}
int XGDMatrixSetInfoFromInterface(DMatrixHandle handle, const char* field, const char* data) {
  API_BEGIN();
  HostArray h = parse_array_interface(data);
  std::vector<float> v = to_float32(h);
  DM(handle)->set_float_info(field, v.data(), v.size());
  API_END();
}

// ---- URI loader in C (data_utils.py:309-313,361 hand "<path>?format=csv&label_column=0[&weight_column=1]" / "?format=libsvm"
// to xgb.DMatrix): every regular file of the directory; CSV text goes to the device parser, libsvm is tokenised here.
namespace {
std::vector<std::string> list_files(const std::string& path) {
  struct stat st;
  if (stat(path.c_str(), &st) != 0) throw Error("Opening " + path + " failed: No such file or directory");
  std::vector<std::string> files;
  if (S_ISDIR(st.st_mode)) {
    DIR* d = opendir(path.c_str());
    if (!d) throw Error("Opening " + path + " failed");
    while (dirent* e = readdir(d)) { std::string f = path + "/" + e->d_name; struct stat fs; if (stat(f.c_str(), &fs) == 0 && S_ISREG(fs.st_mode)) files.push_back(f); }
    closedir(d);
    std::sort(files.begin(), files.end());
    if (files.empty()) throw Error("No files found in " + path);
  } else files.push_back(path);
  return files;
}
std::string read_stripped(const std::string& f) {
  std::ifstream in(f, std::ios::binary);
  std::stringstream ss; ss << in.rdbuf();
  std::string t = ss.str();
  size_t a = 0, b = t.size();
  while (a < b && (t[a] == '\n' || t[a] == '\r' || t[a] == ' ' || t[a] == '\t')) ++a;
  while (b > a && (t[b - 1] == '\n' || t[b - 1] == '\r' || t[b - 1] == ' ' || t[b - 1] == '\t')) --b;
  t = t.substr(a, b - a);
  t.erase(std::remove(t.begin(), t.end(), '\r'), t.end());
  return t;
}
}  // namespace

int XGDMatrixCreateFromURI(const char* config, DMatrixHandle* out) {
  API_BEGIN();
  JPtr cfg = parse_json(config);
  const std::string uri = cfg->at("uri").s;
  const size_t qm = uri.find('?');
  const std::string path = uri.substr(0, qm);
  std::map<std::string, std::string> q;
  if (qm != std::string::npos) {
    std::stringstream ss(uri.substr(qm + 1)); std::string kv;
    while (std::getline(ss, kv, '&')) { size_t eq = kv.find('='); if (eq != std::string::npos) q[kv.substr(0, eq)] = kv.substr(eq + 1); }
  }
  std::string fmt = q.count("format") ? q["format"] : (path.size() > 4 && path.substr(path.size() - 4) == ".csv" ? "csv" : "libsvm");
  std::vector<std::string> files = list_files(path);
  auto box = new DMatrixBox(); std::unique_ptr<DMatrixBox> guard(box);
  if (fmt == "csv") {
    const std::string d = q.count("delimiter") ? q["delimiter"] : ",";
    if (d.size() != 1) throw Error("CSV delimiter must be a single character");
    std::string text;
    for (auto& f : files) { std::string t = read_stripped(f); if (t.empty()) continue; if (!text.empty()) text.push_back('\n'); text += t; }
    if (text.empty()) throw Error("CSV input is empty");
    int st = 0;
    box->dm = DMatrix::from_csv_text_labeled(text.data(), (int64_t)text.size(), d[0], q.count("label_column") ? std::stoi(q["label_column"]) : -1,
                                             q.count("weight_column") ? std::stoi(q["weight_column"]) : -1, &st);
    if (st == 1) throw Error("CSV rows have different numbers of columns");
    if (st != 0) throw Error("CSV contains a field the device parser cannot decide exactly (blank line, > 19 digits or malformed number)");
  } else if (fmt == "libsvm") {
    std::vector<size_t> indptr{0}; std::vector<unsigned> indices; std::vector<float> vals, labels;
    for (auto& f : files) {
      std::ifstream in(f); std::string line;
      while (std::getline(in, line)) {
        size_t hash = line.find('#'); if (hash != std::string::npos) line.resize(hash);
        std::stringstream ls(line); std::string tok;
        if (!(ls >> tok)) continue;
        labels.push_back(std::stof(tok.substr(0, tok.find(':'))));
        while (ls >> tok) {
          size_t c = tok.find(':');
          if (c == std::string::npos) throw Error("Invalid libsvm token " + tok + " in " + f);
          if (tok.compare(0, 4, "qid:") == 0) continue;
          indices.push_back((unsigned)std::stoul(tok.substr(0, c))); vals.push_back(std::stof(tok.substr(c + 1)));
        }
        indptr.push_back(indices.size());
      }
    }
    if (labels.empty()) throw Error("libsvm input is empty");
    box->dm = DMatrix::from_csr(indptr.data(), indices.data(), vals.data(), indptr.size(), indices.size(), 0);
    box->dm->set_float_info("label", labels.data(), labels.size());
  } else throw Error("Unknown data format in URI: " + fmt);
  *out = guard.release();
  API_END();
}

int XGDMatrixFree(DMatrixHandle handle) { API_BEGIN(); delete static_cast<DMatrixBox*>(handle); API_END(); }
int XGDMatrixNumRow(DMatrixHandle handle, bst_ulong* out) { API_BEGIN(); *out = (bst_ulong)DM(handle)->n; API_END(); }
int XGDMatrixNumCol(DMatrixHandle handle, bst_ulong* out) { API_BEGIN(); *out = (bst_ulong)DM(handle)->F; API_END(); }
int XGDMatrixSetFloatInfo(DMatrixHandle handle, const char* field, const float* array, bst_ulong len) {
  API_BEGIN(); DM(handle)->set_float_info(field, array, (size_t)len); API_END();
}
int XGDMatrixGetFloatInfo(DMatrixHandle handle, const char* field, bst_ulong* out_len, const float** out_dptr) {
  API_BEGIN(); const std::vector<float>& v = DM(handle)->get_float_info(field); *out_len = v.size(); *out_dptr = v.data(); API_END();
}
int XGDMatrixSliceDMatrix(DMatrixHandle handle, const int* idxset, bst_ulong len, DMatrixHandle* out) {
  API_BEGIN();
  auto box = new DMatrixBox(); std::unique_ptr<DMatrixBox> guard(box);
  box->dm = DM(handle)->slice(idxset, (int64_t)len);
  *out = guard.release();
  API_END();
}
int XGDMatrixSetStrFeatureInfo(DMatrixHandle handle, const char* field, const char** features, bst_ulong size) {
  API_BEGIN();
  DMatrix* dm = DM(handle);
  std::vector<std::string>& dst = std::string(field) == "feature_name" ? dm->feature_names : dm->feature_types;
  if (std::string(field) != "feature_name" && std::string(field) != "feature_type") throw Error(std::string("Unknown feature info name: ") + field);
  if (size != 0 && (int64_t)size != dm->F) throw Error("Length of " + std::string(field) + " must be equal to the number of columns");
  dst.clear(); for (bst_ulong i = 0; i < size; ++i) dst.emplace_back(features[i]);
  API_END();
}
int XGDMatrixGetStrFeatureInfo(DMatrixHandle handle, const char* field, bst_ulong* size, const char*** out_features) {
  API_BEGIN();
  DMatrixBox* box = static_cast<DMatrixBox*>(handle); DMatrix* dm = DM(handle);
  const std::vector<std::string>& src = std::string(field) == "feature_name" ? dm->feature_names : dm->feature_types;
  box->strs = src; box->str_ptrs.clear(); for (auto& s : box->strs) box->str_ptrs.push_back(s.c_str());
  *size = box->str_ptrs.size(); *out_features = box->str_ptrs.data();
  API_END();
}

// ------------------------------------------------------------------------------------------- Booster
int XGBoosterCreate(const DMatrixHandle dmats[], bst_ulong len, BoosterHandle* out) {
  API_BEGIN();
  (void)dmats; (void)len;      // prediction caches are created lazily per DMatrix
  auto box = new BoosterBox(); box->bst = std::make_unique<Booster>(); *out = box;
  API_END();
}
int XGBoosterFree(BoosterHandle handle) { API_BEGIN(); delete static_cast<BoosterBox*>(handle); API_END(); }
int XGBoosterSetParam(BoosterHandle handle, const char* name, const char* value) { API_BEGIN(); BST(handle)->set_param(name, value ? value : ""); API_END(); }
int XGBoosterUpdateOneIter(BoosterHandle handle, int iter, DMatrixHandle dtrain) { API_BEGIN(); BST(handle)->update_one_iter(iter, DM(dtrain)); API_END(); }
int XGBoosterBoostOneIter(BoosterHandle handle, DMatrixHandle dtrain, float* grad, float* hess, bst_ulong len) {
  API_BEGIN(); BST(handle)->boost_one_iter(DM(dtrain), grad, hess, (size_t)len); API_END();
}
int XGBoosterEvalOneIter(BoosterHandle handle, int iter, DMatrixHandle dmats[], const char* evnames[], bst_ulong len, const char** out_result) {
  API_BEGIN();
  BoosterBox* box = static_cast<BoosterBox*>(handle);
  std::vector<DMatrix*> dms; std::vector<std::string> names;
  for (bst_ulong i = 0; i < len; ++i) { dms.push_back(DM(dmats[i])); names.emplace_back(evnames[i]); }
  box->ret_str = BST(handle)->eval_one_iter(iter, dms, names);
  *out_result = box->ret_str.c_str();
  API_END();
}
int XGBoosterPredictFromDMatrix(BoosterHandle handle, DMatrixHandle dmat, const char* config, bst_ulong const** out_shape,
                                bst_ulong* out_dim, float const** out_result) {
  API_BEGIN();
  BoosterBox* box = static_cast<BoosterBox*>(handle);
  JPtr cfg = parse_json(config ? config : "{}");
  auto geti = [&](const char* k, int64_t def) { auto v = cfg->get(k); return v ? v->as_int() : def; };
  auto getb = [&](const char* k, bool def) { auto v = cfg->get(k); if (!v) return def; return v->type == JValue::kBool ? v->b : v->as_int() != 0; };
  BST(handle)->predict(DM(dmat), (int)geti("type", 0), getb("training", false), (int)geti("iteration_begin", 0), (int)geti("iteration_end", 0),
                       getb("strict_shape", false), &box->ret_vec, &box->ret_shape);
  *out_shape = box->ret_shape.data(); *out_dim = box->ret_shape.size(); *out_result = box->ret_vec.data();
  API_END();
}
static bool ends_with(const std::string& s, const char* suf) { size_t n = strlen(suf); return s.size() >= n && s.compare(s.size() - n, n, suf) == 0; }
int XGBoosterSaveModel(BoosterHandle handle, const char* fname) {
  API_BEGIN();
  std::string f(fname);
  std::string buf = BST(handle)->save_model_buffer(ends_with(f, ".json") ? "json" : "ubj");
  std::ofstream os(f, std::ios::binary);
  if (!os) throw Error("Opening " + f + " failed: cannot write the model file");
  os.write(buf.data(), (std::streamsize)buf.size());
  if (!os) throw Error("Writing " + f + " failed");
  API_END();
}
int XGBoosterLoadModel(BoosterHandle handle, const char* fname) {
  API_BEGIN();
  std::ifstream is(fname, std::ios::binary);
  if (!is) throw Error(std::string("Opening ") + fname + " failed: No such file or directory");
  std::string buf((std::istreambuf_iterator<char>(is)), std::istreambuf_iterator<char>());
  BST(handle)->load_model_buffer(buf.data(), buf.size());
  API_END();
}
int XGBoosterSaveModelToBuffer(BoosterHandle handle, const char* config, bst_ulong* out_len, const char** out_dptr) {
  API_BEGIN();
  BoosterBox* box = static_cast<BoosterBox*>(handle);
  JPtr cfg = parse_json(config ? config : "{}");
  std::string fmt = cfg->has("format") ? cfg->at("format").s : "ubj";
  if (fmt != "json" && fmt != "ubj") throw Error("Unknown model format: " + fmt + " (expected json or ubj)");
  box->ret_str = BST(handle)->save_model_buffer(fmt);
  *out_len = box->ret_str.size(); *out_dptr = box->ret_str.data();
  API_END();
}
int XGBoosterLoadModelFromBuffer(BoosterHandle handle, const void* buf, bst_ulong len) { API_BEGIN(); BST(handle)->load_model_buffer((const char*)buf, (size_t)len); API_END(); }
int XGBoosterSerializeToBuffer(BoosterHandle handle, bst_ulong* out_len, const char** out_dptr) {
  API_BEGIN(); BoosterBox* box = static_cast<BoosterBox*>(handle); box->ret_str = BST(handle)->serialize(); *out_len = box->ret_str.size(); *out_dptr = box->ret_str.data(); API_END();
}
int XGBoosterUnserializeFromBuffer(BoosterHandle handle, const void* buf, bst_ulong len) { API_BEGIN(); BST(handle)->unserialize((const char*)buf, (size_t)len); API_END(); }
int XGBoosterSaveJsonConfig(BoosterHandle handle, bst_ulong* out_len, const char** out_str) {
  API_BEGIN(); BoosterBox* box = static_cast<BoosterBox*>(handle); box->ret_str = BST(handle)->save_config(); *out_len = box->ret_str.size(); *out_str = box->ret_str.c_str(); API_END();
}
int XGBoosterLoadJsonConfig(BoosterHandle handle, const char* config) { API_BEGIN(); BST(handle)->load_config(config); API_END(); }
int XGBoosterGetNumFeature(BoosterHandle handle, bst_ulong* out) { API_BEGIN(); *out = (bst_ulong)BST(handle)->num_features(); API_END(); }
int XGBoosterBoostedRounds(BoosterHandle handle, int* out) { API_BEGIN(); *out = BST(handle)->boosted_rounds(); API_END(); }
int XGBoosterSlice(BoosterHandle handle, int begin_layer, int end_layer, int step, BoosterHandle* out) {
  API_BEGIN();
  auto box = new BoosterBox(); std::unique_ptr<BoosterBox> guard(box);
  box->bst = BST(handle)->slice(begin_layer, end_layer, step);
  *out = guard.release();
  API_END();
}
int XGBoosterGetAttr(BoosterHandle handle, const char* key, const char** out, int* success) {
  API_BEGIN();
  BoosterBox* box = static_cast<BoosterBox*>(handle);
  auto it = BST(handle)->attrs.find(key);
  if (it == BST(handle)->attrs.end()) { *out = nullptr; *success = 0; }
  else { box->ret_str = it->second; *out = box->ret_str.c_str(); *success = 1; }
  API_END();
}
int XGBoosterSetAttr(BoosterHandle handle, const char* key, const char* value) {
  API_BEGIN(); if (value) BST(handle)->attrs[key] = value; else BST(handle)->attrs.erase(key); API_END();
}
int XGBoosterGetAttrNames(BoosterHandle handle, bst_ulong* out_len, const char*** out) {
  API_BEGIN();
  BoosterBox* box = static_cast<BoosterBox*>(handle);
  box->strs.clear(); for (auto& kv : BST(handle)->attrs) box->strs.push_back(kv.first);
  box->str_ptrs.clear(); for (auto& s : box->strs) box->str_ptrs.push_back(s.c_str());
  *out_len = box->str_ptrs.size(); *out = box->str_ptrs.data();
  API_END();
}
int XGBoosterSetStrFeatureInfo(BoosterHandle handle, const char* field, const char** features, bst_ulong size) {
  API_BEGIN();
  Booster* b = BST(handle);
  if (std::string(field) != "feature_name" && std::string(field) != "feature_type") throw Error(std::string("Unknown feature info name: ") + field);
  std::vector<std::string>& dst = std::string(field) == "feature_name" ? b->feature_names : b->feature_types;
  dst.clear(); for (bst_ulong i = 0; i < size; ++i) dst.emplace_back(features[i]);
  API_END();
}
int XGBoosterGetStrFeatureInfo(BoosterHandle handle, const char* field, bst_ulong* len, const char*** out_features) {
  API_BEGIN();
  BoosterBox* box = static_cast<BoosterBox*>(handle); Booster* b = BST(handle);
  box->strs = std::string(field) == "feature_name" ? b->feature_names : b->feature_types;
  box->str_ptrs.clear(); for (auto& s : box->strs) box->str_ptrs.push_back(s.c_str());
  *len = box->str_ptrs.size(); *out_features = box->str_ptrs.data();
  API_END();
}

// ------------------------------------------------------------------------------------------- collective
int XGCommunicatorInit(const char* config) {
  API_BEGIN();
  JPtr cfg = parse_json(config ? config : "{}");
  int rank = cfg->has("rank") ? (int)cfg->at("rank").as_int() : 0;
  int world = cfg->has("world_size") ? (int)cfg->at("world_size").as_int() : 1;
  std::string id = cfg->has("nccl_unique_id") ? hex_decode(cfg->at("nccl_unique_id").s) : std::string();
  engine_stream();            // binds this process to its GPU (LOCAL_RANK) before NCCL initialises
  Comm::get().init(id, rank, world);
  API_END();
}
// host buffer broadcast (distributed.py:119-136 RabitHelper.synchronize reaches it through xgboost.collective.broadcast)
int XGCommunicatorBroadcast(void* send_receive_buffer, size_t size, int root) {
  API_BEGIN();
  Comm& comm = Comm::get();
  if (comm.distributed() && size > 0) {
    cudaStream_t s = engine_stream();
    DevBuf<unsigned char> d; d.alloc(size);
    if (comm.rank() == root) CUDA_OK(cudaMemcpyAsync(d.p, send_receive_buffer, size, cudaMemcpyHostToDevice, s));
    comm.broadcast_bytes(d.p, size, root, s);
    CUDA_OK(cudaMemcpyAsync(send_receive_buffer, d.p, size, cudaMemcpyDeviceToHost, s));
    comm.sync_stream(s);
  }
  API_END();
}
int XGCommunicatorFinalize(void) { API_BEGIN(); Comm::get().finalize(); API_END(); }
int XGCommunicatorGetRank(void) { return Comm::get().rank(); }
int XGCommunicatorGetWorldSize(void) { return Comm::get().world(); }
int XGB200CommPeerReduceActive(void) { return peer_reduce_active() ? 1 : 0; }
int XGCommunicatorGetUniqueId(const char** out_hex) {
  API_BEGIN(); engine_stream(); g_ret_str = hex_encode(Comm::create_unique_id()); *out_hex = g_ret_str.c_str(); API_END();
}

// ------------------------------------------------------------------------------------------- introspection
int XGB200DMatrixGetCuts(DMatrixHandle handle, int max_bin, bst_ulong* n_ptrs, const int** ptrs, bst_ulong* n_vals, const float** vals,
                         const float** mins, int* has_missing) {
  API_BEGIN();
  DMatrix* dm = DM(handle); dm->ensure_binned(max_bin);
  *n_ptrs = dm->cuts.ptrs.size(); *ptrs = dm->cuts.ptrs.data(); *n_vals = dm->cuts.vals.size(); *vals = dm->cuts.vals.data(); *mins = dm->cuts.mins.data();
  if (has_missing) *has_missing = dm->has_missing ? 1 : 0;
  API_END();
}
int XGB200DMatrixSetCuts(DMatrixHandle handle, const int* ptrs, bst_ulong n_ptrs, const float* vals, const float* mins) {
  API_BEGIN();
  HostCuts c; c.ptrs.assign(ptrs, ptrs + n_ptrs); c.vals.assign(vals, vals + (n_ptrs ? ptrs[n_ptrs - 1] : 0)); c.mins.assign(mins, mins + (n_ptrs ? n_ptrs - 1 : 0));
  DM(handle)->set_cuts(c);
  API_END();
}
int XGB200DMatrixGetBins(DMatrixHandle handle, int max_bin, uint8_t* out_row_major) {
  API_BEGIN();
  DMatrix* dm = DM(handle); dm->ensure_binned(max_bin);
  const size_t W = (size_t)dm->ngroups * kSlots;
  std::vector<uint8_t> h((size_t)dm->n * W), t((size_t)dm->n * dm->tw);
  if (!h.empty()) { CUDA_OK(cudaMemcpy(h.data(), dm->bins.p, h.size(), cudaMemcpyDeviceToHost)); }
  if (!t.empty()) { CUDA_OK(cudaMemcpy(t.data(), dm->bins_tail.p, t.size(), cudaMemcpyDeviceToHost)); }
  for (int64_t r = 0; r < dm->n; ++r) for (int f = 0; f < dm->F; ++f)
    out_row_major[r * dm->F + f] = (size_t)f < W ? h[(size_t)r * W + f] : t[(size_t)r * dm->tw + (f - W)];
  API_END();
}
int XGB200BoosterModelShape(BoosterHandle handle, bst_ulong* num_trees, bst_ulong* num_nodes, float* base_score, int* num_class) {
  API_BEGIN();
  Booster* b = BST(handle); const auto& trees = b->trees();
  size_t nn = 0; for (auto& t : trees) nn += t.left.size();
  if (num_trees) *num_trees = trees.size(); if (num_nodes) *num_nodes = nn; if (base_score) *base_score = b->base_score();
  if (num_class) *num_class = b->param().num_class;
  API_END();
}
int XGB200BoosterExportModel(BoosterHandle handle, int64_t* tree_offset, int32_t* tree_info, int32_t* left, int32_t* right, int32_t* parent,
                             int32_t* split_index, int32_t* split_bin, uint8_t* default_left, float* split_cond, float* base_weight,
                             float* loss_chg, float* sum_hess) {
  API_BEGIN();
  Booster* b = BST(handle); const auto& trees = b->trees(); const auto& info = b->tree_info();
  size_t off = 0;
  for (size_t t = 0; t < trees.size(); ++t) {
    const HostTree& h = trees[t]; const size_t nn = h.left.size();
    if (tree_offset) tree_offset[t] = (int64_t)off;
    if (tree_info) tree_info[t] = info[t];
#define CP(dst, src) if (dst) memcpy(dst + off, src.data(), sizeof(src[0]) * nn)
    CP(left, h.left); CP(right, h.right); CP(parent, h.parent); CP(split_index, h.split_index); CP(split_bin, h.split_bin);
    CP(default_left, h.default_left); CP(split_cond, h.split_cond); CP(base_weight, h.base_weight); CP(loss_chg, h.loss_chg); CP(sum_hess, h.sum_hess);
#undef CP
    off += nn;
  }
  if (tree_offset) tree_offset[trees.size()] = (int64_t)off;
  API_END();
}
static void hist_to_feature_major(const DMatrix* dm, const std::vector<long long>& h, int64_t* out_hist) {
  // pool layout [group][bin][slot]{g,h} + tail [bin][tw]{g,h} -> [F][256]{g,h}
  const size_t W = (size_t)dm->ngroups * kSlots, tail0 = (size_t)dm->ngroups * kGroupEntries;
  for (int f = 0; f < dm->F; ++f) {
    for (int b = 0; b < kBins; ++b) {
      const size_t e = (size_t)f < W ? ((size_t)(f / kSlots) * kBins + b) * kSlots + f % kSlots : tail0 + (size_t)b * dm->tw + (f - W);
      const size_t dst = ((size_t)f * kBins + b) * 2;
      out_hist[dst] = h[e * 2]; out_hist[dst + 1] = h[e * 2 + 1];
    }
  }
}
int XGB200DMatrixGetRaw(DMatrixHandle handle, float* out_row_major) {
  API_BEGIN();
  DMatrix* dm = DM(handle);
  if (dm->n * dm->F > 0) CUDA_OK(cudaMemcpy(out_row_major, dm->X.p, sizeof(float) * (size_t)dm->n * dm->F, cudaMemcpyDeviceToHost));
  API_END();
}
int XGB200DMatrixCreateFromCSVEx(const char* text, bst_ulong len, char delimiter, int label_column, int weight_column, int* status, DMatrixHandle* out) {
  API_BEGIN();
  int st = 0;
  auto dm = DMatrix::from_csv_text_labeled(text, (int64_t)len, delimiter, label_column, weight_column, &st);
  if (status) *status = st;
  *out = nullptr;
  if (st == 0) { auto box = new DMatrixBox(); box->dm = std::move(dm); *out = box; }
  API_END();
}
int XGB200DMatrixCreateFromCSV(const char* text, bst_ulong len, char delimiter, int* status, DMatrixHandle* out) {
  API_BEGIN();
  int st = 0;
  auto dm = DMatrix::from_csv_text(text, (int64_t)len, delimiter, &st);
  if (status) *status = st;
  *out = nullptr;
  if (st == 0) { auto box = new DMatrixBox(); box->dm = std::move(dm); *out = box; }
  API_END();
}
int XGB200DMatrixCreateFromLibsvmText(const char* text, bst_ulong len, int whitespace_mode, float absent, int* status, DMatrixHandle* out) {
  API_BEGIN();
  int st = 0;
  auto dm = DMatrix::from_libsvm_text(text, (int64_t)len, whitespace_mode, absent, &st);
  if (status) *status = st;
  *out = nullptr;
  if (st == 0) { auto box = new DMatrixBox(); box->dm = std::move(dm); *out = box; }
  API_END();
}
int XGB200BuildRootHistogram(BoosterHandle handle, DMatrixHandle dmat, const float* gpair, int repeats, int64_t* out_hist, float* scales, float* out_ms) {
  API_BEGIN();
  DMatrix* dm = DM(dmat);
  std::vector<long long> h; float sc[4];
  BST(handle)->debug_build_root_hist(dm, gpair, &h, sc, repeats, out_ms);
  hist_to_feature_major(dm, h, out_hist);
  if (scales) memcpy(scales, sc, sizeof sc);
  API_END();
}
int XGB200BuildHistogramEx(BoosterHandle handle, DMatrixHandle dmat, const float* gpair, int repeats, int mode, const unsigned* row_ids, bst_ulong n_ids,
                           int64_t* out_hist, float* scales, float* out_ms, const char** out_kernel) {
  API_BEGIN();
  DMatrix* dm = DM(dmat);
  std::vector<long long> h; float sc[4];
  BST(handle)->debug_build_root_hist(dm, gpair, &h, sc, repeats, out_ms, mode, row_ids, (int64_t)n_ids);
  hist_to_feature_major(dm, h, out_hist);
  if (scales) memcpy(scales, sc, sizeof sc);
  if (out_kernel) *out_kernel = hist_last_kernel();
  API_END();
}
int XGB200BoosterPredictKernelMs(BoosterHandle handle, DMatrixHandle dmat, int repeats, float* out_ms) {
  API_BEGIN();
  *out_ms = BST(handle)->debug_predict_kernel_ms(DM(dmat), repeats);
  API_END();
}
int XGB200PredictPlan(int data_features, int model_features, const int64_t* node_counts, int tree_begin, int tree_end,
                      int children_adjacent, const char** out_json) {
  API_BEGIN();
  B200_CHECK(out_json != nullptr && tree_begin >= 0 && tree_end >= tree_begin && (node_counts != nullptr || tree_end == tree_begin),
             "XGB200PredictPlan: bad argument");
  g_ret_str = predict_plan_json(plan_predict(data_features, model_features, node_counts, tree_begin, tree_end, children_adjacent != 0));
  *out_json = g_ret_str.c_str();
  API_END();
}
int XGB200BoosterPredictPlan(BoosterHandle handle, DMatrixHandle dmat, int iteration_begin, int iteration_end, const char** out_json) {
  API_BEGIN();
  BoosterBox* box = static_cast<BoosterBox*>(handle);
  box->ret_str = BST(handle)->predict_plan(DM(dmat), iteration_begin, iteration_end); *out_json = box->ret_str.c_str();
  API_END();
}
int XGB200BoosterGetCachedMargin(BoosterHandle handle, DMatrixHandle dmat, float* out) {
  API_BEGIN();
  std::vector<float> v;
  BST(handle)->cached_margin(DM(dmat), &v);
  memcpy(out, v.data(), sizeof(float) * v.size());
  API_END();
}
static cudaEvent_t g_t0 = nullptr, g_t1 = nullptr;
int XGB200TimerStart(void) {
  API_BEGIN();
  if (!g_t0) { CUDA_OK(cudaEventCreate(&g_t0)); CUDA_OK(cudaEventCreate(&g_t1)); }
  CUDA_OK(cudaEventRecord(g_t0, engine_stream()));
  API_END();
}
int XGB200TimerStop(float* out_ms) {
  API_BEGIN();
  if (!g_t0) throw Error("XGB200TimerStop without XGB200TimerStart");
  CUDA_OK(cudaEventRecord(g_t1, engine_stream())); CUDA_OK(cudaEventSynchronize(g_t1));
  CUDA_OK(cudaEventElapsedTime(out_ms, g_t0, g_t1));
  API_END();
}
int XGB200BoosterSetProfile(BoosterHandle handle, int enable) { API_BEGIN(); BST(handle)->set_profile(enable != 0); API_END(); }
int XGB200BoosterGetProfile(BoosterHandle handle, const char** out_json) {
  API_BEGIN(); BoosterBox* box = static_cast<BoosterBox*>(handle); box->ret_str = BST(handle)->get_profile(); *out_json = box->ret_str.c_str(); API_END();
}
int XGB200LaunchCount(long long* out) { API_BEGIN(); *out = g_kernel_launches; API_END(); }
int XGB200Synchronize(void) { API_BEGIN(); CUDA_OK(cudaStreamSynchronize(engine_stream())); API_END(); }
int XGB200DMatrixCreateFromColumns(const void* const* cols, const int* col_types, int ncols, bst_ulong nrow, int label_column, int weight_column, DMatrixHandle* out) {
  API_BEGIN();
  B200_CHECK(out != nullptr && (ncols == 0 || (cols != nullptr && col_types != nullptr)), "XGB200DMatrixCreateFromColumns: NULL argument");
  auto box = new DMatrixBox(); std::unique_ptr<DMatrixBox> guard(box);
  box->dm = DMatrix::from_columns(cols, col_types, ncols, (int64_t)nrow, label_column, weight_column);
  *out = guard.release();
  API_END();
}
int XGB200LegacyModelToUBJ(const void* buf, bst_ulong len, bst_ulong* out_len, const char** out) {
  API_BEGIN();
  B200_CHECK(buf != nullptr && out_len != nullptr && out != nullptr, "XGB200LegacyModelToUBJ: NULL argument");
  const char* p = (const char*)buf; size_t n = (size_t)len;
  auto sect = legacy_serialized_model_section(p, n);
  if (sect.first != nullptr) { p = sect.first; n = sect.second; }
  B200_CHECK(looks_like_legacy_binary(p, n), "XGB200LegacyModelToUBJ: the buffer is not a legacy binary model");
  g_ret_str.clear(); ubj_write(*legacy_binary_to_doc(p, n), &g_ret_str);
  *out_len = g_ret_str.size(); *out = g_ret_str.data();
  API_END();
}

}  // extern "C"
