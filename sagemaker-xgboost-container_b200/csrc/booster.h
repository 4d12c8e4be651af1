// booster.h -- host-side objects behind the C-ABI handles (DMatrixHandle / BoosterHandle).
#pragma once
#include <map>
#include <memory>
#include <string>
#include <vector>
#include "engine.h"
#include "json.h"
#include "misc.h"
#include "tree.h"

namespace b200 {

cudaStream_t engine_stream();
int engine_num_sms();

// ---------------------------------------------------------------------------------------------
// DMatrix: features resident on the device (raw float row-major + lazily the binned feature blocks)
// ---------------------------------------------------------------------------------------------
class DMatrix {
 public:
  int64_t n = 0; int F = 0;
  bool has_missing = false;
  DevBuf<float> X;                                    // n x F, NaN = missing
  std::vector<float> labels, weights, base_margin;    // host copies (returned by GetFloatInfo)
  DevBuf<float> d_labels, d_weights, d_base_margin;
  std::vector<std::string> feature_names, feature_types;
  // binned representation (built on first use as a training matrix)
  bool binned = false; int binned_max_bin = 0;
  HostCuts cuts; DevBuf<int> d_cut_ptrs; DevBuf<float> d_cut_vals, d_min_vals;
  DevBuf<uint8_t> bins, bins_tail, bins_col, bins_gather; int ngroups = 0, tw = 0, ntail = 0, gather_stride = 0;   // engine.h BinnedMatrix layout
  uint64_t binned_version = 0;                        // bumped by every (re)binning: invalidates captured graphs / cached planes
  uint64_t uid;                                       // identity for prediction caches

  DMatrix();
  static std::unique_ptr<DMatrix> from_dense(const float* data, int64_t nrow, int ncol, float missing);
  static std::unique_ptr<DMatrix> from_device(const float* dptr, int64_t nrow, int ncol, float missing);
  // serving path: CSV text parsed on the device (csv.cu); status 0 ok, 1 ragged rows, 2 needs the host parser
  static std::unique_ptr<DMatrix> from_csv_text(const char* text, int64_t len, char delim, int* status);
  // serving path: libsvm request body parsed on the device (csv.cu); whitespace_mode 0 = tokens split on ' ' (serve_utils),
  // 1 = on any whitespace (encoder); absent = value of entries a line does not list (NaN = missing, or 0); status 0 ok,
  // 2 needs the host route, 3 body without a single entry
  static std::unique_ptr<DMatrix> from_libsvm_text(const char* text, int64_t len, int whitespace_mode, float absent, int* status);
  // training channel: columns label_col / weight_col (-1 = none) become the label / weight info, the rest the features
  static std::unique_ptr<DMatrix> from_csv_text_labeled(const char* text, int64_t len, char delim, int label_col, int weight_col, int* status);
  // columnar input (ingest.cu): `ncols` host column buffers of `nrow` items each, type codes as in include/b200xgb.h; columns
  // label_col / weight_col (-1 = none) become the label / weight info, the others the features in order
  static std::unique_ptr<DMatrix> from_columns(const void* const* cols, const int* types, int ncols, int64_t nrow, int label_col, int weight_col);
  static std::unique_ptr<DMatrix> from_csr(const size_t* indptr, const unsigned* indices, const float* data, size_t nindptr, size_t nelem, size_t ncol);
  std::unique_ptr<DMatrix> slice(const int* idx, int64_t len) const;
  void set_float_info(const std::string& field, const float* v, size_t len);
  const std::vector<float>& get_float_info(const std::string& field) const;
  void ensure_binned(int max_bin);
  void set_cuts(const HostCuts& c);                   // external cuts (shared with the oracle in tests)
  BinnedMatrix binned_view() const { BinnedMatrix b; b.bins = bins.p; b.bins_tail = tw ? bins_tail.p : nullptr; b.bins_col = bins_col.p; b.n = n; b.F = F;
    b.bins_gather = bins_gather.p ? bins_gather.p : bins.p; b.gather_stride = gather_stride;
    b.ngroups = ngroups; b.tw = tw; b.ntail = ntail; b.has_missing = has_missing; return b; }
  void finish_upload(float missing);
 private:
  void bin_with_cuts();
};

// ---------------------------------------------------------------------------------------------
// model
// ---------------------------------------------------------------------------------------------
struct HostTree {
  std::vector<int> left, right, parent, split_index, split_bin;
  std::vector<uint8_t> default_left;
  std::vector<float> split_cond, base_weight, loss_chg, sum_hess;
  int num_nodes() const { return (int)left.size(); }
};

struct PendingTree {            // a tree still on its way from the device (async copy into pinned memory)
  void* staging = nullptr; size_t cap_nodes = 0; cudaEvent_t ready = nullptr;
};

struct PredCache { DevBuf<float> margin; int trees_applied = 0; int64_t n = 0; uint64_t model_version = 0; };

// legacy_io.cc: the pre-JSON binary model format -> the 3.x model document
bool looks_like_legacy_binary(const char* buf, size_t len);
JPtr legacy_binary_to_doc(const char* buf, size_t len);
std::pair<const char*, size_t> legacy_serialized_model_section(const char* buf, size_t len);

class Booster {
 public:
  Booster();
  ~Booster();
  // configuration
  void set_param(const std::string& k, const std::string& v);
  std::string save_config();
  void load_config(const std::string& json);
  // training
  void update_one_iter(int iter, DMatrix* dtrain);
  void boost_one_iter(DMatrix* dtrain, const float* grad, const float* hess, size_t len);
  std::string eval_one_iter(int iter, const std::vector<DMatrix*>& dms, const std::vector<std::string>& names);
  // inference; returns host buffer + shape
  void predict(DMatrix* dm, int type, bool training, int iter_begin, int iter_end, bool strict_shape,
               std::vector<float>* out, std::vector<uint64_t>* shape);
  void predict_contribs(DMatrix* dm, int tree_begin, int tree_end, std::vector<float>* out, std::vector<uint64_t>* shape);
  // model IO
  std::string save_model_buffer(const std::string& format);      // "ubj" | "json"
  void load_model_buffer(const char* buf, size_t len);
  std::string serialize();                                         // model + config (pickle)
  void unserialize(const char* buf, size_t len);
  std::unique_ptr<Booster> slice(int begin, int end, int step);
  int boosted_rounds();
  int num_features() const { return num_feature_; }
  std::map<std::string, std::string> attrs;
  std::vector<std::string> feature_names, feature_types;

  // introspection used by tests/bench (build-specific C-ABI entry points)
  void sync_model();                              // materialise pending trees on the host
  void cached_margin(DMatrix* dm, std::vector<float>* out);   // the trainer's prediction cache for dm
  float debug_predict_kernel_ms(DMatrix* dm, int repeats);
  std::string predict_plan(DMatrix* dm, int iter_begin, int iter_end);   // JSON of the plan predict() would run on dm
  const std::vector<HostTree>& trees() { sync_model(); return trees_; }
  const std::vector<int>& tree_info() const { return tree_info_; }
  float base_score() const { return base_score_; }
  int num_class() const { return param_.num_class; }
  const TrainParam& param() { configure(); return param_; }
  void set_profile(bool on);
  std::string get_profile();                      // JSON, see include/b200xgb.h
  // histogram of one node for kernel-level parity tests / the roofline bench
  // mode: 0 = production choice (TMA root kernel), 1 = gather kernel, 2 = G-only TMA root kernel (H plane stays zero).
  // row_ids (optional, n_ids entries): histogram of that row subset, gpair given by POSITION -> exercises the gathered path.
  void debug_build_root_hist(DMatrix* dm, const float* gpair_host, std::vector<long long>* hist_out, float* scales_out,
                             int repeats, float* ms_out, int mode = 0, const unsigned* row_ids = nullptr, int64_t n_ids = 0);

 private:
  friend struct GrowerImpl;
  std::map<std::string, std::string> raw_params_;
  std::vector<std::string> eval_metrics_;
  std::vector<int> monotone_;              // parsed monotone_constraints (empty = none)
  std::vector<std::vector<int>> interaction_;   // parsed interaction_constraints (empty = none)
  bool configured_ = false;
  TrainParam param_;
  std::string objective_name_ = "reg:squarederror";
  bool base_score_set_ = false; float base_score_ = 0.5f; bool base_score_estimated_ = false;
  int num_feature_ = 0;
  std::vector<HostTree> trees_; std::vector<int> tree_info_;
  std::vector<PendingTree> pending_;            // parallel to trees_ (nullptr staging once materialised)
  std::vector<char> on_device_;                 // parallel to trees_: nodes already in d_nodes
  uint64_t model_version_ = 0;
  // device model for prediction
  DevBuf<DevNode> d_nodes; std::vector<int64_t> h_tree_offset; DevBuf<int64_t> d_tree_offset; DevBuf<int> d_tree_info;
  size_t d_nodes_used = 0; int d_trees_uploaded = 0;
  std::map<uint64_t, PredCache> caches_;
  struct GrowerImpl* grower_ = nullptr;
  bool labels_checked_ = false;
  DevBuf<float> pred_margin_, pred_cls_; DevBuf<int> pred_leaf_;      // predict() scratch, grown on demand
  bool children_adjacent_ = true;               // every tree on the device has right child == left child + 1
  bool profile_ = false;
  struct ProfEvent { cudaEvent_t a, b; int level; };
  std::vector<ProfEvent> prof_events_;
  DevBuf<unsigned long long> prof_rows_;       // [0] rows through root launches, [1] rows through deeper launches
  long long prof_launches_ = 0;

  void configure();
  float base_margin() const;
  void estimate_base_score(DMatrix* dtrain);
  void upload_model();
  PredictArgs predict_args(const DMatrix* dm, int tree_begin, int tree_end) const;   // margin / leaf left null
  PredCache& cache_for(DMatrix* dm);
  void bring_cache_up_to_date(DMatrix* dm, PredCache& c);
  void append_device_tree(int class_id, size_t device_offset, int max_nodes, PendingTree pt);
  void grow_one_tree(DMatrix* dtrain, PredCache& cache, int k, int tree_index);
  // root_mode: 0 = accumulate G and H, 1 = G and H + snapshot of the root H plane, 2 = G only on top of the cached H plane
  void enqueue_tree(DMatrix* dtrain, float* margin, int k, const unsigned char* mask, DevNode* packed_out, int root_mode);
  void prof_begin(int level);
  void prof_end();
  JPtr model_to_json();
  void model_from_json(const JValue& doc);
  JPtr config_to_json();
  void config_from_json(const JValue& doc);
  void reset_model();
};

std::string colsample_mask(unsigned seed, int tree_index, int F, float frac);   // bytes, 1 = feature usable
std::string subset_mask(const std::string& parent, float frac, unsigned seed, uint64_t stream);

}  // namespace b200
