// misc.h -- argument blocks and launchers for misc.cu / quantile.cu
#pragma once
#include "engine.h"

namespace b200 {

struct GradArgs {
  const float* margin;      // n x K row-major, nullptr = all zero (base-score stump)
  const float* label; const float* weight;
  float2* gpair;            // [K][gp_stride]
  int64_t gp_stride;        // rows reserved per class (>= n, multiple of 64: keeps class blocks 16 B aligned for the TMA bulk copies)
  unsigned* absmax;         // max|g|, max h as float bits (atomicMax), may be nullptr
  int* err;                 // 1 = logistic label range, 2 = multiclass label range, 3 = squaredlogerror label <= -1, 4 = poisson label < 0,
                            // 5 = gamma label <= 0, 6 = tweedie label < 0
  int64_t n, row_offset;    // row_offset: global index of local row 0 (multi-GPU subsampling stream)
  int K, objective;
  float scale_pos_weight, subsample;
  unsigned seed; unsigned long long iter;
  float aux;                // objective parameter: huber_slope / tweedie_variance_power / the Poisson max_delta_step
};

struct DevNode { float cond; int left; int right; unsigned fidx_dl; };   // 16 B, leaf: left == -1, cond = leaf value

struct PredictArgs {
  const float* X; int64_t n; int F;
  int F_model;              // features of the model; a matrix narrower than that lacks features F..F_model-1 (missing)
  const DevNode* nodes; const int64_t* tree_offset; const int* tree_info;
  int tree_begin, tree_end, K;
  float* margin;            // n x K, pre-initialised with the base margin; may be nullptr
  int* leaf;                // n x (tree_end - tree_begin); may be nullptr
  const int64_t* h_tree_offset;   // host copy of tree_offset (plans the shared-memory tree chunks)
  int has_nan;              // the matrix contains missing values
  int children_adjacent;    // right child == left child + 1 in every tree (true for every tree this engine trains)
};

// Host-side plan of one predictor call: either the thread-per-row kernel, or the tiled kernel run once per chunk of trees,
// each chunk's packed nodes staged in shared memory next to a tile of `rows` rows at `pitch` floats per row.
struct PredictChunk { int tree_lo, tree_hi, rows, threads; size_t head, smem; };   // head: tree offsets + packed nodes (bytes)
struct PredictPlan {
  bool tiled = false;
  int pitch = 0;            // floats per staged row: max(F, F_model) | 1
  bool absent_features = false;    // F < F_model: the staged slots F..F_model-1 hold NaN, so the NaN-aware variant runs
  size_t node_budget = 0;   // bytes of packed nodes one chunk may hold
  std::vector<PredictChunk> chunks;
};
constexpr size_t kPredictSmem = 220 * 1024;       // dynamic shared memory of the tiled predictor (B200: 227 KB per block)
// node_counts[i] = device node slots of tree tree_begin + i; pure host code, touches no device
PredictPlan plan_predict(int F, int F_model, const int64_t* node_counts, int tree_begin, int tree_end, bool children_adjacent);
std::string predict_plan_json(const PredictPlan& p);

enum Metric : int { kMetricRmse = 0, kMetricMae = 1, kMetricLogloss = 2, kMetricError = 3, kMetricMerror = 4, kMetricMlogloss = 5,
                    kMetricAuc = 6, kMetricMse = 7, kMetricRmsle = 8, kMetricMape = 9, kMetricMphe = 10, kMetricPoissonNll = 11,
                    kMetricGammaNll = 12, kMetricGammaDeviance = 13, kMetricTweedieNll = 14 };

struct MetricArgs {
  const float* margin; const float* label; const float* weight; double* out;
  int64_t n; int K, metric, is_logistic; float threshold;
  int transform;            // engine.h Transform applied to the margin first (is_logistic == 1 is kTransformSigmoid)
  float aux;                // huber slope (mphe) / variance power (tweedie-nloglik)
};

// prediction contributions (shap.cu): the model subset [tree_begin, tree_end) repacked with cover and mean value per node
struct ShapNode { float cond; int left; int right; unsigned fidx_dl; float sum_hess; float mean; };   // leaf: left == -1, cond = leaf value
struct ShapArgs {
  const float* X; int64_t n; int F;
  const ShapNode* nodes; const int64_t* tree_offset; const int* tree_info;     // offsets / classes indexed from tree_begin
  int tree_begin, tree_end, K;
  float* out;                      // [n][K][F + 1], zero-initialised by the caller
  const float* base_margin_rows;   // [n][K] user base margins, or nullptr -> base_margin
  float base_margin;
};
void launch_shap(const ShapArgs& a, int max_depth, cudaStream_t s);

void launch_gradient(const GradArgs& a, cudaStream_t s);
void launch_sum_gpair(const float2* gp, int64_t n, double* out, cudaStream_t s);
void launch_bin(const float* X, int64_t n, int F, int ngroups, int tw, const int* cut_ptrs, const float* cut_vals, uint8_t* bins, uint8_t* bins_tail, cudaStream_t s);
void launch_transpose_bins(const uint8_t* bins, const uint8_t* bins_tail, int64_t n, int F, int ngroups, int tw, uint8_t* bins_col, cudaStream_t s);
void launch_pad_rows(const uint8_t* src, int64_t n, int src_stride, uint8_t* dst, int dst_stride, cudaStream_t s);
void launch_count_nan(const float* X, int64_t count, float missing, int use_missing, unsigned long long* out, cudaStream_t s);
void launch_replace_missing(float* X, int64_t count, float missing, cudaStream_t s);
void launch_predict(const PredictArgs& a, cudaStream_t s);
void launch_transform(float* m, int64_t n, int K, int objective, float* out_class, cudaStream_t s);
void launch_fill(float* p, int64_t n, float v, cudaStream_t s);
void launch_metric(const MetricArgs& a, cudaStream_t s);
// auc.cu (experimental): out[0] += unnormalised ROC area, out[1] = positive weight, out[2] = negative weight
void compute_auc_device(const float* margin, const float* label, const float* weight, int64_t n, int is_logistic, double* out, cudaStream_t s);

// quantile.cu: exact weighted-quantile cuts per feature (same definition as oracle/gbt_oracle.c cuts_from_distinct).
// X: device, row-major n x F. Returns host vectors.
struct HostCuts { std::vector<int> ptrs; std::vector<float> vals; std::vector<float> mins; };
// Per-feature summary for distributed merging: distinct values + weights (host), capped.
void compute_cuts_device(const float* dX, int64_t n, int F, const float* dweights, int max_bin, bool has_missing,
                         HostCuts* out, cudaStream_t s);
// Distinct-value summary of one rank (for merging cuts across ranks): per feature the sorted distinct values and
// their weights, exact when a feature has <= cap distinct values, else a cap-point weighted-quantile summary.
struct FeatureSummary { std::vector<float> vals; std::vector<double> weights; };
void compute_summaries_device(const float* dX, int64_t n, int F, const float* dweights, int cap,
                              std::vector<FeatureSummary>* out, cudaStream_t s);
void cuts_from_summaries(const std::vector<FeatureSummary>& sums, int max_bin, bool has_missing, HostCuts* out);

}  // namespace b200
