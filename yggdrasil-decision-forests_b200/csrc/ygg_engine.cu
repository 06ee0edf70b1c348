// ygg_engine.cu — host side of libygg_b200.so: the device-resident boosting loop and the C ABI
// declared in include/ygg_b200.h.
//
// The loop mirrors GradientBoostedTreesLearner::TrainWithStatusImpl
// (learner/gradient_boosted_trees/gradient_boosted_trees.cc:1428-1571) but grows every tree
// level-wise on the GPU with no host synchronisation: all per-node decisions (best split, children,
// stop tests, slot assignment) are taken by kernels that read and write device tables.
#include <algorithm>
#include <mutex>
#include <random>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <map>
#include <queue>
#include <string>
#include <thread>
#include <vector>

#include <cuda_runtime.h>
#include <cub/device/device_radix_sort.cuh>
#include <nvtx3/nvToolsExt.h>   // header-only: the ranges cost nothing unless a profiler injects itself

#include "../../include/ygg_b200.h"
#include "ygg_internal.h"
#include "../../include/ygg_b200_model.h"
#include "ygg_kernels.cuh"

using namespace ygg;

namespace {

thread_local std::string g_last_error;

int set_error(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
  return code;
}

}  // namespace

int ygg_set_error_msg(int code, const char* msg) { return set_error(code, "%s", msg); }

namespace {

#define YGG_CUDA(expr)                                                                          \
  do {                                                                                          \
    cudaError_t _e = (expr);                                                                    \
    if (_e != cudaSuccess)                                                                      \
      return set_error(YGG_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),    \
                       __FILE__, __LINE__);                                                     \
  } while (0)

#define YGG_RETURN_IF_ERROR(expr) \
  do {                            \
    int _s = (expr);              \
    if (_s != YGG_OK) return _s;  \
  } while (0)

// Device memory comes from the device's stream-ordered pool with an unlimited release threshold: a handle
// that is destroyed and re-created in the same process (hyper-parameter sweeps, bench.py's e2e pass) reuses
// the mapped memory instead of paying the driver's map / unmap again (measured: 10-280 ms per create at C3).
// Buffers handed to NCCL (level buffer, shard-best table) stay plain cudaMalloc allocations.
void configure_pool_once(int device) {
  static std::mutex mu;
  static std::vector<char> done;
  std::lock_guard<std::mutex> lock(mu);
  if (static_cast<int>(done.size()) <= device) done.resize(device + 1, 0);
  if (done[device]) return;
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
    unsigned long long threshold = ~0ull;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &threshold);
  }
  cudaGetLastError();
  done[device] = 1;
}

template <typename T>
int dev_alloc(T** p, size_t count) {
  int device = 0;
  cudaGetDevice(&device);
  configure_pool_once(device);
  const size_t bytes = std::max<size_t>(count, 1) * sizeof(T);
  YGG_CUDA(cudaMallocAsync(reinterpret_cast<void**>(p), bytes, nullptr));
  // pool memory is recycled: zero it, so that nothing depends on what a previous handle left behind
  YGG_CUDA(cudaMemsetAsync(*p, 0, bytes, nullptr));
  YGG_CUDA(cudaStreamSynchronize(nullptr));  // usable from any stream from here on
  return YGG_OK;
}
template <typename T>
int dev_alloc_plain(T** p, size_t count) {
  YGG_CUDA(cudaMalloc(reinterpret_cast<void**>(p), std::max<size_t>(count, 1) * sizeof(T)));
  return YGG_OK;
}
// Frees a dev_alloc pointer (callers have synchronised the streams that used it).
inline void dev_free(void* p) {
  if (p != nullptr) cudaFreeAsync(p, nullptr);
}

struct ProfileSlot {
  double ms = 0;
  int64_t launches = 0;
};

}  // namespace


struct LossRec {
  double loss_sum;
  unsigned long long correct;
};

enum ShardMode { kShardNone = 0, kShardFeatures = 1, kShardRows = 2 };

// k_hist launches of one tree level: num_sms persistent CTAs of the instantiation for (mode, hessian planes, passes > 1).
struct HistLevel {
  int mode;           // kHistRootSum / kHistPacked / kHistShared (ygg_hist.cuh)
  int G;              // features per work item
  int S;              // slots in shared memory (windowed: window + 1 dummy slot)
  int passes;         // > 1: the level's slots are accumulated in windows of S - 1 slots, one launch each
  int chunk_blocks;   // 8192-row blocks per work item
  size_t smem;        // dynamic shared memory per CTA
};

struct ygg_gbt {
  ygg_dataset* ds = nullptr;
  int device = 0;   // ds->device: ygg_gbt_destroy must not read `ds`, which may already be destroyed
  ygg_gbt_config cfg{};
  cudaStream_t stream = nullptr;
  bool has_labels = false;
  uint8_t* d_label_u8 = nullptr;
  float* d_label_f32 = nullptr;
  float initial_prediction = 0.f;
  float* d_pred = nullptr;
  float* d_g = nullptr;
  float* d_h = nullptr;
  uint32_t* d_q24 = nullptr;
  uint32_t* d_hq24 = nullptr;
  uint2* d_act = nullptr;
  uint32_t* d_act_h = nullptr;
  int32_t* d_act_count = nullptr;
  uint32_t* d_root_cnt = nullptr;  // [f_count][256] row counts of the root (gradient independent)
  bool root_cnt_valid = false;
  int n_blocks = 0;
  uint16_t* d_node_of_row = nullptr;
  DeviceState* d_st = nullptr;
  LevelDesc* d_levels = nullptr;
  Family* d_fam[2] = {nullptr, nullptr};
  int32_t* d_slot_node[2] = {nullptr, nullptr};
  NodeRec* d_nodes_all = nullptr;   // [tree capacity][max_nodes]
  NodeRec* d_nodes_scratch = nullptr;  // ygg_tree_train_on_gradients
  int tree_capacity = 0;
  unsigned long long* d_hist_sum[2] = {nullptr, nullptr};
  uint32_t* d_hist_cnt[2] = {nullptr, nullptr};
  unsigned long long* d_hist_hsum[2] = {nullptr, nullptr};
  Candidate* d_cand = nullptr;
  uint32_t* d_cand_mask = nullptr;  // [split-level nodes][f_scan][8]
  ShardBest* d_shard_best = nullptr;
  TieRec* d_ties = nullptr;        // [max level nodes] ties of the level being selected (single GPU)
  // stochastic gradient boosting (cfg.subsample < 1): this iteration's sample, drawn on the host from the learner's engine
  uint8_t* d_selected = nullptr;   // [n_pad]
  std::vector<uint8_t> host_selected;
  int64_t n_selected = 0;
  // tie-break replay (cfg.candidate_shuffle): the learner's engine after the trees resolved so far
  std::mt19937 tie_rng;
  bool tie_rng_ready = false;
  int ties_resolved_upto = 0;
  int64_t ties_renamed = 0, ties_unresolved = 0;
  LossRec* d_loss = nullptr;  // [tree capacity] (this rank's rows)
  LossPartials* d_loss_partials = nullptr;   // per-CTA partial sums of the loss kernels (reduce_loss_in_order)
  // Level buffer, one contiguous allocation so that row-sharded runs all-reduce it in one call:
  //   [sum u64 x B][hsum u64 x B (hessian histogram only)][cnt u32 x B][stats u64 x 3 x children]
  // with B = slot bound x hist features x 256.  Counts are summed as u64 pairs (no carry can cross:
  // every count is < 2^31 and so is every total).
  unsigned long long* d_level_buf = nullptr;
  size_t level_buf_bytes = 0;
  size_t slot_elems_cap = 0;      // B for the deepest level
  int stats_cap = 0;              // children capacity of the stats region
  // sharding
  int shard_mode = kShardNone;
  int hist_f_begin = 0, hist_f_end = 0;   // features histogrammed by this rank
  int64_t n_global = 0;                   // rows of the whole job
  ygg_allreduce_fn allreduce = nullptr;
  ygg_reducescatter_fn reducescatter = nullptr;
  bool scatter = false;   // row shards with the level buffer reduce-scattered by feature chunk (and a sharded scan)
  int loss_reduced_upto = 0;
  int max_nodes = 0, max_level_nodes = 0, num_levels = 0;
  int trees_done = 0;
  bool pending = false;  // the last tree's leaves are not yet added to d_pred
  // multinomial loss: K trees per iteration; predictions / gradients are K planes ([K][n] / [K][n_pad])
  int K = 1;
  int iters_done = 0;          // == trees_done / K
  bool pending_loss = false;   // multinomial: the loss of the last iteration is not yet in d_loss
  float* cur_g = nullptr;      // gradient / hessian plane the tree being grown is trained on
  float* cur_h = nullptr;
  float* cur_g2w = nullptr;    // (example weights) plane of (w*g)*g of the tree being grown
  // validation rows (SURVEY §8f N2)
  const ygg_dataset* vds = nullptr;
  float* d_vpred = nullptr;
  uint8_t* d_vlabel_u8 = nullptr;
  float* d_vlabel_f32 = nullptr;
  LossRec* d_vloss = nullptr;     // [tree capacity]
  // example weights (ygg_gbt_set_weights_f32 / ygg_gbt_set_validation_weights_f32)
  float* d_weight = nullptr;      // [n_pad] training weights (null: unweighted)
  float* d_g2w = nullptr;         // [n_pad] (w*g)*g of every row (sum of squares of the nodes)
  unsigned long long* d_wsums = nullptr;   // [max_nodes][2] k_weight_sums_*
  std::vector<float> host_weights;   // kept for the initial predictions (the labels may be set after the weights)
  double sum_weights = 0;         // sum of the training weights, double in row order
  float w_pow2 = 1.f;             // power of two >= max training weight
  // GOSS: sort buffers (|g| keys / row ids, in and out), the iteration's draws, cub's scratch
  float* d_goss_keys[2] = {nullptr, nullptr};
  uint32_t* d_goss_rows[2] = {nullptr, nullptr};
  float* d_goss_u = nullptr;
  void* d_goss_temp = nullptr;
  size_t goss_temp_bytes = 0;
  std::vector<float> host_goss_u;
  int64_t goss_cutoff = 0;
  float* d_vweight = nullptr;     // [validation rows] (null: unweighted)
  double v_sum_weights = 0;
  float v_correct_scale = 0.f;
  bool finalized = false;         // early stopping / truncation applied: no further iterations
  int final_trees = -1;           // model size after truncation
  int log_entries = -1;           // iterations kept in the logs
  float final_validation_loss = 0.f;
  bool early_stopping_triggered = false;
  // feature shard
  int f_begin = 0, f_end = 0, rank = 0, world = 1;
  ygg_allgather_fn exchange = nullptr;
  void* exchange_ctx = nullptr;
  void** d_peer_windows = nullptr;   // [world] best-split windows of every rank as mapped in this process (or null)
  uint32_t exchange_epoch = 0;
  // launch configuration (configure_launches)
  HistLevel hist[32]{};
  int part_smem_children = 0;
  // histogram capture (ygg_gbt_debug_capture_histograms): every level's slot planes of the last tree grown
  bool capture_hist = false;
  unsigned long long* d_capture = nullptr;   // level l's level buffer at capture_off[l]
  size_t capture_u64 = 0;
  std::vector<size_t> capture_off;
  std::vector<ygg_hist_level_info> capture_info;   // launch configuration of every captured level
  float* d_capture_g = nullptr;      // [n_pad] the quantiser's inputs: gradients,
  float* d_capture_h2 = nullptr;     // [n_pad] the second plane's values (hessians or weights),
  uint8_t* d_capture_sel = nullptr;  // [n_pad] the sampled rows
  bool capture_has_h2 = false, capture_has_sel = false;
  DeviceState* d_capture_st = nullptr;
  const NodeRec* capture_nodes = nullptr;   // node table of the captured tree (null: nothing captured)
  // profiling
  bool profiling = false;
  std::map<std::string, ProfileSlot> profile;
  std::vector<std::pair<std::string, std::pair<cudaEvent_t, cudaEvent_t>>> pending_events;
  int64_t launches_total = 0;
};

namespace {

bool use_hess(const ygg_gbt* h) { return h->cfg.use_hessian_gain != 0; }
// IsLogitLoss (loss_utils.cc:41-45): bounded gradients (|g| <= 1, h <= 1/4), leaf clamp.
bool is_logit(const ygg_gbt* h) {
  return h->cfg.loss == YGG_LOSS_BINOMIAL_LOG_LIKELIHOOD || h->cfg.loss == YGG_LOSS_MULTINOMIAL_LOG_LIKELIHOOD;
}
bool is_multinomial(const ygg_gbt* h) { return h->cfg.loss == YGG_LOSS_MULTINOMIAL_LOG_LIKELIHOOD; }
bool weighted(const ygg_gbt* h) { return h->d_weight != nullptr; }
// With example weights every row carries w*h (squared error: w), so the hessian array is always read.
bool has_h(const ygg_gbt* h) { return is_logit(h) || weighted(h); }
float h_pow2_of(const ygg_gbt* h) { return (is_logit(h) ? 0.25f : 1.f) * (weighted(h) ? h->w_pow2 : 1.f); }
// the weight of a correctly classified row is counted in units of 1 / correct_scale
float correct_scale_of(float w_pow2) { return static_cast<float>(1u << kSBits) / w_pow2; }
// A hessian histogram is only accumulated when the hessian varies per row; for squared error
// (h == 1) the per-bin hessian sum is the bin count.
// (example weights, variance gain: the second plane holds the bins' WEIGHT sums, see ScanParams.weighted)
bool hist_hess(const ygg_gbt* h) { return (use_hess(h) && has_h(h)) || weighted(h); }
// SampleTrainingExamples draws nothing for sample >= 1 - eps (gradient_boosted_trees.cc:2936-2940)
// gradient-based one-side sampling: a per-iteration row sample WITH weights (ygg_gbt_config.goss_alpha / goss_beta)
bool goss(const ygg_gbt* h) { return h->cfg.goss_alpha > 0.f || h->cfg.goss_beta > 0.f; }
bool sampling(const ygg_gbt* h) { return h->cfg.subsample < 1.f - std::numeric_limits<float>::epsilon() || goss(h); }
// the caller's example weights (losses, initial predictions); GOSS weights are the engine's own and the losses stay unweighted
bool user_weighted(const ygg_gbt* h) { return h->d_weight != nullptr && !goss(h); }

// Phase scope: CUDA events when ygg_gbt_set_profiling is on (bench.py's kernel_ms_per_step), and an NVTX range named after
// the phase ("hist", "hist_L3", "scan", "select", "partition", "grad", "allreduce", "validation") when YGG_NVTX=1 — the
// host-side enqueue window of the phase, for timeline tools (SURVEY.md §5 tracing).
inline bool nvtx_enabled() {
  static const bool on = [] { const char* v = std::getenv("YGG_NVTX"); return v != nullptr && std::atoi(v) != 0; }();
  return on;
}
struct ProfScope {
  ygg_gbt* h;
  const char* name;
  cudaEvent_t a = nullptr, b = nullptr;
  ProfScope(ygg_gbt* h_, const char* n) : h(h_), name(n) {
    if (nvtx_enabled()) nvtxRangePushA(n);
    if (h->profiling) {
      cudaEventCreate(&a);
      cudaEventCreate(&b);
      cudaEventRecord(a, h->stream);
    }
  }
  ~ProfScope() {
    if (h->profiling) {
      cudaEventRecord(b, h->stream);
      h->pending_events.push_back({name, {a, b}});
    }
    if (nvtx_enabled()) nvtxRangePop();
  }
};

void collect_profile(ygg_gbt* h) {
  for (auto& e : h->pending_events) {
    float ms = 0;
    cudaEventSynchronize(e.second.second);
    cudaEventElapsedTime(&ms, e.second.first, e.second.second);
    auto& s = h->profile[e.first];
    s.ms += ms;
    s.launches++;
    cudaEventDestroy(e.second.first);
    cudaEventDestroy(e.second.second);
  }
  h->pending_events.clear();
}

int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_error(YGG_ERR_CUDA, "launch of %s failed: %s", what, cudaGetErrorString(e));
  return YGG_OK;
}

// Static bound on the histogram slots a level can need.
int level_slot_bound(const ygg_gbt* h, int level) {
  if (level == 0) return 1;
  return h->cfg.sibling_subtraction ? (1 << (level - 1)) : (1 << level);
}

// Level-buffer layout for a level whose slot histograms hold `B` bins (see ygg_gbt::d_level_buf).
struct LevelBuf {
  // chunk 0 (with one chunk: the whole buffer)
  unsigned long long* sum;
  unsigned long long* hsum;
  uint32_t* cnt;
  unsigned long long* stats;
  int W;             // chunks: 1, or the world size when the level buffer is reduce-scattered by feature
  int f_chunk;       // features per chunk
  size_t chunk_u64;  // u64 words per chunk
  size_t planes_u64; // words of a chunk before its stats tail (what is zeroed before k_hist)
  size_t total_u64;  // W * chunk_u64 (for the all-reduce / reduce-scatter)
};
// Layout of the level buffer for `slots` histogram slots and `n_stats_nodes` node statistics:
// per chunk [sum u64 | hsum u64 (hessian) | cnt u32, padded to u64 | stats 3 u64 per node].
LevelBuf level_buf(const ygg_gbt* h, int slots, int n_stats_nodes) {
  LevelBuf lb;
  const int f_hist = h->hist_f_end - h->hist_f_begin;
  lb.W = h->scatter ? h->world : 1;
  lb.f_chunk = (f_hist + lb.W - 1) / lb.W;
  const size_t B = static_cast<size_t>(slots) * lb.f_chunk * kMaxBins;
  lb.sum = h->d_level_buf;
  unsigned long long* p = lb.sum + B;
  lb.hsum = nullptr;
  if (hist_hess(h)) { lb.hsum = p; p += B; }
  lb.cnt = reinterpret_cast<uint32_t*>(p);
  p += (B + 1) / 2;
  lb.stats = p;
  lb.planes_u64 = static_cast<size_t>(p - h->d_level_buf);
  p += static_cast<size_t>(n_stats_nodes) * 3;
  lb.chunk_u64 = static_cast<size_t>(p - h->d_level_buf);
  lb.total_u64 = lb.chunk_u64 * lb.W;
  return lb;
}

// Zeroes the histogram planes of every chunk (not the stats tails) / copies chunk 0's stats to the others.
__global__ void k_zero_planes(unsigned long long* base, size_t chunk_u64, size_t planes_u64) {
  unsigned long long* c = base + static_cast<size_t>(blockIdx.y) * chunk_u64;
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < planes_u64;
       i += static_cast<size_t>(gridDim.x) * blockDim.x)
    c[i] = 0ull;
}
__global__ void k_replicate_stats(unsigned long long* stats0, size_t chunk_u64, int n_words, int W) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_words) return;
  const unsigned long long v = stats0[i];
  for (int c = 1; c < W; c++) stats0[static_cast<size_t>(c) * chunk_u64 + i] = v;
}

int zero_planes(ygg_gbt* h, const LevelBuf& lb) {
  if (lb.W == 1) {
    YGG_CUDA(cudaMemsetAsync(lb.sum, 0, lb.planes_u64 * sizeof(unsigned long long), h->stream));
    return YGG_OK;
  }
  dim3 grid(static_cast<unsigned>(std::min<size_t>((lb.planes_u64 + 255) / 256, 1024)), static_cast<unsigned>(lb.W));
  k_zero_planes<<<grid, 256, 0, h->stream>>>(lb.sum, lb.chunk_u64, lb.planes_u64);
  h->launches_total++;
  return check_launch("k_zero_planes");
}
int replicate_stats(ygg_gbt* h, const LevelBuf& lb, int n_nodes) {
  if (lb.W == 1) return YGG_OK;
  k_replicate_stats<<<(3 * n_nodes + 127) / 128, 128, 0, h->stream>>>(lb.stats, lb.chunk_u64, 3 * n_nodes, lb.W);
  h->launches_total++;
  return check_launch("k_replicate_stats");
}

template <typename F>
int for_hist_kernel(bool hess, int mode, F f, bool multi = false) {
  if (multi) {
    if (hess) return f(k_hist<true, kHistShared, true>);
    if (mode == kHistPacked) return f(k_hist<false, kHistPacked, true>);
    return f(k_hist<false, kHistShared, true>);
  }
  if (hess) return f(k_hist<true, kHistShared>);
  if (mode == kHistRootSum) return f(k_hist<false, kHistRootSum>);
  if (mode == kHistPacked) return f(k_hist<false, kHistPacked>);
  return f(k_hist<false, kHistShared>);
}

// Largest per-bin row count of any (chunk of `chunk_blocks` blocks, histogrammed feature) of this handle's rows;
// `*d_sub` caches the sub-chunk count table between calls (the caller frees it).
// granularity of the packed-bound table and of the chunk sizes it allows: single blocks up to 4M rows (the chunk size is
// then free to fill whole waves of CTAs, which matters when a rank holds few rows), 8 blocks above (table size)
int sub_blocks_of(const ygg_gbt* h) { return h->ds->n_pad / kBlockRows >= 512 ? 8 : 1; }
int chunk_max_count(ygg_gbt* h, int chunk_blocks, uint32_t** d_sub, uint32_t* out_max) {
  const int kSubBlocks = sub_blocks_of(h);
  const ygg_dataset* ds = h->ds;
  const int f_count = h->hist_f_end - h->hist_f_begin;
  const int n_blocks = static_cast<int>(ds->n_pad / kBlockRows);
  const int n_subs = (n_blocks + kSubBlocks - 1) / kSubBlocks;
  if (*d_sub == nullptr) {
    YGG_RETURN_IF_ERROR(dev_alloc(d_sub, static_cast<size_t>(n_subs) * f_count * kMaxBins + 1));
    k_sub_counts<<<dim3(n_subs, f_count), 256>>>(ds->d_bins, ds->n, ds->n_pad, h->hist_f_begin, kSubBlocks, *d_sub);
    YGG_RETURN_IF_ERROR(check_launch("k_sub_counts"));
  }
  uint32_t* d_max = *d_sub + static_cast<size_t>(n_subs) * f_count * kMaxBins;
  YGG_CUDA(cudaMemset(d_max, 0, sizeof(uint32_t)));
  const int subs_per_chunk = chunk_blocks / kSubBlocks;
  const int n_chunks = (n_subs + subs_per_chunk - 1) / subs_per_chunk;
  k_chunk_max<<<dim3(n_chunks, f_count), 256>>>(*d_sub, n_subs, subs_per_chunk, d_max);
  YGG_CUDA(cudaMemcpy(out_max, d_max, sizeof(uint32_t), cudaMemcpyDeviceToHost));
  return YGG_OK;
}

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-kernel cap of the current device, shared by every handle of the
// process (handles with other feature shards, or on other devices, may coexist): raise it to the full budget on every
// k_hist instantiation.  It is only a cap: each launch asks for its level's HistLevel::smem.
int raise_hist_smem_cap(size_t budget) {
  auto cap = [&](auto kern) -> int {
    YGG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(budget)));
    return YGG_OK;
  };
  YGG_RETURN_IF_ERROR(cap(k_hist<false, kHistRootSum>));
  YGG_RETURN_IF_ERROR(cap(k_hist<false, kHistPacked>));
  YGG_RETURN_IF_ERROR(cap(k_hist<false, kHistShared>));
  YGG_RETURN_IF_ERROR(cap(k_hist<true, kHistShared>));
  YGG_RETURN_IF_ERROR(cap(k_hist<false, kHistPacked, true>));
  YGG_RETURN_IF_ERROR(cap(k_hist<false, kHistShared, true>));
  return cap(k_hist<true, kHistShared, true>);
}

// The k_hist launches of every level (HistLevel).  Layout: with the hessian or weight planes, kHistShared; at an
// unsampled root, kHistRootSum (the root's counts are gradient independent and precomputed: no count atomics); else
// kHistPacked (two REDs per element instead of a RED and a returning ATOMS), which falls back to kHistShared when a bin
// could receive more than kPackedMaxUpdates updates inside one work item.
int configure_launches(ygg_gbt* h) {
  const bool hh = hist_hess(h);
  const size_t budget = 224 * 1024;  // dynamic shared memory per CTA we are willing to use (227 KB max)
  const int f_count = h->hist_f_end - h->hist_f_begin;  // features histogrammed by this rank
  const int n_blocks = static_cast<int>(h->ds->n_pad / kBlockRows);
  const int grid = h->ds->num_sms;
  const int kSubBlocks = sub_blocks_of(h);
  // Row blocks per work item of G features (a multiple of `step`): as many as the bin counters allow (the flush to the
  // global histogram is amortised over the chunk), but few enough that every CTA gets at least one item, and among
  // those the size whose item count fills whole waves of the persistent grid (static round-robin over CTAs; measured:
  // whole waves beat many small items on C2, C3 and at 1.25M rows per rank).
  // YGG_HIST_CHUNK_BLOCKS=c (tests: reach the chunk sizes where the bin counters come closest to their limits) forces
  // c row blocks per work item, clamped to [step, kHistMaxChunkBlocks] and rounded down to the step.  Read at every
  // configure.
  const char* env_chunk = std::getenv("YGG_HIST_CHUNK_BLOCKS");
  const int forced_chunk = env_chunk != nullptr ? std::atoi(env_chunk) : 0;
  auto choose_chunk = [&](int G, int step) {
    const int n_fgroups = (f_count + G - 1) / G;
    const int max_c = std::max(step, kHistMaxChunkBlocks / step * step);
    if (forced_chunk > 0) return std::max(step, std::min(forced_chunk, max_c) / step * step);
    const int min_chunks = std::max(1, (n_blocks + max_c - 1) / max_c);
    int best = max_c;
    double best_score = -1;
    for (int nc = min_chunks; nc <= std::max(min_chunks, n_blocks); nc++) {
      // nc chunks of equal size, rounded up to the step (the last chunk may then be shorter: count the real chunks)
      const int c = std::min(max_c, ((n_blocks + nc - 1) / nc + step - 1) / step * step);
      const int real_nc = (n_blocks + c - 1) / c;
      const double per_cta = static_cast<double>(real_nc) * n_fgroups / grid;
      if (per_cta > 8.0 && nc > min_chunks) break;
      // a short last chunk leaves its CTAs idle for the rest of a round: weigh the waves by the rows they carry
      const double fill = static_cast<double>(n_blocks) / (static_cast<double>(real_nc) * c);
      const double eff = per_cta / std::ceil(per_cta) * fill;
      // whole waves first (an unfilled last wave idles the GPU), then at least one item per CTA
      const double score = eff + (per_cta >= 1.0 ? 0.08 : 0.0);
      if (score > best_score + 1e-9) { best_score = score; best = c; }
    }
    return best;
  };
  for (int l = 0; l < h->num_levels; l++) {
    HistLevel& hl = h->hist[l];
    // (a sampled root is not the whole dataset: its counts are not the precomputed ones)
    hl.mode = hh ? kHistShared : (l == 0 && !sampling(h)) ? kHistRootSum : kHistPacked;
    int S = level_slot_bound(h, l);
    hl.passes = 1;
    if (hist_smem_bytes(1, S, hh, hl.mode) > budget) {
      // more slots than shared memory holds: windows of S_pass slots (+ 1 dummy slot for the rows of the other windows),
      // one launch per window.  The slot of a row travels in 8 bits of its active-list entry (0xFF = none).
      if (S > 254)
        return set_error(YGG_ERR_UNIMPLEMENTED, "max_depth=%d needs %d histogram slots at level %d; the active lists carry 8-bit slots",
                         h->cfg.max_depth, S, l);
      int s_pass = 1;
      while (hist_smem_bytes(1, 2 * s_pass + 1, hh, hl.mode) <= budget) s_pass *= 2;
      hl.passes = (S + s_pass - 1) / s_pass;
      S = s_pass + 1;
    }
    int G = 1;
    while (G < 8 && G < f_count && hist_smem_bytes(G + 1, S, hh, hl.mode) <= budget) G++;
    hl.G = G;
    hl.S = S;
    hl.smem = hist_smem_bytes(G, S, hh, hl.mode);
    hl.chunk_blocks = choose_chunk(G, hl.mode == kHistPacked ? kSubBlocks : 1);
  }
  // The packed words' bound: the dataset-level largest count a bin can receive inside one work item (ygg_hist.cuh).
  {
    std::map<int, uint32_t> max_of_chunk;   // chunk size -> largest per-bin count of any (chunk, feature)
    uint32_t* d_sub = nullptr;
    int status = YGG_OK;
    for (int l = 0; l < h->num_levels && status == YGG_OK; l++) {
      HistLevel& hl = h->hist[l];
      if (hl.mode != kHistPacked) continue;
      int chunk = hl.chunk_blocks;
      while (chunk >= kSubBlocks) {
        auto it = max_of_chunk.find(chunk);
        if (it == max_of_chunk.end()) {
          uint32_t m = 0;
          status = chunk_max_count(h, chunk, &d_sub, &m);
          if (status != YGG_OK) break;
          it = max_of_chunk.emplace(chunk, m).first;
        }
        if (it->second <= kPackedMaxUpdates) break;
        // shrink the chunk in proportion (+ margin); below one sub-chunk the flushes would cost more than the RED saves
        const int smaller = static_cast<int>(static_cast<double>(chunk) * 0.9 * kPackedMaxUpdates / it->second) / kSubBlocks * kSubBlocks;
        chunk = std::min(smaller, chunk - kSubBlocks);
      }
      if (chunk < kSubBlocks) {   // heavy bins (a dominant value / category): the carry-detecting layout, any chunk size
        hl.mode = kHistShared;    // (the same shared memory as kHistPacked without the hessian planes)
        hl.chunk_blocks = choose_chunk(hl.G, 1);
      } else {
        hl.chunk_blocks = chunk;
      }
    }
    dev_free(d_sub);
    if (status != YGG_OK) return status;
  }
  YGG_RETURN_IF_ERROR(raise_hist_smem_cap(budget));
  // k_partition shared accumulators: up to 32 KB (one copy) / 14 KB (lane-private, <= 16 children).
  h->part_smem_children = static_cast<int>((32 * 1024) / (kPartWords * sizeof(uint32_t)));
  return YGG_OK;
}

// (Re)allocates everything whose size depends on the feature shard.
int allocate_level_buffers(ygg_gbt* h) {
  const int f_scan = h->f_end - h->f_begin;
  const int f_hist = h->hist_f_end - h->hist_f_begin;
  for (int i = 0; i < 2; i++) {
    dev_free(h->d_hist_sum[i]); dev_free(h->d_hist_cnt[i]); dev_free(h->d_hist_hsum[i]);
    h->d_hist_sum[i] = nullptr; h->d_hist_cnt[i] = nullptr; h->d_hist_hsum[i] = nullptr;
  }
  dev_free(h->d_cand); h->d_cand = nullptr;
  dev_free(h->d_cand_mask); h->d_cand_mask = nullptr;
  cudaFree(h->d_level_buf); h->d_level_buf = nullptr;
  const size_t split_level_nodes = static_cast<size_t>(1) << std::max(0, h->num_levels - 1);
  const size_t node_elems = split_level_nodes * f_scan * kMaxBins;
  for (int i = 0; i < 2; i++) {
    YGG_RETURN_IF_ERROR(dev_alloc(&h->d_hist_sum[i], node_elems));
    YGG_RETURN_IF_ERROR(dev_alloc(&h->d_hist_cnt[i], node_elems));
    if (hist_hess(h)) YGG_RETURN_IF_ERROR(dev_alloc(&h->d_hist_hsum[i], node_elems));
  }
  YGG_RETURN_IF_ERROR(dev_alloc(&h->d_cand, split_level_nodes * f_scan));
  YGG_RETURN_IF_ERROR(dev_alloc(&h->d_cand_mask, split_level_nodes * f_scan * 8));
  if (h->d_shard_best == nullptr)
    YGG_RETURN_IF_ERROR(dev_alloc_plain(&h->d_shard_best, static_cast<size_t>(std::max(1, h->world)) * h->max_level_nodes));
  size_t max_u64 = 16;
  for (int l = 0; l <= h->num_levels; l++) {
    const int slots = l < h->num_levels ? level_slot_bound(h, l) : 0;
    const int stats_nodes = l == 0 ? 1 : (2 << (l - 1));
    max_u64 = std::max(max_u64, level_buf(h, slots, stats_nodes).total_u64);
  }
  (void)f_hist;
  h->level_buf_bytes = max_u64 * sizeof(unsigned long long);
  YGG_RETURN_IF_ERROR(dev_alloc_plain(&h->d_level_buf, max_u64));
  return YGG_OK;
}

int launch_hist(ygg_gbt* h, const HistParams& hp, const HistLevel& hl) {
  return for_hist_kernel(hist_hess(h), hl.mode, [&](auto kern) -> int {
    kern<<<h->ds->num_sms, kHistThreads, hl.smem, h->stream>>>(hp);   // persistent: one CTA per SM
    h->launches_total++;
    return check_launch("k_hist");
  }, hl.passes > 1);
}

// Root count histogram: once per (dataset, shard).
int ensure_root_counts(ygg_gbt* h) {
  if (h->root_cnt_valid) return YGG_OK;
  const int f_count = h->hist_f_end - h->hist_f_begin;
  if (h->d_root_cnt) dev_free(h->d_root_cnt);
  h->d_root_cnt = nullptr;
  const LevelBuf lb = level_buf(h, 1, 1);  // chunk geometry: the array is padded to W * f_chunk features
  const size_t padded = static_cast<size_t>(lb.W) * lb.f_chunk * kMaxBins;
  YGG_RETURN_IF_ERROR(dev_alloc(&h->d_root_cnt, padded));
  YGG_CUDA(cudaMemsetAsync(h->d_root_cnt, 0, padded * sizeof(uint32_t), h->stream));
  dim3 grid(std::max(1, h->ds->num_sms * 8 / std::max(1, f_count)), f_count);
  k_root_counts<<<grid, 256, 0, h->stream>>>(h->ds->d_bins, h->ds->n, h->ds->n_pad, f_count, h->hist_f_begin, h->d_root_cnt);
  h->launches_total++;
  YGG_RETURN_IF_ERROR(check_launch("k_root_counts"));
  h->root_cnt_valid = true;
  return YGG_OK;
}

int elementwise_grid(const ygg_gbt* h) { return h->ds->num_sms * 8; }

int do_allreduce(ygg_gbt* h, void* buf, int64_t count, int dtype, int op) {
  if (h->allreduce == nullptr) return set_error(YGG_ERR_INVALID_ARGUMENT, "row sharding without an all-reduce function");
  const int rc = h->allreduce(h->exchange_ctx, buf, count, dtype, op, h->stream);
  if (rc != 0) return set_error(YGG_ERR_CUDA, "all-reduce failed with code %d", rc);
  return YGG_OK;
}

// Example weights: weight sum and weighted sum of squares of every node of the finished tree (k_weight_sums_*).
int launch_weight_sums(ygg_gbt* h, NodeRec* nodes) {
  ProfScope ps(h, "select");
  WeightSumParams wp{};
  wp.n = h->ds->n; wp.node_of_row = h->d_node_of_row; wp.selected = sampling(h) ? h->d_selected : nullptr;
  wp.weight = h->d_weight; wp.g2w = h->cur_g2w != nullptr ? h->cur_g2w : h->d_g2w; wp.st = h->d_st; wp.w_pow2 = h->w_pow2; wp.nodes = nodes;
  wp.sums = h->d_wsums; wp.levels = h->d_levels; wp.num_levels = h->num_levels + 1;
  wp.smem_nodes = h->max_nodes <= 2048 ? h->max_nodes : 0;
  YGG_CUDA(cudaMemsetAsync(h->d_wsums, 0, static_cast<size_t>(h->max_nodes) * 2 * sizeof(unsigned long long), h->stream));
  const size_t smem = static_cast<size_t>(wp.smem_nodes) * 2 * sizeof(unsigned long long);
  k_weight_sums_rows<<<h->ds->num_sms * 4, 256, smem, h->stream>>>(wp);
  if (h->shard_mode == kShardRows)   // every rank added its rows up; the integer sums make the reduction exact
    YGG_RETURN_IF_ERROR(do_allreduce(h, h->d_wsums, static_cast<int64_t>(h->max_nodes) * 2, 1, 0));
  k_weight_sums_finish<<<1, 1024, 0, h->stream>>>(wp);
  h->launches_total += 2;
  return check_launch("k_weight_sums");
}

// The enum ygg_hist_layout value of a level's launches (the k_hist instantiation for_hist_kernel picks).
int hist_layout(const HistLevel& hl, bool hess) {
  const bool multi = hl.passes > 1;
  if (hess) return multi ? YGG_HIST_LAYOUT_SHARED_HESS_MULTI : YGG_HIST_LAYOUT_SHARED_HESS;
  if (hl.mode == kHistRootSum) return YGG_HIST_LAYOUT_ROOT_SUM;
  if (hl.mode == kHistPacked) return multi ? YGG_HIST_LAYOUT_PACKED_MULTI : YGG_HIST_LAYOUT_PACKED;
  return multi ? YGG_HIST_LAYOUT_SHARED_MULTI : YGG_HIST_LAYOUT_SHARED;
}

// Histogram capture: sizes the buffers for this handle's level geometry and records the launch configuration of every
// level and the quantiser's float inputs `q` of the tree about to be grown.
int begin_capture(ygg_gbt* h, const QuantParams& q) {
  h->capture_nodes = nullptr;
  h->capture_off.assign(h->num_levels, 0);
  size_t total = 0;
  for (int l = 0; l < h->num_levels; l++) {
    h->capture_off[l] = total;
    total += level_buf(h, level_slot_bound(h, l), l == 0 ? 1 : (2 << (l - 1))).total_u64;
  }
  if (h->d_capture == nullptr || h->capture_u64 < total) {
    YGG_CUDA(cudaStreamSynchronize(h->stream));
    dev_free(h->d_capture);
    h->d_capture = nullptr;
    YGG_RETURN_IF_ERROR(dev_alloc(&h->d_capture, total));
    h->capture_u64 = total;
  }
  const int64_t n_pad = h->ds->n_pad;
  if (h->d_capture_st == nullptr) {
    YGG_RETURN_IF_ERROR(dev_alloc(&h->d_capture_st, 1));
    YGG_RETURN_IF_ERROR(dev_alloc(&h->d_capture_g, n_pad));
    YGG_RETURN_IF_ERROR(dev_alloc(&h->d_capture_h2, n_pad));
    YGG_RETURN_IF_ERROR(dev_alloc(&h->d_capture_sel, n_pad));
  }
  const int64_t n = h->ds->n;
  const float* h2 = q.hist_h != nullptr ? q.hist_h : q.h;
  h->capture_has_h2 = h2 != nullptr;
  h->capture_has_sel = q.selected != nullptr;
  YGG_CUDA(cudaMemcpyAsync(h->d_capture_g, q.g, n * sizeof(float), cudaMemcpyDeviceToDevice, h->stream));
  if (h2 != nullptr) YGG_CUDA(cudaMemcpyAsync(h->d_capture_h2, h2, n * sizeof(float), cudaMemcpyDeviceToDevice, h->stream));
  if (q.selected != nullptr)
    YGG_CUDA(cudaMemcpyAsync(h->d_capture_sel, q.selected, n * sizeof(uint8_t), cudaMemcpyDeviceToDevice, h->stream));
  h->capture_info.assign(h->num_levels, ygg_hist_level_info{});
  const bool hess = hist_hess(h);
  for (int l = 0; l < h->num_levels; l++) {
    ygg_hist_level_info& in = h->capture_info[l];
    const HistLevel& hl = h->hist[l];
    in.layout = hist_layout(hl, hess);
    in.features_per_item = hl.G;
    in.smem_slots = hl.S;
    in.passes = hl.passes;
    in.chunk_blocks = hl.chunk_blocks;
    in.feature_begin = h->hist_f_begin;
    in.num_features = h->hist_f_end - h->hist_f_begin;
    in.has_hsum = hess ? 1 : 0;
    in.h2_pow2 = q.hist_h != nullptr ? q.hist_h_pow2 : q.h_pow2;
    in.n_rows = n;
  }
  return YGG_OK;
}

// Grows one tree on the gradients currently in d_g / d_h (gmax_bits must already be in d_st and the
// iteration scalars reset).  Everything is enqueued on h->stream; no host sync.
//
// Per level: k_hist fills the slot histograms of the level buffer from this rank's rows; in
// row-sharded runs ONE all-reduce (NCCL) sums the buffer over the ranks — the integer histograms
// make that exact and order independent — together with the child statistics the previous
// level's k_partition left in the buffer's tail; k_node_stats, k_scan, k_select_*, k_partition follow.
int grow_tree(ygg_gbt* h, NodeRec* nodes) {
  const ygg_dataset* ds = h->ds;
  const int f_count = h->f_end - h->f_begin;                // features scanned by this rank
  const int hist_f_count = h->hist_f_end - h->hist_f_begin;  // features histogrammed by this rank
  const bool rows_sharded = h->shard_mode == kShardRows;
  const int64_t n_job = sampling(h) ? h->n_selected : (rows_sharded ? h->n_global : ds->n);   // rows the tree is trained on
  const int root_candidate = (n_job >= h->cfg.min_examples && 1 < h->cfg.max_depth) ? 1 : 0;
  if (h->num_levels > 0 && h->hist[0].mode == kHistRootSum) YGG_RETURN_IF_ERROR(ensure_root_counts(h));
  const bool hess = hist_hess(h);
  auto slots_of = [&](int l) { return level_slot_bound(h, l); };
  {
    ProfScope ps(h, "grad");
    // root statistics land in the stats tail of the level-0 buffer
    const LevelBuf lb0 = level_buf(h, h->num_levels > 0 ? slots_of(0) : 0, 1);
    YGG_CUDA(cudaMemsetAsync(lb0.stats, 0, 3 * sizeof(unsigned long long), h->stream));
    QuantParams q{};
    q.n = ds->n; q.n_pad = ds->n_pad; q.g = h->cur_g; q.h = has_h(h) ? h->cur_h : nullptr;
    q.q24 = h->d_q24; q.hq24 = hist_hess(h) ? h->d_hq24 : nullptr;
    q.act = h->d_act; q.act_h = h->d_act_h; q.act_count = h->d_act_count;
    q.node_of_row = h->d_node_of_row; q.st = h->d_st; q.stats = lb0.stats; q.root_candidate = root_candidate;
    q.h_pow2 = h_pow2_of(h);
    // binomial: |g| <= 1 always, so P = 1 needs no reduction over rows (or ranks)
    // (with example weights the rows carry w*g: the scale follows max|w*g| of the iteration)
    q.fixed_g_pow2 = (is_logit(h) && !weighted(h)) ? 1.f : 0.f;
    q.selected = sampling(h) ? h->d_selected : nullptr;
    q.hist_h = weighted(h) ? h->d_weight : nullptr; q.hist_h_pow2 = h->w_pow2;
    k_quantize<<<elementwise_grid(h), 256, 0, h->stream>>>(q);
    h->launches_total++;
    YGG_RETURN_IF_ERROR(check_launch("k_quantize"));
    if (sampling(h)) {   // the root's active lists = the sampled rows
      k_compact_root<<<std::min(h->n_blocks, h->ds->num_sms * 4), kCompactThreads, 0, h->stream>>>(
          h->d_act, hist_hess(h) ? h->d_act_h : nullptr, h->d_act_count, h->d_selected, ds->n, h->n_blocks);
      h->launches_total++;
      YGG_RETURN_IF_ERROR(check_launch("k_compact_root"));
    }
    if (h->num_levels > 0) YGG_RETURN_IF_ERROR(replicate_stats(h, lb0, 1));
    if (h->capture_hist) YGG_RETURN_IF_ERROR(begin_capture(h, q));
  }
  StatsParams sp{};
  sp.levels = h->d_levels; sp.nodes = nodes; sp.st = h->d_st;
  sp.use_hessian = use_hess(h); sp.logit_loss = is_logit(h);
  sp.has_h = has_h(h); sp.shrinkage = h->cfg.shrinkage; sp.clamp = h->cfg.clamp_leaf_logit;
  sp.l1 = h->cfg.l1_regularization; sp.l2 = h->cfg.l2_regularization;
  sp.n_rows = n_job; sp.min_examples = h->cfg.min_examples; sp.max_depth = h->cfg.max_depth;
  sp.subtract_parent = h->cfg.hessian_split_score_subtract_parent; sp.l2_categorical = h->cfg.l2_regularization_categorical;
  sp.weighted = weighted(h) ? 1 : 0;
  auto launch_node_stats = [&](int level, const unsigned long long* stats) -> int {
    ProfScope ps(h, "select");
    sp.level = level;
    sp.stats = stats;
    const int bound = level == 0 ? 1 : (2 << (level - 1));
    if (level == 0) k_node_stats<<<1, 32, 0, h->stream>>>(sp);
    else k_node_stats<<<(bound + 127) / 128, 128, 0, h->stream>>>(sp);
    h->launches_total++;
    return check_launch("k_node_stats");
  };
  if (h->num_levels == 0) {
    const LevelBuf lb0 = level_buf(h, 0, 1);
    if (rows_sharded) YGG_RETURN_IF_ERROR(do_allreduce(h, lb0.stats, 3, 1, 0));
    return launch_node_stats(0, lb0.stats);
  }
  for (int l = 0; l < h->num_levels; l++) {
    const int par = l & 1;
    const int level_nodes_bound = 1 << l;
    const int stats_nodes = l == 0 ? 1 : (2 << (l - 1));   // nodes of this level (children of level l-1)
    const LevelBuf lb = level_buf(h, slots_of(l), stats_nodes);
    {
      static const char* kHistLevelNames[16] = {"hist_L0", "hist_L1", "hist_L2", "hist_L3", "hist_L4", "hist_L5",
                                                "hist_L6", "hist_L7", "hist_L8", "hist_L9", "hist_L10", "hist_L11",
                                                "hist_L12", "hist_L13", "hist_L14", "hist_L15"};
      ProfScope ps(h, "hist");
      ProfScope ps_level(h, kHistLevelNames[l & 15]);
      // zero the histogram planes (not the stats tail, which holds this level's node statistics)
      YGG_RETURN_IF_ERROR(zero_planes(h, lb));
      if (h->hist[l].mode == kHistRootSum) {
        // the root's counts do not depend on the gradients: reuse the precomputed (per-rank) ones,
        // d_root_cnt is [W * f_chunk][256] so that every chunk's count plane is one row of a 2-D copy
        const size_t row = static_cast<size_t>(lb.f_chunk) * kMaxBins * sizeof(uint32_t);
        YGG_CUDA(cudaMemcpy2DAsync(lb.cnt, lb.chunk_u64 * sizeof(unsigned long long), h->d_root_cnt, row, row, lb.W,
                                   cudaMemcpyDeviceToDevice, h->stream));
      }
      const HistLevel& hl = h->hist[l];
      HistParams hp{};
      hp.bins = ds->d_bins; hp.n_pad = ds->n_pad; hp.act = h->d_act; hp.act_h = h->d_act_h; hp.q24 = h->d_q24;
      hp.act_count = h->d_act_count; hp.n_blocks = h->n_blocks;
      hp.f_begin = h->hist_f_begin; hp.f_count = hist_f_count; hp.G = hl.G; hp.S = hl.S;
      hp.chunk_blocks = hl.chunk_blocks;
      hp.level = l; hp.levels = h->d_levels;
      hp.hist_sum = lb.sum; hp.hist_cnt = lb.cnt; hp.hist_hsum = lb.hsum;
      hp.f_chunk = lb.f_chunk; hp.chunk_stride = static_cast<long long>(lb.chunk_u64);
      const int window = hl.S - 1;
      for (int pass = 0; pass < hl.passes; pass++) {
        if (hl.passes > 1) hp.level = l | ((pass * window) << 8) | (window << 20);   // slot window of this pass (HistParams.level)
        YGG_RETURN_IF_ERROR(launch_hist(h, hp, hl));
      }
    }
    if (h->capture_hist)   // this rank's own planes, before any collective
      YGG_CUDA(cudaMemcpyAsync(h->d_capture + h->capture_off[l], h->d_level_buf, lb.total_u64 * sizeof(unsigned long long),
                               cudaMemcpyDeviceToDevice, h->stream));
    // after the collective this rank's statistics of the level sit in `level_stats`
    const unsigned long long* level_stats = lb.stats;
    if (rows_sharded && h->scatter) {
      // chunk r (features [r*f_chunk, (r+1)*f_chunk) + a copy of the node statistics) is reduced onto rank r
      ProfScope ps(h, "allreduce");
      const int rc = h->reducescatter(h->exchange_ctx, h->d_level_buf, static_cast<int64_t>(lb.chunk_u64), 1, 0, h->stream);
      if (rc != 0) return set_error(YGG_ERR_CUDA, "reduce-scatter failed with code %d", rc);
      level_stats = lb.stats + static_cast<size_t>(h->rank) * lb.chunk_u64;
    } else if (rows_sharded) {
      ProfScope ps(h, "allreduce");
      YGG_RETURN_IF_ERROR(do_allreduce(h, h->d_level_buf, static_cast<int64_t>(lb.total_u64), 1, 0));
    }
    YGG_RETURN_IF_ERROR(launch_node_stats(l, level_stats));
    {
      ProfScope ps(h, "scan");
      ScanParams sc{};
      sc.level = l; sc.levels = h->d_levels; sc.families = h->d_fam[par]; sc.nodes = nodes;
      sc.f_begin = h->f_begin; sc.f_count = f_count; sc.hist_f_begin = h->hist_f_begin; sc.hist_f_count = hist_f_count;
      sc.num_bins = ds->d_num_bins; sc.na_bin = ds->d_na_bin; sc.feature_type = ds->d_feature_type;
      sc.cand_mask = h->d_cand_mask; sc.l2_categorical = h->cfg.l2_regularization_categorical;
      sc.slot_sum = lb.sum; sc.slot_cnt = lb.cnt; sc.slot_hsum = lb.hsum;
      sc.f_chunk = lb.f_chunk; sc.chunk_stride = static_cast<long long>(lb.chunk_u64);
      sc.hist_sum = h->d_hist_sum[par]; sc.hist_cnt = h->d_hist_cnt[par]; sc.hist_hsum = h->d_hist_hsum[par];
      sc.phist_sum = h->d_hist_sum[par ^ 1]; sc.phist_cnt = h->d_hist_cnt[par ^ 1]; sc.phist_hsum = h->d_hist_hsum[par ^ 1];
      sc.cand = h->d_cand; sc.st = h->d_st;
      sc.min_num_obs = h->cfg.in_split_min_examples_check ? h->cfg.min_examples : 1;  // training.cc:840-841
      sc.use_hessian = use_hess(h); sc.has_h = has_h(h); sc.subtract_parent = h->cfg.hessian_split_score_subtract_parent;
      sc.l1 = h->cfg.l1_regularization; sc.l2 = h->cfg.l2_regularization;
      sc.write_derived = (l + 1 < h->num_levels) ? 1 : 0;
      sc.bucket_values = ds->d_bucket_values; sc.exact_rule = ds->d_exact_rule;
      sc.weighted = weighted(h) ? 1 : 0;
      sc.w_inv = static_cast<double>(h->w_pow2) / static_cast<double>(1u << kQBits);
      dim3 grid(level_slot_bound(h, l), f_count);
      if (hist_hess(h) || use_hess(h)) k_scan<true><<<grid, 256, 0, h->stream>>>(sc);
      else k_scan<false><<<grid, 256, 0, h->stream>>>(sc);
      h->launches_total++;
      YGG_RETURN_IF_ERROR(check_launch("k_scan"));
    }
    {
      ProfScope ps(h, "select");
      SelectParams sel{};
      sel.level = l; sel.levels = h->d_levels; sel.next_families = h->d_fam[par ^ 1];
      sel.next_slot_node = h->d_slot_node[par ^ 1]; sel.nodes = nodes; sel.cand = h->d_cand;
      sel.f_begin = h->f_begin; sel.f_count = f_count; sel.na_bin = ds->d_na_bin;
      sel.cand_mask = h->d_cand_mask; sel.feature_type = ds->d_feature_type;
      sel.shard_best = h->d_shard_best;
      sel.ties = (h->cfg.candidate_shuffle != 0 && h->world == 1) ? h->d_ties : nullptr;
      sel.bucket_values = ds->d_bucket_values; sel.na_replacement = ds->d_na_replacement;
      const bool exchange_bests = (h->shard_mode == kShardFeatures || h->scatter) && h->world > 1;
      sel.rank = exchange_bests ? h->rank : 0; sel.world = exchange_bests ? h->world : 1;
      sel.max_level_nodes = h->max_level_nodes; sel.min_examples = h->cfg.min_examples;
      sel.max_depth = h->cfg.max_depth; sel.sibling_subtraction = h->cfg.sibling_subtraction;
      sel.max_slots = (l + 1 < h->num_levels) ? level_slot_bound(h, l + 1) : 0x7fffffff;
      sel.st = h->d_st; sel.max_nodes = h->max_nodes;
      const int threads = 256, blocks = (level_nodes_bound + (threads / 32) - 1) / (threads / 32);
      k_select_local<<<blocks, threads, 0, h->stream>>>(sel);
      h->launches_total++;
      YGG_RETURN_IF_ERROR(check_launch("k_select_local"));
      sel.peers = nullptr; sel.epoch = 0;
      if (exchange_bests && h->d_peer_windows != nullptr) {
        sel.peers = h->d_peer_windows;   // k_select_global exchanges the records itself over peer memory
        sel.epoch = ++h->exchange_epoch;
      } else if (exchange_bests) {
        if (h->exchange == nullptr) return set_error(YGG_ERR_INVALID_ARGUMENT, "world > 1 without an exchange function");
        const int64_t bytes = static_cast<int64_t>(h->max_level_nodes) * sizeof(ShardBest);
        // in-place all-gather layout: rank r's block lives at offset r*bytes of d_shard_best
        const int rc = h->exchange(h->exchange_ctx,
                                   reinterpret_cast<const char*>(h->d_shard_best) + static_cast<size_t>(h->rank) * bytes,
                                   h->d_shard_best, bytes, h->stream);
        if (rc != 0) return set_error(YGG_ERR_CUDA, "best-split exchange failed with code %d", rc);
      }
      k_select_global<<<1, 256, 0, h->stream>>>(sel);
      h->launches_total++;
      YGG_RETURN_IF_ERROR(check_launch("k_select_global"));
    }
    // children statistics go to the stats tail of the NEXT level's buffer layout
    const int children_bound = 2 << l;
    const LevelBuf lbn = level_buf(h, l + 1 < h->num_levels ? slots_of(l + 1) : 0, children_bound);
    {
      ProfScope ps(h, "partition");
      YGG_CUDA(cudaMemsetAsync(lbn.stats, 0, static_cast<size_t>(children_bound) * 3 * sizeof(unsigned long long), h->stream));
      PartParams pp{};
      pp.n = ds->n; pp.level = l; pp.levels = h->d_levels; pp.nodes = nodes; pp.bins = ds->d_bins;
      pp.n_pad = ds->n_pad; pp.node_of_row = h->d_node_of_row; pp.n_blocks = h->n_blocks;
      pp.q24 = h->d_q24; pp.hq24 = hist_hess(h) ? h->d_hq24 : nullptr;
      pp.act = h->d_act; pp.act_h = h->d_act_h; pp.act_count = h->d_act_count;
      pp.selected = sampling(h) ? h->d_selected : nullptr;
      pp.g = h->cur_g; pp.h = has_h(h) ? h->cur_h : nullptr; pp.st = h->d_st; pp.stats = lbn.stats;
      // Child-statistic accumulators in shared memory: with few children (top levels) every warp
      // hammers the same 2..16 addresses (same-address ATOMS serialise), so each lane gets its own
      // copy; deeper levels use one shared copy to keep the footprint small and occupancy high.
      pp.smem_children = h->part_smem_children;
      // the kernel picks the accumulator layout from the ACTUAL number of children; it must not pick the
      // lane-private one (32 copies) unless the dynamic shared memory was sized for it
      pp.smem_children_private = children_bound <= 16 ? 16 : 0;
      const size_t smem = children_bound <= 16
                              ? static_cast<size_t>(children_bound) * kPartWords * 32 * sizeof(uint32_t)
                              : std::min(children_bound, h->part_smem_children) * kPartWords * sizeof(uint32_t);
      // one wave of resident CTAs (2 per SM at 64 registers): every CTA gets the same number of 8192-row blocks (+-1)
      const int per_cta = (h->n_blocks + h->ds->num_sms * 2 - 1) / (h->ds->num_sms * 2);
      const bool any_cat = std::any_of(ds->feature_type.begin(), ds->feature_type.end(),
                                       [](int32_t t) { return t == YGG_FEATURE_CATEGORICAL; });
      if (any_cat) k_partition<true><<<(h->n_blocks + per_cta - 1) / per_cta, kPartThreads, smem, h->stream>>>(pp);
      else k_partition<false><<<(h->n_blocks + per_cta - 1) / per_cta, kPartThreads, smem, h->stream>>>(pp);
      h->launches_total++;
      YGG_RETURN_IF_ERROR(check_launch("k_partition"));
      if (l + 1 < h->num_levels) YGG_RETURN_IF_ERROR(replicate_stats(h, lbn, children_bound));
    }
    if (l + 1 == h->num_levels) {
      // last level: its children are leaves; reduce their statistics alone and finish them
      if (rows_sharded) {
        ProfScope ps(h, "allreduce");
        YGG_RETURN_IF_ERROR(do_allreduce(h, lbn.stats, static_cast<int64_t>(children_bound) * 3, 1, 0));
      }
      YGG_RETURN_IF_ERROR(launch_node_stats(l + 1, lbn.stats));
    }
  }
  if (weighted(h)) YGG_RETURN_IF_ERROR(launch_weight_sums(h, nodes));
  if (h->capture_hist) {
    YGG_CUDA(cudaMemcpyAsync(h->d_capture_st, h->d_st, sizeof(DeviceState), cudaMemcpyDeviceToDevice, h->stream));
    h->capture_nodes = nodes;
  }
  if (h->cfg.candidate_shuffle != 0 && h->world == 1) {
    // which of the tied candidates recorded by k_select_local cut their node's rows exactly like the chosen split
    ProfScope ps(h, "select");
    k_verify_ties<<<elementwise_grid(h), 256, 0, h->stream>>>(nodes, h->d_node_of_row, ds->d_bins, ds->n, ds->n_pad);
    h->launches_total++;
    YGG_RETURN_IF_ERROR(check_launch("k_verify_ties"));
  }
  return YGG_OK;
}

__global__ void k_store_loss(const DeviceState* st, LossRec* out) {
  out->loss_sum = st->loss_sum;
  out->correct = st->correct;
}

__global__ void k_fill(float* p, int64_t n, float v) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) p[i] = v;
}

__global__ void k_absmax_to(const float* g, int64_t n, unsigned int* target) {
  float m = 0.f;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) m = fmaxf(m, fabsf(g[i]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(target, __float_as_uint(m));
}
__global__ void k_absmax(const float* g, int64_t n, DeviceState* st) {
  float m = 0.f;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) m = fmaxf(m, fabsf(g[i]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(&st->gmax_bits, __float_as_uint(m));
}

// Runs the pred/grad kernel.  apply: add the pending tree to the predictions and account its loss.
// ---- multinomial log-likelihood (loss_imp_multinomial.cc) --------------------------------------------
// Predictions are K planes [K][n]; the reference keeps them interleaved, the arithmetic per example is the same:
// exp of every class score (float, evaluated as for the binomial loss), sequential float sum in class order.
struct McParams {
  int64_t n, n_pad;
  int K;
  const float* pred;        // [K][n]
  const uint8_t* label;     // class index 0..K-1
  float* g;                 // [K][n_pad] or null
  float* h;
  LossRec* out;             // loss record of the iteration or null
  LossPartials* partials;
  // example weights (WEIGHTED instantiation): loss -= w * log(...), accuracy by weight (loss_imp_multinomial.cc:238-256);
  // the gradient planes receive the float products w*g / w*h, g2w the products (w*g)*g (see GradParams)
  const float* weight;
  float* g2w;               // [K][n_pad]
  float correct_scale;
};
template <bool WEIGHTED>
__global__ void __launch_bounds__(256) k_mc_grad(McParams p) {
  double loss = 0;
  unsigned long long correct = 0;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r < p.n; r += stride) {
    float e[32];
    float sum_exp = 0.f;
    int predicted = -1;
    float predicted_exp = 0.f;
    const int label = p.label[r];
    for (int k = 0; k < p.K; k++) {
      const float v = exp_rn(p.pred[static_cast<int64_t>(k) * p.n + r]);
      e[k] = v;
      sum_exp += v;
      if (v > predicted_exp) { predicted_exp = v; predicted = k; }   // TemplatedLossImp :258-265
    }
    float w = 1.f;
    if (WEIGHTED) w = p.weight[r];
    if (p.out != nullptr) {
      const float term = log_rn(e[label] / sum_exp);                  // :268-272
      loss -= WEIGHTED ? w * term : term;
      if (predicted == label) correct += WEIGHTED ? static_cast<unsigned long long>(__float2ull_rn(w * p.correct_scale)) : 1ull;
    }
    if (p.g != nullptr) {
      const float normalization = 1.f / sum_exp;                      // TemplatedUpdateGradients :163-189
      for (int k = 0; k < p.K; k++) {
        const float grad = (label == k ? 1.f : 0.f) - e[k] * normalization;
        const float a = fabsf(grad);
        if (WEIGHTED) {
          const float wg = grad * w;
          p.g[static_cast<int64_t>(k) * p.n_pad + r] = wg;
          p.h[static_cast<int64_t>(k) * p.n_pad + r] = w * (a * (1 - a));
          p.g2w[static_cast<int64_t>(k) * p.n_pad + r] = wg * grad;
        } else {
          p.g[static_cast<int64_t>(k) * p.n_pad + r] = grad;
          p.h[static_cast<int64_t>(k) * p.n_pad + r] = a * (1 - a);
        }
      }
    }
  }
  if (p.out == nullptr) return;
  loss = warp_sum_f64(loss);
  correct = warp_sum_u64(correct);
  __shared__ double s_loss[8];
  __shared__ unsigned long long s_cor[8];
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) { s_loss[w] = loss; s_cor[w] = correct; }
  __syncthreads();
  if (threadIdx.x == 0)
    for (int i = 1; i < 8; i++) { loss += s_loss[i]; correct += s_cor[i]; }
  reduce_loss_in_order(p.partials, loss, correct, &p.out->loss_sum, &p.out->correct);
}

// UpdatePredictions for the tree just grown: the leaf of a training row is its final node id.
__global__ void __launch_bounds__(256) k_apply_leaves(float* __restrict__ pred, const uint16_t* __restrict__ node_of_row,
                                                      const NodeRec* __restrict__ tree, int64_t n) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r < n; r += stride)
    pred[r] += tree[node_of_row[r]].leaf_value;
}

// Validation rows: UpdatePredictions on the held-out rows by tree traversal (loss_utils.cc:214-229,
// gradient_boosted_trees.cc:1556-1566) fused with the validation loss of the iteration
// (:1610-1626; loss_imp_binomial.cc:204-234, metric/metric.cc:2173-2199).
template <int LOSS>
__global__ void __launch_bounds__(256) k_valid_update(const uint8_t* __restrict__ bins, int64_t n, int64_t n_pad,
                                                      const NodeRec* __restrict__ tree, float* __restrict__ pred,
                                                      const uint8_t* __restrict__ label_u8,
                                                      const float* __restrict__ label_f32, LossRec* out, LossPartials* partials,
                                                      const float* __restrict__ weight, float correct_scale) {
  double loss = 0;
  unsigned long long correct = 0;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r < n; r += stride) {
    int node = 0;
    while (true) {
      const int f = tree[node].feature;
      if (f < 0) break;
      const uint32_t b = bins[static_cast<int64_t>(f) * n_pad + r];
      const bool pos = tree[node].cond_type == 1 ? ((tree[node].mask[b >> 5] >> (b & 31)) & 1u) != 0
                                                 : static_cast<int>(b) >= tree[node].thr;
      node = pos ? tree[node].pos_child : tree[node].neg_child;
    }
    const float p = pred[r] + tree[node].leaf_value;
    pred[r] = p;
    if (LOSS == 2) continue;  // multinomial: the loss needs all K planes (k_mc_grad after the K-th tree)
    if (LOSS == 0) {
      const float label = label_u8[r] ? 1.f : 0.f;
      const float inner = label * p - log_rn(1.f + exp_rn(p));
      const bool hit = (p > 0.f) == (label_u8[r] != 0);
      if (weight != nullptr) {   // loss_imp_binomial.cc:218-224
        const float w = weight[r];
        loss -= 2 * w * inner;
        if (hit) correct += static_cast<unsigned long long>(__float2ull_rn(w * correct_scale));
      } else {
        loss -= 2 * inner;
        correct += hit ? 1ull : 0ull;
      }
    } else {
      const float d = label_f32[r] - p;
      loss += weight != nullptr ? weight[r] * d * d : d * d;   // metric/metric.cc:2097-2115
    }
  }
  if (LOSS == 2) return;
  loss = warp_sum_f64(loss);
  correct = warp_sum_u64(correct);
  __shared__ double s_loss[8];
  __shared__ unsigned long long s_cor[8];
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) { s_loss[w] = loss; s_cor[w] = correct; }
  __syncthreads();
  if (threadIdx.x == 0)
    for (int i = 1; i < 8; i++) { loss += s_loss[i]; correct += s_cor[i]; }
  reduce_loss_in_order(partials, loss, correct, &out->loss_sum, &out->correct);
}

// Raw scores of the model's first `n_trees` trees on any dataset with the training dataset's features (ComputePredictions,
// gradient_boosted_trees.cc:2872-2930: the predictions a resumed training starts from): initial prediction + the leaves
// reached in every tree of the row's class plane.  One thread per row, trees in order (float sums in the reference's order).
__global__ void __launch_bounds__(256) k_predict(const uint8_t* __restrict__ bins, int64_t n, int64_t n_pad, const NodeRec* __restrict__ trees,
                                                int max_nodes, int n_trees, int K, float initial, float* __restrict__ out /*[K][n]*/) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r < n; r += stride) {
    for (int k = 0; k < K; k++) {
      float acc = initial;
      for (int t = k; t < n_trees; t += K) {
        const NodeRec* tree = trees + static_cast<size_t>(t) * max_nodes;
        int node = 0;
        while (true) {
          const int f = tree[node].feature;
          if (f < 0) break;
          const uint32_t b = bins[static_cast<int64_t>(f) * n_pad + r];
          const bool pos = tree[node].cond_type == 1 ? ((tree[node].mask[b >> 5] >> (b & 31)) & 1u) != 0
                                                     : static_cast<int>(b) >= tree[node].thr;
          node = pos ? tree[node].pos_child : tree[node].neg_child;
        }
        acc += tree[node].leaf_value;
      }
      out[static_cast<int64_t>(k) * n + r] = acc;
    }
  }
}

// `tree_idx`: the tree just grown; `plane`: its class (0 unless multinomial).
int launch_valid_update(ygg_gbt* h, int tree_idx, int plane = 0) {
  if (h->vds == nullptr) return YGG_OK;
  ProfScope ps(h, "validation");
  const NodeRec* tree = h->d_nodes_all + static_cast<size_t>(tree_idx) * h->max_nodes;
  const int64_t nv = h->vds->n;
  const int grid = static_cast<int>(std::min<int64_t>((nv + 255) / 256, static_cast<int64_t>(h->ds->num_sms) * 8));
  if (is_multinomial(h)) {
    k_valid_update<2><<<grid, 256, 0, h->stream>>>(h->vds->d_bins, nv, h->vds->n_pad, tree, h->d_vpred + static_cast<int64_t>(plane) * nv,
                                                   nullptr, nullptr, nullptr, nullptr, nullptr, 0.f);
    h->launches_total++;
    YGG_RETURN_IF_ERROR(check_launch("k_valid_update"));
    if (plane + 1 == h->K) {  // all K trees of the iteration applied: validation loss of the iteration
      McParams p{};
      p.n = nv; p.n_pad = nv; p.K = h->K; p.pred = h->d_vpred; p.label = h->d_vlabel_u8; p.out = h->d_vloss + h->iters_done;
      p.partials = h->d_loss_partials;
      p.weight = h->d_vweight; p.correct_scale = h->v_correct_scale;
      if (h->d_vweight != nullptr) k_mc_grad<true><<<grid, 256, 0, h->stream>>>(p);
      else k_mc_grad<false><<<grid, 256, 0, h->stream>>>(p);
      h->launches_total++;
      YGG_RETURN_IF_ERROR(check_launch("k_mc_grad"));
    }
    return YGG_OK;
  }
  if (h->cfg.loss == YGG_LOSS_BINOMIAL_LOG_LIKELIHOOD)
    k_valid_update<0><<<grid, 256, 0, h->stream>>>(h->vds->d_bins, nv, h->vds->n_pad, tree, h->d_vpred, h->d_vlabel_u8,
                                                   h->d_vlabel_f32, h->d_vloss + h->iters_done, h->d_loss_partials,
                                                   h->d_vweight, h->v_correct_scale);
  else
    k_valid_update<1><<<grid, 256, 0, h->stream>>>(h->vds->d_bins, nv, h->vds->n_pad, tree, h->d_vpred, h->d_vlabel_u8,
                                                   h->d_vlabel_f32, h->d_vloss + h->iters_done, h->d_loss_partials,
                                                   h->d_vweight, h->v_correct_scale);
  h->launches_total++;
  return check_launch("k_valid_update");
}

// `n`: rows, or the weight sum of a weighted set; `correct_scale`: units of rec.correct per unit of weight (1: rows).
float loss_value(const ygg_gbt* h, const LossRec& rec, double n, float* secondary, double correct_scale = 1.0) {
  if (is_logit(h)) {  // multinomial: sum_loss / n and accuracy (loss_imp_multinomial.cc:336-341)
    *secondary = static_cast<float>(static_cast<double>(rec.correct) / correct_scale / n);
    return static_cast<float>(rec.loss_sum / n);  // loss_imp_binomial.cc:289-291
  }
  const float v = static_cast<float>(std::sqrt(rec.loss_sum / n));  // metric/metric.cc:2164
  *secondary = v;
  return v;
}

float validation_loss_value(const ygg_gbt* h, const LossRec& rec, float* secondary) {
  if (h->d_vweight != nullptr) return loss_value(h, rec, h->v_sum_weights, secondary, h->v_correct_scale);
  return loss_value(h, rec, static_cast<double>(h->vds->n), secondary);
}

// EarlyStopping::Update / ShouldStop (early_stopping/early_stopping.cc:30-62), one tree per iteration.
struct EarlyStoppingState {
  float best_loss = 0.f, last_loss = 0.f;
  int best_num_trees = -1, last_num_trees = 0;
  int look_ahead = 30, initial_iteration = 10;
  void update(float validation_loss, int num_trees, int iter) {
    if (iter >= initial_iteration && (best_num_trees == -1 || validation_loss < best_loss)) {
      best_loss = validation_loss;
      best_num_trees = num_trees;
    }
    last_loss = validation_loss;
    last_num_trees = num_trees;
  }
  bool should_stop(int iter) const { return iter >= initial_iteration && last_num_trees - best_num_trees >= look_ahead; }
};

int launch_mc(ygg_gbt* h, bool with_loss, bool with_grad) {
  ProfScope ps(h, "grad");
  McParams p{};
  p.n = h->ds->n; p.n_pad = h->ds->n_pad; p.K = h->K; p.pred = h->d_pred; p.label = h->d_label_u8;
  p.g = with_grad ? h->d_g : nullptr; p.h = with_grad ? h->d_h : nullptr;
  p.out = with_loss ? h->d_loss + (h->iters_done - 1) : nullptr;
  p.partials = h->d_loss_partials;
  p.weight = h->d_weight; p.g2w = h->d_g2w; p.correct_scale = correct_scale_of(h->w_pow2);
  if (user_weighted(h)) k_mc_grad<true><<<elementwise_grid(h), 256, 0, h->stream>>>(p);
  else k_mc_grad<false><<<elementwise_grid(h), 256, 0, h->stream>>>(p);
  h->launches_total++;
  return check_launch("k_mc_grad");
}

int launch_pred_grad(ygg_gbt* h, bool apply, bool compute_grad) {
  ProfScope ps(h, "grad");
  GradParams g{};
  g.n = h->ds->n; g.pred = h->d_pred; g.label_u8 = h->d_label_u8; g.label_f32 = h->d_label_f32;
  g.node_of_row = h->d_node_of_row;
  g.pending_tree = apply ? h->d_nodes_all + static_cast<size_t>(h->trees_done - 1) * h->max_nodes : nullptr;
  g.g = h->d_g; g.h = h->d_h; g.st = h->d_st; g.compute_grad = compute_grad ? 1 : 0;
  g.partials = h->d_loss_partials;
  g.weight = h->d_weight; g.g2w = h->d_g2w; g.correct_scale = correct_scale_of(h->w_pow2);
  if (apply) { k_reset_loss<<<1, 1, 0, h->stream>>>(h->d_st); h->launches_total++; }
  const bool binomial = h->cfg.loss == YGG_LOSS_BINOMIAL_LOG_LIKELIHOOD;
  if (user_weighted(h)) {
    if (binomial) k_pred_grad<0, true><<<elementwise_grid(h), 256, 0, h->stream>>>(g);
    else k_pred_grad<1, true><<<elementwise_grid(h), 256, 0, h->stream>>>(g);
  } else if (binomial) k_pred_grad<0><<<elementwise_grid(h), 256, 0, h->stream>>>(g);
  else k_pred_grad<1><<<elementwise_grid(h), 256, 0, h->stream>>>(g);
  h->launches_total++;
  YGG_RETURN_IF_ERROR(check_launch("k_pred_grad"));
  if (apply) { k_store_loss<<<1, 1, 0, h->stream>>>(h->d_st, h->d_loss + (h->trees_done - 1)); h->launches_total++; }
  return YGG_OK;
}

// Row-sharded runs: the per-tree loss records hold this rank's rows only; sum the records that have
// not been reduced yet over the ranks.  A LossRec is {double, u64}: the two columns are reduced
// through a strided copy into two dense arrays.  Every rank must call this collectively.
__global__ void k_loss_split(const LossRec* rec, int n, double* a, unsigned long long* b) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) { a[i] = rec[i].loss_sum; b[i] = rec[i].correct; }
}
__global__ void k_loss_merge(LossRec* rec, int n, const double* a, const unsigned long long* b) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) { rec[i].loss_sum = a[i]; rec[i].correct = b[i]; }
}
int reduce_losses(ygg_gbt* h) {
  if (h->shard_mode != kShardRows) return YGG_OK;
  const int first = h->loss_reduced_upto, n = h->iters_done - first;
  if (n <= 0) return YGG_OK;
  double* a = reinterpret_cast<double*>(h->d_level_buf);
  unsigned long long* b = h->d_level_buf + n;
  if (static_cast<size_t>(2 * n) * 8 > h->level_buf_bytes) return set_error(YGG_ERR_INVALID_ARGUMENT, "too many unreduced loss records");
  k_loss_split<<<(n + 127) / 128, 128, 0, h->stream>>>(h->d_loss + first, n, a, b);
  YGG_RETURN_IF_ERROR(do_allreduce(h, a, n, 2, 0));
  YGG_RETURN_IF_ERROR(do_allreduce(h, b, n, 1, 0));
  k_loss_merge<<<(n + 127) / 128, 128, 0, h->stream>>>(h->d_loss + first, n, a, b);
  YGG_RETURN_IF_ERROR(check_launch("k_loss_merge"));
  h->loss_reduced_upto = h->iters_done;
  return YGG_OK;
}

int apply_pending(ygg_gbt* h) {
  if (is_multinomial(h)) {  // the trees are already in the predictions; only the loss of the iteration is due
    if (!h->pending_loss) return YGG_OK;
    YGG_RETURN_IF_ERROR(launch_mc(h, true, false));
    h->pending_loss = false;
    return YGG_OK;
  }
  if (!h->pending) return YGG_OK;
  YGG_RETURN_IF_ERROR(launch_pred_grad(h, true, false));
  h->pending = false;
  return YGG_OK;
}

int check_device_error(ygg_gbt* h) {
  DeviceState st;
  YGG_CUDA(cudaMemcpyAsync(&st, h->d_st, sizeof(st), cudaMemcpyDeviceToHost, h->stream));
  YGG_CUDA(cudaStreamSynchronize(h->stream));
  if (st.error_flag != 0) return set_error(YGG_ERR_CUDA, "device invariant violated (code %d)", st.error_flag);
  return YGG_OK;
}

// libc++'s std::shuffle (llvm libcxx/include/__algorithm/shuffle.h): for every position but the last, draw i in [0, d]
// with its uniform_int_distribution — the low w bits of one engine word, redrawn while > d (w = bits of d + 1) — and
// swap.  The reference's golden models were built against libc++ (DESIGN.md §6); libstdc++'s differs.
void shuffle_libcxx(std::vector<int32_t>* v, std::mt19937* g) {
  const int64_t n = static_cast<int64_t>(v->size());
  int64_t d = n - 1;
  for (int64_t first = 0; first < n - 1; ++first, --d) {
    const uint64_t rp = static_cast<uint64_t>(d) + 1;
    int w = 63 - __builtin_clzll(rp);
    if (rp & ((1ull << w) - 1)) ++w;
    uint32_t u;
    do { u = (*g)() & static_cast<uint32_t>((1ull << w) - 1); } while (u >= rp);
    if (u != 0) std::swap((*v)[first], (*v)[first + u]);
  }
}

// Tie-break replay (cfg.candidate_shuffle != 0).  The reference decides between features whose best splits have equal
// float scores by the order of its per-node shuffle of the candidate features (training.cc:4293-4306, consumed at
// :1658 / :1781), drawn from the learner's engine while it visits the nodes depth-first, positive child first.  The
// k-th node that reaches FindBestCondition takes the k-th shuffle of the stream whatever the data are, so the stream
// can be replayed on FINISHED trees: the level-wise engine grows them with the lowest-index tie-break, records up to
// kMaxTieAlts tied candidates per split (k_select_local), and this pass gives every tied node the candidate the
// reference would have taken — a rename when the two candidates cut the node's rows identically (twin features: equal
// score and equal positive count), counted as unresolved otherwise (the subtree would have to be regrown).
void ensure_tie_rng(ygg_gbt* h) {
  if (h->tie_rng_ready) return;
  h->tie_rng.seed(h->cfg.random_seed);   // utils::RandomEngine random(config.random_seed()), gradient_boosted_trees.cc:1198
  h->tie_rng.discard(h->cfg.rng_words_consumed);
  h->tie_rng_ready = true;
}

// One finished tree (host copy of its node table), the handle's stream positioned where the reference's engine
// was when it started that tree.  Returns true if a node was renamed.
bool resolve_tree_on_host(ygg_gbt* h, NodeRec* tree) {
  const int F = h->ds->F;
  std::vector<int32_t> perm(F), rank_of(F);
  std::vector<int> stack(1, 0);
  bool changed = false;
  while (!stack.empty()) {
    NodeRec& nd = tree[stack.back()];
    stack.pop_back();
    if (!nd.candidate) continue;                       // NodeTrain returned before FindBestCondition (training.cc:4909-4914)
    for (int f = 0; f < F; f++) perm[f] = f;
    if (h->cfg.candidate_shuffle == 2) shuffle_libcxx(&perm, &h->tie_rng);
    else std::shuffle(perm.begin(), perm.end(), h->tie_rng);
    if (h->cfg.split_jobs_draw_seeds) h->tie_rng.discard(F);   // one seed per feature job (training.cc:1658)
    if (nd.feature < 0) continue;
    if (nd.tie_count > 0) {
      for (int i = 0; i < F; i++) rank_of[perm[i]] = i;
      int best = -1, best_rank = rank_of[nd.feature];
      for (int i = 0; i < std::min(nd.tie_count, kMaxTieAlts); i++)
        if (rank_of[nd.tie[i].feature] < best_rank) { best_rank = rank_of[nd.tie[i].feature]; best = i; }
      if (nd.tie_count > kMaxTieAlts) {
        h->ties_unresolved++;                          // more ties than recorded: the first in the shuffle may be unknown
      } else if (best >= 0) {
        const TieAlt a = nd.tie[best];
        if (a.n_pos == nd.n_pos) {
          // keep the old choice among the alternatives, so that the record stays complete
          TieAlt old{};
          old.feature = nd.feature; old.thr = nd.thr; old.n_pos = static_cast<int32_t>(nd.n_pos); old.cond_type = nd.cond_type;
          old.na_value = nd.na_value; old.thr_value = nd.thr_value;
          std::memcpy(old.mask, nd.mask, sizeof(old.mask));
          nd.feature = a.feature; nd.thr = a.thr; nd.cond_type = a.cond_type; nd.na_value = a.na_value; nd.thr_value = a.thr_value;
          std::memcpy(nd.mask, a.mask, sizeof(nd.mask));
          nd.tie[best] = old;
          h->ties_renamed++;
          changed = true;
        } else {
          h->ties_unresolved++;
        }
      }
    }
    stack.push_back(nd.neg_child);                     // positive child first (training.cc:5031-5046)
    stack.push_back(nd.pos_child);
  }
  return changed;
}

int resolve_ties(ygg_gbt* h, int upto) {
  if (h->cfg.candidate_shuffle == 0 || upto <= h->ties_resolved_upto) return YGG_OK;
  ensure_tie_rng(h);
  const int first = h->ties_resolved_upto, count = upto - first;
  std::vector<NodeRec> nodes(static_cast<size_t>(count) * h->max_nodes);
  YGG_CUDA(cudaMemcpyAsync(nodes.data(), h->d_nodes_all + static_cast<size_t>(first) * h->max_nodes,
                           nodes.size() * sizeof(NodeRec), cudaMemcpyDeviceToHost, h->stream));
  YGG_CUDA(cudaStreamSynchronize(h->stream));
  for (int t = 0; t < count; t++) {
    NodeRec* tree = nodes.data() + static_cast<size_t>(t) * h->max_nodes;
    if (resolve_tree_on_host(h, tree))
      YGG_CUDA(cudaMemcpyAsync(h->d_nodes_all + static_cast<size_t>(first + t) * h->max_nodes, tree, sizeof(NodeRec) * h->max_nodes,
                               cudaMemcpyHostToDevice, h->stream));
  }
  YGG_CUDA(cudaStreamSynchronize(h->stream));
  h->ties_resolved_upto = upto;
  return YGG_OK;
}

// SampleTrainingExamples (gradient_boosted_trees.cc:2932-2956): stochastic gradient boosting.  One word of the learner's
// engine per row (std::uniform_real_distribution<float>, the same library call as the reference), drawn at the start of
// the iteration — after the candidate shuffles of the previous iteration's trees, which is why the tie-break replay of
// those trees has to be done first when it is on.  The row is in the sample iff the draw is < subsample; an empty sample
// gets one row drawn uniformly.  The draw runs on the host (the stream is sequential): ~3 ns per row.
int draw_sample(ygg_gbt* h) {
  if (h->shard_mode != kShardNone) return set_error(YGG_ERR_UNIMPLEMENTED, "subsample < 1 is not combined with sharding");
  if (h->cfg.candidate_shuffle != 0) YGG_RETURN_IF_ERROR(resolve_ties(h, h->trees_done));
  ensure_tie_rng(h);
  const int64_t n = h->ds->n;
  h->host_selected.resize(n);
  std::uniform_real_distribution<float> unif_dist_unit;
  int64_t count = 0;
  uint8_t* sel = h->host_selected.data();
  for (int64_t r = 0; r < n; r++) {
    const uint8_t in = unif_dist_unit(h->tie_rng) < h->cfg.subsample ? 1 : 0;
    sel[r] = in;
    count += in;
  }
  if (count == 0) {   // at least one example
    sel[std::uniform_int_distribution<uint32_t>(0u, static_cast<uint32_t>(n - 1))(h->tie_rng)] = 1;
    count = 1;
  }
  YGG_CUDA(cudaMemcpyAsync(h->d_selected, sel, n, cudaMemcpyHostToDevice, h->stream));
  h->n_selected = count;
  return YGG_OK;
}

// Gradient-based one-side sampling, host part (before the iteration is enqueued): the draws of the rows outside the top
// alpha fraction — one engine word each, consumed in sorted order whatever the rows turn out to be — and with them the
// size of the sample.  Same place in the learner's stream as SampleTrainingExamples' draws (draw_sample).
int draw_goss(ygg_gbt* h) {
  if (h->shard_mode != kShardNone) return set_error(YGG_ERR_UNIMPLEMENTED, "GOSS is not combined with sharding");
  if (h->cfg.candidate_shuffle != 0) YGG_RETURN_IF_ERROR(resolve_ties(h, h->trees_done));
  ensure_tie_rng(h);
  const int64_t n = h->ds->n;
  const float alpha = h->cfg.goss_alpha, beta = h->cfg.goss_beta;
  // int cutoff = std::ceil(alpha * num_rows): float times UnsignedExampleIdx (gradient_boosted_trees.cc:2983)
  int64_t cutoff = static_cast<int64_t>(std::ceil(alpha * static_cast<float>(static_cast<uint32_t>(n))));
  cutoff = std::min(cutoff, n);
  int64_t count = cutoff;
  const int64_t m = beta > 0.f ? n - cutoff : 0;
  h->host_goss_u.resize(std::max<int64_t>(m, 1));
  std::uniform_real_distribution<float> unif_dist_unit;
  for (int64_t j = 0; j < m; j++) {
    const float u = unif_dist_unit(h->tie_rng);
    h->host_goss_u[j] = u;
    count += u < beta ? 1 : 0;
  }
  if (count == 0) {
    // "at least one example" draws a row uniformly; with no row kept by rank or by draw (alpha = 0 and an unlucky tail)
    // the tree would be trained on that one row.  Not reproduced: refuse rather than diverge silently.
    return set_error(YGG_ERR_UNIMPLEMENTED, "GOSS selected no row in this iteration (goss_alpha = 0 and no tail row drawn)");
  }
  if (m > 0) YGG_CUDA(cudaMemcpyAsync(h->d_goss_u, h->host_goss_u.data(), m * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  h->goss_cutoff = cutoff;
  h->n_selected = count;
  return YGG_OK;
}

// Device part, after the iteration's unit gradients are in d_g / d_h: order the rows by decreasing |g| (stable: equal keys
// by row index), mark the sample and its weights, and turn g / h into the weighted products the tree trainer sums.
int apply_goss(ygg_gbt* h) {
  ProfScope ps(h, "grad");
  const int64_t n = h->ds->n;
  const int grid = elementwise_grid(h);
  k_goss_keys<<<grid, 256, 0, h->stream>>>(h->d_g, n, h->d_goss_keys[0], h->d_goss_rows[0]);
  YGG_CUDA(cub::DeviceRadixSort::SortPairsDescending(h->d_goss_temp, h->goss_temp_bytes, h->d_goss_keys[0], h->d_goss_keys[1],
                                                    h->d_goss_rows[0], h->d_goss_rows[1], static_cast<int>(n), 0, 32, h->stream));
  const float amplification = h->cfg.goss_beta > 0.f ? (1.f - h->cfg.goss_alpha) / h->cfg.goss_beta : 1.f;
  k_goss_apply<<<grid, 256, 0, h->stream>>>(h->d_goss_rows[1], h->d_goss_u, n, h->goss_cutoff, h->cfg.goss_beta, amplification,
                                            h->d_selected, h->d_weight);
  DeviceState* st = h->d_st;
  YGG_CUDA(cudaMemsetAsync(&st->gmax_bits, 0, sizeof(unsigned int), h->stream));   // now: max |w*g|
  k_apply_weights<<<grid, 256, 0, h->stream>>>(n, h->d_g, h->d_h, is_logit(h) ? 0 : 1, h->d_weight, h->d_g2w, h->d_st);
  h->launches_total += 5;
  return check_launch("k_apply_weights");
}

// growing_strategy = BEST_FIRST_GLOBAL (GrowTreeBestFirstGlobal, training.cc:4499-4656).  The reference keeps a max-heap of
// candidate splits keyed by split_score * num_examples (float), splits the best one, ingests its children (positive first: leaf
// value + FindBestCondition), until max_num_nodes leaves exist.  A node's best split does not depend on when it is found, so the
// result is a SUBTREE of the tree grown to the depth limit: the engine grows that tree level-wise as usual and replays the heap on
// it — same container, same push order as the reference — turning the splits the heap never reached into leaves.  The rows below
// such a leaf keep their deep node ids; their nodes take the leaf's value, so that the prediction update needs no other change.
int best_first_prune(ygg_gbt* h, NodeRec* d_tree) {
  std::vector<NodeRec> tree(h->max_nodes);
  YGG_CUDA(cudaMemcpyAsync(tree.data(), d_tree, sizeof(NodeRec) * h->max_nodes, cudaMemcpyDeviceToHost, h->stream));
  YGG_CUDA(cudaStreamSynchronize(h->stream));
  struct Cand {
    float key; int node;
    bool operator<(const Cand& o) const { return key < o.key; }
  };
  std::priority_queue<Cand> heap;
  std::vector<char> keep(h->max_nodes, 0);
  auto ingest = [&](int node) {
    const NodeRec& nd = tree[node];
    if (nd.feature >= 0) heap.push({nd.score * static_cast<float>(nd.n), node});
  };
  ingest(0);
  int leaves = 1;
  const int limit = h->cfg.max_num_nodes;
  while (!heap.empty() && (limit < 0 || leaves < limit)) {
    while (limit >= 0 && static_cast<int>(heap.size()) > limit) heap.pop();   // (:4571-4575)
    const Cand c = heap.top();
    heap.pop();
    keep[c.node] = 1;
    ingest(tree[c.node].pos_child);
    ingest(tree[c.node].neg_child);
    leaves++;
  }
  // splits never taken become leaves; everything below them answers with their value
  std::vector<int> stack(1, 0);
  while (!stack.empty()) {
    const int node = stack.back();
    stack.pop_back();
    NodeRec& nd = tree[node];
    if (nd.feature < 0) continue;
    if (keep[node]) { stack.push_back(nd.neg_child); stack.push_back(nd.pos_child); continue; }
    std::vector<int> below = {nd.pos_child, nd.neg_child};
    while (!below.empty()) {
      const int d = below.back();
      below.pop_back();
      if (tree[d].feature >= 0) { below.push_back(tree[d].pos_child); below.push_back(tree[d].neg_child); }
      tree[d].leaf_value = nd.leaf_value;
    }
    nd.feature = -1;
    nd.tie_count = 0;
  }
  YGG_CUDA(cudaMemcpyAsync(d_tree, tree.data(), sizeof(NodeRec) * h->max_nodes, cudaMemcpyHostToDevice, h->stream));
  YGG_CUDA(cudaStreamSynchronize(h->stream));
  return YGG_OK;
}

// Position of every node id in preorder()'s output (-1: not in the tree).
void preorder_positions(const std::vector<NodeRec>& nodes, int idx, int* next, std::vector<int>* pos) {
  (*pos)[idx] = (*next)++;
  if (nodes[idx].feature < 0) return;
  preorder_positions(nodes, nodes[idx].neg_child, next, pos);
  preorder_positions(nodes, nodes[idx].pos_child, next, pos);
}

void preorder(const std::vector<NodeRec>& nodes, int idx, std::vector<ygg_node>* out) {
  const NodeRec& n = nodes[idx];
  const int my = static_cast<int>(out->size());
  out->emplace_back();
  ygg_node o;
  std::memset(&o, 0, sizeof(o));
  const bool leaf = n.feature < 0;
  o.feature = leaf ? -1 : n.feature;
  o.threshold_bin = leaf ? 0 : n.thr;
  o.na_value = leaf ? 0 : n.na_value;
  o.depth = n.depth;
  o.neg_child = o.pos_child = -1;
  o.split_score = leaf ? 0.f : n.score;
  o.leaf_value = n.leaf_value;
  o.num_examples = n.n;
  o.num_pos_examples = leaf ? 0 : n.n_pos;
  o.stat[0] = n.stat[0]; o.stat[1] = n.stat[1]; o.stat[2] = n.stat[2];
  o.threshold_value = leaf ? std::numeric_limits<float>::quiet_NaN() : n.thr_value;
  if (!leaf && n.cond_type == YGG_FEATURE_CATEGORICAL) {
    o.condition_type = YGG_FEATURE_CATEGORICAL;
    o.threshold_bin = 0;
    for (int i = 0; i < 8; i++) o.cat_mask[i] = n.mask[i];
  }
  if (!leaf) {
    o.neg_child = static_cast<int>(out->size());
    preorder(nodes, n.neg_child, out);
    o.pos_child = static_cast<int>(out->size());
    preorder(nodes, n.pos_child, out);
  }
  (*out)[my] = o;
}

// resolve: the tree is not one of the handle's own (ygg_tree_train_on_gradients): break its ties here, with the
// handle's stream where it stands.
int fetch_tree(ygg_gbt* h, const NodeRec* d_nodes, std::vector<ygg_node>* out, bool resolve = false) {
  // The node count of a finished tree: walk from the root (children ids are < max_nodes).
  std::vector<NodeRec> nodes(h->max_nodes);
  YGG_CUDA(cudaMemcpyAsync(nodes.data(), d_nodes, sizeof(NodeRec) * h->max_nodes, cudaMemcpyDeviceToHost, h->stream));
  YGG_CUDA(cudaStreamSynchronize(h->stream));
  if (resolve && h->cfg.candidate_shuffle != 0) {
    ensure_tie_rng(h);
    resolve_tree_on_host(h, nodes.data());
  }
  out->clear();
  preorder(nodes, 0, out);
  return YGG_OK;
}

int require_device() {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    cudaGetLastError();
    return set_error(YGG_ERR_NO_DEVICE, "no CUDA device available: libygg_b200 has no CPU fallback");
  }
  return YGG_OK;
}

}  // namespace

// Allocates the device-resident dataset (bins zeroed, every feature DISCRETIZED_NUMERICAL with one bin);
// the caller fills ds->num_bins / na_bin / feature_type and the bins, then calls _finalize.
int ygg_internal_dataset_alloc(ygg_dataset** out, int64_t n_rows, int32_t n_features, int32_t device) {
  if (n_rows <= 0 || n_features <= 0) return set_error(YGG_ERR_INVALID_ARGUMENT, "empty dataset (%lld rows, %d features)", static_cast<long long>(n_rows), n_features);
  if (n_rows >= (1ll << 31)) return set_error(YGG_ERR_INVALID_ARGUMENT, "at most 2^31-1 rows (UnsignedExampleIdx is 32-bit in the reference)");
  YGG_RETURN_IF_ERROR(require_device());
  YGG_CUDA(cudaSetDevice(device));
  auto* ds = new ygg_dataset();
  ds->device = device;
  ds->n = n_rows;
  ds->n_pad = (n_rows + kBlockRows - 1) / kBlockRows * kBlockRows;
  ds->F = n_features;
  ds->num_bins.assign(n_features, 1);
  ds->na_bin.assign(n_features, 0);
  ds->feature_type.assign(n_features, YGG_FEATURE_DISCRETIZED_NUMERICAL);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { delete ds; return set_error(YGG_ERR_CUDA, "cudaGetDeviceProperties failed"); }
  ds->num_sms = prop.multiProcessorCount;
  const size_t bytes = static_cast<size_t>(ds->n_pad) * n_features;
  int st = dev_alloc(&ds->d_bins, bytes);
  if (st == YGG_OK) st = dev_alloc(&ds->d_num_bins, n_features);
  if (st == YGG_OK) st = dev_alloc(&ds->d_na_bin, n_features);
  if (st == YGG_OK) st = dev_alloc(&ds->d_feature_type, n_features);
  // the columns may be filled from other (non-blocking) streams: the zero fill must have completed
  if (st == YGG_OK && (cudaMemset(ds->d_bins, 0, bytes) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess))
    st = set_error(YGG_ERR_CUDA, "cudaMemset failed");
  if (st != YGG_OK) { ygg_dataset_destroy(ds); return st; }
  *out = ds;
  return YGG_OK;
}

int ygg_internal_dataset_finalize(ygg_dataset* ds) {
  YGG_CUDA(cudaSetDevice(ds->device));
  YGG_CUDA(cudaMemcpy(ds->d_num_bins, ds->num_bins.data(), sizeof(int32_t) * ds->F, cudaMemcpyHostToDevice));
  YGG_CUDA(cudaMemcpy(ds->d_na_bin, ds->na_bin.data(), sizeof(int32_t) * ds->F, cudaMemcpyHostToDevice));
  YGG_CUDA(cudaMemcpy(ds->d_feature_type, ds->feature_type.data(), sizeof(int32_t) * ds->F, cudaMemcpyHostToDevice));
  return YGG_OK;
}

extern "C" {

int ygg_abi_version(void) { return YGG_ABI_VERSION; }
const char* ygg_last_error(void) { return g_last_error.c_str(); }

int ygg_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int ygg_dataset_create(ygg_dataset** out, int64_t n_rows, int32_t n_features, const uint8_t* bins,
                       int64_t column_stride, const int32_t* num_bins, const int32_t* na_bin,
                       int32_t device) {
  if (!out || !bins || !num_bins || !na_bin) return set_error(YGG_ERR_INVALID_ARGUMENT, "null argument");
  if (column_stride < n_rows) return set_error(YGG_ERR_INVALID_ARGUMENT, "column_stride < n_rows");
  for (int f = 0; f < n_features; f++) {
    if (num_bins[f] < 1 || num_bins[f] > kMaxBins)
      return set_error(YGG_ERR_INVALID_ARGUMENT, "feature %d: num_bins=%d outside [1, 256]", f, num_bins[f]);
    if (na_bin[f] < 0 || na_bin[f] >= num_bins[f])
      return set_error(YGG_ERR_INVALID_ARGUMENT, "feature %d: na_bin=%d outside [0, num_bins)", f, na_bin[f]);
  }
  ygg_dataset* ds = nullptr;
  YGG_RETURN_IF_ERROR(ygg_internal_dataset_alloc(&ds, n_rows, n_features, device));
  ds->num_bins.assign(num_bins, num_bins + n_features);
  ds->na_bin.assign(na_bin, na_bin + n_features);
  cudaError_t e = cudaMemcpy2D(ds->d_bins, ds->n_pad, bins, column_stride, n_rows, n_features, cudaMemcpyHostToDevice);
  int st = e == cudaSuccess ? ygg_internal_dataset_finalize(ds)
                            : set_error(YGG_ERR_CUDA, "upload of the bins failed: %s", cudaGetErrorString(e));
  if (st != YGG_OK) {
    ygg_dataset_destroy(ds);
    return st;
  }
  *out = ds;
  return YGG_OK;
}

int ygg_dataset_set_feature_types(ygg_dataset* ds, const int32_t* feature_types, int32_t n_features) {
  if (!ds || !feature_types) return set_error(YGG_ERR_INVALID_ARGUMENT, "null argument");
  if (n_features != ds->F) return set_error(YGG_ERR_INVALID_ARGUMENT, "n_features=%d, dataset has %d", n_features, ds->F);
  for (int f = 0; f < n_features; f++)
    if (feature_types[f] != YGG_FEATURE_DISCRETIZED_NUMERICAL && feature_types[f] != YGG_FEATURE_CATEGORICAL)
      return set_error(YGG_ERR_INVALID_ARGUMENT, "feature %d: unknown feature type %d", f, feature_types[f]);
  YGG_CUDA(cudaSetDevice(ds->device));
  ds->feature_type.assign(feature_types, feature_types + n_features);
  YGG_CUDA(cudaMemcpy(ds->d_feature_type, feature_types, sizeof(int32_t) * n_features, cudaMemcpyHostToDevice));
  return YGG_OK;
}

int ygg_dataset_set_bucket_values(ygg_dataset* ds, int32_t feature, const float* values, int32_t n, float na_replacement) {
  if (!ds || !values) return set_error(YGG_ERR_INVALID_ARGUMENT, "null argument");
  if (feature < 0 || feature >= ds->F) return set_error(YGG_ERR_INVALID_ARGUMENT, "feature %d out of range", feature);
  if (ds->feature_type[feature] != YGG_FEATURE_DISCRETIZED_NUMERICAL) return set_error(YGG_ERR_INVALID_ARGUMENT, "feature %d is not numerical", feature);
  if (n != ds->num_bins[feature]) return set_error(YGG_ERR_INVALID_ARGUMENT, "feature %d has %d bins, %d values given", feature, ds->num_bins[feature], n);
  for (int i = 0; i < n; i++)
    if (!std::isfinite(values[i]) || (i > 0 && !(values[i] > values[i - 1])))
      return set_error(YGG_ERR_INVALID_ARGUMENT, "feature %d: bucket values must be finite and strictly ascending", feature);
  YGG_CUDA(cudaSetDevice(ds->device));
  if (ds->d_bucket_values == nullptr) {
    YGG_RETURN_IF_ERROR(dev_alloc(&ds->d_bucket_values, static_cast<size_t>(ds->F) * kMaxBins));
    YGG_RETURN_IF_ERROR(dev_alloc(&ds->d_exact_rule, ds->F));
    YGG_RETURN_IF_ERROR(dev_alloc(&ds->d_na_replacement, ds->F));
  }
  YGG_CUDA(cudaMemcpy(ds->d_na_replacement + feature, &na_replacement, sizeof(float), cudaMemcpyHostToDevice));
  const int32_t one = 1;
  YGG_CUDA(cudaMemcpy(ds->d_bucket_values + static_cast<size_t>(feature) * kMaxBins, values, sizeof(float) * n, cudaMemcpyHostToDevice));
  YGG_CUDA(cudaMemcpy(ds->d_exact_rule + feature, &one, sizeof(one), cudaMemcpyHostToDevice));
  return YGG_OK;
}

int ygg_dataset_destroy(ygg_dataset* ds) {
  if (!ds) return YGG_OK;
  cudaSetDevice(ds->device);
  dev_free(ds->d_bins);
  dev_free(ds->d_num_bins);
  dev_free(ds->d_na_bin);
  dev_free(ds->d_feature_type);
  dev_free(ds->d_bucket_values);
  dev_free(ds->d_exact_rule);
  dev_free(ds->d_na_replacement);
  delete ds;
  return YGG_OK;
}

int64_t ygg_dataset_num_rows(const ygg_dataset* ds) { return ds ? ds->n : 0; }
int32_t ygg_dataset_num_features(const ygg_dataset* ds) { return ds ? ds->F : 0; }

void ygg_gbt_config_init(ygg_gbt_config* cfg) {
  std::memset(cfg, 0, sizeof(*cfg));
  cfg->abi_version = YGG_ABI_VERSION;
  cfg->loss = YGG_LOSS_BINOMIAL_LOG_LIKELIHOOD;
  cfg->num_trees = 300;
  cfg->shrinkage = 0.1f;
  cfg->max_depth = 6;
  cfg->min_examples = 5;
  cfg->in_split_min_examples_check = 1;
  cfg->use_hessian_gain = 0;
  cfg->l1_regularization = 0.f;
  cfg->l2_regularization = 0.f;
  cfg->l2_regularization_categorical = 1.f;
  cfg->clamp_leaf_logit = 5.f;
  cfg->hessian_split_score_subtract_parent = 0;
  cfg->random_seed = 123456;
  cfg->subsample = 1.f;
  cfg->validation_ratio = 0.f;
  cfg->sibling_subtraction = 1;
  cfg->early_stopping = YGG_EARLY_STOPPING_LOSS_INCREASE;  // gradient_boosted_trees.proto:150-182
  cfg->early_stopping_num_trees_look_ahead = 30;
  cfg->early_stopping_initial_iteration = 10;
  cfg->growing_strategy = 0;
  cfg->max_num_nodes = 31;
}

static int init_handle(ygg_gbt* h);

int ygg_gbt_create(ygg_gbt** out, ygg_dataset* ds, const ygg_gbt_config* cfg) {
  if (!out || !ds || !cfg) return set_error(YGG_ERR_INVALID_ARGUMENT, "null argument");
  if (cfg->abi_version != YGG_ABI_VERSION) return set_error(YGG_ERR_INVALID_ARGUMENT, "abi_version %d != %d", cfg->abi_version, YGG_ABI_VERSION);
  if (cfg->loss != YGG_LOSS_BINOMIAL_LOG_LIKELIHOOD && cfg->loss != YGG_LOSS_SQUARED_ERROR &&
      cfg->loss != YGG_LOSS_MULTINOMIAL_LOG_LIKELIHOOD)
    return set_error(YGG_ERR_UNIMPLEMENTED, "loss %d is outside the hot path (binomial / multinomial log-likelihood and squared error only)", cfg->loss);
  if (cfg->loss == YGG_LOSS_MULTINOMIAL_LOG_LIKELIHOOD && (cfg->num_classes < 2 || cfg->num_classes > 32))
    return set_error(YGG_ERR_INVALID_ARGUMENT, "multinomial loss: num_classes=%d outside [2, 32]", cfg->num_classes);
  if (cfg->growing_strategy != 0 && cfg->growing_strategy != 1) return set_error(YGG_ERR_INVALID_ARGUMENT, "unknown growing_strategy %d", cfg->growing_strategy);
  if (cfg->growing_strategy == 1 && cfg->candidate_shuffle != 0)
    return set_error(YGG_ERR_UNIMPLEMENTED, "the tie-break replay follows the depth-first order of the local growth; not combined with best-first growth");
  if (cfg->growing_strategy == 1 && (cfg->max_num_nodes == 0 || cfg->max_num_nodes < -1)) return set_error(YGG_ERR_INVALID_ARGUMENT, "max_num_nodes=%d", cfg->max_num_nodes);
  if (cfg->candidate_shuffle < 0 || cfg->candidate_shuffle > 2) return set_error(YGG_ERR_INVALID_ARGUMENT, "candidate_shuffle=%d outside {0, 1, 2}", cfg->candidate_shuffle);
  if (!(cfg->subsample > 0.f) || cfg->subsample > 1.f) return set_error(YGG_ERR_INVALID_ARGUMENT, "subsample=%g outside (0, 1]", cfg->subsample);
  if (cfg->early_stopping < 0 || cfg->early_stopping > 2) return set_error(YGG_ERR_INVALID_ARGUMENT, "unknown early_stopping policy %d", cfg->early_stopping);
  if (cfg->early_stopping_num_trees_look_ahead < 1 || cfg->early_stopping_initial_iteration < 0)
    return set_error(YGG_ERR_INVALID_ARGUMENT, "bad early stopping parameters");
  if (cfg->goss_alpha < 0.f || cfg->goss_alpha > 1.f || cfg->goss_beta < 0.f || cfg->goss_beta > 1.f)
    return set_error(YGG_ERR_INVALID_ARGUMENT, "goss_alpha=%g / goss_beta=%g outside [0, 1]", cfg->goss_alpha, cfg->goss_beta);
  if (cfg->goss_alpha > 0.f || cfg->goss_beta > 0.f) {
    if (cfg->subsample < 1.f) return set_error(YGG_ERR_INVALID_ARGUMENT, "GOSS and subsample < 1 are alternative sampling methods");
    if (cfg->use_hessian_gain) return set_error(YGG_ERR_UNIMPLEMENTED, "GOSS trains on weighted rows: variance gain only (use_hessian_gain = 0)");
    if (cfg->loss == YGG_LOSS_MULTINOMIAL_LOG_LIKELIHOOD) return set_error(YGG_ERR_UNIMPLEMENTED, "GOSS is not combined with the multinomial loss");
  }
  if (cfg->max_depth < 1 || cfg->max_depth > 16) return set_error(YGG_ERR_INVALID_ARGUMENT, "max_depth=%d outside [1, 16]", cfg->max_depth);
  if (cfg->num_trees < 1) return set_error(YGG_ERR_INVALID_ARGUMENT, "num_trees < 1");
  if (cfg->min_examples < 1) return set_error(YGG_ERR_INVALID_ARGUMENT, "min_examples < 1");
  if (cfg->shrinkage <= 0.f) return set_error(YGG_ERR_INVALID_ARGUMENT, "shrinkage <= 0");
  YGG_RETURN_IF_ERROR(require_device());
  YGG_CUDA(cudaSetDevice(ds->device));
  auto* h = new ygg_gbt();
  h->ds = ds;
  h->device = ds->device;
  h->cfg = *cfg;
  // any failure below releases everything the handle already owns (stream, device buffers: the pool would otherwise
  // keep them for the life of the process and a retry with smaller settings could fail again)
  const int status = init_handle(h);
  if (status != YGG_OK) {
    const std::string msg = g_last_error;
    ygg_gbt_destroy(h);
    g_last_error = msg;
    return status;
  }
  *out = h;
  return YGG_OK;
}

static int init_handle(ygg_gbt* h) {
  ygg_dataset* ds = h->ds;
  const ygg_gbt_config* cfg = &h->cfg;
  // best-first growth counts depth from 0 (training.cc:4530, :4606): one more level than the local growth
  if (cfg->growing_strategy == 1) h->cfg.max_depth += 1;
  h->f_begin = 0;
  h->f_end = ds->F;
  h->hist_f_begin = 0;
  h->hist_f_end = ds->F;
  h->n_global = ds->n;
  h->num_levels = cfg->max_depth - 1;
  h->max_nodes = (1 << cfg->max_depth) - 1;
  h->max_level_nodes = 1 << std::max(0, cfg->max_depth - 1);
  h->K = cfg->loss == YGG_LOSS_MULTINOMIAL_LOG_LIKELIHOOD ? cfg->num_classes : 1;
  h->tree_capacity = cfg->num_trees * h->K;
  const int64_t n = ds->n, n_pad = ds->n_pad;
  if (goss(h)) {
    // GOSS = a row sample + per-iteration weights: the weighted kernels with the engine's own weight array
    YGG_RETURN_IF_ERROR(dev_alloc(&h->d_weight, n_pad));
    YGG_RETURN_IF_ERROR(dev_alloc(&h->d_g2w, n_pad));
    YGG_RETURN_IF_ERROR(dev_alloc(&h->d_wsums, static_cast<size_t>(h->max_nodes) * 2));
    YGG_CUDA(cudaMemset(h->d_weight, 0, n_pad * sizeof(float)));
    YGG_CUDA(cudaMemset(h->d_g2w, 0, n_pad * sizeof(float)));
    const float amplification = cfg->goss_beta > 0.f ? (1.f - cfg->goss_alpha) / cfg->goss_beta : 1.f;
    h->w_pow2 = 1.f;
    while (h->w_pow2 < amplification) h->w_pow2 *= 2.f;
    for (int i = 0; i < 2; i++) {
      YGG_RETURN_IF_ERROR(dev_alloc(&h->d_goss_keys[i], n));
      YGG_RETURN_IF_ERROR(dev_alloc(&h->d_goss_rows[i], n));
    }
    YGG_RETURN_IF_ERROR(dev_alloc(&h->d_goss_u, n));
    YGG_CUDA(cub::DeviceRadixSort::SortPairsDescending(nullptr, h->goss_temp_bytes, h->d_goss_keys[0], h->d_goss_keys[1], h->d_goss_rows[0],
                                                      h->d_goss_rows[1], static_cast<int>(n)));
    YGG_CUDA(cudaMalloc(&h->d_goss_temp, h->goss_temp_bytes));
  }
  YGG_RETURN_IF_ERROR(configure_launches(h));
  YGG_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  YGG_RETURN_IF_ERROR(dev_alloc(&h->d_pred, n * h->K));
  YGG_RETURN_IF_ERROR(dev_alloc(&h->d_g, n_pad * h->K));   // padded: k_partition reads 16 rows per thread with 128-bit loads
  YGG_RETURN_IF_ERROR(dev_alloc(&h->d_h, n_pad * h->K));
  h->cur_g = h->d_g;
  h->cur_h = h->d_h;
  h->n_blocks = static_cast<int>(n_pad / kBlockRows);
  YGG_RETURN_IF_ERROR(dev_alloc(&h->d_q24, n_pad));
  YGG_RETURN_IF_ERROR(dev_alloc(&h->d_act, n_pad));
  YGG_RETURN_IF_ERROR(dev_alloc(&h->d_act_count, h->n_blocks));
  if (hist_hess(h)) {
    YGG_RETURN_IF_ERROR(dev_alloc(&h->d_hq24, n_pad));
    YGG_RETURN_IF_ERROR(dev_alloc(&h->d_act_h, n_pad));
  }
  YGG_RETURN_IF_ERROR(dev_alloc(&h->d_node_of_row, n_pad));
  YGG_CUDA(cudaMemset(h->d_node_of_row, 0, n_pad * sizeof(uint16_t)));
  YGG_CUDA(cudaMemset(h->d_g, 0, n_pad * h->K * sizeof(float)));
  YGG_CUDA(cudaMemset(h->d_h, 0, n_pad * h->K * sizeof(float)));
  YGG_CUDA(cudaMemset(h->d_q24, 0, n_pad * sizeof(uint32_t)));
  YGG_RETURN_IF_ERROR(dev_alloc(&h->d_st, 1));
  YGG_CUDA(cudaMemset(h->d_st, 0, sizeof(DeviceState)));
  YGG_RETURN_IF_ERROR(dev_alloc(&h->d_levels, 32));
  YGG_CUDA(cudaMemset(h->d_levels, 0, sizeof(LevelDesc) * 32));
  for (int i = 0; i < 2; i++) {
    YGG_RETURN_IF_ERROR(dev_alloc(&h->d_fam[i], h->max_level_nodes));
    YGG_RETURN_IF_ERROR(dev_alloc(&h->d_slot_node[i], h->max_level_nodes));
  }
  YGG_RETURN_IF_ERROR(dev_alloc(&h->d_nodes_all, static_cast<size_t>(h->tree_capacity) * h->max_nodes));
  YGG_RETURN_IF_ERROR(dev_alloc(&h->d_nodes_scratch, h->max_nodes));
  YGG_RETURN_IF_ERROR(dev_alloc(&h->d_loss, h->tree_capacity));
  YGG_RETURN_IF_ERROR(dev_alloc(&h->d_loss_partials, 1));
  YGG_RETURN_IF_ERROR(dev_alloc(&h->d_ties, h->max_level_nodes));
  if (sampling(h)) YGG_RETURN_IF_ERROR(dev_alloc(&h->d_selected, n_pad));
  YGG_CUDA(cudaMemset(h->d_loss, 0, sizeof(LossRec) * h->tree_capacity));
  YGG_RETURN_IF_ERROR(allocate_level_buffers(h));
  return YGG_OK;
}

int ygg_gbt_destroy(ygg_gbt* h) {
  if (!h) return YGG_OK;
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  collect_profile(h);
  dev_free(h->d_label_u8); dev_free(h->d_label_f32); dev_free(h->d_pred); dev_free(h->d_g); dev_free(h->d_h);
  dev_free(h->d_q24); dev_free(h->d_hq24); dev_free(h->d_act); dev_free(h->d_act_h);
  dev_free(h->d_act_count); dev_free(h->d_root_cnt); dev_free(h->d_node_of_row); dev_free(h->d_st); dev_free(h->d_levels);
  for (int i = 0; i < 2; i++) {
    dev_free(h->d_fam[i]); dev_free(h->d_slot_node[i]); dev_free(h->d_hist_sum[i]); dev_free(h->d_hist_cnt[i]);
    dev_free(h->d_hist_hsum[i]);
  }
  dev_free(h->d_nodes_all); dev_free(h->d_nodes_scratch); dev_free(h->d_cand); dev_free(h->d_cand_mask); cudaFree(h->d_shard_best); dev_free(h->d_loss); dev_free(h->d_loss_partials); dev_free(h->d_ties); dev_free(h->d_selected); dev_free(h->d_peer_windows);
  dev_free(h->d_vpred); dev_free(h->d_vlabel_u8); dev_free(h->d_vlabel_f32); dev_free(h->d_vloss);
  dev_free(h->d_weight); dev_free(h->d_g2w); dev_free(h->d_wsums); dev_free(h->d_vweight);
  for (int i = 0; i < 2; i++) { dev_free(h->d_goss_keys[i]); dev_free(h->d_goss_rows[i]); }
  dev_free(h->d_goss_u);
  dev_free(h->d_capture); dev_free(h->d_capture_g); dev_free(h->d_capture_h2); dev_free(h->d_capture_sel); dev_free(h->d_capture_st);
  cudaFree(h->d_goss_temp);
  cudaFree(h->d_level_buf);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
  return YGG_OK;
}

static int set_initial_predictions(ygg_gbt* h) {
  (void)cudaGetLastError();  // stale foreign error, see ygg_gbt_step
  k_fill<<<elementwise_grid(h), 256, 0, h->stream>>>(h->d_pred, h->ds->n * h->K, h->initial_prediction);
  h->launches_total++;
  YGG_RETURN_IF_ERROR(check_launch("k_fill"));
  h->trees_done = 0;
  h->iters_done = 0;
  h->tie_rng_ready = false;
  h->ties_resolved_upto = 0;
  h->ties_renamed = h->ties_unresolved = 0;
  h->finalized = false;
  h->final_trees = -1;
  h->log_entries = -1;
  h->pending_loss = false;
  h->loss_reduced_upto = 0;
  h->pending = false;
  h->has_labels = true;
  return YGG_OK;
}

int ygg_gbt_set_labels_i32(ygg_gbt* h, const int32_t* labels, int64_t n) {
  if (!h || !labels) return set_error(YGG_ERR_INVALID_ARGUMENT, "null argument");
  if (n != h->ds->n) return set_error(YGG_ERR_INVALID_ARGUMENT, "label count %lld != rows %lld", static_cast<long long>(n), static_cast<long long>(h->ds->n));
  if (!is_logit(h)) return set_error(YGG_ERR_INVALID_ARGUMENT, "integer labels need a log-likelihood loss");
  YGG_CUDA(cudaSetDevice(h->ds->device));
  if (is_multinomial(h)) {
    std::vector<uint8_t> cls(n);
    for (int64_t i = 0; i < n; i++) {
      if (labels[i] < 1 || labels[i] > h->K)  // loss_imp_multinomial.cc:84-90
        return set_error(YGG_ERR_INVALID_ARGUMENT, "Label value at example_idx %lld is invalid: %d. Expected value between 1 and %d",
                         static_cast<long long>(i), labels[i], h->K);
      cls[i] = static_cast<uint8_t>(labels[i] - 1);
    }
    h->initial_prediction = 0.f;  // initialize_with_class_priors = false (:64-66)
    if (!h->d_label_u8) YGG_RETURN_IF_ERROR(dev_alloc(&h->d_label_u8, n));
    YGG_CUDA(cudaMemcpy(h->d_label_u8, cls.data(), n, cudaMemcpyHostToDevice));
    return set_initial_predictions(h);
  }
  std::vector<uint8_t> u8(n);
  int64_t pos = 0;
  {
    // 10M labels: the check / conversion / count is integer work, split over a few host threads (it sits between the
    // dataset upload and the first iteration of an end-to-end run)
    const int T = static_cast<int>(std::min<int64_t>(8, std::max<int64_t>(1, n / (1 << 20))));
    std::vector<int64_t> part_pos(T, 0), part_bad(T, -1);
    auto work = [&](int t) {
      const int64_t b = n * t / T, e = n * (t + 1) / T;
      int64_t c = 0;
      for (int64_t i = b; i < e; i++) {
        const int32_t v = labels[i];
        if (v != 1 && v != 2) { if (part_bad[t] < 0) part_bad[t] = i; continue; }
        u8[i] = v == 2;
        c += v == 2;
      }
      part_pos[t] = c;
    };
    std::vector<std::thread> threads;
    for (int t = 1; t < T; t++) threads.emplace_back(work, t);
    work(0);
    for (auto& th : threads) th.join();
    for (int t = 0; t < T; t++) {
      if (part_bad[t] >= 0)
        return set_error(YGG_ERR_INVALID_ARGUMENT, "binary label %d at row %lld is not in {1, 2} (loss_imp_binomial.cc:58-61)", labels[part_bad[t]],
                         static_cast<long long>(part_bad[t]));
      pos += part_pos[t];
    }
  }
  // BinomialLogLikelihoodLoss::InitialPredictions (loss_imp_binomial.cc:65-99).
  double ratio = static_cast<double>(pos) / static_cast<double>(n);
  if (user_weighted(h)) {   // :83-88: double sums of the float weights, in row order
    double sum_weights = 0, weighted_sum_positive = 0;
    for (int64_t i = 0; i < n; i++) {
      sum_weights += h->host_weights[i];
      weighted_sum_positive += h->host_weights[i] * static_cast<float>(u8[i]);
    }
    ratio = weighted_sum_positive / sum_weights;
  }
  if (ratio == 0.0) h->initial_prediction = -std::numeric_limits<float>::max();
  else if (ratio == 1.0) h->initial_prediction = std::numeric_limits<float>::max();
  else h->initial_prediction = static_cast<float>(std::log(ratio / (1. - ratio)));
  if (!h->d_label_u8) YGG_RETURN_IF_ERROR(dev_alloc(&h->d_label_u8, n));
  YGG_CUDA(cudaMemcpy(h->d_label_u8, u8.data(), n, cudaMemcpyHostToDevice));
  return set_initial_predictions(h);
}

int ygg_gbt_set_labels_f32(ygg_gbt* h, const float* labels, int64_t n) {
  if (!h || !labels) return set_error(YGG_ERR_INVALID_ARGUMENT, "null argument");
  if (n != h->ds->n) return set_error(YGG_ERR_INVALID_ARGUMENT, "label count %lld != rows %lld", static_cast<long long>(n), static_cast<long long>(h->ds->n));
  if (h->cfg.loss != YGG_LOSS_SQUARED_ERROR) return set_error(YGG_ERR_INVALID_ARGUMENT, "float labels need the squared-error loss");
  YGG_CUDA(cudaSetDevice(h->ds->device));
  // MeanSquaredErrorLoss::InitialPredictions (loss_imp_mean_square_error.cc:56-88).
  double s = 0;
  for (int64_t i = 0; i < n; i++) {
    if (!std::isfinite(labels[i])) return set_error(YGG_ERR_INVALID_ARGUMENT, "non-finite label at row %lld", static_cast<long long>(i));
    s += labels[i];
  }
  h->initial_prediction = static_cast<float>(s / static_cast<double>(n));
  if (user_weighted(h)) {   // loss_imp_mean_square_error.cc:72-77
    double sum_weights = 0, weighted_sum_values = 0;
    for (int64_t i = 0; i < n; i++) {
      sum_weights += h->host_weights[i];
      weighted_sum_values += h->host_weights[i] * labels[i];
    }
    h->initial_prediction = static_cast<float>(weighted_sum_values / sum_weights);
  }
  if (!h->d_label_f32) YGG_RETURN_IF_ERROR(dev_alloc(&h->d_label_f32, n));
  YGG_CUDA(cudaMemcpy(h->d_label_f32, labels, n * sizeof(float), cudaMemcpyHostToDevice));
  return set_initial_predictions(h);
}

// Example weights (TrainingConfig.weight_definition; dataset::GetWeights -> the `weights` spans of the losses and of
// the tree trainer).  Call BEFORE ygg_gbt_set_labels_*: the initial predictions are weighted means.
static float pow2_cover_host(float v) {
  float p = 1.f;
  while (p < v) p *= 2.f;
  while (p * 0.5f >= v && p > 1e-30f) p *= 0.5f;
  return p;
}
static int check_weights(const float* weights, int64_t n, double* sum, float* wmax) {
  double s = 0;
  float m = 0.f;
  for (int64_t i = 0; i < n; i++) {
    // negative weights are rejected when the reference infers the dataspec (data_spec_inference / weight.cc)
    if (!std::isfinite(weights[i]) || weights[i] < 0.f)
      return set_error(YGG_ERR_INVALID_ARGUMENT, "weight %g at row %lld is negative or not finite", weights[i], static_cast<long long>(i));
    s += weights[i];
    m = std::max(m, weights[i]);
  }
  if (!(s > 0)) return set_error(YGG_ERR_INVALID_ARGUMENT, "the sum of the weights is null (loss_imp_mean_square_error.cc:80-84)");
  *sum = s;
  *wmax = m;
  return YGG_OK;
}

int ygg_gbt_set_weights_f32(ygg_gbt* h, const float* weights, int64_t n) {
  if (!h || !weights) return set_error(YGG_ERR_INVALID_ARGUMENT, "null argument");
  if (n != h->ds->n) return set_error(YGG_ERR_INVALID_ARGUMENT, "weight count %lld != rows %lld", static_cast<long long>(n), static_cast<long long>(h->ds->n));
  if (goss(h)) return set_error(YGG_ERR_UNIMPLEMENTED, "example weights are not combined with GOSS");
  if (h->has_labels) return set_error(YGG_ERR_INVALID_ARGUMENT, "set the weights before the labels (the initial predictions depend on them)");
  if (use_hess(h)) return set_error(YGG_ERR_UNIMPLEMENTED, "example weights are implemented for the variance gain only (use_hessian_gain = 0)");
  if (h->shard_mode != kShardNone) return set_error(YGG_ERR_INVALID_ARGUMENT, "set the weights before the shard");
  double sum = 0;
  float wmax = 0.f;
  YGG_RETURN_IF_ERROR(check_weights(weights, n, &sum, &wmax));
  YGG_CUDA(cudaSetDevice(h->ds->device));
  const int64_t n_pad = h->ds->n_pad;
  if (!h->d_weight) {
    YGG_RETURN_IF_ERROR(dev_alloc(&h->d_weight, n_pad));
    YGG_RETURN_IF_ERROR(dev_alloc(&h->d_g2w, n_pad * h->K));
    YGG_RETURN_IF_ERROR(dev_alloc(&h->d_wsums, static_cast<size_t>(h->max_nodes) * 2));
  }
  YGG_CUDA(cudaMemset(h->d_weight, 0, n_pad * sizeof(float)));
  YGG_CUDA(cudaMemset(h->d_g2w, 0, n_pad * h->K * sizeof(float)));
  h->cur_g2w = h->d_g2w;
  YGG_CUDA(cudaMemcpy(h->d_weight, weights, n * sizeof(float), cudaMemcpyHostToDevice));
  h->host_weights.assign(weights, weights + n);
  h->sum_weights = sum;
  h->w_pow2 = pow2_cover_host(wmax);
  // the histograms now carry a second plane (weight sums): launch shapes and level buffers follow
  if (!h->d_hq24) {
    YGG_RETURN_IF_ERROR(dev_alloc(&h->d_hq24, n_pad));
    YGG_RETURN_IF_ERROR(dev_alloc(&h->d_act_h, n_pad));
  }
  h->root_cnt_valid = false;
  YGG_RETURN_IF_ERROR(configure_launches(h));
  return allocate_level_buffers(h);
}

int ygg_gbt_set_validation_weights_f32(ygg_gbt* h, const float* weights, int64_t n) {
  if (!h || !weights) return set_error(YGG_ERR_INVALID_ARGUMENT, "null argument");
  if (h->vds == nullptr) return set_error(YGG_ERR_INVALID_ARGUMENT, "no validation rows attached");
  if (n != h->vds->n) return set_error(YGG_ERR_INVALID_ARGUMENT, "weight count %lld != validation rows %lld", static_cast<long long>(n), static_cast<long long>(h->vds->n));
  if (h->iters_done > 0) return set_error(YGG_ERR_INVALID_ARGUMENT, "validation weights must be set before training");
  double sum = 0;
  float wmax = 0.f;
  YGG_RETURN_IF_ERROR(check_weights(weights, n, &sum, &wmax));
  YGG_CUDA(cudaSetDevice(h->ds->device));
  dev_free(h->d_vweight); h->d_vweight = nullptr;
  YGG_RETURN_IF_ERROR(dev_alloc(&h->d_vweight, n));
  YGG_CUDA(cudaMemcpy(h->d_vweight, weights, n * sizeof(float), cudaMemcpyHostToDevice));
  h->v_sum_weights = sum;
  h->v_correct_scale = correct_scale_of(pow2_cover_host(wmax));
  return YGG_OK;
}

int ygg_gbt_set_feature_shard(ygg_gbt* h, int32_t feature_begin, int32_t feature_end, int32_t rank,
                              int32_t world, ygg_allgather_fn exchange, void* ctx) {
  if (!h) return set_error(YGG_ERR_INVALID_ARGUMENT, "null handle");
  if (feature_begin < 0 || feature_end > h->ds->F || feature_begin >= feature_end)
    return set_error(YGG_ERR_INVALID_ARGUMENT, "bad feature shard [%d, %d) of %d", feature_begin, feature_end, h->ds->F);
  if (world < 1 || rank < 0 || rank >= world) return set_error(YGG_ERR_INVALID_ARGUMENT, "bad rank %d / world %d", rank, world);
  if (world > 1 && !exchange) return set_error(YGG_ERR_INVALID_ARGUMENT, "world > 1 needs an exchange function");
  if (h->trees_done > 0) return set_error(YGG_ERR_INVALID_ARGUMENT, "shard must be set before training");
  if (world > 1 && h->cfg.candidate_shuffle != 0) return set_error(YGG_ERR_UNIMPLEMENTED, "candidate_shuffle is not combined with sharding");
  YGG_CUDA(cudaSetDevice(h->ds->device));
  h->f_begin = feature_begin; h->f_end = feature_end; h->rank = rank; h->world = world;
  h->hist_f_begin = feature_begin; h->hist_f_end = feature_end;
  h->shard_mode = world > 1 ? kShardFeatures : kShardNone;
  h->exchange = exchange; h->exchange_ctx = ctx;
  h->root_cnt_valid = false;
  cudaFree(h->d_shard_best);
  h->d_shard_best = nullptr;
  YGG_RETURN_IF_ERROR(dev_alloc_plain(&h->d_shard_best, static_cast<size_t>(world) * h->max_level_nodes));
  YGG_RETURN_IF_ERROR(configure_launches(h));
  return allocate_level_buffers(h);
}

int ygg_gbt_set_row_shard(ygg_gbt* h, int32_t rank, int32_t world, int64_t n_rows_global,
                          float initial_prediction, ygg_allreduce_fn allreduce, void* ctx) {
  if (!h) return set_error(YGG_ERR_INVALID_ARGUMENT, "null handle");
  if (world < 1 || rank < 0 || rank >= world) return set_error(YGG_ERR_INVALID_ARGUMENT, "bad rank %d / world %d", rank, world);
  if (world > 1 && !allreduce) return set_error(YGG_ERR_INVALID_ARGUMENT, "world > 1 needs an all-reduce function");
  if (n_rows_global < h->ds->n) return set_error(YGG_ERR_INVALID_ARGUMENT, "n_rows_global < local rows");
  if (!h->has_labels) return set_error(YGG_ERR_INVALID_ARGUMENT, "set the labels before the row shard");

  if (world > 1 && h->cfg.candidate_shuffle != 0) return set_error(YGG_ERR_UNIMPLEMENTED, "candidate_shuffle is not combined with sharding");
  if (h->trees_done > 0) return set_error(YGG_ERR_INVALID_ARGUMENT, "shard must be set before training");
  YGG_CUDA(cudaSetDevice(h->ds->device));
  (void)cudaGetLastError();  // stale foreign error, see ygg_gbt_step
  h->rank = rank; h->world = world;
  h->shard_mode = world > 1 ? kShardRows : kShardNone;
  h->n_global = n_rows_global;
  h->allreduce = allreduce; h->exchange_ctx = ctx;
  h->initial_prediction = initial_prediction;
  k_fill<<<elementwise_grid(h), 256, 0, h->stream>>>(h->d_pred, h->ds->n, h->initial_prediction);
  h->launches_total++;
  YGG_RETURN_IF_ERROR(check_launch("k_fill"));
  if (user_weighted(h) && world > 1) {
    // example weights: the fixed-point scale (largest weight) and the weight sum are the job's, not this rank's
    uint32_t bits;
    std::memcpy(&bits, &h->w_pow2, sizeof(bits));
    unsigned long long* scratch = h->d_wsums;   // >= 2 words, unused until the first tree is finished
    YGG_CUDA(cudaMemcpyAsync(scratch, &bits, sizeof(bits), cudaMemcpyHostToDevice, h->stream));
    YGG_CUDA(cudaMemcpyAsync(scratch + 1, &h->sum_weights, sizeof(double), cudaMemcpyHostToDevice, h->stream));
    YGG_RETURN_IF_ERROR(do_allreduce(h, scratch, 1, 0, 1));       // positive floats order like their bit patterns
    YGG_RETURN_IF_ERROR(do_allreduce(h, scratch + 1, 1, 2, 0));
    YGG_CUDA(cudaMemcpyAsync(&bits, scratch, sizeof(bits), cudaMemcpyDeviceToHost, h->stream));
    YGG_CUDA(cudaMemcpyAsync(&h->sum_weights, scratch + 1, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    YGG_CUDA(cudaStreamSynchronize(h->stream));
    std::memcpy(&h->w_pow2, &bits, sizeof(bits));
  }
  return YGG_OK;
}

int ygg_gbt_set_row_shard_scatter(ygg_gbt* h, int32_t rank, int32_t world, int64_t n_rows_global,
                                  float initial_prediction, ygg_allreduce_fn allreduce,
                                  ygg_reducescatter_fn reducescatter, ygg_allgather_fn allgather, void* ctx) {
  if (!h) return set_error(YGG_ERR_INVALID_ARGUMENT, "null handle");
  if (world > 1 && (!reducescatter || !allgather)) return set_error(YGG_ERR_INVALID_ARGUMENT, "world > 1 needs reduce-scatter and all-gather functions");
  if (world > h->ds->F) return set_error(YGG_ERR_INVALID_ARGUMENT, "more ranks (%d) than features (%d)", world, h->ds->F);
  YGG_RETURN_IF_ERROR(ygg_gbt_set_row_shard(h, rank, world, n_rows_global, initial_prediction, allreduce, ctx));
  if (world <= 1) return YGG_OK;
  // histograms cover every feature; the scan / best-split search covers this rank's chunk of them
  const int f_chunk = (h->ds->F + world - 1) / world;
  if (static_cast<int64_t>(world - 1) * f_chunk >= h->ds->F)
    return set_error(YGG_ERR_INVALID_ARGUMENT, "%d features do not split into %d non-empty chunks of %d", h->ds->F, world, f_chunk);
  h->scatter = true;
  h->reducescatter = reducescatter;
  h->exchange = allgather;
  h->hist_f_begin = 0; h->hist_f_end = h->ds->F;
  h->f_begin = std::min(h->ds->F, rank * f_chunk);
  h->f_end = std::min(h->ds->F, (rank + 1) * f_chunk);
  h->root_cnt_valid = false;
  cudaFree(h->d_shard_best);
  h->d_shard_best = nullptr;
  YGG_RETURN_IF_ERROR(dev_alloc_plain(&h->d_shard_best, static_cast<size_t>(world) * h->max_level_nodes));
  YGG_RETURN_IF_ERROR(configure_launches(h));
  return allocate_level_buffers(h);
}

namespace {
__global__ void k_gather_rows(const uint8_t* __restrict__ in, int64_t in_pad, const uint32_t* __restrict__ rows, int64_t n_out,
                              int64_t out_pad, uint8_t* __restrict__ out) {
  const int f = blockIdx.y;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n_out; i += stride)
    out[static_cast<int64_t>(f) * out_pad + i] = in[static_cast<int64_t>(f) * in_pad + rows[i]];
}

int attach_validation(ygg_gbt* h, const ygg_dataset* valid, int64_t n) {
  (void)cudaGetLastError();  // stale foreign error, see ygg_gbt_step
  if (h->trees_done > 0) return set_error(YGG_ERR_INVALID_ARGUMENT, "validation rows must be attached before training");
  if (h->shard_mode != kShardNone) return set_error(YGG_ERR_UNIMPLEMENTED, "validation rows are not combined with sharding");
  if (!h->has_labels) return set_error(YGG_ERR_INVALID_ARGUMENT, "set the training labels first (the initial prediction comes from them)");
  if (valid->device != h->ds->device) return set_error(YGG_ERR_INVALID_ARGUMENT, "the validation dataset lives on another device");
  if (valid->F != h->ds->F || valid->num_bins != h->ds->num_bins || valid->feature_type != h->ds->feature_type)
    return set_error(YGG_ERR_INVALID_ARGUMENT, "the validation dataset does not have the features / binning of the training dataset");
  if (n != valid->n) return set_error(YGG_ERR_INVALID_ARGUMENT, "label count %lld != validation rows %lld", static_cast<long long>(n), static_cast<long long>(valid->n));
  YGG_CUDA(cudaSetDevice(h->ds->device));
  dev_free(h->d_vpred); dev_free(h->d_vloss);
  h->d_vpred = nullptr; h->d_vloss = nullptr;
  YGG_RETURN_IF_ERROR(dev_alloc(&h->d_vpred, n * h->K));
  YGG_RETURN_IF_ERROR(dev_alloc(&h->d_vloss, h->tree_capacity));
  YGG_CUDA(cudaMemsetAsync(h->d_vloss, 0, sizeof(LossRec) * h->tree_capacity, h->stream));
  // the validation predictions start from the initial prediction of the TRAINING rows
  k_fill<<<static_cast<int>(std::min<int64_t>((n + 255) / 256, 4096)), 256, 0, h->stream>>>(h->d_vpred, n * h->K, h->initial_prediction);
  h->launches_total++;
  h->vds = valid;
  return check_launch("k_fill");
}
}  // namespace

int ygg_validation_split_mask(uint32_t random_seed, int64_t n_rows, float validation_ratio, uint8_t* out_in_training) {
  if (!out_in_training || n_rows < 0) return set_error(YGG_ERR_INVALID_ARGUMENT, "bad argument");
  if (validation_ratio < 0.f || validation_ratio > 1.f)
    return set_error(YGG_ERR_INVALID_ARGUMENT, "The validation set ratio should be in [0,1].");  // :2724-2727
  // utils::RandomEngine = std::mt19937 seeded with random_seed; this is its first consumer
  // (gradient_boosted_trees.cc:1198, :2731-2738).  Same standard-library calls as the reference.
  std::mt19937 random(random_seed);
  std::uniform_real_distribution<float> unif_dist_01;
  for (int64_t r = 0; r < n_rows; r++)
    out_in_training[r] = validation_ratio == 0.f ? 1 : (unif_dist_01(random) > validation_ratio ? 1 : 0);
  return YGG_OK;
}

int ygg_dataset_split_rows(const ygg_dataset* ds, const uint8_t* select, ygg_dataset** selected, ygg_dataset** rest) {
  if (!ds || !select || !selected || !rest) return set_error(YGG_ERR_INVALID_ARGUMENT, "null argument");
  std::vector<uint32_t> rows[2];
  for (int64_t r = 0; r < ds->n; r++) rows[select[r] ? 0 : 1].push_back(static_cast<uint32_t>(r));
  if (rows[0].empty() || rows[1].empty()) return set_error(YGG_ERR_INVALID_ARGUMENT, "one side of the split is empty");
  YGG_CUDA(cudaSetDevice(ds->device));
  ygg_dataset* out[2] = {nullptr, nullptr};
  uint32_t* d_rows = nullptr;
  int st = YGG_OK;
  for (int k = 0; k < 2 && st == YGG_OK; k++) {
    const int64_t n = static_cast<int64_t>(rows[k].size());
    st = ygg_internal_dataset_alloc(&out[k], n, ds->F, ds->device);
    if (st != YGG_OK) break;
    out[k]->num_bins = ds->num_bins; out[k]->na_bin = ds->na_bin; out[k]->feature_type = ds->feature_type;
    if (cudaMalloc(&d_rows, sizeof(uint32_t) * n) != cudaSuccess ||
        cudaMemcpy(d_rows, rows[k].data(), sizeof(uint32_t) * n, cudaMemcpyHostToDevice) != cudaSuccess) {
      st = set_error(YGG_ERR_CUDA, "row index upload failed");
      break;
    }
    dim3 grid(static_cast<unsigned>(std::min<int64_t>((n + 255) / 256, 2048)), static_cast<unsigned>(ds->F));
    k_gather_rows<<<grid, 256>>>(ds->d_bins, ds->n_pad, d_rows, n, out[k]->n_pad, out[k]->d_bins);
    if (cudaDeviceSynchronize() != cudaSuccess) st = set_error(YGG_ERR_CUDA, "row gather failed: %s", cudaGetErrorString(cudaGetLastError()));
    cudaFree(d_rows);
    d_rows = nullptr;
    if (st == YGG_OK) st = ygg_internal_dataset_finalize(out[k]);
    if (st == YGG_OK && ds->d_bucket_values != nullptr) {   // the exact threshold rule travels with the columns
      st = dev_alloc(&out[k]->d_bucket_values, static_cast<size_t>(ds->F) * kMaxBins);
      if (st == YGG_OK) st = dev_alloc(&out[k]->d_exact_rule, ds->F);
      if (st == YGG_OK) st = dev_alloc(&out[k]->d_na_replacement, ds->F);
      if (st == YGG_OK && cudaMemcpy(out[k]->d_na_replacement, ds->d_na_replacement, sizeof(float) * ds->F, cudaMemcpyDeviceToDevice) != cudaSuccess)
        st = set_error(YGG_ERR_CUDA, "copy of the bucket values failed");
      if (st == YGG_OK && (cudaMemcpy(out[k]->d_bucket_values, ds->d_bucket_values, sizeof(float) * ds->F * kMaxBins, cudaMemcpyDeviceToDevice) != cudaSuccess ||
                           cudaMemcpy(out[k]->d_exact_rule, ds->d_exact_rule, sizeof(int32_t) * ds->F, cudaMemcpyDeviceToDevice) != cudaSuccess))
        st = set_error(YGG_ERR_CUDA, "copy of the bucket values failed");
    }
  }
  if (st != YGG_OK) {
    cudaFree(d_rows);
    ygg_dataset_destroy(out[0]);
    ygg_dataset_destroy(out[1]);
    return st;
  }
  *selected = out[0];
  *rest = out[1];
  return YGG_OK;
}

int ygg_gbt_set_validation_i32(ygg_gbt* h, const ygg_dataset* valid, const int32_t* labels, int64_t n) {
  if (!h || !valid || !labels) return set_error(YGG_ERR_INVALID_ARGUMENT, "null argument");
  if (!is_logit(h)) return set_error(YGG_ERR_INVALID_ARGUMENT, "integer labels need a log-likelihood loss");
  std::vector<uint8_t> u8(std::max<int64_t>(n, 0));
  const int top = is_multinomial(h) ? h->K : 2;
  for (int64_t i = 0; i < n; i++) {
    if (labels[i] < 1 || labels[i] > top) return set_error(YGG_ERR_INVALID_ARGUMENT, "label %d at validation row %lld is not in [1, %d]", labels[i], static_cast<long long>(i), top);
    u8[i] = is_multinomial(h) ? static_cast<uint8_t>(labels[i] - 1) : static_cast<uint8_t>(labels[i] == 2);
  }
  YGG_RETURN_IF_ERROR(attach_validation(h, valid, n));
  dev_free(h->d_vlabel_u8); h->d_vlabel_u8 = nullptr;
  YGG_RETURN_IF_ERROR(dev_alloc(&h->d_vlabel_u8, n));
  YGG_CUDA(cudaMemcpy(h->d_vlabel_u8, u8.data(), n, cudaMemcpyHostToDevice));
  return YGG_OK;
}

int ygg_gbt_set_validation_f32(ygg_gbt* h, const ygg_dataset* valid, const float* labels, int64_t n) {
  if (!h || !valid || !labels) return set_error(YGG_ERR_INVALID_ARGUMENT, "null argument");
  if (h->cfg.loss != YGG_LOSS_SQUARED_ERROR) return set_error(YGG_ERR_INVALID_ARGUMENT, "float labels need the squared-error loss");
  YGG_RETURN_IF_ERROR(attach_validation(h, valid, n));
  dev_free(h->d_vlabel_f32); h->d_vlabel_f32 = nullptr;
  YGG_RETURN_IF_ERROR(dev_alloc(&h->d_vlabel_f32, n));
  YGG_CUDA(cudaMemcpy(h->d_vlabel_f32, labels, n * sizeof(float), cudaMemcpyHostToDevice));
  return YGG_OK;
}

int ygg_gbt_validation_loss(ygg_gbt* h, int32_t iter, float* loss, float* secondary) {
  if (!h || !loss || !secondary) return set_error(YGG_ERR_INVALID_ARGUMENT, "null argument");
  if (h->vds == nullptr) return set_error(YGG_ERR_INVALID_ARGUMENT, "no validation rows attached");
  if (iter < 0 || iter >= h->iters_done) return set_error(YGG_ERR_INVALID_ARGUMENT, "iteration %d not trained", iter);
  YGG_CUDA(cudaSetDevice(h->ds->device));
  LossRec rec;
  YGG_CUDA(cudaMemcpyAsync(&rec, h->d_vloss + iter, sizeof(rec), cudaMemcpyDeviceToHost, h->stream));
  YGG_CUDA(cudaStreamSynchronize(h->stream));
  *loss = validation_loss_value(h, rec, secondary);
  return YGG_OK;
}

int ygg_gbt_final_validation(ygg_gbt* h, float* validation_loss, int32_t* early_stopping_triggered) {
  if (!h || !validation_loss || !early_stopping_triggered) return set_error(YGG_ERR_INVALID_ARGUMENT, "null argument");
  if (h->vds == nullptr || h->trees_done == 0) return set_error(YGG_ERR_INVALID_ARGUMENT, "no validation result");
  if (h->finalized) {
    *validation_loss = h->final_validation_loss;
    *early_stopping_triggered = h->early_stopping_triggered ? 1 : 0;
    return YGG_OK;
  }
  float sec;  // early_stopping = NONE: the loss of the full model (gradient_boosted_trees.cc:273-290)
  *early_stopping_triggered = 0;
  return ygg_gbt_validation_loss(h, h->iters_done - 1, validation_loss, &sec);
}

int ygg_feature_shard(int32_t n_features, int32_t rank, int32_t world, int32_t* begin, int32_t* end) {
  if (!begin || !end || world < 1 || rank < 0 || rank >= world || n_features < world)
    return set_error(YGG_ERR_INVALID_ARGUMENT, "bad shard request: %d features, rank %d of %d", n_features, rank, world);
  *begin = static_cast<int32_t>(static_cast<int64_t>(n_features) * rank / world);
  *end = static_cast<int32_t>(static_cast<int64_t>(n_features) * (rank + 1) / world);
  return YGG_OK;
}

int ygg_merge_shard_best(const ygg_shard_best* records, int32_t world, int32_t nodes, ygg_shard_best* out) {
  if (!records || !out || world < 1 || nodes < 0) return set_error(YGG_ERR_INVALID_ARGUMENT, "bad argument");
  static_assert(sizeof(ygg_shard_best) == sizeof(ShardBest), "layout");
  for (int j = 0; j < nodes; j++) {
    const ShardBest b = merge_shard_bests(reinterpret_cast<const ShardBest*>(records), world, nodes, j);
    std::memcpy(&out[j], &b, sizeof(b));
  }
  return YGG_OK;
}

int ygg_gbt_initial_prediction(ygg_gbt* h, float* out) {
  if (!h || !out) return set_error(YGG_ERR_INVALID_ARGUMENT, "null argument");
  if (!h->has_labels) return set_error(YGG_ERR_INVALID_ARGUMENT, "labels not set");
  *out = h->initial_prediction;
  return YGG_OK;
}

int ygg_gbt_step(ygg_gbt* h) {
  if (!h) return set_error(YGG_ERR_INVALID_ARGUMENT, "null handle");
  if (!h->has_labels) return set_error(YGG_ERR_INVALID_ARGUMENT, "labels not set");
  if (h->trees_done + h->K > h->tree_capacity) return set_error(YGG_ERR_INVALID_ARGUMENT, "all %d trees already trained", h->tree_capacity);
  if (h->finalized) return set_error(YGG_ERR_INVALID_ARGUMENT, "training was finalized by early stopping");
  YGG_CUDA(cudaSetDevice(h->ds->device));
  (void)cudaGetLastError();  // drop a stale, non-sticky error of an earlier foreign runtime call (see check_launch)
  if (goss(h)) YGG_RETURN_IF_ERROR(draw_goss(h));
  else if (sampling(h)) YGG_RETURN_IF_ERROR(draw_sample(h));
  const int64_t n_job = sampling(h) ? h->n_selected : (h->shard_mode == kShardRows ? h->n_global : h->ds->n);
  const int root_candidate = (n_job >= h->cfg.min_examples && 1 < h->cfg.max_depth) ? 1 : 0;
  if (is_multinomial(h)) {
    // One iteration = K trees on the gradients taken at its start (gradient_boosted_trees.cc:1445, :1490-1511),
    // each added to its class plane as soon as it is grown (the next tree does not read the predictions).
    if (h->shard_mode != kShardNone) return set_error(YGG_ERR_UNIMPLEMENTED, "the multinomial loss is not combined with sharding");
    YGG_RETURN_IF_ERROR(launch_mc(h, h->pending_loss, true));
    h->pending_loss = false;
    for (int k = 0; k < h->K; k++) {
      h->cur_g = h->d_g + static_cast<int64_t>(k) * h->ds->n_pad;
      h->cur_h = h->d_h + static_cast<int64_t>(k) * h->ds->n_pad;
      k_begin_iteration<<<1, 1, 0, h->stream>>>(h->d_st, h->d_levels, h->d_fam[0], h->d_slot_node[0], root_candidate);
      h->launches_total++;
      if (weighted(h)) {
        // the fixed-point scales of this class's tree: max |w*g| and max (w*g)*g over its plane
        h->cur_g2w = h->d_g2w + static_cast<int64_t>(k) * h->ds->n_pad;
        DeviceState* st = h->d_st;
        k_absmax_to<<<elementwise_grid(h), 256, 0, h->stream>>>(h->cur_g, h->ds->n, &st->gmax_bits);
        k_absmax_to<<<elementwise_grid(h), 256, 0, h->stream>>>(h->cur_g2w, h->ds->n, &st->g2w_max_bits);
        h->launches_total += 2;
      }
      NodeRec* nodes = h->d_nodes_all + static_cast<size_t>(h->trees_done) * h->max_nodes;
      YGG_RETURN_IF_ERROR(grow_tree(h, nodes));
      if (h->cfg.growing_strategy == 1) YGG_RETURN_IF_ERROR(best_first_prune(h, nodes));
      k_apply_leaves<<<elementwise_grid(h), 256, 0, h->stream>>>(h->d_pred + static_cast<int64_t>(k) * h->ds->n, h->d_node_of_row,
                                                                 nodes, h->ds->n);
      h->launches_total++;
      YGG_RETURN_IF_ERROR(check_launch("k_apply_leaves"));
      if (h->vds != nullptr && h->cfg.candidate_shuffle != 0) { h->trees_done++; const int st = resolve_ties(h, h->trees_done); h->trees_done--; YGG_RETURN_IF_ERROR(st); }
      YGG_RETURN_IF_ERROR(launch_valid_update(h, h->trees_done, k));
      h->trees_done++;
    }
    h->cur_g = h->d_g;
    h->cur_h = h->d_h;
    h->cur_g2w = h->d_g2w;
    h->iters_done++;
    h->pending_loss = true;
    return YGG_OK;
  }
  k_begin_iteration<<<1, 1, 0, h->stream>>>(h->d_st, h->d_levels, h->d_fam[0], h->d_slot_node[0], root_candidate);
  h->launches_total++;
  YGG_RETURN_IF_ERROR(check_launch("k_begin_iteration"));
  YGG_RETURN_IF_ERROR(launch_pred_grad(h, h->pending, true));
  if (goss(h)) YGG_RETURN_IF_ERROR(apply_goss(h));
  if (h->shard_mode == kShardRows && (!is_logit(h) || weighted(h))) {
    // squared error / example weights: the quantisation scale P needs max|g| (max|w*g|) over ALL rows
    DeviceState* st = h->d_st;
    YGG_RETURN_IF_ERROR(do_allreduce(h, &st->gmax_bits, 1, 0, 1));
    if (weighted(h)) YGG_RETURN_IF_ERROR(do_allreduce(h, &st->g2w_max_bits, 1, 0, 1));
  }
  NodeRec* nodes = h->d_nodes_all + static_cast<size_t>(h->trees_done) * h->max_nodes;
  YGG_RETURN_IF_ERROR(grow_tree(h, nodes));
  if (h->cfg.growing_strategy == 1) YGG_RETURN_IF_ERROR(best_first_prune(h, nodes));
  // held-out rows are routed by the FINAL conditions: twins agree on the training rows only
  if (h->vds != nullptr && h->cfg.candidate_shuffle != 0) { h->trees_done++; const int st = resolve_ties(h, h->trees_done); h->trees_done--; YGG_RETURN_IF_ERROR(st); }
  YGG_RETURN_IF_ERROR(launch_valid_update(h, h->trees_done));
  h->trees_done++;
  h->iters_done++;
  h->pending = true;
  return YGG_OK;
}

int ygg_gbt_sync(ygg_gbt* h) {
  if (!h) return set_error(YGG_ERR_INVALID_ARGUMENT, "null handle");
  YGG_CUDA(cudaSetDevice(h->ds->device));
  YGG_RETURN_IF_ERROR(apply_pending(h));
  YGG_RETURN_IF_ERROR(reduce_losses(h));
  YGG_RETURN_IF_ERROR(check_device_error(h));
  collect_profile(h);
  return YGG_OK;
}

int ygg_gbt_train(ygg_gbt* h, int32_t num_iters, const volatile int32_t* stop_flag) {
  if (!h) return set_error(YGG_ERR_INVALID_ARGUMENT, "null handle");
  const bool watch = h->vds != nullptr && h->cfg.early_stopping != YGG_EARLY_STOPPING_NONE;
  if (!watch) {
    for (int i = 0; i < num_iters; i++) {
      if (stop_flag && *stop_flag) {
        ygg_gbt_sync(h);
        return set_error(YGG_ERR_CANCELLED, "training stopped by the caller after %d iterations", h->trees_done);
      }
      YGG_RETURN_IF_ERROR(ygg_gbt_step(h));
    }
    return ygg_gbt_sync(h);
  }
  // Early stopping (gradient_boosted_trees.cc:1628-1647).  The validation losses stay on the device; they
  // are read back every kBatch iterations and the reference's per-iteration policy is replayed on them, so
  // the level loop never waits for the host.  Trees trained past the stopping point are dropped — the
  // final model and logs are the ones the reference produces.
  if (h->iters_done != 0) return set_error(YGG_ERR_INVALID_ARGUMENT, "early stopping needs a fresh handle");
  constexpr int kBatch = 8;
  EarlyStoppingState es;
  es.look_ahead = h->cfg.early_stopping_num_trees_look_ahead;
  es.initial_iteration = h->cfg.early_stopping_initial_iteration;
  const double nv = static_cast<double>(h->vds->n);
  int replayed = 0, stop_iter = -1;
  std::vector<LossRec> rec(kBatch);
  while (h->iters_done < num_iters && stop_iter < 0) {
    const int todo = std::min(kBatch, num_iters - h->iters_done);
    for (int i = 0; i < todo; i++) {
      if (stop_flag && *stop_flag) {
        ygg_gbt_sync(h);
        return set_error(YGG_ERR_CANCELLED, "training stopped by the caller after %d iterations", h->trees_done);
      }
      YGG_RETURN_IF_ERROR(ygg_gbt_step(h));
    }
    const int n_new = h->iters_done - replayed;
    YGG_CUDA(cudaMemcpyAsync(rec.data(), h->d_vloss + replayed, sizeof(LossRec) * n_new, cudaMemcpyDeviceToHost, h->stream));
    YGG_CUDA(cudaStreamSynchronize(h->stream));
    for (int i = 0; i < n_new && stop_iter < 0; i++) {
      const int iter = replayed + i;
      float sec;
      es.update(validation_loss_value(h, rec[i], &sec), (iter + 1) * h->K, iter);  // EarlyStopping counts trees
      if (h->cfg.early_stopping == YGG_EARLY_STOPPING_LOSS_INCREASE && es.should_stop(iter)) stop_iter = iter;
    }
    replayed = h->iters_done;
  }
  YGG_RETURN_IF_ERROR(ygg_gbt_sync(h));
  // FinalizeModelWithValidationDataset (gradient_boosted_trees.cc:212-272)
  const int trained = stop_iter >= 0 ? stop_iter + 1 : h->iters_done;   // iterations
  h->log_entries = trained;
  h->finalized = true;
  if (trained < es.initial_iteration + 1) {
    h->final_trees = trained * h->K;
    h->final_validation_loss = es.last_loss;
    h->early_stopping_triggered = false;
  } else {
    h->final_trees = es.best_num_trees;
    h->final_validation_loss = es.best_loss;
    h->early_stopping_triggered = true;
  }
  return YGG_OK;
}

int ygg_gbt_train_timed(ygg_gbt* h, int32_t num_iters, double* device_ms, int64_t* kernel_launches) {
  if (!h || !device_ms) return set_error(YGG_ERR_INVALID_ARGUMENT, "null argument");
  YGG_CUDA(cudaSetDevice(h->ds->device));
  cudaEvent_t a, b;
  YGG_CUDA(cudaEventCreate(&a));
  YGG_CUDA(cudaEventCreate(&b));
  const int64_t l0 = h->launches_total;
  YGG_CUDA(cudaStreamSynchronize(h->stream));
  YGG_CUDA(cudaEventRecord(a, h->stream));
  for (int i = 0; i < num_iters; i++) YGG_RETURN_IF_ERROR(ygg_gbt_step(h));
  YGG_RETURN_IF_ERROR(apply_pending(h));
  YGG_RETURN_IF_ERROR(reduce_losses(h));
  YGG_CUDA(cudaEventRecord(b, h->stream));
  YGG_CUDA(cudaEventSynchronize(b));
  float ms = 0;
  YGG_CUDA(cudaEventElapsedTime(&ms, a, b));
  cudaEventDestroy(a);
  cudaEventDestroy(b);
  *device_ms = ms;
  if (kernel_launches) *kernel_launches = h->launches_total - l0;
  YGG_RETURN_IF_ERROR(check_device_error(h));
  collect_profile(h);
  return YGG_OK;
}

int32_t ygg_gbt_num_trees(const ygg_gbt* h) { return !h ? 0 : (h->final_trees >= 0 ? h->final_trees : h->trees_done); }
int32_t ygg_gbt_num_iterations(const ygg_gbt* h) { return !h ? 0 : (h->log_entries >= 0 ? h->log_entries : h->iters_done); }

int ygg_gbt_get_tree(ygg_gbt* h, int32_t iter, ygg_node* out, int32_t capacity, int32_t* n_nodes) {
  if (!h || !out || !n_nodes) return set_error(YGG_ERR_INVALID_ARGUMENT, "null argument");
  if (iter < 0 || iter >= h->trees_done) return set_error(YGG_ERR_INVALID_ARGUMENT, "tree %d not trained (have %d)", iter, h->trees_done);
  YGG_CUDA(cudaSetDevice(h->ds->device));
  YGG_RETURN_IF_ERROR(resolve_ties(h, h->trees_done));
  std::vector<ygg_node> flat;
  YGG_RETURN_IF_ERROR(fetch_tree(h, h->d_nodes_all + static_cast<size_t>(iter) * h->max_nodes, &flat));
  *n_nodes = static_cast<int32_t>(flat.size());
  if (static_cast<int32_t>(flat.size()) > capacity) return set_error(YGG_ERR_INVALID_ARGUMENT, "capacity %d < %zu nodes", capacity, flat.size());
  std::memcpy(out, flat.data(), flat.size() * sizeof(ygg_node));
  return YGG_OK;
}

int ygg_gbt_train_loss(ygg_gbt* h, int32_t iter, float* loss, float* secondary) {
  if (!h || !loss || !secondary) return set_error(YGG_ERR_INVALID_ARGUMENT, "null argument");
  if (iter < 0 || iter >= h->iters_done) return set_error(YGG_ERR_INVALID_ARGUMENT, "iteration %d not trained", iter);
  YGG_CUDA(cudaSetDevice(h->ds->device));
  YGG_RETURN_IF_ERROR(apply_pending(h));
  YGG_RETURN_IF_ERROR(reduce_losses(h));
  LossRec rec;
  YGG_CUDA(cudaMemcpyAsync(&rec, h->d_loss + iter, sizeof(rec), cudaMemcpyDeviceToHost, h->stream));
  YGG_CUDA(cudaStreamSynchronize(h->stream));
  const double n = static_cast<double>(h->shard_mode == kShardRows ? h->n_global : h->ds->n);
  if (user_weighted(h)) *loss = loss_value(h, rec, h->sum_weights, secondary, correct_scale_of(h->w_pow2));
  else *loss = loss_value(h, rec, n, secondary);
  return YGG_OK;
}

int ygg_gbt_get_predictions(ygg_gbt* h, float* out, int64_t n) {
  if (!h || !out) return set_error(YGG_ERR_INVALID_ARGUMENT, "null argument");
  if (n != h->ds->n * h->K) return set_error(YGG_ERR_INVALID_ARGUMENT, "n mismatch (rows x classes expected)");
  YGG_CUDA(cudaSetDevice(h->ds->device));
  YGG_RETURN_IF_ERROR(apply_pending(h));
  YGG_CUDA(cudaMemcpyAsync(out, h->d_pred, n * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  YGG_CUDA(cudaStreamSynchronize(h->stream));
  return YGG_OK;
}

int ygg_gbt_predict(ygg_gbt* h, const ygg_dataset* ds, float* out, int64_t n) {
  if (!h || !ds || !out) return set_error(YGG_ERR_INVALID_ARGUMENT, "null argument");
  if (ds->device != h->ds->device) return set_error(YGG_ERR_INVALID_ARGUMENT, "the dataset lives on another device");
  if (ds->F != h->ds->F || ds->num_bins != h->ds->num_bins || ds->feature_type != h->ds->feature_type)
    return set_error(YGG_ERR_INVALID_ARGUMENT, "the dataset does not have the features / binning of the training dataset");
  if (n != ds->n * h->K) return set_error(YGG_ERR_INVALID_ARGUMENT, "n mismatch (rows x classes expected)");
  YGG_CUDA(cudaSetDevice(h->ds->device));
  (void)cudaGetLastError();
  YGG_RETURN_IF_ERROR(resolve_ties(h, h->trees_done));
  float* d_out = nullptr;
  YGG_RETURN_IF_ERROR(dev_alloc(&d_out, static_cast<size_t>(n)));
  const int n_trees = ygg_gbt_num_trees(h);
  k_predict<<<static_cast<int>(std::min<int64_t>((ds->n + 255) / 256, static_cast<int64_t>(h->ds->num_sms) * 16)), 256, 0, h->stream>>>(
      ds->d_bins, ds->n, ds->n_pad, h->d_nodes_all, h->max_nodes, n_trees, h->K, h->initial_prediction, d_out);
  h->launches_total++;
  int st = check_launch("k_predict");
  if (st == YGG_OK && (cudaMemcpyAsync(out, d_out, sizeof(float) * n, cudaMemcpyDeviceToHost, h->stream) != cudaSuccess ||
                       cudaStreamSynchronize(h->stream) != cudaSuccess))
    st = set_error(YGG_ERR_CUDA, "prediction read-back failed: %s", cudaGetErrorString(cudaGetLastError()));
  dev_free(d_out);
  return st;
}

int ygg_gbt_set_predictions(ygg_gbt* h, const float* pred, int64_t n) {
  if (!h || !pred) return set_error(YGG_ERR_INVALID_ARGUMENT, "null argument");
  if (n != h->ds->n) return set_error(YGG_ERR_INVALID_ARGUMENT, "n mismatch");
  YGG_CUDA(cudaSetDevice(h->ds->device));
  YGG_RETURN_IF_ERROR(apply_pending(h));
  YGG_CUDA(cudaMemcpyAsync(h->d_pred, pred, n * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  YGG_CUDA(cudaStreamSynchronize(h->stream));
  return YGG_OK;
}

int ygg_tree_train_on_gradients(ygg_gbt* h, const float* gradients, const float* hessians, ygg_node* out,
                                int32_t capacity, int32_t* n_nodes) {
  if (!h || !gradients || !out || !n_nodes) return set_error(YGG_ERR_INVALID_ARGUMENT, "null argument");
  if (weighted(h)) return set_error(YGG_ERR_UNIMPLEMENTED, "ygg_tree_train_on_gradients takes unit gradients; not combined with example weights");
  if (has_h(h) && !hessians) return set_error(YGG_ERR_INVALID_ARGUMENT, "hessians required for this loss");
  YGG_CUDA(cudaSetDevice(h->ds->device));
  (void)cudaGetLastError();  // stale foreign error, see ygg_gbt_step
  YGG_RETURN_IF_ERROR(apply_pending(h));
  const int64_t n = h->ds->n;
  YGG_CUDA(cudaMemcpyAsync(h->d_g, gradients, n * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  if (has_h(h)) YGG_CUDA(cudaMemcpyAsync(h->d_h, hessians, n * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  const int root_candidate = (n >= h->cfg.min_examples && 1 < h->cfg.max_depth) ? 1 : 0;
  k_begin_iteration<<<1, 1, 0, h->stream>>>(h->d_st, h->d_levels, h->d_fam[0], h->d_slot_node[0], root_candidate);
  h->launches_total++;
  k_absmax<<<elementwise_grid(h), 256, 0, h->stream>>>(h->d_g, n, h->d_st);
  h->launches_total++;
  YGG_RETURN_IF_ERROR(check_launch("k_absmax"));
  YGG_RETURN_IF_ERROR(grow_tree(h, h->d_nodes_scratch));
  if (h->cfg.growing_strategy == 1) YGG_RETURN_IF_ERROR(best_first_prune(h, h->d_nodes_scratch));
  YGG_RETURN_IF_ERROR(check_device_error(h));
  std::vector<ygg_node> flat;
  YGG_RETURN_IF_ERROR(fetch_tree(h, h->d_nodes_scratch, &flat, true));
  *n_nodes = static_cast<int32_t>(flat.size());
  if (static_cast<int32_t>(flat.size()) > capacity) return set_error(YGG_ERR_INVALID_ARGUMENT, "capacity %d < %zu nodes", capacity, flat.size());
  std::memcpy(out, flat.data(), flat.size() * sizeof(ygg_node));
  return YGG_OK;
}

int ygg_gbt_debug_capture_histograms(ygg_gbt* h, int32_t enabled) {
  if (!h) return set_error(YGG_ERR_INVALID_ARGUMENT, "null handle");
  h->capture_hist = enabled != 0;
  return YGG_OK;
}

int ygg_gbt_debug_level_histograms(ygg_gbt* h, int32_t level, ygg_hist_level_info* info, uint64_t* sum, uint64_t* hsum,
                                   uint32_t* cnt, int32_t* slot_node, int32_t capacity) {
  if (!h || !info) return set_error(YGG_ERR_INVALID_ARGUMENT, "null argument");
  if (h->capture_nodes == nullptr) return set_error(YGG_ERR_INVALID_ARGUMENT, "no tree was grown with the histogram capture on");
  if (level < 0 || level >= static_cast<int>(h->capture_info.size()))
    return set_error(YGG_ERR_INVALID_ARGUMENT, "level %d: the captured tree has %zu histogram levels", level, h->capture_info.size());
  YGG_CUDA(cudaSetDevice(h->ds->device));
  YGG_CUDA(cudaStreamSynchronize(h->stream));
  float* in_g = info->g;
  float* in_h2 = info->h2;
  uint8_t* in_sel = info->selected;
  *info = h->capture_info[level];
  info->g = in_g; info->h2 = in_h2; info->selected = in_sel;
  DeviceState st;
  YGG_CUDA(cudaMemcpy(&st, h->d_capture_st, sizeof(st), cudaMemcpyDeviceToHost));
  info->g_pow2 = st.g_pow2;
  const int64_t n = h->ds->n;
  if (in_g) YGG_CUDA(cudaMemcpy(in_g, h->d_capture_g, n * sizeof(float), cudaMemcpyDeviceToHost));
  if (in_h2) {
    if (h->capture_has_h2) YGG_CUDA(cudaMemcpy(in_h2, h->d_capture_h2, n * sizeof(float), cudaMemcpyDeviceToHost));
    else std::fill(in_h2, in_h2 + n, 1.f);
  }
  if (in_sel) {
    if (h->capture_has_sel) YGG_CUDA(cudaMemcpy(in_sel, h->d_capture_sel, n, cudaMemcpyDeviceToHost));
    else std::memset(in_sel, 1, n);
  }
  // slots of the level: its nodes (depth level + 1) whose histogram was accumulated from rows
  std::vector<NodeRec> nodes(h->max_nodes);
  YGG_CUDA(cudaMemcpy(nodes.data(), h->capture_nodes, sizeof(NodeRec) * h->max_nodes, cudaMemcpyDeviceToHost));
  std::vector<int> pos(h->max_nodes, -1);
  int next = 0;
  preorder_positions(nodes, 0, &next, &pos);
  std::vector<int> node_of_slot;
  for (int i = 0; i < h->max_nodes; i++) {
    if (pos[i] < 0 || nodes[i].depth != level + 1 || nodes[i].slot < 0) continue;
    if (nodes[i].slot >= static_cast<int>(node_of_slot.size())) node_of_slot.resize(nodes[i].slot + 1, -1);
    node_of_slot[nodes[i].slot] = pos[i];
  }
  info->num_slots = static_cast<int32_t>(node_of_slot.size());
  if (!sum && !hsum && !cnt && !slot_node) return YGG_OK;
  if (capacity < info->num_slots) return set_error(YGG_ERR_INVALID_ARGUMENT, "capacity %d < %d slots", capacity, info->num_slots);
  if (hsum && !info->has_hsum) return set_error(YGG_ERR_INVALID_ARGUMENT, "the level has no second histogram plane");
  if (slot_node) std::copy(node_of_slot.begin(), node_of_slot.end(), slot_node);
  // the level buffer as k_hist left it, [slot][feature][256] per plane once the chunking is undone
  const LevelBuf lb = level_buf(h, level_slot_bound(h, level), level == 0 ? 1 : (2 << (level - 1)));
  std::vector<unsigned long long> buf(lb.total_u64);
  YGG_CUDA(cudaMemcpy(buf.data(), h->d_capture + h->capture_off[level], lb.total_u64 * sizeof(unsigned long long),
                      cudaMemcpyDeviceToHost));
  const unsigned long long* b_sum = buf.data();
  const unsigned long long* b_hsum = lb.hsum ? buf.data() + (lb.hsum - lb.sum) : nullptr;
  const uint32_t* b_cnt = reinterpret_cast<const uint32_t*>(buf.data()) + (lb.cnt - reinterpret_cast<uint32_t*>(lb.sum));
  const int F = info->num_features;
  for (int s = 0; s < info->num_slots; s++)
    for (int f = 0; f < F; f++)
      for (int b = 0; b < kMaxBins; b++) {
        size_t oc;
        const size_t o = slot_hist_offset(s, f, b, lb.f_chunk, static_cast<long long>(lb.chunk_u64), &oc);
        const size_t i = (static_cast<size_t>(s) * F + f) * kMaxBins + b;
        if (sum) sum[i] = b_sum[o];
        if (hsum) hsum[i] = b_hsum[o];
        if (cnt) cnt[i] = b_cnt[oc];
      }
  return YGG_OK;
}

int ygg_partition_rows(ygg_dataset* ds, const uint32_t* rows_in, int64_t n, int32_t feature,
                       int32_t threshold_bin, uint32_t* rows_out, int64_t* n_pos) {
  if (!ds || !rows_in || !rows_out || !n_pos) return set_error(YGG_ERR_INVALID_ARGUMENT, "null argument");
  if (feature < 0 || feature >= ds->F) return set_error(YGG_ERR_INVALID_ARGUMENT, "feature %d out of range", feature);
  if (n < 0 || n >= (1ll << 32)) return set_error(YGG_ERR_INVALID_ARGUMENT, "bad row count");
  if (n == 0) { *n_pos = 0; return YGG_OK; }
  for (int64_t i = 0; i < n; i++)
    if (rows_in[i] >= ds->n) return set_error(YGG_ERR_INVALID_ARGUMENT, "row id %u out of range", rows_in[i]);
  YGG_RETURN_IF_ERROR(require_device());
  YGG_CUDA(cudaSetDevice(ds->device));
  (void)cudaGetLastError();  // stale foreign error, see ygg_gbt_step
  uint32_t *d_in = nullptr, *d_out = nullptr, *d_cnt = nullptr;
  const int blocks = static_cast<int>((n + 255) / 256);
  YGG_RETURN_IF_ERROR(dev_alloc(&d_in, n));
  YGG_RETURN_IF_ERROR(dev_alloc(&d_out, n));
  YGG_RETURN_IF_ERROR(dev_alloc(&d_cnt, blocks));
  YGG_CUDA(cudaMemcpy(d_in, rows_in, n * sizeof(uint32_t), cudaMemcpyHostToDevice));
  const uint8_t* col = ds->d_bins + static_cast<int64_t>(feature) * ds->n_pad;
  k_partition_count<<<blocks, 256>>>(col, d_in, n, threshold_bin, d_cnt);
  YGG_RETURN_IF_ERROR(check_launch("k_partition_count"));
  std::vector<uint32_t> cnt(blocks);
  YGG_CUDA(cudaMemcpy(cnt.data(), d_cnt, blocks * sizeof(uint32_t), cudaMemcpyDeviceToHost));
  uint32_t total = 0;
  for (int i = 0; i < blocks; i++) { const uint32_t c = cnt[i]; cnt[i] = total; total += c; }
  YGG_CUDA(cudaMemcpy(d_cnt, cnt.data(), blocks * sizeof(uint32_t), cudaMemcpyHostToDevice));
  k_partition_scatter<<<blocks, 256>>>(col, d_in, n, threshold_bin, d_cnt, total, d_out);
  YGG_RETURN_IF_ERROR(check_launch("k_partition_scatter"));
  YGG_CUDA(cudaMemcpy(rows_out, d_out, n * sizeof(uint32_t), cudaMemcpyDeviceToHost));
  dev_free(d_in); dev_free(d_out); dev_free(d_cnt);
  *n_pos = total;
  return YGG_OK;
}

int ygg_gbt_set_tie_rng_position(ygg_gbt* h, uint64_t words) {
  if (!h) return set_error(YGG_ERR_INVALID_ARGUMENT, "null handle");
  h->tie_rng.seed(h->cfg.random_seed);
  h->tie_rng.discard(words);
  h->tie_rng_ready = true;
  return YGG_OK;
}

int64_t ygg_gbt_best_split_window_bytes(const ygg_gbt* h) {
  if (!h) return 0;
  return 2ll * h->world * h->max_level_nodes * static_cast<int64_t>(sizeof(ShardBest)) + 2ll * h->world * 4 + 64;
}

int ygg_gbt_set_best_split_window(ygg_gbt* h, void* const* peer_windows, int32_t world) {
  if (!h || !peer_windows) return set_error(YGG_ERR_INVALID_ARGUMENT, "null argument");
  if (world != h->world || world < 2) return set_error(YGG_ERR_INVALID_ARGUMENT, "the windows of %d ranks for a handle sharded over %d", world, h->world);
  if (h->trees_done > 0) return set_error(YGG_ERR_INVALID_ARGUMENT, "the window must be set before training");
  YGG_CUDA(cudaSetDevice(h->ds->device));
  dev_free(h->d_peer_windows);
  h->d_peer_windows = nullptr;
  YGG_RETURN_IF_ERROR(dev_alloc(&h->d_peer_windows, world));
  YGG_CUDA(cudaMemcpy(h->d_peer_windows, peer_windows, sizeof(void*) * world, cudaMemcpyHostToDevice));
  h->exchange_epoch = 0;
  return YGG_OK;
}

int ygg_gbt_tie_stats(ygg_gbt* h, int64_t* renamed, int64_t* unresolved) {
  if (!h || !renamed || !unresolved) return set_error(YGG_ERR_INVALID_ARGUMENT, "null argument");
  YGG_CUDA(cudaSetDevice(h->ds->device));
  YGG_RETURN_IF_ERROR(resolve_ties(h, h->trees_done));
  *renamed = h->ties_renamed;
  *unresolved = h->ties_unresolved;
  return YGG_OK;
}

int ygg_gbt_set_profiling(ygg_gbt* h, int32_t enabled) {
  if (!h) return set_error(YGG_ERR_INVALID_ARGUMENT, "null handle");
  h->profiling = enabled != 0;
  h->profile.clear();
  h->launches_total = 0;
  return YGG_OK;
}

int ygg_gbt_get_profile(ygg_gbt* h, const char* name, double* ms, int64_t* launches) {
  if (!h || !name || !ms || !launches) return set_error(YGG_ERR_INVALID_ARGUMENT, "null argument");
  collect_profile(h);
  if (std::strcmp(name, "total") == 0) {
    double t = 0;
    for (auto& kv : h->profile)
      if (kv.first.rfind("hist_L", 0) != 0) t += kv.second.ms;
    *ms = t;
    *launches = h->launches_total;
    return YGG_OK;
  }
  auto it = h->profile.find(name);
  if (it == h->profile.end()) { *ms = 0; *launches = 0; return YGG_OK; }
  *ms = it->second.ms;
  *launches = it->second.launches;
  return YGG_OK;
}

int ygg_gbt_save_ydf(ygg_gbt* h, const char* directory, const char* label_name, const uint8_t* data_spec_pb,
                     int64_t data_spec_len, int32_t label_col_idx, const int32_t* feature_col_idx) {
  (void)label_name;
  if (!h || !directory || !data_spec_pb || !feature_col_idx) return set_error(YGG_ERR_INVALID_ARGUMENT, "null argument");
  YGG_CUDA(cudaSetDevice(h->ds->device));
  YGG_RETURN_IF_ERROR(apply_pending(h));
  YGG_RETURN_IF_ERROR(resolve_ties(h, h->trees_done));
  std::vector<ygg_node> all;
  std::vector<int64_t> offsets(1, 0);
  const int n_trees = ygg_gbt_num_trees(h), n_logs = ygg_gbt_num_iterations(h);
  std::vector<float> loss(n_logs), sec(n_logs), vloss, vsec;
  for (int t = 0; t < n_trees; t++) {
    std::vector<ygg_node> flat;
    YGG_RETURN_IF_ERROR(fetch_tree(h, h->d_nodes_all + static_cast<size_t>(t) * h->max_nodes, &flat));
    all.insert(all.end(), flat.begin(), flat.end());
    offsets.push_back(static_cast<int64_t>(all.size()));
  }
  for (int t = 0; t < n_logs; t++) YGG_RETURN_IF_ERROR(ygg_gbt_train_loss(h, t, &loss[t], &sec[t]));
  float final_vloss = 0.f;
  int32_t triggered = 0;
  if (h->vds != nullptr) {
    vloss.resize(n_logs); vsec.resize(n_logs);
    for (int t = 0; t < n_logs; t++) YGG_RETURN_IF_ERROR(ygg_gbt_validation_loss(h, t, &vloss[t], &vsec[t]));
    YGG_RETURN_IF_ERROR(ygg_gbt_final_validation(h, &final_vloss, &triggered));
  }
  ygg_model_desc d;
  std::memset(&d, 0, sizeof(d));
  d.directory = directory;
  d.task = is_logit(h) ? 1 : 2;
  d.num_trees_per_iter = h->K;
  d.loss = h->cfg.loss;
  d.use_hessian_gain = h->cfg.use_hessian_gain;
  d.initial_prediction = h->initial_prediction;
  d.num_trees = n_trees;
  d.num_log_entries = n_logs;
  d.valid_loss = vloss.empty() ? nullptr : vloss.data();
  d.valid_secondary = vsec.empty() ? nullptr : vsec.data();
  d.has_validation_loss = h->vds != nullptr ? 1 : 0;
  d.validation_loss = final_vloss;
  d.early_stopping_triggered = triggered;
  d.trees = all.data();
  d.tree_offsets = offsets.data();
  d.num_features = h->ds->F;
  d.feature_col_idx = feature_col_idx;
  d.label_col_idx = label_col_idx;
  d.data_spec_pb = data_spec_pb;
  d.data_spec_len = data_spec_len;
  d.train_loss = loss.data();
  d.train_secondary = sec.data();
  d.feature_num_values = h->ds->num_bins.data();
  const int st = ygg_model_write_ydf(&d);
  if (st != YGG_OK) return set_error(st, "could not write the model directory %s", directory);
  return YGG_OK;
}

}  // extern "C"
