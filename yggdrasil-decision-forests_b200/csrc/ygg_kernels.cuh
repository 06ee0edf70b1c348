// ygg_kernels.cuh — hand-written sm_100a kernels of the GBT histogram split finder.
//
// Kernel inventory (DESIGN.md §4), one boosting iteration = pred/grad -> quantise -> per level
// {hist, scan, select, partition, node_stats}:
//   k_pred_grad   UpdatePredictions + Loss + UpdateGradients, fused (gradient_boosted_trees.cc:1445,
//                 :1544, :1575; loss_imp_binomial.cc:124-144, loss_imp_mean_square_error.cc:96-120)
//   k_quantize    fixed-point encoding of g/h, root statistics (loss_utils.cc:49-132 for the root)
//   k_hist        FillExampleBucketSet for all open nodes x features of one level
//                 (splitter_scanner.h:859-909) — the HBM-bound hot kernel
//   k_scan        ScanSplits<bucket_interpolation=true> (splitter_scanner.h:931-1101)
//   k_select      FindBestConditionConcurrentManager's ordered arg-max (training.cc:1728-1746) + NodeTrain
//                 bookkeeping (training.cc:4865-5049)
//   k_partition   SplitExamplesInPlace (training.cc:5243-5305) as a node-id relabel + child statistics
//   k_node_stats  SetLeafValueWithNewtonRaphsonStep (loss_utils.cc:49-132)
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "ygg_device.cuh"
#include "ygg_hist.cuh"

namespace ygg {

// ---------------------------------------------------------------------------------------------
// small helpers
__device__ __forceinline__ unsigned long long warp_sum_u64(unsigned long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Exponent e of the gradient scale P = 2^e: the smallest power of two STRICTLY above max|g| (from its float bits; 1 when
// every g is 0).  Strictly above, so that g = +max|g| quantises to rint(g * 2^23 / P) + 2^23 < 2^24 instead of being
// clamped one unit short (the biased 24-bit code has no room for +P).
__device__ __forceinline__ int pow2_above_exp(unsigned int max_bits) {
  if (max_bits == 0u) return 0;
  const int be = static_cast<int>(max_bits >> 23);          // biased exponent; 0: subnormal m * 2^-149
  return be != 0 ? be - 126 : 32 - __clz(static_cast<int>(max_bits)) - 149;
}
// 2^k as a double, k in [-1022, 1023].  The quantisers scale by 2^(23-e), 2^(30-e), 2^(31-2e): for tiny or huge P these
// leave float range (2^(31-2e) overflows once P <= 2^-49), never double range.
__device__ __forceinline__ double pow2_d(int k) { return __longlong_as_double(static_cast<long long>(1023 + k) << 52); }

// Power of two P with v <= P, from the float bits of max v (inclusive: the caller's quantiser keeps v = P exact).
__device__ __forceinline__ float pow2_cover(unsigned int max_bits) {
  if (max_bits == 0u) return 1.f;
  const int e = static_cast<int>(max_bits >> 23) - 127;
  const bool exact = (max_bits & 0x7FFFFFu) == 0u;
  return exact ? exp2f(static_cast<float>(e)) : exp2f(static_cast<float>(e + 1));
}

// Deterministic loss reduction (ADVICE r01): every CTA leaves its partial sums in its own slot, the CTA that finishes
// last adds the slots in index order.  For a given grid the result is the same bit pattern on every run (a double
// atomicAdd across CTAs is not), so early stopping cannot flip on summation noise.
constexpr int kLossParts = 4096;
struct LossPartials {
  double loss[kLossParts];
  unsigned long long correct[kLossParts];
  unsigned int done;
};
// Called by ALL threads of every CTA (256 threads) of a grid of <= kLossParts CTAs, with the CTA's sums in thread 0; the CTA
// that arrives last adds the slots: thread t the slots t, t + 256, ... in that order, thread 0 the 256 partial sums in thread
// order — a fixed association, whatever the arrival order.
__device__ __forceinline__ void reduce_loss_in_order(LossPartials* part, double loss, unsigned long long correct, double* out_loss,
                                                     unsigned long long* out_correct) {
  __shared__ bool s_last;
  __shared__ double s_l[256];
  __shared__ unsigned long long s_c[256];
  if (threadIdx.x == 0) {
    part->loss[blockIdx.x] = loss;
    part->correct[blockIdx.x] = correct;
    __threadfence();
    s_last = atomicInc(&part->done, gridDim.x - 1) == gridDim.x - 1;   // wraps to 0 for the next use
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  double l = 0;
  unsigned long long c = 0;
  for (unsigned int i = threadIdx.x; i < gridDim.x; i += 256) {
    l += reinterpret_cast<volatile double*>(part->loss)[i];
    c += reinterpret_cast<volatile unsigned long long*>(part->correct)[i];
  }
  s_l[threadIdx.x] = l;
  s_c[threadIdx.x] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < 256; i++) { l += s_l[i]; c += s_c[i]; }
    *out_loss = l;
    *out_correct = c;
  }
}

struct GradParams {
  int64_t n;
  float* pred;
  const uint8_t* label_u8;   // binomial: 1 if the row's class is the positive one ("2")
  const float* label_f32;    // regression target
  const uint16_t* node_of_row;
  const NodeRec* pending_tree;  // tree whose leaves are still to be added to pred (or null)
  float* g;
  float* h;
  DeviceState* st;
  int compute_grad;
  LossPartials* partials;
  // example weights (WEIGHTED instantiation; loss_utils.cc:81-89, splitter_accumulator.h:1552-1560): g / h receive the
  // float products w*g / w*h the reference accumulates, g2w the product (w*g)*g of its sum of squares
  const float* weight;
  float* g2w;
  float correct_scale;       // the weight of a correctly classified row is counted as rint(w * correct_scale)
};

// expf / logf evaluated in double and rounded once: within the reference's glibc (<1 ulp,
// correctly rounded for all but ~1e-3 of inputs) far more often than the 2-ulp device expf.
__device__ __forceinline__ float exp_rn(float x) { return static_cast<float>(exp(static_cast<double>(x))); }
__device__ __forceinline__ float log_rn(float x) { return static_cast<float>(log(static_cast<double>(x))); }

template <int LOSS, bool WEIGHTED = false>
__global__ void __launch_bounds__(256) k_pred_grad(GradParams p) {
  double loss = 0;
  unsigned long long correct = 0;
  float gmax = 0.f, g2max = 0.f;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r < p.n; r += stride) {
    float pred = p.pred[r];
    float weight = 1.f;
    if (WEIGHTED) weight = p.weight[r];
    if (p.pending_tree != nullptr) {
      // UpdatePredictionWithSingleUnivariateTree (loss_utils.cc:214-229): the leaf of a row is its
      // final node id, no traversal needed.
      pred += p.pending_tree[p.node_of_row[r]].leaf_value;
      p.pred[r] = pred;
      if (LOSS == 0) {
        // loss_imp_binomial.cc:204-234, float arithmetic as in the reference.
        const float label = p.label_u8[r] ? 1.f : 0.f;
        const float inner = label * pred - log_rn(1.f + exp_rn(pred));
        const float term = WEIGHTED ? 2 * weight * inner : 2 * inner;   // :221-223 / :228-229
        loss -= term;
        const bool predicted_pos = pred > 0.f;
        if (predicted_pos == (p.label_u8[r] != 0))
          correct += WEIGHTED ? static_cast<unsigned long long>(__float2ull_rn(weight * p.correct_scale)) : 1ull;
      } else {
        const float d = p.label_f32[r] - pred;  // metric/metric.cc:2097-2115
        loss += WEIGHTED ? weight * d * d : d * d;
      }
    }
    if (p.compute_grad) {
      float g, h;
      if (LOSS == 0) {
        const float label = p.label_u8[r] ? 1.f : 0.f;
        const float proba = 1.f / (1.f + exp_rn(-pred));
        g = label - proba;
        h = proba * (1 - proba);
      } else {
        g = p.label_f32[r] - pred;
        h = 1.f;
      }
      if (WEIGHTED) {
        const float wg = g * weight;          // value * weight (distribution.h:58-64) == weight * unit_gradient
        const float g2 = wg * g;
        p.g[r] = wg;
        p.h[r] = weight * h;
        p.g2w[r] = g2;
        gmax = fmaxf(gmax, fabsf(wg));
        g2max = fmaxf(g2max, g2);
      } else {
        p.g[r] = g;
        if (LOSS == 0) p.h[r] = h;
        gmax = fmaxf(gmax, fabsf(g));
      }
    }
  }
  // block reduction
  loss = warp_sum_f64(loss);
  correct = warp_sum_u64(correct);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    gmax = fmaxf(gmax, __shfl_xor_sync(0xffffffffu, gmax, o));
    if (WEIGHTED) g2max = fmaxf(g2max, __shfl_xor_sync(0xffffffffu, g2max, o));
  }
  __shared__ double s_loss[8];
  __shared__ unsigned long long s_cor[8];
  __shared__ float s_gmax[8], s_g2max[8];
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) { s_loss[w] = loss; s_cor[w] = correct; s_gmax[w] = gmax; s_g2max[w] = g2max; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < 8; i++) { loss += s_loss[i]; correct += s_cor[i]; gmax = fmaxf(gmax, s_gmax[i]); g2max = fmaxf(g2max, s_g2max[i]); }
    if (p.compute_grad) atomicMax(&p.st->gmax_bits, __float_as_uint(gmax));
    if (WEIGHTED && p.compute_grad) atomicMax(&p.st->g2w_max_bits, __float_as_uint(g2max));
  }
  if (p.pending_tree != nullptr) reduce_loss_in_order(p.partials, loss, correct, &p.st->loss_sum, &p.st->correct);
}

// ---------------------------------------------------------------------------------------------
struct QuantParams {
  int64_t n;
  int64_t n_pad;
  const float* g;
  const float* h;          // null for squared error (h == 1)
  uint32_t* q24;           // [n_pad]  biased 24-bit quantised gradient of every row
  uint32_t* hq24;          // [n_pad]  24-bit quantised hessian (hessian histogram only, else null)
  uint2* act;              // root level active lists (dense): (q24 | slot 0, row offset)
  uint32_t* act_h;
  int32_t* act_count;
  uint16_t* node_of_row;
  DeviceState* st;
  unsigned long long* stats;  // [3] root statistics (fixed point sums of g, h, g^2 over this rank's rows)
  int root_candidate;
  float h_pow2;
  float fixed_g_pow2;      // > 0: use this P instead of the one derived from max|g| (binomial: |g| <= 1)
  const uint8_t* selected; // stochastic gradient boosting: 1 = the row is in this iteration's sample (null: all rows)
  const float* hist_h;     // example weights: the second histogram plane sums THESE (the weights) instead of h (null: h)
  float hist_h_pow2;       // power of two >= max hist_h
};

__device__ __forceinline__ uint32_t quant_biased(float v, double scale, uint32_t bias, uint32_t vmax) {
  // rint(v * scale) + bias, clamped to [0, vmax]; scale is a power of two so v*scale is exact.
  const double t = rint(static_cast<double>(v) * scale) + static_cast<double>(bias);
  return static_cast<uint32_t>(fmin(fmax(t, 0.0), static_cast<double>(vmax)));
}
// 31-bit statistics quantisers.  `scale` is a power of two, so v*scale is exact; the conversion rounds to the nearest
// integer.  Saturating.  (A float scale gives the same results wherever it is finite: the product is exact either way.)
__device__ __forceinline__ uint32_t quant_stat_signed(float v, double scale) {   // -> [0, 2^31], bias 2^30
  const int t = __double2int_rn(static_cast<double>(v) * scale);                 // |v*scale| <= 2^30
  return static_cast<uint32_t>(min(max(t, -(1 << 30)), (1 << 30)) + (1 << 30));
}
__device__ __forceinline__ uint32_t quant_stat_unsigned(float v, double scale) {  // v >= 0 -> [0, 2^31]
  return min(__double2uint_rn(static_cast<double>(v) * scale), 0x80000000u);  // v == its power-of-two cover stays exact
}

__global__ void __launch_bounds__(256) k_quantize(QuantParams p) {
  const int e = p.fixed_g_pow2 > 0.f ? ilogbf(p.fixed_g_pow2) : pow2_above_exp(p.st->gmax_bits);   // P = 2^e
  const float P = ldexpf(1.f, e);
  const double qscale = pow2_d(kQBits - 1 - e);    // 2^23 / P
  const double sscale = pow2_d(kSBits - 1 - e);    // 2^30 / P
  const double s2scale = pow2_d(kSBits - 2 * e);   // g^2 in [0, P^2]
  const float hscale = static_cast<float>(1u << kSBits) / p.h_pow2;    // h in [0, h_pow2]
  const float hqscale = static_cast<float>(1u << kQBits) / (p.hist_h != nullptr ? p.hist_h_pow2 : p.h_pow2);
  unsigned long long sg = 0, sh = 0, sg2 = 0;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r < p.n_pad; r += stride) {
    if ((r & (kBlockRows - 1)) == 0) {
      // one thread per block publishes the block's active-row count: every real row at the root
      const int64_t left = p.n - r;
      p.act_count[r / kBlockRows] = p.root_candidate ? static_cast<int32_t>(left < 0 ? 0 : (left > kBlockRows ? kBlockRows : left)) : 0;
    }
    if (r < p.n) {
      const float g = p.g[r];
      const uint32_t q = quant_biased(g, qscale, kQBias, kQMax);
      p.q24[r] = q;
      p.act[r] = make_uint2(q, static_cast<uint32_t>(r & (kBlockRows - 1)));  // slot 0
      p.node_of_row[r] = 0;
      const bool sel = p.selected == nullptr || p.selected[r] != 0;   // the tree is trained on the sampled rows only
      if (sel) {
        sg += quant_stat_signed(g, sscale);
        sg2 += quant_stat_unsigned(g * g, s2scale);  // float product, as loss_utils.cc:94
      }
      if (p.h != nullptr) {
        const float h = p.h[r];
        if (sel) sh += quant_stat_unsigned(h, hscale);
        if (p.hq24 != nullptr) {
          // [0, 2^24] inclusive: h == h_pow2 (binomial p = 1/2) must stay exact, or categories whose
          // hessian priorities tie in exact arithmetic would be ordered by rounding noise
          const float hh = p.hist_h != nullptr ? p.hist_h[r] : h;
          const uint32_t hq = static_cast<uint32_t>(fminf(rintf(hh * hqscale), static_cast<float>(kQMax + 1u)));
          p.hq24[r] = hq;
          p.act_h[r] = hq;
        }
      }
    }
  }
  sg = warp_sum_u64(sg); sh = warp_sum_u64(sh); sg2 = warp_sum_u64(sg2);
  __shared__ unsigned long long s[3][8];
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) { s[0][w] = sg; s[1][w] = sh; s[2][w] = sg2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < 8; i++) { sg += s[0][i]; sh += s[1][i]; sg2 += s[2][i]; }
    atomicAdd(&p.stats[0], sg);
    atomicAdd(&p.stats[1], sh);
    atomicAdd(&p.stats[2], sg2);
    if (blockIdx.x == 0) { p.st->g_pow2 = P; p.st->h_pow2 = p.h_pow2; }
  }
}

// Stochastic gradient boosting (SampleTrainingExamples, gradient_boosted_trees.cc:2932-2956): the root's active lists
// hold the sampled rows only.  k_quantize wrote them dense; one CTA per 8192-row block compacts them in place, in row
// order (entries go to registers first, so reading and writing the same list is safe).
constexpr int kCompactThreads = 512;
__global__ void __launch_bounds__(kCompactThreads) k_compact_root(uint2* act, uint32_t* act_h, int32_t* act_count,
                                                                  const uint8_t* __restrict__ selected, int64_t n, int n_blocks) {
  constexpr int R = kBlockRows / kCompactThreads;   // 16 consecutive rows per thread
  __shared__ int s_warp_tot[kCompactThreads / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int blk = blockIdx.x; blk < n_blocks; blk += gridDim.x) {
    const int64_t base = static_cast<int64_t>(blk) * kBlockRows;
    uint2 e[R];
    uint32_t eh[R];
    uint32_t mask = 0;
#pragma unroll
    for (int j = 0; j < R; j++) {
      const int64_t r = base + threadIdx.x * R + j;
      e[j] = act[r];
      eh[j] = act_h != nullptr ? act_h[r] : 0u;
      if (r < n && selected[r] != 0) mask |= 1u << j;
    }
    const int mine = __popc(mask);
    int incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    if (lane == 31) s_warp_tot[warp] = incl;
    __syncthreads();
    int offset = incl - mine, total = 0;
    for (int w = 0; w < kCompactThreads / 32; w++) {
      const int t = s_warp_tot[w];
      if (w < warp) offset += t;
      total += t;
    }
    if (threadIdx.x == 0) act_count[blk] = total;
    __syncthreads();
#pragma unroll
    for (int j = 0; j < R; j++) {
      if (mask & (1u << j)) {
        act[base + offset] = e[j];
        if (act_h != nullptr) act_h[base + offset] = eh[j];
        offset++;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// k_scan: one CTA of 256 threads (thread b = bin b) per (family, feature).
struct ScanParams {
  int level;
  const LevelDesc* levels;
  const Family* families;     // families of this level
  NodeRec* nodes;
  int f_begin, f_count;       // features scanned by this rank
  int hist_f_begin, hist_f_count;  // features present in the slot histograms
  int f_chunk;                     // chunked slot-histogram layout, see HistParams
  long long chunk_stride;
  const int32_t* num_bins;    // per dataset feature
  const int32_t* na_bin;
  const int32_t* feature_type;  // per dataset feature: 0 discretized numerical, 1 categorical
  uint32_t* cand_mask;        // [level nodes][f_count][8] positive-category masks of categorical candidates
  double l2_categorical;
  // direct histograms of this level, accumulated from rows: [slot][hist_f_count][256]
  const unsigned long long* slot_sum;
  const uint32_t* slot_cnt;
  const unsigned long long* slot_hsum;
  // per-node histograms (parents of the next level): [level nodes][f_count][256]
  unsigned long long* hist_sum;
  uint32_t* hist_cnt;
  unsigned long long* hist_hsum;
  const unsigned long long* phist_sum; // parent level
  const uint32_t* phist_cnt;
  const unsigned long long* phist_hsum;
  Candidate* cand;            // [level nodes][f_count]
  const DeviceState* st;
  int min_num_obs;
  int use_hessian;
  int has_h;                  // 0: h == 1 for every row, the hessian sum of a bin is its count
  int subtract_parent;
  double l1, l2;
  int write_derived;          // 0 on the last level (no histogram of this level is ever a parent)
  const float* bucket_values; // [F][256] value of every bucket of the features under the exact threshold rule (or null)
  const int32_t* exact_rule;  // [F] 1: the feature has bucket values
  // example weights (variance gain): the hessian plane holds the bins' weight sums in units of w_inv; they take the
  // place of the counts in the score (LabelNumericalBucket<weighted>: value.count = sum of weights), the integer
  // counts keep deciding min_examples
  int weighted;
  double w_inv;
};

__device__ __forceinline__ double l1_threshold_d(double v, double l1) {
  if (l1 == 0.0) return v;
  const double len = fmax(0.0, fabs(v) - l1);
  return v > 0 ? len : -len;
}

// Block-wide inclusive scan of (count, sum, hsum) over 256 threads.
struct Scan3 { long long c; long long s; long long h; };
__device__ __forceinline__ Scan3 block_inclusive_scan(Scan3 v, Scan3* s_warp /*[8]*/, Scan3* total) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const long long c = __shfl_up_sync(0xffffffffu, v.c, o);
    const long long s = __shfl_up_sync(0xffffffffu, v.s, o);
    const long long h = __shfl_up_sync(0xffffffffu, v.h, o);
    if (lane >= o) { v.c += c; v.s += s; v.h += h; }
  }
  if (lane == 31) s_warp[w] = v;
  __syncthreads();
  Scan3 off{0, 0, 0}, tot{0, 0, 0};
  for (int i = 0; i < 8; i++) {
    if (i < w) { off.c += s_warp[i].c; off.s += s_warp[i].s; off.h += s_warp[i].h; }
    tot.c += s_warp[i].c; tot.s += s_warp[i].s; tot.h += s_warp[i].h;
  }
  __syncthreads();
  v.c += off.c; v.s += off.s; v.h += off.h;
  *total = tot;
  return v;
}

// Scans one node's 256-bin histogram held one bin per thread; thread 0 writes the Candidate.
__device__ void scan_node(const ScanParams& p, const NodeRec& node, int f_global, long long cnt,
                          long long sq /*unbiased quantised sum*/, long long hq, Candidate* out) {
  __shared__ Scan3 s_warp[8];
  __shared__ double s_best_score[8];
  __shared__ int s_best_b[8];
  __shared__ int s_interp[8];
  const int b = threadIdx.x;
  const int B = p.num_bins[f_global];
  Scan3 tot;
  const Scan3 inc = block_inclusive_scan(Scan3{cnt, sq, hq}, s_warp, &tot);
  const double ginv = static_cast<double>(p.st->g_pow2) / static_cast<double>(1u << (kQBits - 1));
  const double hinv = static_cast<double>(p.st->h_pow2) / static_cast<double>(1u << kQBits);
  const long long n_neg = inc.c, n_pos = tot.c - inc.c;
  bool valid = (b <= B - 2) && (n_pos >= p.min_num_obs) && (n_neg >= p.min_num_obs);
  double score = 0.0;
  double min_score = 0.0;
  if (!p.use_hessian) {
    // Variance reduction (V0 - V_pos - V_neg) / c0 (splitter_scanner.h:911-926,
    // splitter_accumulator.h:1517-1519).  With consistent sums the sum-of-squares terms cancel and
    // the numerator is the between-group sum of squares n_pos*n_neg/c0 * (mean_pos - mean_neg)^2,
    // evaluated from the integer sums as d^2 / (n_pos*n_neg*c0) with d = S_pos*n_neg - S_neg*n_pos:
    // non-negative by construction and exactly 0 for equal means (DESIGN.md §5).
    double c0 = static_cast<double>(tot.c);
    double np_ = static_cast<double>(n_pos), nn_ = static_cast<double>(n_neg);
    if (p.weighted) {   // weight sums instead of counts (exact integers in units of w_inv)
      c0 = static_cast<double>(tot.h) * p.w_inv;
      np_ = static_cast<double>(tot.h - inc.h) * p.w_inv;
      nn_ = static_cast<double>(inc.h) * p.w_inv;
      valid = valid && np_ > 0.0 && nn_ > 0.0;
    }
    if (valid) {
      double dq = static_cast<double>(tot.s - inc.s) * nn_ - static_cast<double>(inc.s) * np_;
      if (p.weighted) {
        // Every sum is a sum of ROUNDED products (w*g and w at 2^-24 of their scales), so a node whose rows all carry the
        // same gradient gives d = 0 only up to +-half a unit per row: below that bound d is not distinguishable from 0 and
        // the split would be decided by rounding (the reference's doubles flip the same coin at 1e-16).  Unweighted sums
        // are exact integers and need no such floor.
        const double half_units = 0.5 * (static_cast<double>(n_pos) * nn_ + static_cast<double>(n_neg) * np_ +
                                         (fabs(static_cast<double>(tot.s - inc.s)) * static_cast<double>(n_neg) +
                                          fabs(static_cast<double>(inc.s)) * static_cast<double>(n_pos)) * p.w_inv);
        if (fabs(dq) <= half_units) dq = 0.0;
      }
      const double d = dq * ginv;
      score = (d / np_) * (d / nn_) / (c0 * c0);
    }
  } else {
    // splitter_accumulator.h:755-773 (Score), :1706-1727 (parent / minimum score).
    // the parent's term from the SAME histogram sums as the children's (the totals over the bins are the node's sums at
    // the histogram's resolution): a gain is then a difference of like-rounded numbers, and exactly the rounding noise of
    // the formula — as in the reference — on a pure node, instead of the offset between 24-bit and 31-bit sums
    const double g0 = l1_threshold_d(static_cast<double>(tot.s) * ginv, p.l1);
    const double parent_full = g0 * g0 / (fmax(static_cast<double>(tot.h) * hinv, kMinHessianForNewtonStep) + p.l2);
    const double parent_score = p.subtract_parent ? parent_full : 0.0;
    min_score = p.subtract_parent ? 0.0 : parent_full;
    if (valid) {
      const double gn = l1_threshold_d(static_cast<double>(inc.s) * ginv, p.l1);
      const double gp = l1_threshold_d(static_cast<double>(tot.s - inc.s) * ginv, p.l1);
      const double hn = fmax(static_cast<double>(inc.h) * hinv, kMinHessianForNewtonStep) + p.l2;
      const double hp = fmax(static_cast<double>(tot.h - inc.h) * hinv, kMinHessianForNewtonStep) + p.l2;
      score = gp * gp / hp + gn * gn / hn - parent_score;
    }
  }
  // best_score starts at max(condition.split_score (0), MinimumScore()) and needs strict '>'.
  valid = valid && (score > min_score) && (score > 0.0 || p.use_hessian);
  // arg-max with the lowest bin on ties (sequential strict '>' keeps the first maximum).
  double bs = valid ? score : -1.0;
  int bb = valid ? b : 0x7fffffff;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double os = __shfl_xor_sync(0xffffffffu, bs, o);
    const int ob = __shfl_xor_sync(0xffffffffu, bb, o);
    if (os > bs || (os == bs && ob < bb)) { bs = os; bb = ob; }
  }
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { s_best_score[w] = bs; s_best_b[w] = bb; }
  __syncthreads();
  bs = s_best_score[0]; bb = s_best_b[0];
  for (int i = 1; i < 8; i++) {
    if (s_best_score[i] > bs || (s_best_score[i] == bs && s_best_b[i] < bb)) { bs = s_best_score[i]; bb = s_best_b[i]; }
  }
  const bool found = bb != 0x7fffffff;
  // Bucket interpolation (splitter_scanner.h:993-1000, :1076-1086): first non-empty bucket after the
  // best one that the sequential scan visits (indices <= B-2).
  // (hi: the same over ALL buckets, for the exact threshold rule; the scan itself never visits bucket B-1)
  int cand_i = (found && b > bb && b <= B - 1 && cnt > 0) ? b : 0x7fffffff;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cand_i = min(cand_i, __shfl_xor_sync(0xffffffffu, cand_i, o));
  if (lane == 0) s_interp[w] = cand_i;
  __syncthreads();
  int hi = s_interp[0];
  for (int i = 1; i < 8; i++) hi = min(hi, s_interp[i]);
  const int interp = hi <= B - 2 ? hi : 0x7fffffff;
  // n_pos at the best boundary lives in thread bb.
  __shared__ long long s_npos;
  if (found && b == bb) s_npos = n_pos;
  __syncthreads();
  if (threadIdx.x == 0) {
    Candidate c;
    c.found = found ? 1 : 0;
    c.score = found ? static_cast<float>(bs) : 0.f;
    int idx = bb;
    if (found && interp != 0x7fffffff && interp != bb + 1) idx = (bb + interp) / 2;
    c.thr = found ? idx + 1 : 0;
    if (found && p.exact_rule != nullptr && p.exact_rule[f_global] && hi != 0x7fffffff) {
      // exact numerical splitter: threshold = middle of the two values PRESENT in the node around the cut; the bin
      // threshold is the first bucket whose value reaches it (every bucket in between is empty in this node)
      const float* values = p.bucket_values + static_cast<size_t>(f_global) * kMaxBins;
      const float threshold = mid_threshold(values[bb], values[hi]);
      int k = bb + 1;
      while (k < hi && values[k] < threshold) k++;
      c.thr = pack_exact_thr(k, bb, hi);
    }
    c.n_pos = found ? static_cast<int32_t>(s_npos) : 0;
    *out = c;
  }
  __syncthreads();
}

// Categorical feature: FindBestSplit<..., require_label_sorting=true> (splitter_scanner.h:1823-1826,
// :1978-1981).  The buckets (one per category) are sorted by label mean (variance gain,
// splitter_accumulator.h:1492-1494) or by the float hessian priority (:1797-1804, :1699-1701), then
// scanned like a numerical feature without bucket interpolation; the buckets after the best boundary
// form the positive set (splitter_accumulator.h:391-411).  Equal keys are ordered by category
// index (the reference's std::sort leaves that order unspecified; DESIGN.md §6).
__device__ void scan_node_categorical(const ScanParams& p, const NodeRec& node, int f_global, long long cnt,
                                      long long sq, long long hq, Candidate* out, uint32_t* mask_out) {
  __shared__ double s_key[kMaxBins];
  __shared__ int s_idx[kMaxBins];
  __shared__ long long s_cnt[kMaxBins], s_sq[kMaxBins], s_hq[kMaxBins];
  __shared__ Scan3 s_warp[8];
  __shared__ double s_best_score[8];
  __shared__ int s_best_b[8];
  __shared__ uint32_t s_mask[8];
  __shared__ long long s_npos;
  const int b = threadIdx.x;
  const int B = p.num_bins[f_global];
  const double ginv = static_cast<double>(p.st->g_pow2) / static_cast<double>(1u << (kQBits - 1));
  const double hinv = static_cast<double>(p.st->h_pow2) / static_cast<double>(1u << kQBits);
  const double l2 = p.l2_categorical;
  double key;
  if (b >= B) {
    key = __longlong_as_double(0x7FF0000000000000ll);  // +inf: not a category of this feature
  } else if (!p.use_hessian) {
    // Mean() = sum / count, count = the weight sum when weighted (distribution.h; 0 for an empty bucket)
    const double den = p.weighted ? static_cast<double>(hq) * p.w_inv : static_cast<double>(cnt);
    key = (cnt == 0 || den == 0.0) ? 0.0 : (static_cast<double>(sq) * ginv) / den;
  } else {
    const double H = static_cast<double>(hq) * hinv;
    key = H > 0 ? static_cast<double>(static_cast<float>(l1_threshold_d(static_cast<double>(sq) * ginv, p.l1) / (H + l2))) : 0.0;
  }
  s_key[b] = key; s_idx[b] = b; s_cnt[b] = cnt; s_sq[b] = sq; s_hq[b] = hq;
  if (b < 8) s_mask[b] = 0u;
  __syncthreads();
  // bitonic sort of (key, index) pairs, ascending
  for (int k = 2; k <= kMaxBins; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      const int partner = b ^ j;
      if (partner > b) {
        const double ka = s_key[b], kb = s_key[partner];
        const int ia = s_idx[b], ib = s_idx[partner];
        const bool a_gt_b = ka > kb || (ka == kb && ia > ib);
        const bool ascending = (b & k) == 0;
        if (a_gt_b == ascending) { s_key[b] = kb; s_key[partner] = ka; s_idx[b] = ib; s_idx[partner] = ia; }
      }
      __syncthreads();
    }
  }
  const int my = s_idx[b];  // category at sorted position b
  Scan3 tot;
  const Scan3 inc = block_inclusive_scan(Scan3{s_cnt[my], s_sq[my], s_hq[my]}, s_warp, &tot);
  const long long n_neg = inc.c, n_pos = tot.c - inc.c;
  bool valid = (b <= B - 2) && (n_pos >= p.min_num_obs) && (n_neg >= p.min_num_obs);
  double score = 0.0, min_score = 0.0;
  if (!p.use_hessian) {
    double c0 = static_cast<double>(tot.c);
    double np_ = static_cast<double>(n_pos), nn_ = static_cast<double>(n_neg);
    if (p.weighted) {   // weight sums instead of counts (exact integers in units of w_inv)
      c0 = static_cast<double>(tot.h) * p.w_inv;
      np_ = static_cast<double>(tot.h - inc.h) * p.w_inv;
      nn_ = static_cast<double>(inc.h) * p.w_inv;
      valid = valid && np_ > 0.0 && nn_ > 0.0;
    }
    if (valid) {
      double dq = static_cast<double>(tot.s - inc.s) * nn_ - static_cast<double>(inc.s) * np_;
      if (p.weighted) {
        // Every sum is a sum of ROUNDED products (w*g and w at 2^-24 of their scales), so a node whose rows all carry the
        // same gradient gives d = 0 only up to +-half a unit per row: below that bound d is not distinguishable from 0 and
        // the split would be decided by rounding (the reference's doubles flip the same coin at 1e-16).  Unweighted sums
        // are exact integers and need no such floor.
        const double half_units = 0.5 * (static_cast<double>(n_pos) * nn_ + static_cast<double>(n_neg) * np_ +
                                         (fabs(static_cast<double>(tot.s - inc.s)) * static_cast<double>(n_neg) +
                                          fabs(static_cast<double>(inc.s)) * static_cast<double>(n_pos)) * p.w_inv);
        if (fabs(dq) <= half_units) dq = 0.0;
      }
      const double d = dq * ginv;
      score = (d / np_) * (d / nn_) / (c0 * c0);
    }
  } else {
    const double g0 = l1_threshold_d(static_cast<double>(tot.s) * ginv, p.l1);   // see scan_node
    const double parent_full = g0 * g0 / (fmax(static_cast<double>(tot.h) * hinv, kMinHessianForNewtonStep) + l2);
    const double parent_score = p.subtract_parent ? parent_full : 0.0;
    min_score = p.subtract_parent ? 0.0 : parent_full;
    if (valid) {
      const double gn = l1_threshold_d(static_cast<double>(inc.s) * ginv, p.l1);
      const double gp = l1_threshold_d(static_cast<double>(tot.s - inc.s) * ginv, p.l1);
      const double hn = fmax(static_cast<double>(inc.h) * hinv, kMinHessianForNewtonStep) + l2;
      const double hp = fmax(static_cast<double>(tot.h - inc.h) * hinv, kMinHessianForNewtonStep) + l2;
      score = gp * gp / hp + gn * gn / hn - parent_score;
    }
  }
  valid = valid && (score > min_score) && (score > 0.0 || p.use_hessian);
  double bs = valid ? score : -1.0;
  int bb = valid ? b : 0x7fffffff;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double os = __shfl_xor_sync(0xffffffffu, bs, o);
    const int ob = __shfl_xor_sync(0xffffffffu, bb, o);
    if (os > bs || (os == bs && ob < bb)) { bs = os; bb = ob; }
  }
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { s_best_score[w] = bs; s_best_b[w] = bb; }
  __syncthreads();
  bs = s_best_score[0]; bb = s_best_b[0];
  for (int i = 1; i < 8; i++)
    if (s_best_score[i] > bs || (s_best_score[i] == bs && s_best_b[i] < bb)) { bs = s_best_score[i]; bb = s_best_b[i]; }
  const bool found = bb != 0x7fffffff;
  if (found && b > bb && b < B) atomicOr(&s_mask[my >> 5], 1u << (my & 31));
  if (found && b == bb) s_npos = n_pos;
  __syncthreads();
  if (threadIdx.x == 0) {
    Candidate c;
    c.found = found ? 1 : 0;
    c.score = found ? static_cast<float>(bs) : 0.f;
    c.thr = 0;
    c.n_pos = found ? static_cast<int32_t>(s_npos) : 0;
    *out = c;
  }
  if (threadIdx.x < 8) mask_out[threadIdx.x] = found ? s_mask[threadIdx.x] : 0u;
  __syncthreads();
}

template <bool HESS>
__global__ void __launch_bounds__(256) k_scan(ScanParams p) {
  const LevelDesc lv = p.levels[p.level];
  const int fam_idx = blockIdx.x;
  if (fam_idx >= lv.num_families) return;
  const int fl = blockIdx.y;  // local feature
  const Family fam = p.families[fam_idx];
  const int f_global = p.f_begin + fl;
  const int b = threadIdx.x;
  const NodeRec direct = p.nodes[fam.direct];
  size_t osc;
  const size_t os = slot_hist_offset(direct.slot, f_global - p.hist_f_begin, b, p.f_chunk, p.chunk_stride, &osc);
  const long long cnt_d = p.slot_cnt[osc];
  const unsigned long long sum_d = p.slot_sum[os];
  // hessian sums in units of h_pow2 * 2^-24; with h == 1 (h_pow2 = 1) a row contributes 2^24
  const unsigned long long hs_d =
      HESS ? (p.has_h ? p.slot_hsum[os] : (static_cast<unsigned long long>(cnt_d) << kQBits)) : 0ull;
  if (p.write_derived) {
    // keep the direct histogram under its node: it is a parent at the next level
    const size_t od = (static_cast<size_t>(fam.direct - lv.first_node) * p.f_count + fl) * kMaxBins + b;
    p.hist_cnt[od] = static_cast<uint32_t>(cnt_d);
    p.hist_sum[od] = sum_d;
    if (HESS && p.has_h) p.hist_hsum[od] = hs_d;
  }
  const bool categorical = p.feature_type[f_global] == 1;
  if (direct.candidate) {
    const size_t ci = static_cast<size_t>(fam.direct - lv.first_node) * p.f_count + fl;
    if (categorical)
      scan_node_categorical(p, direct, f_global, cnt_d, static_cast<long long>(sum_d) - cnt_d * static_cast<long long>(kQBias),
                            static_cast<long long>(hs_d), &p.cand[ci], p.cand_mask + ci * 8);
    else
      scan_node(p, direct, f_global, cnt_d, static_cast<long long>(sum_d) - cnt_d * static_cast<long long>(kQBias),
                static_cast<long long>(hs_d), &p.cand[ci]);
  }
  if (fam.derived >= 0) {
    const NodeRec derived = p.nodes[fam.derived];
    if (derived.candidate) {
      const LevelDesc plv = p.levels[p.level - 1];
      const size_t op = (static_cast<size_t>(fam.parent - plv.first_node) * p.f_count + fl) * kMaxBins + b;
      const long long cnt_x = static_cast<long long>(p.phist_cnt[op]) - cnt_d;
      const unsigned long long sum_x = p.phist_sum[op] - sum_d;
      const unsigned long long hs_x =
          HESS ? (p.has_h ? p.phist_hsum[op] - hs_d : (static_cast<unsigned long long>(cnt_x) << kQBits)) : 0ull;
      if (p.write_derived) {
        const size_t ox = (static_cast<size_t>(fam.derived - lv.first_node) * p.f_count + fl) * kMaxBins + b;
        p.hist_cnt[ox] = static_cast<uint32_t>(cnt_x);
        p.hist_sum[ox] = sum_x;
        if (HESS && p.has_h) p.hist_hsum[ox] = hs_x;
      }
      const size_t cx = static_cast<size_t>(fam.derived - lv.first_node) * p.f_count + fl;
      if (categorical)
        scan_node_categorical(p, derived, f_global, cnt_x, static_cast<long long>(sum_x) - cnt_x * static_cast<long long>(kQBias),
                              static_cast<long long>(hs_x), &p.cand[cx], p.cand_mask + cx * 8);
      else
        scan_node(p, derived, f_global, cnt_x, static_cast<long long>(sum_x) - cnt_x * static_cast<long long>(kQBias),
                  static_cast<long long>(hs_x), &p.cand[cx]);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// k_select_local: per node of the level, ordered arg-max over this shard's features
// (FindBestConditionConcurrentManager, training.cc:1728-1746: float scores, strict '>', candidate
// order = feature index order).
struct SelectParams {
  int level;
  LevelDesc* levels;
  Family* next_families;
  int32_t* next_slot_node;
  NodeRec* nodes;
  const Candidate* cand;
  const uint32_t* cand_mask;
  const int32_t* feature_type;
  int f_begin, f_count;
  const int32_t* na_bin;
  TieRec* ties;                // [max level nodes] ties of the best split (single GPU; null: not recorded)
  const float* bucket_values;  // see ScanParams (null: no feature under the exact threshold rule)
  const float* na_replacement; // [F] column means of those features
  // best-split exchange over peer memory (ygg_gbt_set_best_split_window): every rank's window, as mapped here;
  // window = [2 parities][world sources][max level nodes] ShardBest, then [2][world] epoch flags
  void* const* peers;          // [world] device array (null: the records were exchanged by the caller's all-gather)
  uint32_t epoch;              // > 0, the same on every rank for this (tree, level)
  ShardBest* shard_best;       // [world][max level nodes] (this rank writes its row; exchange fills the rest)
  int rank, world, max_level_nodes;
  int min_examples, max_depth;
  int sibling_subtraction;
  int max_slots;               // capacity of one histogram pass
  DeviceState* st;
  int max_nodes;
};

__global__ void __launch_bounds__(256) k_select_local(SelectParams p) {
  // One warp per node: lane l scans features l, l+32, ... in increasing order with strict '>'
  // (= first maximum among its features), then the warp keeps the maximum score, lowest feature
  // index on ties — the first maximum in feature order, as the sequential fold gives.
  const LevelDesc lv = p.levels[p.level];
  const int lane = threadIdx.x & 31;
  const int warps_per_block = blockDim.x >> 5;
  for (int j = blockIdx.x * warps_per_block + (threadIdx.x >> 5); j < lv.num_nodes; j += gridDim.x * warps_per_block) {
    float best_score = 0.f;  // NodeCondition.split_score default: a split needs score > 0
    int best_f = 0x7fffffff;
    Candidate best_c{0.f, 0, 0, 0};
    if (p.nodes[lv.first_node + j].candidate) {
      for (int fl = lane; fl < p.f_count; fl += 32) {
        const Candidate c = p.cand[static_cast<size_t>(j) * p.f_count + fl];
        if (c.found && c.score > best_score) { best_score = c.score; best_f = fl; best_c = c; }
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float os = __shfl_xor_sync(0xffffffffu, best_score, o);
      const int of = __shfl_xor_sync(0xffffffffu, best_f, o);
      const int othr = __shfl_xor_sync(0xffffffffu, best_c.thr, o);
      const int onp = __shfl_xor_sync(0xffffffffu, best_c.n_pos, o);
      if (of != 0x7fffffff && (best_f == 0x7fffffff || os > best_score || (os == best_score && of < best_f))) {
        best_score = os; best_f = of; best_c.thr = othr; best_c.n_pos = onp;
      }
    }
    if (p.ties != nullptr) {
      // the other features whose best split has the same float score, in feature order
      int n_ties = 0;
      if (best_f != 0x7fffffff) {
        for (int f0 = 0; f0 < p.f_count; f0 += 32) {
          const int fl = f0 + lane;
          Candidate c{0.f, 0, 0, 0};
          bool tie = false;
          if (fl < p.f_count && fl != best_f) {
            c = p.cand[static_cast<size_t>(j) * p.f_count + fl];
            tie = c.found && c.score == best_score;
          }
          const uint32_t bal = __ballot_sync(0xffffffffu, tie);
          const int pos = n_ties + __popc(bal & ((1u << lane) - 1u));
          if (tie && pos < kMaxTieAlts) {
            TieAlt a{};
            const int fg = p.f_begin + fl;
            a.feature = fg; a.thr = thr_bin_of(c.thr); a.n_pos = c.n_pos; a.cond_type = p.feature_type[fg];
            a.thr_value = p.bucket_values != nullptr ? thr_value_of(c.thr, p.bucket_values + static_cast<size_t>(fg) * kMaxBins) : __builtin_nanf("");
            if (a.cond_type == 1) {
              const uint32_t* m = p.cand_mask + (static_cast<size_t>(j) * p.f_count + fl) * 8;
              const int na = p.na_bin[fg];
              for (int i = 0; i < 8; i++) a.mask[i] = m[i];
              a.na_value = (m[na >> 5] >> (na & 31)) & 1u;
            } else {
              a.na_value = (p.na_bin[fg] >= a.thr) ? 1 : 0;   // na_bin > thr - 1
              if (a.thr_value == a.thr_value) a.na_value = p.na_replacement[fg] >= a.thr_value ? 1 : 0;   // exact rule (:218)
            }
            p.ties[j].alt[pos] = a;
          }
          n_ties += __popc(bal);
        }
      }
      if (lane == 0) p.ties[j].count = n_ties;
    }
    if (lane == 0) {
      ShardBest out{};
      out.feature = -1;
      if (best_f != 0x7fffffff) {
        const int fg = p.f_begin + best_f;
        out.score = best_score; out.feature = fg; out.thr = best_c.thr; out.n_pos = best_c.n_pos;
        out.cond_type = p.feature_type[fg];
        if (out.cond_type == 1) {
          const uint32_t* m = p.cand_mask + (static_cast<size_t>(j) * p.f_count + best_f) * 8;
          const int na = p.na_bin[fg];
#pragma unroll
          for (int i = 0; i < 8; i++) out.mask[i] = m[i];
          out.na_value = (m[na >> 5] >> (na & 31)) & 1u;  // NA replacement in the positive set
        }
      }
      p.shard_best[static_cast<size_t>(p.rank) * p.max_level_nodes + j] = out;
    }
  }
}

// k_select_global: merges the shards' bests in rank order (== global feature order), applies the
// split to the node table, creates the children and lays out the next level.  One CTA.
// Block-wide exclusive scan of one int per thread (blockDim.x <= 1024); returns the exclusive
// prefix and the block total.
__device__ __forceinline__ int block_exclusive_scan(int v, int* s_warp /*[32]*/, int* total) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  int incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) s_warp[w] = incl;
  __syncthreads();
  int off = 0, tot = 0;
  for (int i = 0; i < nw; i++) {
    if (i < w) off += s_warp[i];
    tot += s_warp[i];
  }
  __syncthreads();
  *total = tot;
  return off + incl - v;
}

__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* a) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(a) : "memory");
  return v;
}

__global__ void __launch_bounds__(256) k_select_global(SelectParams p) {
  __shared__ int s_warp[32];
  __shared__ int s_next, s_slots, s_fams;
  const LevelDesc lv = p.levels[p.level];
  if (p.peers != nullptr) {
    // Best-split exchange fused into this kernel: push this rank's records of the level into every rank's window
    // (NVLink peer stores), publish the epoch, wait for every source's epoch in the local window, merge from there.
    // Two parities: a rank can only be one level ahead of the slowest one (it needs everybody's records to go on).
    const size_t mail = static_cast<size_t>(p.world) * p.max_level_nodes * sizeof(ShardBest);
    const size_t par = p.epoch & 1u;
    const uint32_t* mine = reinterpret_cast<const uint32_t*>(p.shard_best + static_cast<size_t>(p.rank) * p.max_level_nodes);
    const int words = lv.num_nodes * static_cast<int>(sizeof(ShardBest) / 4);
    for (int r = 0; r < p.world; r++) {
      uint32_t* dst = reinterpret_cast<uint32_t*>(static_cast<char*>(p.peers[r]) + par * mail +
                                                  static_cast<size_t>(p.rank) * p.max_level_nodes * sizeof(ShardBest));
      for (int i = threadIdx.x; i < words; i += blockDim.x) dst[i] = mine[i];
    }
    __threadfence_system();
    __syncthreads();
    if (static_cast<int>(threadIdx.x) < p.world) {
      uint32_t* flag = reinterpret_cast<uint32_t*>(static_cast<char*>(p.peers[threadIdx.x]) + 2 * mail) + par * p.world + p.rank;
      asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(flag), "r"(p.epoch) : "memory");
      const uint32_t* wait = reinterpret_cast<const uint32_t*>(static_cast<char*>(p.peers[p.rank]) + 2 * mail) + par * p.world + threadIdx.x;
      const long long t0 = clock64();
      while (ld_acquire_sys(wait) < p.epoch) {
        if (clock64() - t0 > 20000000000ll) { p.st->error_flag = 4; break; }   // ~10 s: a peer is gone
      }
    }
    __syncthreads();
    p.shard_best = reinterpret_cast<ShardBest*>(static_cast<char*>(p.peers[p.rank]) + par * mail);
  }
  const int first_next = lv.first_node + lv.num_nodes;
  if (threadIdx.x == 0) { s_next = first_next; s_slots = 0; s_fams = 0; }
  __syncthreads();
  // Nodes are processed in chunks of blockDim.x in node order, so child ids, slots and families are
  // assigned exactly as a serial pass over the level would assign them.
  for (int j0 = 0; j0 < lv.num_nodes; j0 += blockDim.x) {
    const int j = j0 + threadIdx.x;
    const bool in = j < lv.num_nodes;
    bool split = false;
    NodeRec* nd = in ? &p.nodes[lv.first_node + j] : nullptr;
    int depth = 0;
    long long n = 0, n_pos = 0;
    if (in) {
      ShardBest best{};
      best.feature = -1;
      if (nd->candidate) best = merge_shard_bests(p.shard_best, p.world, p.max_level_nodes, j);
      if (best.feature >= 0 && best.n_pos > 0 && best.n_pos < nd->n) {
        nd->feature = best.feature;
        nd->thr_value = p.bucket_values != nullptr && best.cond_type == 0
                            ? thr_value_of(best.thr, p.bucket_values + static_cast<size_t>(best.feature) * kMaxBins) : __builtin_nanf("");
        best.thr = thr_bin_of(best.thr);
        nd->thr = best.thr;
        nd->cond_type = best.cond_type;
#pragma unroll
        for (int i = 0; i < 8; i++) nd->mask[i] = best.mask[i];
        nd->na_value = best.cond_type == 1 ? best.na_value
                                           : ((p.na_bin[best.feature] >= best.thr) ? 1 : 0);  // na_bin > thr - 1
        // exact rule: na_value = na_replacement >= threshold (splitter_accumulator.h:218)
        if (nd->thr_value == nd->thr_value) nd->na_value = p.na_replacement[best.feature] >= nd->thr_value ? 1 : 0;
        nd->score = best.score;
        nd->n_pos = best.n_pos;
        nd->tie_count = 0;
        if (p.ties != nullptr) {
          const TieRec& tr = p.ties[j];
          nd->tie_count = tr.count;
          for (int i = 0; i < min(tr.count, kMaxTieAlts); i++) nd->tie[i] = tr.alt[i];
        }
        split = true;
        depth = nd->depth; n = nd->n; n_pos = best.n_pos;
      } else {
        nd->feature = -1;
      }
    }
    int n_split_total;
    const int rank = block_exclusive_scan(split ? 1 : 0, s_warp, &n_split_total);
    const int base_next = s_next;
    bool want_pair = false, cand_p = false, cand_n = false, pos_small = false;
    int pos = -1, neg = -1;
    if (split) {
      pos = base_next + 2 * rank;
      neg = pos + 1;
      if (neg >= p.max_nodes) {   // cannot happen for depth-bounded trees; keep the tree consistent
        p.st->error_flag = 2;
        nd->feature = -1;
        split = false;
      }
    }
    if (split) {
      nd->pos_child = pos;
      nd->neg_child = neg;
      NodeRec cp{}, cn{};
      cp.parent = cn.parent = lv.first_node + j;
      cp.depth = cn.depth = depth + 1;
      cp.feature = cn.feature = -1;
      cp.pos_child = cp.neg_child = cn.pos_child = cn.neg_child = -1;
      cp.sibling = neg; cn.sibling = pos;
      cp.n = n_pos;
      cn.n = n - n_pos;
      cp.slot = cn.slot = -1;
      // NodeTrain stop tests (training.cc:4909-4914).
      cand_p = (cp.n >= p.min_examples && cp.depth < p.max_depth);
      cand_n = (cn.n >= p.min_examples && cn.depth < p.max_depth);
      cp.candidate = cand_p ? 1 : 0;
      cn.candidate = cand_n ? 1 : 0;
      pos_small = cp.n <= cn.n;
      p.nodes[pos] = cp;
      p.nodes[neg] = cn;
      want_pair = cand_p || cand_n;
    }
    // Slots / families: with sibling subtraction one slot (the smaller child) and one family per
    // split that has a candidate child; without it one slot and one family per candidate child.
    const int my_slots = !split ? 0 : (p.sibling_subtraction ? (want_pair ? 1 : 0) : (cand_p ? 1 : 0) + (cand_n ? 1 : 0));
    int slots_total;
    const int slot_rank = block_exclusive_scan(my_slots, s_warp, &slots_total);
    const int base_slots = s_slots;
    if (my_slots > 0) {
      int sl = base_slots + slot_rank;
      if (sl + my_slots > p.max_slots) {
        p.st->error_flag = 3;
      } else if (p.sibling_subtraction) {
        const int small = pos_small ? pos : neg, large = pos_small ? neg : pos;
        p.nodes[small].slot = sl;
        p.next_slot_node[sl] = small;
        p.next_families[sl] = Family{lv.first_node + j, small, large};
      } else {
        if (cand_p) { p.nodes[pos].slot = sl; p.next_slot_node[sl] = pos; p.next_families[sl] = Family{-1, pos, -1}; sl++; }
        if (cand_n) { p.nodes[neg].slot = sl; p.next_slot_node[sl] = neg; p.next_families[sl] = Family{-1, neg, -1}; }
      }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      s_next = base_next + 2 * n_split_total;
      s_slots = base_slots + slots_total;
      s_fams = s_slots;  // one family per slot in both modes
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    LevelDesc nl;
    nl.first_node = first_next;
    nl.num_nodes = s_next - first_next;
    nl.num_slots = s_slots;
    nl.num_families = s_fams;
    p.levels[p.level + 1] = nl;
    p.st->num_nodes = s_next;
  }
}

// ---------------------------------------------------------------------------------------------
// k_partition: SplitExamplesInPlace (training.cc:5243-5305 -> decision_tree.cc:957-1012) on the
// node-id representation.  One CTA iteration = one block of 8192 rows (16 consecutive rows per
// thread).  Every row of a split node is relabelled with its child id; the rows whose child is
// histogrammed at the next level are compacted, in row order, into the block's active list
// (block-wide exclusive scan = the stable scatter of example indices); the children's exact
// statistics are accumulated on the way.
struct PartParams {
  int64_t n;
  int n_blocks;
  int level;
  const LevelDesc* levels;
  NodeRec* nodes;
  const uint8_t* bins;
  int64_t n_pad;
  uint16_t* node_of_row;
  const uint32_t* q24;
  const uint32_t* hq24;   // hessian histogram only
  uint2* act;
  uint32_t* act_h;
  int32_t* act_count;
  const uint8_t* selected;    // stochastic gradient boosting: rows outside the sample are routed but not counted (null: all rows)
  const float* g;
  const float* h;   // null: h == 1
  const DeviceState* st;
  unsigned long long* stats;  // [children of this level][3] fixed-point sums of g, h, g^2 (this rank's rows)
  int smem_children;          // capacity of the shared accumulators (children of this level)
  int smem_children_private;  // capacity with one accumulator copy per lane
};

// Shared accumulators per child: cnt, g_lo, g_hi, h_lo, h_hi, g2_lo, g2_hi.
constexpr int kPartWords = 7;
constexpr int kPartThreads = 512;
constexpr int kPartRows = 8;                                   // consecutive rows per thread per pass
constexpr int kPartPassRows = kPartThreads * kPartRows;        // 4096
constexpr int kPartPasses = kBlockRows / kPartPassRows;        // 2 passes per 8192-row block
static_assert(kPartPasses * kPartPassRows == kBlockRows, "a block is a whole number of passes");

__device__ __forceinline__ void add64_smem(uint32_t* lo, uint32_t* hi, uint32_t v) {
  const uint32_t old = atomicAdd(lo, v);
  if (old + v < old) atomicAdd(hi, 1u);
}

// Split table of the current level, staged in shared memory once per CTA (16 bytes per node).
struct PartNode {
  int32_t feature;   // -1: the node is a leaf
  int32_t thr;       // >= 0: bin >= thr ; -1: categorical (positive set in s_masks)
  uint32_t kids;     // pos child | neg child << 16
  uint32_t meta;     // pos slot (0xFF none) | neg slot << 8 | (the positive child is the smaller one) << 16
};
constexpr int kPartMaxLevelNodes = 512;  // levels with more nodes read the node table from global memory

// The child whose statistics are accumulated from rows: the SMALLER one (positive on ties); the other child's are
// parent - smaller, exact on the integer sums (k_node_stats).  Halves the statistics atomics of the pass.
__device__ __forceinline__ bool pos_child_is_smaller(const NodeRec* nodes, const NodeRec& nd) {
  return nodes[nd.pos_child].n <= nodes[nd.neg_child].n;
}
template <bool CAT>
__device__ __forceinline__ PartNode make_part_node(const NodeRec* nodes, const NodeRec& nd) {
  PartNode pn;
  pn.feature = nd.feature;
  pn.thr = (CAT && nd.cond_type == 1) ? -1 : nd.thr;
  pn.kids = 0u; pn.meta = 0u;
  if (nd.feature >= 0) {
    pn.kids = static_cast<uint32_t>(nd.pos_child) | (static_cast<uint32_t>(nd.neg_child) << 16);
    pn.meta = (static_cast<uint32_t>(nodes[nd.pos_child].slot) & 0xFFu) | ((static_cast<uint32_t>(nodes[nd.neg_child].slot) & 0xFFu) << 8) |
              (pos_child_is_smaller(nodes, nd) ? 1u << 16 : 0u);
  }
  return pn;
}

// CAT: the dataset has categorical features (numerical-only datasets keep the leaner hot loop).
// One CTA iteration = one block of 8192 rows in two passes of 4096 (8 consecutive rows per thread): per pass the
// node ids (one 128-bit load), the byte gathers of the split columns, then — only for threads that own a row of a
// node being split — g / h / q24 (128-bit loads), the relabel, the statistics of the smaller children and the
// stable compaction of the rows histogrammed at the next level (block-wide exclusive scan; the list stays in ROW
// ORDER, which k_hist relies on for conflict-free LDS.U8 reads of its bins tile).
template <bool CAT>
__global__ void __launch_bounds__(kPartThreads, 2) k_partition(PartParams p) {
  extern __shared__ __align__(16) uint32_t smem[];
  __shared__ int s_warp_tot[kPartThreads / 32];
  __shared__ __align__(16) PartNode s_nodes[kPartMaxLevelNodes];
  __shared__ uint32_t s_masks[CAT ? kPartMaxLevelNodes : 1][8];
  const LevelDesc lv = p.levels[p.level];
  const LevelDesc nl = p.levels[p.level + 1];
  const int n_children = nl.num_nodes;
  // Accumulator layout: lane-private copies ([child][word][lane]) while they fit, else one shared
  // copy, else global atomics.
  const bool use_priv = n_children <= p.smem_children_private;
  const bool use_smem = use_priv || n_children <= p.smem_children;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int copies = use_priv ? 32 : 1;
  const bool nodes_in_smem = lv.num_nodes <= kPartMaxLevelNodes;
  if (use_smem)
    for (int i = threadIdx.x; i < n_children * kPartWords * copies; i += blockDim.x) smem[i] = 0u;
  if (nodes_in_smem) {
    for (int j = threadIdx.x; j < lv.num_nodes; j += blockDim.x) {
      const NodeRec& nd = p.nodes[lv.first_node + j];
      s_nodes[j] = make_part_node<CAT>(p.nodes, nd);
      if (CAT)
        for (int i = 0; i < 8; i++) s_masks[j][i] = nd.mask[i];
    }
  }
  __syncthreads();
  const int e = ilogbf(p.st->g_pow2);             // P = 2^e, see k_quantize
  const double sscale = pow2_d(kSBits - 1 - e);
  const double s2scale = pow2_d(kSBits - 2 * e);
  const float hscale = static_cast<float>(1u << kSBits) / p.st->h_pow2;
  for (int blk = blockIdx.x; blk < p.n_blocks; blk += gridDim.x) {
    const int64_t base = static_cast<int64_t>(blk) * kBlockRows;
    int written = 0;  // active rows of this block compacted so far
    if (nl.num_nodes == 0) {
      if (threadIdx.x == 0) p.act_count[blk] = 0;
      continue;
    }
#pragma unroll 1
    for (int pass = 0; pass < kPartPasses; pass++) {
      const int row0 = pass * kPartPassRows + threadIdx.x * kPartRows;  // first row of this thread, inside the block
      const int64_t rh = base + row0;
      // node ids of the 8 rows (arrays are padded to n_pad; rows >= n are masked below)
      uint32_t nodew[4];
      {
        const uint4 a = *reinterpret_cast<const uint4*>(p.node_of_row + rh);
        nodew[0] = a.x; nodew[1] = a.y; nodew[2] = a.z; nodew[3] = a.w;
      }
      // level-local node index (or -1) and the gathered split byte, packed: index << 8 | byte
      int32_t lb[kPartRows];
      bool any = false;
#pragma unroll
      for (int j = 0; j < kPartRows; j++) {
        const int node = static_cast<int>((nodew[j >> 1] >> (16 * (j & 1))) & 0xFFFFu);
        lb[j] = -1;
        if (rh + j < p.n && node >= lv.first_node) {  // else: padding, or a row in a finished leaf
          const int li = node - lv.first_node;
          const int feature = nodes_in_smem ? s_nodes[li].feature : p.nodes[node].feature;
          if (feature >= 0) {
            lb[j] = (li << 8) | static_cast<int32_t>(p.bins[static_cast<int64_t>(feature) * p.n_pad + rh + j]);
            any = true;
          }
        }
      }
      uint32_t out_info[kPartRows];
      uint32_t active_mask = 0;
      // rows outside the iteration's sample follow the splits (their predictions need the leaf) but carry no statistics
      // and are never histogrammed
      unsigned long long sel8 = 0x0101010101010101ull;
      if (p.selected != nullptr && any) sel8 = *reinterpret_cast<const unsigned long long*>(p.selected + rh);
      if (any) {
#pragma unroll
        for (int half = 0; half < 2; half++) {
          // g / h / q24 of 4 rows
          const float4 g4 = __ldg(reinterpret_cast<const float4*>(p.g + rh + 4 * half));
          const uint4 q4 = __ldg(reinterpret_cast<const uint4*>(p.q24 + rh + 4 * half));
          float4 h4 = make_float4(0.f, 0.f, 0.f, 0.f);
          if (p.h) h4 = __ldg(reinterpret_cast<const float4*>(p.h + rh + 4 * half));
          const float gv[4] = {g4.x, g4.y, g4.z, g4.w};
          const float hv[4] = {h4.x, h4.y, h4.z, h4.w};
          const uint32_t qv[4] = {q4.x, q4.y, q4.z, q4.w};
#pragma unroll
          for (int k = 0; k < 4; k++) {
            const int j = 4 * half + k;
            out_info[j] = 0u;
            if (lb[j] < 0) continue;
            const int li = lb[j] >> 8;
            const uint32_t bin = static_cast<uint32_t>(lb[j]) & 0xFFu;
            const PartNode pn = nodes_in_smem ? s_nodes[li] : make_part_node<CAT>(p.nodes, p.nodes[lv.first_node + li]);
            // EvalConditionDiscretizedHigher (decision_tree.cc:724-743) / Contains (:766-812); NA is
            // already folded into na_bin.
            bool go_pos;
            if (!CAT || pn.thr >= 0) {
              go_pos = static_cast<int>(bin) >= pn.thr;
            } else {
              const uint32_t mw = nodes_in_smem ? s_masks[li][bin >> 5] : p.nodes[lv.first_node + li].mask[bin >> 5];
              go_pos = ((mw >> (bin & 31)) & 1u) != 0;
            }
            const uint32_t child = go_pos ? (pn.kids & 0xFFFFu) : (pn.kids >> 16);
            const uint32_t slot = go_pos ? (pn.meta & 0xFFu) : ((pn.meta >> 8) & 0xFFu);
            nodew[j >> 1] = (j & 1) ? ((nodew[j >> 1] & 0x0000FFFFu) | (child << 16)) : ((nodew[j >> 1] & 0xFFFF0000u) | child);
            if (((sel8 >> (8 * j)) & 0xFFull) == 0ull) continue;
            if (slot != 0xFFu) {
              active_mask |= 1u << j;
              out_info[j] = qv[k] | (slot << 24);
            }
            if (go_pos != (((pn.meta >> 16) & 1u) != 0u)) continue;   // statistics: rows of the smaller child only
            const float g = gv[k];
            const uint32_t qg = quant_stat_signed(g, sscale);
            const uint32_t qg2 = quant_stat_unsigned(g * g, s2scale);
            const uint32_t qh = p.h ? quant_stat_unsigned(hv[k], hscale) : 0u;
            const int c = static_cast<int>(child) - nl.first_node;
            if (use_smem) {
              // word w of child c lives at (c*kPartWords + w) * copies + (private ? lane : 0)
              uint32_t* a = smem + static_cast<size_t>(c) * kPartWords * copies + (use_priv ? lane : 0);
              atomicAdd(&a[0], 1u);
              add64_smem(&a[1 * copies], &a[2 * copies], qg);
              if (p.h) add64_smem(&a[3 * copies], &a[4 * copies], qh);
              add64_smem(&a[5 * copies], &a[6 * copies], qg2);
            } else {
              unsigned long long* cs = p.stats + static_cast<size_t>(c) * 3;
              atomicAdd(&cs[0], static_cast<unsigned long long>(qg));
              if (p.h) atomicAdd(&cs[1], static_cast<unsigned long long>(qh));
              atomicAdd(&cs[2], static_cast<unsigned long long>(qg2));
            }
          }
        }
        // new node ids of the 8 rows: one 128-bit store (rows past n are padding)
        *reinterpret_cast<uint4*>(p.node_of_row + rh) = make_uint4(nodew[0], nodew[1], nodew[2], nodew[3]);
      }
      // Block-wide exclusive scan of the per-thread active counts.
      const int mine = __popc(active_mask);
      int incl = mine;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
      }
      if (lane == 31) s_warp_tot[warp] = incl;
      __syncthreads();
      int offset = written + incl - mine;
      int total = 0;
#pragma unroll
      for (int w = 0; w < kPartThreads / 32; w++) {
        const int t = s_warp_tot[w];
        if (w < warp) offset += t;
        total += t;
      }
      __syncthreads();
      written += total;
      if (mine > 0) {
#pragma unroll
        for (int j = 0; j < kPartRows; j++) {
          if (active_mask & (1u << j)) {
            p.act[base + offset] = make_uint2(out_info[j], static_cast<uint32_t>(row0 + j));
            if (p.hq24 != nullptr) p.act_h[base + offset] = p.hq24[rh + j];
            offset++;
          }
        }
      }
    }
    if (threadIdx.x == 0) p.act_count[blk] = written;
  }
  if (use_smem) {
    __syncthreads();
    for (int c = threadIdx.x; c < n_children; c += blockDim.x) {
      unsigned long long w[kPartWords];
#pragma unroll
      for (int k = 0; k < kPartWords; k++) {
        unsigned long long t = 0;
        const uint32_t* a = smem + (static_cast<size_t>(c) * kPartWords + k) * copies;
        for (int l = 0; l < copies; l++) t += a[(l + threadIdx.x) & (copies - 1)];  // staggered: fewer bank conflicts
        w[k] = t;
      }
      if (w[0] == 0ull) continue;
      unsigned long long* cs = p.stats + static_cast<size_t>(c) * 3;
      atomicAdd(&cs[0], (w[2] << 32) + w[1]);
      if (p.h) atomicAdd(&cs[1], (w[4] << 32) + w[3]);
      atomicAdd(&cs[2], (w[6] << 32) + w[5]);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// k_node_stats: fixed-point sums -> the doubles the reference stores, and the Newton leaf value.
// SetLeafValueWithNewtonRaphsonStep<false> (loss_utils.cc:49-132).
struct StatsParams {
  int level;            // nodes of level `level` are finalised (level 0: the root)
  const LevelDesc* levels;
  NodeRec* nodes;
  DeviceState* st;
  int use_hessian, logit_loss, has_h;
  float shrinkage, clamp;
  double l1, l2;
  const unsigned long long* stats;  // [nodes of the level][3] (root: [3])
  int64_t n_rows;       // rows of the whole job (all ranks)
  int min_examples, max_depth;
  // the score of a split is re-evaluated from its children's 31-bit statistics (the scan works on 24-bit histograms)
  int subtract_parent;
  double l2_categorical;
  int weighted;         // example weights: the weight sums only exist once the tree is finished (k_weight_sums_finish)
};

__global__ void k_node_stats(StatsParams p) {
  if (p.level == 0 && blockIdx.x == 0 && threadIdx.x == 0) {
    // Root record (NodeTrain on the root, training.cc:4880-4894).
    NodeRec root{};
    root.parent = -1; root.depth = 1; root.feature = -1; root.pos_child = root.neg_child = -1;
    root.sibling = -1;
    root.n = p.n_rows;
    root.candidate = (p.n_rows >= p.min_examples && 1 < p.max_depth) ? 1 : 0;
    root.slot = root.candidate ? 0 : -1;
    p.nodes[0] = root;
  }
  __syncthreads();
  const LevelDesc lv = p.levels[p.level];
  const double P = p.st->g_pow2;
  const double ginv = P / static_cast<double>(1u << (kSBits - 1));
  const double g2inv = P * P / static_cast<double>(1u << kSBits);
  const double hinv = static_cast<double>(p.st->h_pow2) / static_cast<double>(1u << kSBits);
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < lv.num_nodes; j += gridDim.x * blockDim.x) {
    NodeRec& nd = p.nodes[lv.first_node + j];
    const double n = static_cast<double>(nd.n);
    const unsigned long long* cs = p.stats + static_cast<size_t>(j) * 3;
    if (p.level == 0) {
      nd.sg = cs[0]; nd.sh = cs[1]; nd.sg2 = cs[2];
    } else {
      // k_partition accumulated the SMALLER child of every split from its rows; the other child is
      // parent - smaller, exact on the biased integer sums (every row carries the same bias).
      const NodeRec& par = p.nodes[nd.parent];
      const bool i_am_pos = par.pos_child == lv.first_node + j;
      const bool pos_smaller = p.nodes[par.pos_child].n <= p.nodes[par.neg_child].n;
      if (i_am_pos == pos_smaller) {
        nd.sg = cs[0]; nd.sh = cs[1]; nd.sg2 = cs[2];
      } else {
        const unsigned long long* ss = p.stats + static_cast<size_t>(nd.sibling - lv.first_node) * 3;
        nd.sg = par.sg - ss[0]; nd.sh = par.sh - ss[1]; nd.sg2 = par.sg2 - ss[2];
      }
    }
    if (p.level > 0 && !p.weighted) {
      // The parent's split score, as the scan computes it (scan_node) but from the children's node statistics: the
      // argmax was taken on the 24-bit histogram sums, whose rounding shows in scores that are small against P^2.
      NodeRec& par = p.nodes[nd.parent];
      if (par.pos_child == lv.first_node + j) {
        const unsigned long long* ss = p.stats + static_cast<size_t>(nd.sibling - lv.first_node) * 3;
        const NodeRec& sib = p.nodes[nd.sibling];
        const bool pos_smaller = nd.n <= sib.n;
        const unsigned long long sg_n = pos_smaller ? par.sg - nd.sg : ss[0];
        const unsigned long long sh_n = pos_smaller ? par.sh - nd.sh : ss[1];
        const double np_ = n, nn_ = static_cast<double>(sib.n);
        const double Sp = (static_cast<double>(static_cast<long long>(nd.sg)) - np_ * static_cast<double>(kSBias)) * ginv;
        const double Sn = (static_cast<double>(static_cast<long long>(sg_n)) - nn_ * static_cast<double>(kSBias)) * ginv;
        double score;
        if (!p.use_hessian) {
          const double c0 = np_ + nn_;
          const double d = Sp * nn_ - Sn * np_;
          score = (d / np_) * (d / nn_) / (c0 * c0);
        } else {
          const double l2 = par.cond_type == 1 ? p.l2_categorical : p.l2;
          const double Hp = p.has_h ? static_cast<double>(nd.sh) * hinv : np_;
          const double Hn = p.has_h ? static_cast<double>(sh_n) * hinv : nn_;
          const double gp = l1_threshold_d(Sp, p.l1), gn = l1_threshold_d(Sn, p.l1);
          const double g0 = l1_threshold_d(par.stat[0], p.l1);
          score = gp * gp / (fmax(Hp, kMinHessianForNewtonStep) + l2) + gn * gn / (fmax(Hn, kMinHessianForNewtonStep) + l2) -
                  (p.subtract_parent ? g0 * g0 / (par.stat[1] + l2) : 0.0);
        }
        // (a split exists because its 24-bit score was positive; keep it so)
        if (score > 0.0) par.score = static_cast<float>(score);
      }
    }
    const double sum_g = (static_cast<double>(static_cast<long long>(nd.sg)) - n * static_cast<double>(kSBias)) * ginv;
    double sum_h = p.has_h ? static_cast<double>(nd.sh) * hinv : n;
    const double sum_g2 = static_cast<double>(nd.sg2) * g2inv;
    if (sum_h <= kMinHessianForNewtonStep) sum_h = kMinHessianForNewtonStep;
    if (p.use_hessian) { nd.stat[0] = sum_g; nd.stat[1] = sum_h; nd.stat[2] = n; }
    else { nd.stat[0] = sum_g; nd.stat[1] = sum_g2; nd.stat[2] = n; }
    const double numerator = l1_threshold_d(sum_g, p.l1);
    const double denominator = sum_h + p.l2;
    float value = static_cast<float>(static_cast<double>(p.shrinkage) * numerator / denominator);
    if (p.logit_loss) value = fminf(fmaxf(value, -p.clamp), p.clamp);
    nd.leaf_value = value;
  }
}

// ---------------------------------------------------------------------------------------------
// Gradient-based one-side sampling (SampleTrainingExamplesWithGoss, gradient_boosted_trees.cc:2958-3007).
// keys = |g| (the L1 norm of a one-dimensional gradient), values = row ids; sorted by the caller (descending, stable).
__global__ void __launch_bounds__(256) k_goss_keys(const float* __restrict__ g, int64_t n, float* __restrict__ keys, uint32_t* __restrict__ rows) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r < n; r += stride) {
    keys[r] = fabsf(g[r]);
    rows[r] = static_cast<uint32_t>(r);
  }
}
// Position i of the sorted order: the first `cutoff` rows are kept with weight 1, row i >= cutoff iff its draw u[i - cutoff]
// is below beta, with weight (1 - alpha) / beta (the dataset's weights are all 1 with GOSS, :1236-1242).
__global__ void __launch_bounds__(256) k_goss_apply(const uint32_t* __restrict__ sorted_rows, const float* __restrict__ u, int64_t n,
                                                    int64_t cutoff, float beta, float amplification, uint8_t* __restrict__ selected,
                                                    float* __restrict__ weight) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
    const uint32_t row = sorted_rows[i];
    bool in = true;
    float w = 1.f;
    if (i >= cutoff) {
      in = beta > 0.f && u[i - cutoff] < beta;
      if (in) w = 1.f * amplification;
    }
    selected[row] = in ? 1 : 0;
    weight[row] = w;
  }
}
// The rows' unit gradients / hessians times this iteration's weights, as k_pred_grad<., WEIGHTED> leaves them.
__global__ void __launch_bounds__(256) k_apply_weights(int64_t n, float* __restrict__ g, float* __restrict__ h, int unit_hessian,
                                                       const float* __restrict__ weight, float* __restrict__ g2w, DeviceState* st) {
  float gmax = 0.f, g2max = 0.f;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r < n; r += stride) {
    const float w = weight[r], gu = g[r];
    const float wg = gu * w, g2 = wg * gu;
    g[r] = wg;
    h[r] = unit_hessian ? w : w * h[r];
    g2w[r] = g2;
    gmax = fmaxf(gmax, fabsf(wg));
    g2max = fmaxf(g2max, g2);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    gmax = fmaxf(gmax, __shfl_xor_sync(0xffffffffu, gmax, o));
    g2max = fmaxf(g2max, __shfl_xor_sync(0xffffffffu, g2max, o));
  }
  if ((threadIdx.x & 31) == 0) {
    atomicMax(&st->gmax_bits, __float_as_uint(gmax));
    atomicMax(&st->g2w_max_bits, __float_as_uint(g2max));
  }
}

// Example weights: the two node statistics the growth itself never needs — the weight sum (the node's `count`) and the
// weighted sum of squared gradients — are added up once per tree from the rows' final leaves and propagated to the
// ancestors (loss_utils.cc:81-89 stores them in the node; scores and leaf values do not read them).
struct WeightSumParams {
  int64_t n;
  const uint16_t* node_of_row;
  const uint8_t* selected;     // see QuantParams
  const float* weight;
  const float* g2w;            // (w*g)*g of every row
  const DeviceState* st;
  float w_pow2;                // power of two >= max weight
  NodeRec* nodes;
  unsigned long long* sums;    // [max_nodes][2], zeroed: fixed-point sums of w and (w*g)*g per node
  const LevelDesc* levels;
  int num_levels;              // levels of the level table that may hold nodes
  int smem_nodes;              // nodes whose accumulators fit the dynamic shared memory (0: global atomics)
};
__global__ void __launch_bounds__(256) k_weight_sums_rows(WeightSumParams p) {
  extern __shared__ unsigned long long s_acc[];
  const int n_nodes = p.st->num_nodes;
  const bool in_smem = n_nodes <= p.smem_nodes;
  if (in_smem)
    for (int i = threadIdx.x; i < 2 * n_nodes; i += blockDim.x) s_acc[i] = 0ull;
  __syncthreads();
  const float wscale = static_cast<float>(1u << kSBits) / p.w_pow2;
  const float g2scale = static_cast<float>(1u << kSBits) / pow2_cover(p.st->g2w_max_bits);
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r < p.n; r += stride) {
    if (p.selected != nullptr && p.selected[r] == 0) continue;
    const int node = p.node_of_row[r];
    unsigned long long* a = (in_smem ? s_acc : p.sums) + 2 * static_cast<size_t>(node);
    atomicAdd(&a[0], static_cast<unsigned long long>(quant_stat_unsigned(p.weight[r], wscale)));
    atomicAdd(&a[1], static_cast<unsigned long long>(quant_stat_unsigned(p.g2w[r], g2scale)));
  }
  if (!in_smem) return;
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * n_nodes; i += blockDim.x)
    if (s_acc[i] != 0ull) atomicAdd(&p.sums[i], s_acc[i]);
}
// One CTA: levels from the deepest up, every split node = the sum of its two children.
__global__ void __launch_bounds__(1024) k_weight_sums_finish(WeightSumParams p) {
  const double winv = static_cast<double>(p.w_pow2) / static_cast<double>(1u << kSBits);
  const double g2inv = static_cast<double>(pow2_cover(p.st->g2w_max_bits)) / static_cast<double>(1u << kSBits);
  for (int l = p.num_levels - 1; l >= 0; l--) {
    const LevelDesc lv = p.levels[l];
    for (int j = threadIdx.x; j < lv.num_nodes; j += blockDim.x) {
      const int id = lv.first_node + j;
      NodeRec& nd = p.nodes[id];
      unsigned long long* a = p.sums + 2 * static_cast<size_t>(id);
      if (nd.feature >= 0) {
        const unsigned long long* x = p.sums + 2 * static_cast<size_t>(nd.pos_child);
        const unsigned long long* y = p.sums + 2 * static_cast<size_t>(nd.neg_child);
        a[0] = x[0] + y[0];
        a[1] = x[1] + y[1];
        // the split's score from the children's 31-bit sums (see k_node_stats), with weight sums for counts
        const NodeRec& pc = p.nodes[nd.pos_child];
        const NodeRec& nc = p.nodes[nd.neg_child];
        const double ginv = static_cast<double>(p.st->g_pow2) / static_cast<double>(1u << (kSBits - 1));
        const double Sp = (static_cast<double>(static_cast<long long>(pc.sg)) - static_cast<double>(pc.n) * static_cast<double>(kSBias)) * ginv;
        const double Sn = (static_cast<double>(static_cast<long long>(nc.sg)) - static_cast<double>(nc.n) * static_cast<double>(kSBias)) * ginv;
        const double Wp = static_cast<double>(x[0]) * winv, Wn = static_cast<double>(y[0]) * winv;
        if (Wp > 0.0 && Wn > 0.0) {
          const double W0 = Wp + Wn;
          const double d = Sp * Wn - Sn * Wp;
          const double score = (d / Wp) * (d / Wn) / (W0 * W0);
          if (score > 0.0) nd.score = static_cast<float>(score);
        }
      }
      nd.stat[1] = static_cast<double>(a[1]) * g2inv;
      nd.stat[2] = static_cast<double>(a[0]) * winv;
    }
    __threadfence_block();
    __syncthreads();
  }
}

// Tie-break replay, device part: a tied candidate may only take the place of the chosen split if it sends EVERY row of
// the node to the same side (twin columns); equal float scores and equal positive counts do not prove that.  Every
// row walks from its leaf to the root; at each ancestor with recorded ties it knows on which side it went and
// evaluates the alternatives' conditions: a disagreement disqualifies the alternative (n_pos = -1).
__global__ void __launch_bounds__(256) k_verify_ties(NodeRec* nodes, const uint16_t* __restrict__ node_of_row,
                                                     const uint8_t* __restrict__ bins, int64_t n, int64_t n_pad) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r < n; r += stride) {
    int child = node_of_row[r];
    int node = nodes[child].parent;
    while (node >= 0) {
      const int tc = nodes[node].tie_count;
      if (tc > 0) {
        const bool went_pos = nodes[node].pos_child == child;
        for (int i = 0; i < min(tc, kMaxTieAlts); i++) {
          const TieAlt& a = nodes[node].tie[i];
          if (a.n_pos < 0) continue;
          const uint32_t b = bins[static_cast<int64_t>(a.feature) * n_pad + r];
          const bool alt_pos = a.cond_type == 1 ? ((a.mask[b >> 5] >> (b & 31)) & 1u) != 0 : static_cast<int>(b) >= a.thr;
          if (alt_pos != went_pos) nodes[node].tie[i].n_pos = -1;
        }
      }
      child = node;
      node = nodes[node].parent;
    }
  }
}

// Resets the per-iteration scalars and the level table.
__global__ void k_begin_iteration(DeviceState* st, LevelDesc* levels, Family* fam0, int32_t* slot_node0,
                                  int root_candidate) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    st->gmax_bits = 0u;
    st->g2w_max_bits = 0u;
    st->num_nodes = 1;
    levels[0] = LevelDesc{0, 1, root_candidate ? 1 : 0, root_candidate ? 1 : 0};
    fam0[0] = Family{-1, 0, -1};
    slot_node0[0] = 0;
  }
}

__global__ void k_reset_loss(DeviceState* st) {
  st->loss_sum = 0.0;
  st->correct = 0ull;
}

// ---------------------------------------------------------------------------------------------
// Debug / seam kernels.

// SplitExamplesInPlace as a standalone stable partition of a row-id list (single CTA per 2048-row
// tile + decoupled offsets are overkill for a test seam: two-pass count/scatter with a global scan).
__global__ void k_partition_count(const uint8_t* col, const uint32_t* rows, int64_t n, int thr,
                                  uint32_t* block_pos_counts) {
  __shared__ uint32_t s[8];
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const bool pos = i < n && col[rows[i]] >= thr;
  const uint32_t bal = __ballot_sync(0xffffffffu, pos);
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = __popc(bal);
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t t = 0;
    for (int k = 0; k < 8; k++) t += s[k];
    block_pos_counts[blockIdx.x] = t;
  }
}

__global__ void k_partition_scatter(const uint8_t* col, const uint32_t* rows, int64_t n, int thr,
                                    const uint32_t* block_pos_offsets, uint32_t total_pos,
                                    uint32_t* out) {
  __shared__ uint32_t s[8];
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const bool in = i < n;
  const uint32_t row = in ? rows[i] : 0u;
  const bool pos = in && col[row] >= thr;
  const uint32_t bal = __ballot_sync(0xffffffffu, pos);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) s[w] = __popc(bal);
  __syncthreads();
  uint32_t warp_off = 0;
  for (int k = 0; k < w; k++) warp_off += s[k];
  const uint32_t pos_before = block_pos_offsets[blockIdx.x] + warp_off + __popc(bal & ((1u << lane) - 1u));
  if (in) {
    if (pos) out[pos_before] = row;
    else out[total_pos + (static_cast<uint32_t>(i) - pos_before)] = row;
  }
}

}  // namespace ygg
