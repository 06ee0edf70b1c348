// ygg_hist.cuh — k_hist, the hot kernel: FillExampleBucketSet (learner/decision_tree/
// splitter_scanner.h:859-909) for every open node x feature of one tree level.
//
// Data in HBM (DESIGN.md §2):
//   bins[f][row]            one byte per value, column-major, row stride n_pad (multiple of 8192)
//   act_info[block][k]      per 8192-row block, the compacted list of ACTIVE rows of this level
//                           (rows whose node's histogram is accumulated from rows, i.e. not a leaf
//                           and not the sibling derived by subtraction): q24 | slot << 24
//   act_ridx[block][k]      the row's offset inside its block (uint16)
//   act_count[block]        number of active rows of the block
// The lists are written by k_quantize (root) / k_partition (deeper levels), in ascending row order.
//
// Work item = (chunk of consecutive row blocks) x (group of G consecutive features).  Per item a
// CTA zeroes G*S*256 shared-memory bins, streams the chunk block by block — the G x 8192-byte bins
// tile of each block is staged into shared memory by the TMA engine (cp.async.bulk, mbarrier
// pipeline, kStages deep) — and flushes its non-empty bins to the 64-bit global histogram.
//
// Shared-memory bin = two 32-bit words updated with native ATOMS.ADD (the only shared-memory
// atomic add sm_100a executes natively; 64-bit and float adds compile to CAS loops):
//   word0 = count (bits 0..19) + carries of the sum (bits 20..31), word1 = low 32 bits of sum(q24).
// A chunk has < 2^20 rows, so count < 2^20 and carries <= count * 2^24 / 2^32 < 2^12: the pair is
// an exact 44-bit sum.  A carry is detected from the value ATOMS.ADD returns; it happens once per
// ~256 updates of a bin and is handled off the hot path.
//
// Because every lane of a warp works on an ACTIVE row, the inner loop has no predication and no
// divergence, and sibling subtraction halves the number of shared-memory atomics, which — not HBM
// bandwidth — is what bounds this kernel (profiles/atoms_microbench_r01.txt).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "ygg_device.cuh"

namespace ygg {

#ifndef YGG_HIST_THREADS
#define YGG_HIST_THREADS 1024
#endif
#ifndef YGG_HIST_UNROLL
#define YGG_HIST_UNROLL 4
#endif
constexpr int kHistThreads = YGG_HIST_THREADS;
constexpr int kBlockRows = 8192;                 // rows per block (TMA tile = G x 8192 bytes)
constexpr int kHistStages = 3;
constexpr int kHistCntBits = 20;
constexpr int kHistMaxChunkBlocks = ((1 << kHistCntBits) - 1) / kBlockRows;  // 127 blocks = 1,040,384 rows
constexpr int kHistUnroll = YGG_HIST_UNROLL;                   // active rows per thread per inner iteration

struct HistParams {
  const uint8_t* bins;
  int64_t n_pad;
  const uint32_t* q24;        // [n_pad] quantised gradient of every row (dense root path)
  const uint2* act;           // [n_pad] per block: (q24 | slot << 24, row offset in block)
  const uint32_t* act_h;      // hq24 per active row (hessian histogram only)
  const int32_t* act_count;
  int n_blocks;
  int f_begin;        // first feature (dataset index) of this shard
  int f_count;        // features in this shard
  int G;              // features per work item
  int S;              // shared-memory slots (>= slots used at this level; multi-pass: slots of a pass + 1 dummy)
  int chunk_blocks;   // row blocks per work item (<= kHistMaxChunkBlocks)
  int level;          // multi-pass launches (k_hist<., ., MULTI>) also carry their slot window here: level | slot_base << 8 |
                      // slot_count << 20 — the struct keeps the size and layout the single-pass kernels were tuned with (two more
                      // words in it cost k_hist<., kHistPacked> 3.5 % on levels 1-6, measured A/B on one B200)
  const LevelDesc* levels;
  // Histograms of the level's slots.  One chunk: [slot][f_count][256].  Row-sharded runs with a
  // reduce-scatter cut the features into `world` chunks of f_chunk features, each chunk a contiguous
  // block [sum | hsum | cnt | stats] of chunk_stride u64 words (so that rank r receives chunk r):
  // element (slot, f_local, bin) lives at chunk (f_local / f_chunk), offset (slot*f_chunk + f_local % f_chunk)*256 + bin.
  unsigned long long* hist_sum;
  uint32_t* hist_cnt;
  unsigned long long* hist_hsum;  // hessian histogram only
  int f_chunk;                    // features per chunk (= f_count when there is a single chunk)
  long long chunk_stride;         // u64 words between chunks
};

// Offset (in elements of the sum plane; the u32 count plane uses 2 * chunk part) of a slot-histogram bin.
__host__ __device__ __forceinline__ size_t slot_hist_offset(int slot, int f_local, int bin, int f_chunk,
                                                            long long chunk_stride, size_t* cnt_offset) {
  const int ch = f_local / f_chunk, fi = f_local - ch * f_chunk;
  const size_t in_chunk = (static_cast<size_t>(slot) * f_chunk + fi) * 256 + bin;
  *cnt_offset = static_cast<size_t>(ch) * chunk_stride * 2 + in_chunk;
  return static_cast<size_t>(ch) * chunk_stride + in_chunk;
}

// ---- PTX wrappers: mbarrier + TMA bulk copy (SASS: SYNCS / UBLKCP) and shared-memory atomics ----
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t"
      "}\n" ::"r"(bar), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(dst),
      "l"(src), "r"(bytes), "r"(bar)
      : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
}
__device__ __forceinline__ void smem_red(uint32_t addr, uint32_t v) {
  asm volatile("red.shared.add.u32 [%0], %1;\n" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t smem_add(uint32_t addr, uint32_t v) {
  uint32_t old;
  asm volatile("atom.shared.add.u32 %0, [%1], %2;\n" : "=r"(old) : "r"(addr), "r"(v) : "memory");
  return old;
}
__device__ __forceinline__ uint32_t smem_ld_u32(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];\n" : "=r"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ uint32_t smem_ld_u8(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u8 %0, [%1];\n" : "=r"(v) : "r"(addr));
  return v;
}

// Histogram layouts in shared memory (words of 32 bits; B = G*S*256 bins):
//   kHistShared  : [cnt B][lo B]([hlo B][hhi B])          any S; random bank conflicts (~3.3 wavefronts / ATOMS)
//   kHistRootSum : [lo B][carry B]                        shared layout without counts: the root's counts do not
//                                                         depend on the gradients and are precomputed once
// Measured on B200 (profiles/atoms_microbench_r01.txt, A/B runs in profiles/k_hist_tuning_r01.md): the
// shared-memory atomic pipe retires one ATOMS warp-instruction per ~4 cycles per SM whether or not its
// lanes conflict (up to ~4-way), so bank-conflict-free layouts (a lane-private copy of every bin was measured) buy
// nothing; only the NUMBER of atomic instructions matters.
//   kHistPacked  : [w0 B][w1 B]                            TWO NON-RETURNING atomics (RED) per element and no carry
//                                                         handling at all: w0 += 1 | (q >> 18) << 13 holds the count
//                                                         (bits 0..12) and a coarse sum (bits 13..31), w1 += q holds the
//                                                         sum modulo 2^32.  While a bin receives <= 8191 updates per work
//                                                         item both fields are carry-free, and the coarse sum pins the exact
//                                                         sum to a window of n * 2^18 < 2^31, so w1 identifies it uniquely:
//                                                         sum = base + ((w1 - base) mod 2^32), base = coarse << 18.
//                                                         The bound is a property of the DATASET (rows of a chunk that share
//                                                         a bin of a feature, over all rows >= over any node's rows): the
//                                                         host checks it once with k_chunk_max_count and falls back to
//                                                         kHistShared for levels / datasets where it does not hold.
// A RED warp-instruction costs ~2.7 clk of the SM's atomic pipe, a returning ATOMS ~5 (tools/atoms_bench.cu), so the
// packed layout needs 5.4 clk per 32 elements where kHistShared needs 7.7 + the carry fix-ups.
enum HistMode { kHistShared = 0, kHistRootSum = 1, kHistPacked = 2, kHistModes = 3 };
constexpr int kPackedCntBits = 13;
constexpr uint32_t kPackedMaxUpdates = (1u << kPackedCntBits) - 1u;   // 8191 updates of a bin per work item
constexpr int kPackedCoarseShift = 18;                                // coarse = q >> 18 (6 bits), field 19 bits

__host__ __device__ inline size_t hist_bins_bytes(int G, int S, bool hess, int mode) {
  const size_t B = static_cast<size_t>(G) * S * kMaxBins;
  if (mode == kHistShared) return (hess ? 4 : 2) * B * 4;
  return 2 * B * 4;
}
// Shared-memory layout (dynamic):  [histogram][kHistStages x G x 8192 B tiles][mbarriers]
__host__ __device__ inline size_t hist_smem_bytes(int G, int S, bool hess, int mode) {
  return hist_bins_bytes(G, S, hess, mode) + static_cast<size_t>(kHistStages) * G * kBlockRows + 2 * kHistStages * 8 + 16;
}

// MULTI: a level with more histogram slots than shared memory holds (max_depth 10: 128 slots at the last level) is
// accumulated in several launches, each over a window of slots; a separate instantiation, so that the single-pass hot
// loop is compiled exactly as before.
template <bool HESS, int MODE, bool MULTI = false>
__global__ void __launch_bounds__(kHistThreads, 1) k_hist(HistParams p) {
  static_assert(!(HESS && MODE != kHistShared), "hessian histograms use the shared layout");
  static_assert(kPackedCntBits + (kQBits - kPackedCoarseShift) + kPackedCntBits == 32, "w0 = count | coarse sum");
  static_assert(kPackedCntBits + kPackedCoarseShift < 32, "the coarse sum must pin the sum to a window < 2^32");
  extern __shared__ __align__(128) uint8_t smem_raw[];
  __shared__ int s_counts[kHistMaxChunkBlocks + 1];
  int win_base = 0, win_count = 0;   // MULTI: this launch accumulates the slots [win_base, win_base + win_count)
  if constexpr (MULTI) {
    win_base = (p.level >> 8) & 0xFFF;
    win_count = (p.level >> 20) & 0xFFF;
  }
  const LevelDesc lv = p.levels[MULTI ? (p.level & 0xFF) : p.level];
  if (lv.num_slots == 0) return;
  if constexpr (MULTI) {
    if (lv.num_slots <= win_base) return;
  }
  const int S = p.S;
  const int G = p.G;
  const int bins_per_feature = S * kMaxBins;
  const int B = G * bins_per_feature;
  uint32_t* hist = reinterpret_cast<uint32_t*>(smem_raw);
  uint32_t s_hist = static_cast<uint32_t>(__cvta_generic_to_shared(smem_raw));
  // keep the shared window base in a register: otherwise ptxas rematerialises it (S2UR + ULEA ...)
  // in front of every shared-memory atomic of the hot loops
  asm volatile("mov.u32 %0, %0;" : "+r"(s_hist));
  const uint32_t hist_bytes = static_cast<uint32_t>(hist_bins_bytes(G, S, HESS, MODE));
  // byte offsets of the planes
  const uint32_t plane_bytes = static_cast<uint32_t>(B) * 4u;
  const uint32_t s_tiles = s_hist + hist_bytes;
  const uint32_t stage_bytes = static_cast<uint32_t>(G) * kBlockRows;
  const uint32_t s_full = s_tiles + kHistStages * stage_bytes;  // kHistStages full barriers
  const uint32_t s_empty = s_full + kHistStages * 8;            // kHistStages empty barriers

  const int tid = threadIdx.x;
  const uint32_t lane = tid & 31;
  const int n_fgroups = (p.f_count + G - 1) / G;
  const int n_chunks = (p.n_blocks + p.chunk_blocks - 1) / p.chunk_blocks;
  const int64_t n_items = static_cast<int64_t>(n_chunks) * n_fgroups;

  if (tid == 0) {
    for (int s = 0; s < kHistStages; s++) {
      mbar_init(s_full + 8 * s, 1);
      mbar_init(s_empty + 8 * s, kHistThreads / 32);
    }
    fence_barrier_init();
  }
  __syncthreads();

  // Pipeline bookkeeping persists across work items: `produced` / `consumed` count tiles.
  uint32_t produced = 0, consumed = 0;

  // One (row, feature) update.  `a` = byte offset of the bin inside a plane (layout dependent).
  // Returns true if a carry out of the low word has to be recorded (rare).
  auto bin_offset = [&](uint32_t info, uint32_t b) -> uint32_t {
    if constexpr (MULTI) {
      // outside the window: dummy slot
      const uint32_t slot = min((info >> 24) - static_cast<uint32_t>(win_base), static_cast<uint32_t>(S - 1));
      return ((slot << 8) | b) << 2;
    } else {
      return (((info >> 24) << 8) | b) << 2;
    }
  };

  for (int64_t item = blockIdx.x; item < n_items; item += gridDim.x) {
    const int chunk = static_cast<int>(item / n_fgroups);
    const int fg = static_cast<int>(item - static_cast<int64_t>(chunk) * n_fgroups);
    const int f0 = fg * G;
    const int gcount = min(G, p.f_count - f0);
    const int b0 = chunk * p.chunk_blocks;
    const int b1 = min(b0 + p.chunk_blocks, p.n_blocks);
    const int nb = b1 - b0;

    {
      uint4* z = reinterpret_cast<uint4*>(hist);
      const int n4 = hist_bytes / 16;
      for (int i = tid; i < n4; i += kHistThreads) z[i] = make_uint4(0u, 0u, 0u, 0u);
    }
    __syncthreads();

    // producer (thread 0): issue the TMA copies of tile `t` of this item
    auto issue = [&](int t) {
      const uint32_t s = produced % kHistStages;
      const uint32_t use = produced / kHistStages;
      if (use > 0) mbar_wait(s_empty + 8 * s, (use - 1) & 1u);  // consumers released the slot
      mbar_expect_tx(s_full + 8 * s, static_cast<uint32_t>(gcount) * kBlockRows);
      const uint8_t* src = p.bins + static_cast<int64_t>(p.f_begin + f0) * p.n_pad + static_cast<int64_t>(b0 + t) * kBlockRows;
      for (int gi = 0; gi < gcount; gi++)
        tma_bulk_g2s(s_tiles + s * stage_bytes + gi * kBlockRows, src + static_cast<int64_t>(gi) * p.n_pad, kBlockRows, s_full + 8 * s);
      produced++;
    };
    if (tid == 0) {
      const int pre = min(nb, kHistStages - 1);
      for (int t = 0; t < pre; t++) issue(t);
    }

    // Per-block active counts of this item, so that the software pipeline below can look ahead.
    for (int i = tid; i < nb; i += kHistThreads) s_counts[i] = p.act_count[b0 + i];
    __syncthreads();

    const int warp_first = tid & ~31;  // first list index handled by this warp in an iteration
    if (MODE == kHistRootSum) {
      // ---- Root: every row of a block is active and sits in slot 0, so no active list is needed.
      // A thread takes groups of 4 consecutive rows: one 128-bit load of their gradients (prefetched
      // one iteration ahead), one 32-bit shared load of their bins per feature, conflict-free
      // one returning atomic per element; counts come from the precomputed root count histogram.
      auto load_q = [&](int tt, int g) -> uint4 {
        const int ng = (s_counts[tt] + 3) >> 2;
        return g < ng ? __ldg(reinterpret_cast<const uint4*>(p.q24 + static_cast<int64_t>(b0 + tt) * kBlockRows) + g)
                      : make_uint4(0u, 0u, 0u, 0u);
      };
      uint4 cur = load_q(0, tid);
      for (int t = 0; t < nb; t++) {
        if (tid == 0 && t + kHistStages - 1 < nb) issue(t + kHistStages - 1);
        const uint32_t s = consumed % kHistStages;
        const uint32_t parity = (consumed / kHistStages) & 1u;
        const int n_act = s_counts[t];
        const int n_groups = (n_act + 3) >> 2;
        mbar_wait(s_full + 8 * s, parity);
        const uint32_t tile = s_tiles + s * stage_bytes;
        int wb = warp_first;
        if (wb >= n_groups) {
          if (t + 1 < nb) cur = load_q(t + 1, tid);
        } else {
          while (true) {
            const int nwb = wb + kHistThreads;
            const bool more = nwb < n_groups;
            uint4 nxt = make_uint4(0u, 0u, 0u, 0u);
            if (more) nxt = load_q(t, nwb + lane);
            else if (t + 1 < nb) nxt = load_q(t + 1, tid);
            const int g0 = wb + lane;
            const int valid = min(4, n_act - g0 * 4);  // <= 0 for lanes past the end
            const uint32_t q[4] = {cur.x, cur.y, cur.z, cur.w};
            // all 4 rows of every lane of this warp valid => no predication in the hot path
            const bool full = (wb + 31) * 4 + 3 < n_act;
            if (full) {
              for (int gi = 0; gi < gcount; gi++) {
                const uint32_t fbase = s_hist + static_cast<uint32_t>(gi * bins_per_feature) * 4u;
                const uint32_t w = smem_ld_u32(tile + gi * kBlockRows + (g0 << 2));
                uint32_t old[4], a[4];
#pragma unroll
                for (int j = 0; j < 4; j++) a[j] = fbase + (((w >> (8 * j)) & 0xFFu) << 2);
#pragma unroll
                for (int j = 0; j < 4; j++) old[j] = smem_add(a[j], q[j]);
                bool carry = false;
#pragma unroll
                for (int j = 0; j < 4; j++) carry |= (old[j] + q[j] < old[j]);
                if (carry) {
#pragma unroll
                  for (int j = 0; j < 4; j++)
                    if (old[j] + q[j] < old[j]) smem_red(a[j] + plane_bytes, 1u);
                }
              }
            } else {
              for (int gi = 0; gi < gcount; gi++) {
                const uint32_t fbase = s_hist + static_cast<uint32_t>(gi * bins_per_feature) * 4u;
                const uint32_t w = smem_ld_u32(tile + gi * kBlockRows + (min(g0, kBlockRows / 4 - 1) << 2));
                for (int j = 0; j < valid; j++) {
                  const uint32_t a = fbase + (((w >> (8 * j)) & 0xFFu) << 2);
                  const uint32_t o = smem_add(a, q[j]);
                  if (o + q[j] < o) smem_red(a + plane_bytes, 1u);
                }
              }
            }
            cur = nxt;
            if (!more) break;
            wb = nwb;
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(s_empty + 8 * s);
        consumed++;
      }
    } else {
      // ---- General path: compacted active lists, kHistUnroll rows per thread per iteration, the
      // next iteration's list entries prefetched into registers (hides the L2 latency that
      // dominated the first version's stalls: profiles/k_hist_ncu_r01.md).
      auto load_act = [&](int tt, int wb, uint2* dst) {
        const int n = s_counts[tt];
        const uint2* base = p.act + static_cast<int64_t>(b0 + tt) * kBlockRows;
#pragma unroll
        for (int u = 0; u < kHistUnroll; u++) {
          const int e = wb + static_cast<int>(lane) + u * kHistThreads;
          dst[u] = e < n ? __ldg(base + e) : make_uint2(0u, 0u);
        }
      };
      uint2 cur[kHistUnroll];
      load_act(0, warp_first, cur);
      for (int t = 0; t < nb; t++) {
        if (tid == 0 && t + kHistStages - 1 < nb) issue(t + kHistStages - 1);
        const uint32_t s = consumed % kHistStages;
        const uint32_t parity = (consumed / kHistStages) & 1u;
        const int n_act = s_counts[t];
        const uint32_t* h_p = HESS ? p.act_h + static_cast<int64_t>(b0 + t) * kBlockRows : nullptr;
        mbar_wait(s_full + 8 * s, parity);
        const uint32_t tile = s_tiles + s * stage_bytes;
        int wb = warp_first;
        if (wb >= n_act) {
          if (t + 1 < nb) load_act(t + 1, warp_first, cur);
        } else {
          while (true) {
            const int nwb = wb + kHistThreads * kHistUnroll;
            const bool more = nwb < n_act;
            uint2 nxt[kHistUnroll];
#pragma unroll
            for (int u = 0; u < kHistUnroll; u++) nxt[u] = make_uint2(0u, 0u);
            if (more) load_act(t, nwb, nxt);
            else if (t + 1 < nb) load_act(t + 1, warp_first, nxt);

            uint32_t hq[kHistUnroll];
            bool ok[kHistUnroll];
#pragma unroll
            for (int u = 0; u < kHistUnroll; u++) {
              const int e = wb + static_cast<int>(lane) + u * kHistThreads;
              ok[u] = e < n_act;
              hq[u] = (HESS && ok[u]) ? __ldg(h_p + e) : 0u;
            }
            // the last row of the warp's window valid => all rows of all lanes valid: no predication
            const bool full = (wb + 31 + (kHistUnroll - 1) * kHistThreads) < n_act;
            if (full) {
              for (int gi = 0; gi < gcount; gi++) {
                const uint32_t fbase = s_hist + static_cast<uint32_t>(gi * bins_per_feature) * 4u;
                const uint32_t tbase = tile + gi * kBlockRows;
                uint32_t addr[kHistUnroll], old[kHistUnroll], hold[kHistUnroll];
#pragma unroll
                for (int u = 0; u < kHistUnroll; u++) addr[u] = fbase + bin_offset(cur[u].x, smem_ld_u8(tbase + cur[u].y));
                if constexpr (MODE == kHistPacked) {
#pragma unroll
                  for (int u = 0; u < kHistUnroll; u++) {
                    smem_red(addr[u], (((cur[u].x >> kPackedCoarseShift) & 0x3Fu) << kPackedCntBits) | 1u);
                    smem_red(addr[u] + plane_bytes, cur[u].x & kQMax);
                  }
                } else {
#pragma unroll
                for (int u = 0; u < kHistUnroll; u++) {
                  smem_red(addr[u], 1u);
                  old[u] = smem_add(addr[u] + plane_bytes, cur[u].x & kQMax);
                  if (HESS) hold[u] = smem_add(addr[u] + 2u * plane_bytes, hq[u]);
                }
                bool carry = false;
#pragma unroll
                for (int u = 0; u < kHistUnroll; u++) {
                  const uint32_t q = cur[u].x & kQMax;
                  carry |= (old[u] + q < old[u]);
                  if (HESS) carry |= (hold[u] + hq[u] < hold[u]);
                }
                if (carry) {
#pragma unroll
                  for (int u = 0; u < kHistUnroll; u++) {
                    const uint32_t q = cur[u].x & kQMax;
                    if (old[u] + q < old[u]) smem_red(addr[u], 1u << kHistCntBits);
                    if (HESS) {
                      if (hold[u] + hq[u] < hold[u]) smem_red(addr[u] + 3u * plane_bytes, 1u);
                    }
                  }
                }
                }
              }
            } else {
              // tail of the block's active list
              for (int gi = 0; gi < gcount; gi++) {
                const uint32_t fbase = s_hist + static_cast<uint32_t>(gi * bins_per_feature) * 4u;
                const uint32_t tbase = tile + gi * kBlockRows;
#pragma unroll
                for (int u = 0; u < kHistUnroll; u++) {
                  if (!ok[u]) continue;
                  const uint32_t a = fbase + bin_offset(cur[u].x, smem_ld_u8(tbase + cur[u].y));
                  const uint32_t q = cur[u].x & kQMax;
                  if (MODE == kHistPacked) {
                    smem_red(a, (((cur[u].x >> kPackedCoarseShift) & 0x3Fu) << kPackedCntBits) | 1u);
                    smem_red(a + plane_bytes, q);
                    continue;
                  }
                  smem_red(a, 1u);
                  const uint32_t o = smem_add(a + plane_bytes, q);
                  if (o + q < o) smem_red(a, 1u << kHistCntBits);
                  if (HESS) {
                    const uint32_t ho = smem_add(a + 2u * plane_bytes, hq[u]);
                    if (ho + hq[u] < ho) smem_red(a + 3u * plane_bytes, 1u);
                  }
                }
              }
            }
#pragma unroll
            for (int u = 0; u < kHistUnroll; u++) cur[u] = nxt[u];
            if (!more) break;
            wb = nwb;
          }
        }
        // release the tile: one arrival per warp
        __syncwarp();
        if (lane == 0) mbar_arrive(s_empty + 8 * s);
        consumed++;
      }
    }
    __syncthreads();
    // Flush non-empty bins to the global 64-bit histogram.
    int slot_base = 0;
    int used = lv.num_slots * kMaxBins;
    if constexpr (MULTI) {
      slot_base = win_base;
      used = min(lv.num_slots - slot_base, win_count) * kMaxBins;
    }
    {
      const uint32_t* s_cnt = hist;              // kHistRootSum: plane 0 = lo, plane 1 = carries
      const uint32_t* s_lo = hist + B;
      const uint32_t* s_hlo = hist + 2 * B;
      const uint32_t* s_hhi = hist + 3 * B;
      for (int gi = 0; gi < gcount; gi++) {
        const int f_local = f0 + gi;
        for (int i = tid; i < used; i += kHistThreads) {
          const int sl = MULTI ? (i >> 8) + slot_base : (i >> 8), b = i & 0xFF;
          if (MODE == kHistRootSum) {
            const unsigned long long sum =
                (static_cast<unsigned long long>(hist[B + gi * bins_per_feature + i]) << 32) + hist[gi * bins_per_feature + i];
            size_t oc;
            if (sum != 0ull) atomicAdd(&p.hist_sum[slot_hist_offset(sl, f_local, b, p.f_chunk, p.chunk_stride, &oc)], sum);
            continue;
          }
          const uint32_t c = s_cnt[gi * bins_per_feature + i];
          if (MODE == kHistPacked) {
            if (c != 0u) {
              size_t oc;
              const size_t o = slot_hist_offset(sl, f_local, b, p.f_chunk, p.chunk_stride, &oc);
              const unsigned long long base = static_cast<unsigned long long>(c >> kPackedCntBits) << kPackedCoarseShift;
              const uint32_t lo = s_lo[gi * bins_per_feature + i];
              atomicAdd(&p.hist_sum[o], base + static_cast<uint32_t>(lo - static_cast<uint32_t>(base)));
              atomicAdd(&p.hist_cnt[oc], c & kPackedMaxUpdates);
            }
            continue;
          }
          if (c != 0u) {
            size_t oc;
            const size_t o = slot_hist_offset(sl, f_local, b, p.f_chunk, p.chunk_stride, &oc);
            const unsigned long long sum =
                (static_cast<unsigned long long>(c >> kHistCntBits) << 32) + s_lo[gi * bins_per_feature + i];
            atomicAdd(&p.hist_sum[o], sum);
            atomicAdd(&p.hist_cnt[oc], c & ((1u << kHistCntBits) - 1u));
            if (HESS) {
              const unsigned long long hsum =
                  (static_cast<unsigned long long>(s_hhi[gi * bins_per_feature + i]) << 32) +
                  s_hlo[gi * bins_per_feature + i];
              atomicAdd(&p.hist_hsum[o], hsum);
            }
          }
        }
      }
    }
    __syncthreads();
  }
}

// Row counts per (feature, bin) over ALL rows: the root's count histogram, which does not depend
// on the gradients.  Computed once per dataset (plain global atomics; not on the per-iteration path).
__global__ void __launch_bounds__(256) k_root_counts(const uint8_t* bins, int64_t n, int64_t n_pad, int f_count,
                                                    int f_begin, uint32_t* root_cnt /*[f_count][256]*/) {
  __shared__ uint32_t h[kMaxBins];
  const int fl = blockIdx.y;
  h[threadIdx.x] = 0u;
  __syncthreads();
  const uint8_t* col = bins + static_cast<int64_t>(f_begin + fl) * n_pad;  // n_pad is a multiple of 8192: 16-byte aligned
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  const int64_t n16 = n / 16;
  const uint4* col16 = reinterpret_cast<const uint4*>(col);
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n16; i += stride) {
    const uint4 v = col16[i];
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 4; k++) {
      atomicAdd(&h[w[k] & 0xFFu], 1u);
      atomicAdd(&h[(w[k] >> 8) & 0xFFu], 1u);
      atomicAdd(&h[(w[k] >> 16) & 0xFFu], 1u);
      atomicAdd(&h[w[k] >> 24], 1u);
    }
  }
  for (int64_t r = n16 * 16 + static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r < n; r += stride)
    atomicAdd(&h[col[r]], 1u);
  __syncthreads();
  if (h[threadIdx.x] != 0u) atomicAdd(&root_cnt[static_cast<size_t>(fl) * kMaxBins + threadIdx.x], h[threadIdx.x]);
}

// The bound kHistPacked needs: the largest number of rows of one chunk of row blocks that share a bin of one feature
// (any node's rows are a subset of all rows).  Two steps, once per handle: k_sub_counts builds the count histogram of
// every (sub-chunk of row blocks, feature) in one pass over the matrix; k_chunk_max sums the sub-chunks of a
// chunk (chunk sizes are multiples of the sub-chunk: 8 blocks, 1 for small datasets) and takes the maximum over the bins, for every chunk size in use.
__global__ void __launch_bounds__(256) k_sub_counts(const uint8_t* bins, int64_t n, int64_t n_pad, int f_begin, int kSubBlocks,
                                                   uint32_t* out /*[subs][gridDim.y][256]*/) {
  __shared__ uint32_t h[kMaxBins];
  const int fl = blockIdx.y, sub = blockIdx.x;
  h[threadIdx.x] = 0u;
  __syncthreads();
  const int64_t r0 = static_cast<int64_t>(sub) * kSubBlocks * kBlockRows;
  const int64_t r1 = min(n, r0 + static_cast<int64_t>(kSubBlocks) * kBlockRows);
  const uint8_t* col = bins + static_cast<int64_t>(f_begin + fl) * n_pad;
  const int64_t n16 = r1 > r0 ? (r1 - r0) / 16 : 0;   // r0 is a multiple of 8192: 16-byte aligned
  const uint4* col16 = reinterpret_cast<const uint4*>(col + r0);
  for (int64_t i = threadIdx.x; i < n16; i += blockDim.x) {
    const uint4 v = col16[i];
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 4; k++) {
      atomicAdd(&h[w[k] & 0xFFu], 1u);
      atomicAdd(&h[(w[k] >> 8) & 0xFFu], 1u);
      atomicAdd(&h[(w[k] >> 16) & 0xFFu], 1u);
      atomicAdd(&h[w[k] >> 24], 1u);
    }
  }
  for (int64_t r = r0 + n16 * 16 + threadIdx.x; r < r1; r += blockDim.x) atomicAdd(&h[col[r]], 1u);
  __syncthreads();
  out[(static_cast<size_t>(sub) * gridDim.y + fl) * kMaxBins + threadIdx.x] = h[threadIdx.x];
}
__global__ void __launch_bounds__(256) k_chunk_max(const uint32_t* sub_counts, int n_subs, int subs_per_chunk,
                                                  uint32_t* out_max /*one word*/) {
  __shared__ uint32_t s_max[8];
  const int fl = blockIdx.y, chunk = blockIdx.x;
  uint32_t c = 0;
  for (int s = chunk * subs_per_chunk; s < min(n_subs, (chunk + 1) * subs_per_chunk); s++)
    c += sub_counts[(static_cast<size_t>(s) * gridDim.y + fl) * kMaxBins + threadIdx.x];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c = max(c, __shfl_xor_sync(0xffffffffu, c, o));
  if ((threadIdx.x & 31) == 0) s_max[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < 8; i++) c = max(c, s_max[i]);
    atomicMax(out_max, c);
  }
}

}  // namespace ygg
