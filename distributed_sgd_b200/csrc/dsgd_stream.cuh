// dsgd_stream.cuh -- streaming pass over many row windows: Master.localLoss/localAccuracy (core/Master.scala:
// 100-107), SlaveImpl.forward (core/Slave.scala:129-140) and large-batch SlaveImpl.gradient (142-157).
//
// This is the HBM-bound form of the hot path (roofline: 8*nnz + 16 bytes per sample, SURVEY.md 8d).
//   * The weight vector is staged ONCE per CTA into shared memory as fp32 (47 236 x 4 B = 189 KB of the 227 KB),
//     so the ~94 gathers per row hit shared-memory banks, not 32-byte L2 sectors.  One persistent CTA per SM.
//   * FLAT STREAM.  A warp owns blocks of 32 rows and walks their 16-byte units (2 pairs) as ONE virtual
//     stream: unit v of the block belongs to the row whose prefix-sum interval contains v, found with one ballot
//     and one or-reduction per 32 units -- every lane loads a useful unit whatever the row lengths are (round 1
//     walked a row per 16-lane group: 47 of 64 load slots used on the mean row, long rows serialised), kUnroll
//     128-bit loads per lane are in flight before the first is used (64 KB per SM), and consecutive rows of an
//     evaluation pass make every warp load one contiguous 512-byte request.
//   * The dot is needed for its SIGN only (prediction, gate: SparseSVM.scala:14,28), so it is accumulated with fp32
//     FMAs against the fp32 weights -- no fp32->fp64 conversions (ncu, round 1: the XU pipe they run on was 46 %
//     busy).  A lane accumulates its units of the open row; the warp reduces once per ROW END (one 5-step butterfly
//     of ONE float), not per load, and the row's lane just keeps the sum: predictions, counters and gates of the 32
//     rows are worked out by 32 lanes in parallel after the block's stream.  The kernel is ISSUE-bound before it is
//     HBM-bound (ncu: round 2's first cut 108 warp instructions per 64 pairs = 131 us per evaluation pass; 100.8 us at
//     70; 88.7 us at ~55, profiles/r2_streaming.md), so every per-slot instruction counts: groups that lie inside the block
//     carry no bounds predicates (only a block's last group does), a slot without a row end adds its products with one
//     FADD, and a pass over CONSECUTIVE rows (kContig: evaluation) needs no row lookup for its loads at all -- the windows
//     are back to back in the pair array -- so its four loads leave before the row-end masks are even computed.
//   * Blocks are dealt dynamically (one atomic per block, requested a block ahead); the last fifth of a pass goes out in
//     blocks of half the size so the warps run dry together.
//   * Exactness against the fp64 arithmetic of the reference.  That arithmetic sums filt(x_j * w_j): values with
//     |x| <= 1e-20 never enter a row (math/Sparse.scala:108-118; k_repack stores them as 0 and leaves them out of sum|x|),
//     and products with |x w| <= 1e-20 are dropped.  The fp32 result differs from that sum by at most
//       (D + 1) * 2^-24 * max|w| * sum|x|      relative rounding: D = units/32 + 9 roundings on the longest add chain,
//                                              + 1 for rounding w to fp32 (first-order bound)
//     + 2^-150 * sum|x|                        absolute rounding of weights that become fp32 subnormals (or 0)
//     + 1e-20 * pairs                          the products the filter drops; this term also covers the absolute
//                                              rounding of subnormal fp32 products and sums (2^-150 per operation)
//     and the threshold is that bound with 1.5x slack, computed in fp64 so that no term underflows (an fp32 band of
//     2^-24 * max|w| is subnormal below max|w| ~ 1e-31); a dot that overflowed fp32 is never trusted.  sum|x| per row is
//     computed once when the rows are loaded (k_repack, rounded up, stored with the label in its sign bit: one 4-byte
//     load per row).  Rows whose |dot| is inside the band are recomputed with the fp64 weights from L2 after the block's
//     stream, so every prediction and gate decision is that of the fp64 arithmetic
//     (tests/test_gpu_parity.py::test_streaming_exact_fallback_decides_like_fp64, tests/test_gpu_edge_regimes.py).
//   * Scatter (gradient): rows that pass the gate are re-walked after the block's stream (their units are in
//     L1/L2) and y*x goes to g with fp64 REDs.  On trained weights few rows pass (the misclassified ones) and the pass
//     runs at the streaming rate; on untrained weights every row passes and the fp64 RED rate at L2 bounds it
//     (0.45 per SM-cycle, tools/microbench.cu).  Per-CTA fixed-point accumulators in shared memory for the most
//     frequent columns were measured and dropped: 162 -> 160 us on 262 144 rows, 58 -> 64 us on 65 536
//     (profiles/r2_streaming.md).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "dsgd_kernels.cuh"

namespace dsgd {

struct TrueTag { static constexpr bool value = true; };
struct FalseTag { static constexpr bool value = false; };

constexpr int kStreamThreads = 1024;
constexpr int kStreamUnroll = 4;

struct StreamParams {
  const uint32_t *rp16;
  const uint4 *units;      // the pair array viewed as 16-byte units (2 pairs)
  const float *yabs;       // per row: label * sum_j |x_j| (rounded up); the sign bit is the label
  const int32_t *samples;  // nullptr: rows [row_begin, row_begin + n)
  int64_t row_begin, n;
  const double *w;         // fp64 weights (exact fallback, L2)
  const float *w32;        // fp32 shadow of the same weights
  int dim;
  double *g;               // scatter target (fp64, L2) or nullptr
  double *preds;           // per-sample predictions or nullptr
  unsigned long long *cnt; // kCntHinge / kCntCorrect
  unsigned long long *n_exact;     // rows that took the exact fallback (diagnostic)
  unsigned long long *next_block;  // work counter (zero on entry): blocks beyond the first wave are claimed dynamically
  int rows_log2;               // rows per block = 1 << rows_log2 (5, 4 or 3): the host picks it so that every warp gets
                               // several blocks (a block is the unit of the dynamic work distribution)
  int64_t n_big;               // blocks [0, n_big) have 1 << rows_log2 rows, the blocks after them 1 << tail_log2: the
  int tail_log2;               // last part of a pass is dealt in smaller pieces, so the warps run dry together
};

__host__ __device__ constexpr size_t stream_smem_bytes(int dim) { return (((size_t)dim + 3) & ~(size_t)3) * sizeof(float); }

// kContig: the rows of the pass are consecutive (samples == nullptr), hence so are their windows in the pair array: unit v
// of a block sits at (first window) + v and the loads need no row lookup (5 instructions per slot less, and the row-end
// masks are worked out while the loads are in flight).
template <bool kScatter, bool kPreds, bool kContig>
__global__ void __launch_bounds__(kStreamThreads, 1) k_stream_rows(const StreamParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float *ws = reinterpret_cast<float *>(smem_raw);
  __shared__ float s_wmax[kStreamThreads / 32];
  __shared__ unsigned long long s_cnt[2];

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned lt_mask = (1u << lane) - 1u;
  const int rlog = p.rows_log2, tlog = p.tail_log2;
  const int64_t tail_row0 = p.n_big << rlog;   // first row of the smaller tail blocks
  const int64_t n_blocks = p.n_big + ((p.n - tail_row0 + (1 << tlog) - 1) >> tlog);
  const int64_t warp_global = (int64_t)blockIdx.x * (kStreamThreads / 32) + warp;
  const int64_t n_warps = (int64_t)gridDim.x * (kStreamThreads / 32);
  unsigned hinge = 0, correct = 0, n_exact = 0;

  // bounds of the block being processed / the next one: lane l holds row l of the block
  auto load_block = [&](int64_t blk, int64_t &first, uint32_t &b, uint32_t &e, float &ya, bool &valid) {
    const bool big = blk < p.n_big;
    first = big ? (blk << rlog) : tail_row0 + ((blk - p.n_big) << tlog);
    const int64_t i = first + lane;
    b = 0u; e = 0u; ya = 0.f;
    valid = blk < n_blocks && lane < (1 << (big ? rlog : tlog)) && i < p.n;
    if (valid) {
      const int64_t rid = (!kContig && p.samples) ? (int64_t)__ldg(&p.samples[i]) : p.row_begin + i;
      b = __ldg(&p.rp16[rid]);
      e = __ldg(&p.rp16[rid + 1]);
      ya = __ldg(&p.yabs[rid]);
    }
  };
  // Work distribution: the first wave is static (block = warp id), later blocks are claimed from a global counter one
  // step ahead; the ticket (an atomic with a return value) is requested when a block starts and read when it ends, the
  // next block's bounds were prefetched a block earlier.
  unsigned long long ticket = 0;   // lane 0: the pending claim
  auto claim_issue = [&]() {
    if (lane == 0) ticket = atomicAdd(p.next_block, 1ull);
  };
  auto claim_get = [&]() -> int64_t { return (int64_t)__shfl_sync(0xffffffffu, ticket, 0) + n_warps; };
  uint32_t nb, ne; float nya; bool nvalid; int64_t nfirst;
  int64_t blk = warp_global;
  int64_t blk_next = n_blocks;
  if (blk < n_blocks) claim_issue();
  load_block(blk, nfirst, nb, ne, nya, nvalid);   // (requested before the weights are staged: latency off the path)

  // ---- stage the fp32 weights, find max|w| ----
  float wmax = 0.f;
  {
    const float4 *src = reinterpret_cast<const float4 *>(p.w32);
    float4 *dst = reinterpret_cast<float4 *>(ws);
    const int n4 = p.dim >> 2;
    for (int i = threadIdx.x; i < n4; i += kStreamThreads) {
      const float4 v = __ldg(&src[i]);
      dst[i] = v;
      wmax = fmaxf(wmax, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
    }
    for (int i = (n4 << 2) + threadIdx.x; i < p.dim; i += kStreamThreads) {
      const float v = __ldg(&p.w32[i]);
      ws[i] = v;
      wmax = fmaxf(wmax, fabsf(v));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) wmax = fmaxf(wmax, __shfl_xor_sync(0xffffffffu, wmax, o));
    if (lane == 0) s_wmax[warp] = wmax;
    if (threadIdx.x < 2) s_cnt[threadIdx.x] = 0ull;
    __syncthreads();
    wmax = 0.f;
#pragma unroll
    for (int i = 0; i < kStreamThreads / 32; ++i) wmax = fmaxf(wmax, s_wmax[i]);
  }
  const double band_rel = 1.5 * 0x1p-24 * (double)wmax;   // 1.5 * 2^-24 * max|w|, in fp64: no underflow for any fp32 wmax
  // one gradient entry (SparseSVM.scala:26-29): a reduction without a return value
  auto scatter_one = [&](uint32_t col, double gv) {
    if (gv != 0.0) red_add_f64(&p.g[col], gv);
  };

  if (blk < n_blocks) blk_next = claim_get();
  for (; blk < n_blocks;) {
    uint32_t b = nb;
    int len = (int)(ne - nb);   // units
    float ya = nya;
    bool valid = nvalid;
    const int64_t first = nfirst;   // first row (position in the pass) of this block
    load_block(blk_next, nfirst, nb, ne, nya, nvalid);
    if (blk_next < n_blocks) claim_issue();   // for the block after next: read at the end of this block
    int opos = lane;            // position of this lane's row inside the block (before compaction)
    // empty rows: dot 0 -> prediction 0, hinge 1, never correct, nothing to scatter (SparseSVM.scala:14-16)
    if (valid && len == 0) {
      hinge += 1u;
      if (kPreds) p.preds[first + lane] = 0.0;
    }
    const unsigned ne_mask = __ballot_sync(0xffffffffu, valid && len > 0);
    if (ne_mask != 0xffffffffu) {   // compact the non-empty rows to lanes 0 .. n-1 (order kept)
      const unsigned src = __fns(ne_mask, 0, lane + 1);
      const bool has = src < 32u;
      const int sl = has ? (int)src : 0;
      b = __shfl_sync(0xffffffffu, b, sl);
      len = __shfl_sync(0xffffffffu, len, sl);
      ya = __shfl_sync(0xffffffffu, ya, sl);
      opos = sl;
      valid = has;
      if (!has) len = 0;
    } else {
      valid = true;
    }
    const int y = (__float_as_uint(ya) >> 31) ? -1 : 1;
    // P = inclusive prefix sum of the row lengths: row l covers virtual units [P - len, P)
    int P = len;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int a = __shfl_up_sync(0xffffffffu, P, o);
      if (lane >= o) P += a;
    }
    const int total = __shfl_sync(0xffffffffu, P, 31);
    const uint32_t base = b - (uint32_t)(P - len);   // unit address of virtual unit v of this row = base + v (mod 2^32)
    const uint32_t base0 = __shfl_sync(0xffffffffu, base, 0);   // kContig: the same for every row of the block
    const int my_end = len > 0 ? P - 1 : -1;          // virtual position of this row's LAST unit
    float acc_p = 0.f;                                // this lane's share of the OPEN row: sum x*w
    float dot_mine = 0.f;                             // this lane's row: x.w in fp32 once the row is closed
    int row0 = 0;                                     // rows closed so far (warp-uniform)

    // One GROUP = kStreamUnroll slots of 32 units: where rows end inside the group (one or-reduction per slot), hence the
    // row of each lane's unit, then the 128-bit loads -- all issued before the first is used (64 KB in flight per SM).
    // Groups that lie entirely inside the block (kFull) carry no bounds predicates; the block's last group does.
    // (A software-prefetched form -- group g + 1 fetched before group g is processed, 768 threads x 80 registers -- was
    // measured SLOWER: 118.9 us against 107.4 us per evaluation pass, profiles/r2_streaming.md: the lost warps cost more
    // latency hiding than the deeper queue bought.)
    auto do_group = [&](auto full_tag, const int v0) {
      constexpr bool kFull = decltype(full_tag)::value;
      uint4 q[kStreamUnroll];
      unsigned ends[kStreamUnroll];   // bit j: a row's LAST unit sits at lane j of this slot
      const unsigned pos = (unsigned)(my_end - v0);          // < 32 * kStreamUnroll iff the row ends in this group
      const unsigned bit = 1u << (pos & 31u);
      if constexpr (kContig) {
#pragma unroll
        for (int i = 0; i < kStreamUnroll; ++i) {
          if (kFull || v0 + 32 * i + lane < total) q[i] = __ldg(&p.units[base0 + (uint32_t)(v0 + 32 * i + lane)]);
          else q[i] = make_uint4(0u, 0u, 0u, 0u);  // col 0, val +0.0f
        }
#pragma unroll
        for (int i = 0; i < kStreamUnroll; ++i)
          ends[i] = __reduce_or_sync(0xffffffffu, (pos >> 5) == (unsigned)i ? bit : 0u);
      } else {
        int r0 = row0;
#pragma unroll
        for (int i = 0; i < kStreamUnroll; ++i) {
          ends[i] = __reduce_or_sync(0xffffffffu, (pos >> 5) == (unsigned)i ? bit : 0u);
          const int rmy = r0 + __popc(ends[i] & lt_mask);      // row of this lane's unit
          r0 += __popc(ends[i]);
          const uint32_t bs = __shfl_sync(0xffffffffu, base, rmy & 31);
          if (kFull || v0 + 32 * i + lane < total) q[i] = __ldg(&p.units[bs + (uint32_t)(v0 + 32 * i + lane)]);
          else q[i] = make_uint4(0u, 0u, 0u, 0u);
        }
      }
#pragma unroll
      for (int i = 0; i < kStreamUnroll; ++i) {
        float pp = __fmaf_rn(__uint_as_float(q[i].w), ws[q[i].z], __uint_as_float(q[i].y) * ws[q[i].x]);
        if (!kFull && !(v0 + 32 * i + lane < total)) pp = 0.f;   // a masked unit reads ws[0]: keep a NaN / inf weight out
        unsigned m = ends[i];
        if (m == 0u) {   // warp-uniform: no row ends inside this slot
          acc_p += pp;
        } else {
          const int rmy = row0 + __popc(m & lt_mask);           // row0 == rows closed before this slot
          do {   // close the rows that end inside this slot, in order
            m &= m - 1u;
            float sp = acc_p + (rmy == row0 ? pp : 0.f);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) sp += __shfl_xor_sync(0xffffffffu, sp, o);
            if (lane == row0) dot_mine = sp;
            acc_p = 0.f;
            ++row0;
          } while (m);
          acc_p = (rmy == row0) ? pp : 0.f;
        }
      }
    };
    {
      int v0 = 0;
      for (; v0 + 32 * kStreamUnroll <= total; v0 += 32 * kStreamUnroll) do_group(TrueTag{}, v0);
      if (v0 < total) do_group(FalseTag{}, v0);
    }
    // ---- 32 rows decided by 32 lanes: inside the rounding band -> exact recomputation; else the sign is certain ----
    bool need_exact = false, do_scatter = false;
    int pred_mine = 0;
    // prediction known for this lane's row: counters and the gate (y * dot < 0  <=>  pred == y)
    auto finalize = [&](int pr) {
      pred_mine = pr;
      hinge += (unsigned)(1 - y * pr);
      correct += (unsigned)(pr == y);
      do_scatter = kScatter && (pr != y);
    };
    if (valid) {
      // the band of the header comment: relative rounding (D + 1) * 2^-24 * max|w| * sum|x|, absolute rounding of fp32
      // weights below 2^-126 (2^-150 per unit of sum|x|), and the products of at most 1e-20 that the fp64 arithmetic drops
      // (<= 2 * len pairs); all with 1.5x slack, in fp64 so that no term underflows
      const double thresh = (double)fabsf(ya) * (band_rel * (double)((len >> 5) + 10) + 1.5 * 0x1p-150) + 3e-20 * (double)len;
      const float ad = fabsf(dot_mine);
      if (!((double)ad > thresh && ad <= 3.4028235e38f)) need_exact = true;   // also catches NaN and an fp32 overflow
      else finalize(dot_mine > 0.f ? -1 : 1);
    }
    // ---- exact recomputation of the rows the fp32 sign could not decide ----
    unsigned ex = __ballot_sync(0xffffffffu, need_exact);
    while (ex) {
      const int r = __ffs(ex) - 1;
      ex &= ex - 1u;
      const uint32_t rb = __shfl_sync(0xffffffffu, b, r);
      const int rl = __shfl_sync(0xffffffffu, len, r);
      double acc = 0.0;
      for (int u = lane; u < rl; u += 32) {
        const uint4 qq = __ldg(&p.units[rb + (uint32_t)u]);
        acc += filt(filt((double)__uint_as_float(qq.y)) * __ldcg(&p.w[qq.x]));
        acc += filt(filt((double)__uint_as_float(qq.w)) * __ldcg(&p.w[qq.z]));
      }
      const double dot = warp_sum(acc);
      if (lane == r) {
        finalize(pred_of(dot));
        ++n_exact;
      }
    }
    if (kPreds) {
      if (valid) p.preds[first + opos] = (double)pred_mine;
    }
    // ---- scatter y*x of the rows that passed the gate (SparseSVM.scala:28) ----
    if (kScatter) {
      unsigned sc = __ballot_sync(0xffffffffu, do_scatter);
      while (sc) {
        const int r = __ffs(sc) - 1;
        sc &= sc - 1u;
        const uint32_t rb = __shfl_sync(0xffffffffu, b, r);
        const int rl = __shfl_sync(0xffffffffu, len, r);
        const double yy = (double)__shfl_sync(0xffffffffu, y, r);
        for (int u = lane; u < rl; u += 32) {
          const uint4 qq = __ldg(&p.units[rb + (uint32_t)u]);
          scatter_one(qq.x, filt(filt((double)__uint_as_float(qq.y)) * yy));
          scatter_one(qq.z, filt(filt((double)__uint_as_float(qq.w)) * yy));
        }
      }
    }
    blk = blk_next;
    if (blk < n_blocks) blk_next = claim_get();
  }
  // ---- counters: lane -> warp -> CTA -> one atomic per CTA ----
  hinge = __reduce_add_sync(0xffffffffu, hinge);
  correct = __reduce_add_sync(0xffffffffu, correct);
  n_exact = __reduce_add_sync(0xffffffffu, n_exact);
  if (lane == 0) {
    atomicAdd(&s_cnt[0], (unsigned long long)hinge);
    atomicAdd(&s_cnt[1], (unsigned long long)correct);
    if (p.n_exact && n_exact) atomicAdd(p.n_exact, (unsigned long long)n_exact);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    if (s_cnt[0]) atomicAdd(&p.cnt[kCntHinge], s_cnt[0]);
    if (s_cnt[1]) atomicAdd(&p.cnt[kCntCorrect], s_cnt[1]);
  }
}

}  // namespace dsgd
