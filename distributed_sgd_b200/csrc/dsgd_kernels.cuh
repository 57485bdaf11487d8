// dsgd_kernels.cuh -- sm_100a kernels of the SGD hot path (see DESIGN.md for the layout and rooflines).
//
// Device layout of the rows ("row windows"): one array of 8-byte (col:int32, val:fp32) pairs, each row
// padded with (col = last col, val = 0) pairs to a multiple of 2 pairs so that every row window starts on
// a 16-byte boundary and is a multiple of 16 bytes long (what cp.async.bulk / 128-bit loads need).
// rp16[r] is the window start in 16-byte units.  A val == 0 pair is arithmetically inert everywhere:
// it adds 0 to the dot product and is skipped by the scatter.
//
// State vectors (w, g, d) are fp64 and live in L2 (3 x 378 KB on a 126 MB L2); the HBM stream is the
// row windows only.  All reference arithmetic cited as path:line under
// /root/reference/src/main/scala/epfl/distributed/.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace dsgd {

constexpr double kEps = 1e-20;  // math/Sparse.scala:104

// Slots of the per-ctx scalar block (double[kNumScal]) kept on the device.
enum Scal : int {
  kScalC = 0,      // c = 2*lambda*(w . d) of the CURRENT resident weights (SparseSVM.scala:31)
  kScalNrm2 = 1,   // ||w||^2 of the current resident weights (SparseSVM.scala:21)
  kScalReqC = 2,   // same two for a request-supplied weight vector (GradientRequest.weights)
  kScalReqNrm2 = 3,
  kNumScal = 8
};
// Slots of the per-ctx counter block (unsigned long long[kNumCnt]).
enum Cnt : int {
  kCntHinge = 0,    // sum of per-sample hinge losses of the running batch (integers: 0, 1 or 2 each)
  kCntCorrect = 1,  // #{pred == y}
  kCntTicket = 2,   // last-block ticket of k_update
  kNumCnt = 8
};

__device__ __forceinline__ double filt(double v) { return fabs(v) > kEps ? v : 0.0; }  // Sparse.scala:108-118

// Gradient scatter: a reduction WITHOUT a return value.  Written as PTX `red` because nvcc 12.9 compiles atomicAdd(double *)
// with an unused result to ATOMG (result discarded, but the response still travels back: ncu counted 1.9 M returned sectors
// per 300 steps) inside the large persistent kernels, and to REDG only in small ones.
__device__ __forceinline__ void red_add_f64(double *p, double v) {
  asm volatile("red.relaxed.gpu.global.add.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}
__device__ __forceinline__ void red_add_f64_sys(double *p, double v) {   // peer replicas over NVLink
  asm volatile("red.relaxed.sys.global.add.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}
__device__ __forceinline__ void red_add_u64_sys(unsigned long long *p, unsigned long long v) {
  asm volatile("red.relaxed.sys.global.add.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// prediction = -signum(x . w)  (core/ml/SparseSVM.scala:14)
__device__ __forceinline__ int pred_of(double dot) { return (dot > 0.0) ? -1 : ((dot < 0.0) ? 1 : 0); }

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Block-wide sum in a fixed order (deterministic run to run). Result valid in thread 0.
template <int kThreads>
__device__ __forceinline__ double block_sum(double v, double *smem /* kThreads/32 */) {
  v = warp_sum(v);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) smem[wid] = v;
  __syncthreads();
  double s = 0.0;
  if (threadIdx.x == 0) {
#pragma unroll
    for (int i = 0; i < kThreads / 32; ++i) s += smem[i];
  }
  __syncthreads();
  return s;
}

// ---------------------------------------------------------------------------------------------------
// k_prepare: c = lambda*2*(w . d) and ||w||^2 for a weight vector (SparseSVM.scala:31,21).  One block,
// fixed-order reduction.  47 236 elements: ~2 us; only used when the host installs weights -- in the
// step loop k_update produces both numbers for the next step.
// ---------------------------------------------------------------------------------------------------
template <int kThreads>
__global__ void __launch_bounds__(kThreads) k_prepare(const double *__restrict__ w, const double *__restrict__ d,
                                                      int dim, double lambda, double *__restrict__ scal_c,
                                                      double *__restrict__ scal_nrm2) {
  __shared__ double red[kThreads / 32];
  double sd = 0.0, sn = 0.0;
  for (int j = threadIdx.x; j < dim; j += kThreads) {
    const double wj = w[j];
    sd += filt(wj * d[j]);  // (w * d).sum: products below 1e-20 are dropped by the Sparse constructor
    sn += wj * wj;
  }
  sd = block_sum<kThreads>(sd, red);
  sn = block_sum<kThreads>(sn, red);
  if (threadIdx.x == 0) {
    *scal_c = lambda * 2.0 * sd;
    *scal_nrm2 = sn;
  }
}

// ---------------------------------------------------------------------------------------------------
// k_rows: the per-sample body of SlaveImpl.gradient / SlaveImpl.forward (core/Slave.scala:129-157):
// one warp per row window; fp64 dot with the L2-resident weights; prediction, hinge loss, gate; scatter
// y*x into the dense gradient with fp64 reductions at L2 (no return value -> RED, not ATOM).
//   kScatter: accumulate backward() into g            (SparseSVM.scala:26-29)
//   kPreds:   write p = -signum(x.w) per sample       (SparseSVM.scala:14)
// samples == nullptr walks rows [row_begin, row_begin + n).
// Hinge losses are integers (y, p in {-1,0,1}), so batch loss and accuracy are accumulated as exact
// integer counters: deterministic regardless of the order in which warps finish.
// ---------------------------------------------------------------------------------------------------
template <bool kScatter, bool kPreds>
__global__ void __launch_bounds__(256) k_rows(const uint32_t *__restrict__ rp16, const uint2 *__restrict__ pairs,
                                              const int8_t *__restrict__ label, const int32_t *__restrict__ samples,
                                              int64_t row_begin, int64_t n, const double *__restrict__ w,
                                              double *__restrict__ g, double *__restrict__ preds,
                                              unsigned long long *__restrict__ cnt) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  unsigned hinge = 0, correct = 0;  // lane 0 only
  for (int64_t i = warp0; i < n; i += nwarps) {
    const int64_t r = samples ? (int64_t)samples[i] : row_begin + i;
    const int64_t b = (int64_t)rp16[r] * 2, e = (int64_t)rp16[r + 1] * 2;
    double dot = 0.0;
    for (int64_t k = b + lane; k < e; k += 32) {
      const uint2 pr = pairs[k];
      const double xv = filt((double)__uint_as_float(pr.y));
      dot += filt(xv * w[pr.x]);  // (x * w).sum  (math/Vec.scala:58; math/Sparse.scala:46)
    }
    dot = warp_sum(dot);
    const double y = (double)label[r];
    const int p = (dot > 0.0) ? -1 : ((dot < 0.0) ? 1 : 0);  // -signum(dot)
    if (lane == 0) {
      const int l = 1 - (int)y * p;  // max(0, 1 - y*p), never negative for y,p in {-1,0,1}
      hinge += (unsigned)l;
      correct += (unsigned)(p == (int)y);
      if (kPreds) preds[i] = (double)p;
    }
    if (kScatter) {
      if (!(y * dot < 0.0)) {  // SparseSVM.scala:28: gradient is y*x unless activity < 0
        for (int64_t k = b + lane; k < e; k += 32) {
          const uint2 pr = pairs[k];
          const double gv = filt(filt((double)__uint_as_float(pr.y)) * y);
          if (gv != 0.0) atomicAdd(&g[pr.x], gv);
        }
      }
    }
  }
  if (lane == 0 && (hinge | correct)) {
    atomicAdd(&cnt[kCntHinge], (unsigned long long)hinge);
    atomicAdd(&cnt[kCntCorrect], (unsigned long long)correct);
  }
}

// ---------------------------------------------------------------------------------------------------
// k_finish: regularize in place -- r_j = g_j + c on the keys that survived the 1e-20 filter
// (SparseSVM.scala:31; math/Vec.scala:65-75).  Also publishes the batch's hinge sum and size in
// g[dim], g[dim+1] so that they ride along in the gradient allreduce.
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_finish(double *__restrict__ g, int dim, const double *__restrict__ scal_c,
                                                const unsigned long long *__restrict__ cnt, double n_samples) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const double c = *scal_c;
  const bool add_c = (c != 0.0) && (fabs(c) > kEps);
  if (j < dim) {
    double v = filt(g[j]);
    if (v != 0.0 && add_c) v = filt(v + c);
    g[j] = v;
  } else if (j == dim) {
    g[dim] = (double)cnt[kCntHinge];
    g[dim + 1] = n_samples;
  }
}

// ---------------------------------------------------------------------------------------------------
// k_finish_acc: one logical worker's reply folded into the master's running sum.  r = regularize(g) on the
// worker's own support (SparseSVM.scala:31), then sum <- sum + r with the constructor filter after the
// addition (Vec.sum is a left fold of `+`, math/Vec.scala:128-131), g cleared for the next worker.
// Slots [dim], [dim+1] of `sum` carry the hinge total and the sample count of the step.
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_finish_acc(double *__restrict__ g, double *__restrict__ sum, int dim,
                                                    const double *__restrict__ scal_c,
                                                    unsigned long long *__restrict__ cnt, double n_samples, int first) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const double c = *scal_c;
  const bool add_c = (c != 0.0) && (fabs(c) > kEps);
  if (j < dim) {
    const double raw = g[j];
    double v = filt(raw);
    if (v != 0.0 && add_c) v = filt(v + c);
    if (raw != 0.0) g[j] = 0.0;
    sum[j] = first ? v : filt(sum[j] + v);
  } else if (j == dim) {
    const double h = (double)cnt[kCntHinge];
    sum[dim] = first ? h : sum[dim] + h;
    sum[dim + 1] = first ? n_samples : sum[dim + 1] + n_samples;
    cnt[kCntHinge] = 0ull;
    cnt[kCntCorrect] = 0ull;
  }
}

// ---------------------------------------------------------------------------------------------------
// k_update: the master's aggregate + SGD update (core/Master.scala:194,197) fused with the bookkeeping
// for the next step:  w_j <- w_j - lr * (sum_j / K);  gradient buffer zeroed;  c and ||w||^2 of the NEW
// weights reduced (fixed order: per-block partial -> last block sums the slots in index order) so that the
// next step needs no separate reduction; per-step loss = lambda*||w_before||^2 + hinge/total written.
//   kFuseRegularize: the buffer holds the raw local sum (single worker): apply regularize() here.
//   otherwise it holds sum_k r^(k) (already regularized per worker, then allreduced).
// ---------------------------------------------------------------------------------------------------
template <bool kFuseRegularize>
__global__ void __launch_bounds__(256) k_update(double *__restrict__ w, float *__restrict__ w32,
                                                double *__restrict__ g, const double *__restrict__ d, int dim,
                                                double lambda, double lr, double inv_k_den, double *__restrict__ scal,
                                                unsigned long long *__restrict__ cnt, double *__restrict__ partial,
                                                double n_samples_local, double *__restrict__ loss_out) {
  __shared__ double red[8];
  __shared__ bool is_last;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const double c = scal[kScalC];
  const bool add_c = (c != 0.0) && (fabs(c) > kEps);
  double pd = 0.0, pn = 0.0;
  if (j < dim) {
    const double raw = g[j];
    double v = raw;
    if (kFuseRegularize) {
      v = filt(v);
      if (v != 0.0 && add_c) v = filt(v + c);
    }
    double wn = w[j];
    if (raw != 0.0) g[j] = 0.0;
    if (v != 0.0) {
      const double mean = filt(v / inv_k_den);  // Vec.mean: sum / K
      const double step = filt(mean * lr);      // learningRate * grad
      wn = filt(wn - step);                     // batchWeights - ...
      w[j] = wn;
      w32[j] = (float)wn;
    }
    pd = filt(wn * d[j]);
    pn = wn * wn;
  }
  pd = block_sum<256>(pd, red);
  pn = block_sum<256>(pn, red);
  if (threadIdx.x == 0) {
    partial[2 * blockIdx.x] = pd;
    partial[2 * blockIdx.x + 1] = pn;
    __threadfence();
    const unsigned long long t = atomicAdd(&cnt[kCntTicket], 1ull);
    is_last = (t == (unsigned long long)gridDim.x - 1);
  }
  __syncthreads();
  if (is_last) {
    __threadfence();
    double sd = 0.0, sn = 0.0;
    if (threadIdx.x == 0) {
      for (unsigned b = 0; b < gridDim.x; ++b) {
        sd += __ldcg(&partial[2 * b]);
        sn += __ldcg(&partial[2 * b + 1]);
      }
      // per-step loss on the weights the gradient was taken at (SparseSVM.scala:20-23; SURVEY.md F5)
      double hinge, total;
      if (kFuseRegularize) {
        hinge = (double)cnt[kCntHinge];
        total = n_samples_local;
      } else {
        hinge = g[dim];
        total = g[dim + 1];
        g[dim] = 0.0;
        g[dim + 1] = 0.0;
      }
      if (loss_out) *loss_out = lambda * scal[kScalNrm2] + hinge / total;
      scal[kScalC] = lambda * 2.0 * sd;
      scal[kScalNrm2] = sn;
      cnt[kCntHinge] = 0ull;
      cnt[kCntCorrect] = 0ull;
      cnt[kCntTicket] = 0ull;
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// k_loss_scalar: loss = lambda*||w||^2 + hinge/n, acc = correct/n from the integer counters.
// ---------------------------------------------------------------------------------------------------
__global__ void k_loss_scalar(const double *__restrict__ scal_nrm2, unsigned long long *__restrict__ cnt,
                              double lambda, double n, double *__restrict__ out2) {
  out2[0] = lambda * (*scal_nrm2) + (double)cnt[kCntHinge] / n;
  out2[1] = (double)cnt[kCntCorrect] / n;
  out2[2] = (double)cnt[kCntHinge];   // exact: counts are far below 2^53
  out2[3] = (double)cnt[kCntCorrect];
  out2[4] = *scal_nrm2;
  cnt[kCntHinge] = 0ull;
  cnt[kCntCorrect] = 0ull;
}

// ---------------------------------------------------------------------------------------------------
// K0: document frequencies and dimSparsity (Main.scala:54-65).
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_col_hist(const uint2 *__restrict__ pairs, int64_t n_pairs,
                                                  unsigned *__restrict__ df) {
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n_pairs; k += (int64_t)gridDim.x * blockDim.x) {
    const uint2 pr = pairs[k];
    if (fabs((double)__uint_as_float(pr.y)) > kEps) atomicAdd(&df[pr.x], 1u);  // padding pairs have val == 0
  }
}
__global__ void __launch_bounds__(256) k_dim_sparsity(const unsigned *__restrict__ df, int dim, double *__restrict__ d) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < dim) {
    // reference key c of d holds 1/(df_c + 1); weight column c is reference key c+1, so it meets d key c+1 (Q3)
    const int src = c + 1;
    d[c] = (src < dim && df[src] != 0u) ? 1.0 / ((double)df[src] + 1.0) : 0.0;
  }
}

// ---------------------------------------------------------------------------------------------------
// Repack: host CSR (row_ptr int64, col, val) -> aligned pair windows.  One thread per destination pair.
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_repack(const int64_t *__restrict__ row_ptr, const int32_t *__restrict__ col,
                                                const float *__restrict__ val, const uint32_t *__restrict__ rp16,
                                                const int8_t *__restrict__ label, int64_t n_rows, uint2 *__restrict__ pairs,
                                                float *__restrict__ yabs) {
  // one warp per row keeps the writes coalesced
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t r = warp0; r < n_rows; r += nwarps) {
    const int64_t sb = row_ptr[r], se = row_ptr[r + 1];
    const int64_t db = (int64_t)rp16[r] * 2, de = (int64_t)rp16[r + 1] * 2;
    const int64_t len = se - sb;
    double asum = 0.0;
    for (int64_t k = lane; k < de - db; k += 32) {
      uint2 pr;
      if (k < len) {
        // a value the Sparse constructor drops (|x| <= 1e-20, math/Sparse.scala:108-118) is stored as +0: every fp64
        // consumer applies filt(x) first and sees the same absent key, and the fp32 dot of the streaming pass no longer
        // adds a product the fp64 arithmetic never forms (its rounding band, dsgd_stream.cuh, relies on this)
        const double xv = filt((double)val[sb + k]);
        pr.x = (uint32_t)col[sb + k];
        pr.y = __float_as_uint((float)xv);
        asum += fabs(xv);
      } else {
        pr.x = len > 0 ? (uint32_t)col[se - 1] : 0u;
        pr.y = 0u;
      }
      pairs[db + k] = pr;
    }
    // yabs[r] = label * sum_j |x_j| rounded UP to fp32 (the sign bit carries the label, also on a zero sum): the streaming
    // pass reads the label and the rounding-band scale of a row with one 4-byte load
    asum = warp_sum(asum);
    if (lane == 0) {
      const float a = __double2float_ru(asum);
      yabs[r] = label[r] < 0 ? -a : a;
    }
  }
}

__global__ void __launch_bounds__(256) k_to_f32(const double *__restrict__ src, float *__restrict__ dst, int n) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < n) dst[j] = (float)src[j];
}

}  // namespace dsgd
