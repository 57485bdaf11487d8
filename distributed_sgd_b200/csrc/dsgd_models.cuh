// dsgd_models.cuh -- a MODEL SET: M SparseSVMs with their own (lambda, learning rate) trained on the same batch draws by
// ONE persistent cooperative kernel, one grid barrier per SGD step for all of them.
//
// The reference trains one `new SparseSVM(config.lambda, ...)` per run (Main.scala:68) with Master.fit's batch loop
// (core/Master.scala:179-198); a sweep over lambda / learning rate reruns all of it.  The batch draws do not depend on
// the model, so the models of a set share what a step of k_sync_persistent (dsgd_persistent.cuh) spends most of its time
// on: the sample ids, the TMA row loads, the launch and the grid barrier.  Each model pays for its own gathers, gate and
// scatter and for its own update.
//
// Layout (one GPU, one worker per step; interval I_t between grid barrier t-1 and t, as in k_sync_persistent):
//   PRODUCER warp : produce_stages() below (the producer of k_sync_persistent) -- a step's rows are staged ONCE for all models.
//   CONSUMER warps: the work unit is (chunk of a row, model), dealt round-robin to the warps: a CTA holds ~2 rows of a
//                   batch-256 step, so the models of one chunk go to different warps and their gathers overlap instead of
//                   queueing behind one warp.  Per unit: one 16-byte {W, g} gather per non-zero from the model's records,
//                   W_t applied on the fly (FetchLocal), dot, gate, RED of y*x into the model's g_t.
//   UPDATE warps  : W_t <- update(W_{t-1}, g_{t-1}, c_{t-1}) for every model and every column (dense: the records of 4
//                   models are requested together), W_t stored into the record arrays that need it, the CTA's partial
//                   {W_t . d, ||W_t||^2} of each model pushed into that model's exact accumulator (acc_push).
//   After the barrier, update warp 0 reads every model's accumulator with one request per lane (lane k ends with model
//   k's sums) and publishes c_t of all models through one mbarrier.
//
// Records of model k: three rotating arrays {W, g} like the single-model kernel, but with no weights held in registers
// (M x columns would not fit): in interval t the update thread of column j reads {W_{t-1}, g_{t-1}} (buffer t-1), stores
// W_t into buffer t where g_{t-1} != 0 (elsewhere buffer t already holds W_{t-1} == W_t) and {W_t, 0} into buffer t+1,
// which nobody reads in interval t and which the consumers RED g_{t+1} into during interval t+1.
#pragma once
#include "dsgd_persistent.cuh"

namespace dsgd {

constexpr int kMaxModels = 32;   // DSGD_MAX_MODELS: 3 record arrays of 16 bytes per column and model stay inside the L2

struct ModelsParams {
  const uint32_t *rp16;
  const uint2 *pairs;
  const int8_t *label;
  const int32_t *samples;  // n_steps * batch ids, step-major
  int64_t n_steps;
  int32_t batch;
  int32_t dim;
  int32_t n_act;            // models of this launch (the active ones), slot k = 0 .. n_act-1
  int64_t rec_stride;       // records between two record arrays
  double2 *rec;             // slot k, buffer i: rec + (3 * k + i) * rec_stride; on entry all three = {W_init, 0}
  const double *d;
  unsigned long long *acc;  // [3 rotating][n_act][kAccStride]: exact accumulators of {W.d, ||W||^2}; zero on entry
  unsigned *hinge;          // [n_steps][n_act], zero on entry
  double *losses;           // [n_steps][n_act] or nullptr
  double *w_res;            // resident weights of the whole set, [n_models][dim]
  unsigned *bar;            // grid barrier: arrival counter, zero on entry
  int *abort_flag;          // set to 1 if a wait hit the watchdog
  long long timeout_cycles;
  int32_t id[kMaxModels];   // slot -> model index in w_res
  double lambda[kMaxModels], lr[kMaxModels];
};
static_assert(sizeof(ModelsParams) <= 4000, "kernel parameter space is 4 KB");

template <int kCons, int kUpd, int kStages, int kStagePairs, int kMaxChunks>
struct ModelsSmem {
  uint2 ring[kStages][kStagePairs];
  StageMeta<kMaxChunks> meta[kStages];
  uint64_t full[kStages];
  uint64_t empty[kStages];
  uint64_t c_bar[2];                       // c of every model for the interval's updates
  uint64_t u_bar;                          // every update warp has left its partials in red[]
  double part[kMaxChunks][kMaxModels];     // pass-1 partial dots of the stage being consumed (rows of several chunks)
  double red[kMaxModels][kUpd][2];
  double c_val[2][kMaxModels];
  unsigned hinge_acc[kMaxModels];
  int ok;
};

// ---- the producer warp: runs ahead of everybody else, bounded only by the empty[] barriers.  Lane m owns row m. --------
// The producer of k_sync_persistent as a function (same stage layout, same chunk list).  k_sync_persistent keeps its inline
// copy: calling this function from it changed that kernel's register allocation and cost 0.45 % of its bench throughput
// on a B200 (5.994e7 -> 5.969e7 samples/s, two alternated runs each, spread 0.05 %).
template <int kStages, int kStagePairs, int kMaxChunks, class Smem>
__device__ __forceinline__ void produce_stages(const ModelsParams &p, Smem &sm, const int64_t S, const int B, const int G,
                                               const int n_r, const int lane) {
  auto load_id = [&](int64_t t) -> int32_t {
    return (t < S && lane < n_r) ? __ldg(&p.samples[t * B + blockIdx.x + lane * G]) : -1;
  };
  uint32_t b0 = 0, e0 = 0, b1 = 0, e1 = 0;
  int y0 = 0, y1 = 0;
  auto load_win = [&](int32_t id, uint32_t &b, uint32_t &e, int &y) {
    b = 0u; e = 0u; y = 0;
    if (id >= 0) {
      b = __ldg(&p.rp16[id]);
      e = __ldg(&p.rp16[id + 1]);
      y = (int)__ldg(&p.label[id]);
    }
  };
  load_win(load_id(0), b0, e0, y0);   // window of step t      (stage C input)
  load_win(load_id(1), b1, e1, y1);   // window of step t + 1  (stage B)
  int32_t id_next = load_id(2);       // sample id of step t + 2 (stage A)
  for (int64_t t = 0; t < S; ++t) {
    const int st = (int)t & (kStages - 1);
    if (t >= kStages) {
      mbar_wait(&sm.empty[st], (unsigned)(((t / kStages) - 1) & 1), p.abort_flag, p.timeout_cycles);
      if (*(volatile int *)p.abort_flag) return;  // the barrier-synchronised warps gave up (watchdog)
    }
    auto &mt = sm.meta[st];
    // lay the rows out: exclusive scans over the CTA's rows of pairs and chunks
    const int len = (lane < n_r) ? (int)(e0 - b0) * 2 : 0;
    const int nch = (len + kChunkPairs - 1) / kChunkPairs;
    int ps = len, cs = nch;  // inclusive warp scans
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int a = __shfl_up_sync(0xffffffffu, ps, o), c2 = __shfl_up_sync(0xffffffffu, cs, o);
      if (lane >= o) { ps += a; cs += c2; }
    }
    const int my_pair = ps - len, my_chunk = cs - nch;
    const bool listed = (my_chunk + nch) <= kMaxChunks;           // prefix property: later rows miss too
    const bool in_ring = listed && (my_pair + len) <= kStagePairs;
    if (lane < n_r) {
      mt.row_y[lane] = y0;
      mt.row_b[lane] = b0;
      mt.row_len[lane] = len;
      mt.row_first[lane] = (short)my_chunk;
      mt.row_nch[lane] = (short)(listed ? nch : -1);
      if (listed) {
        for (int c = 0; c < nch; ++c) {
          const int n = min(kChunkPairs, len - c * kChunkPairs);
          mt.ch_off[my_chunk + c] = in_ring ? (uint32_t)(my_pair + c * kChunkPairs)
                                            : (kChunkGlobal | (b0 * 2u + (uint32_t)(c * kChunkPairs)));
          mt.ch_n[my_chunk + c] = (short)n;
          mt.ch_row[my_chunk + c] = (short)lane;
        }
      }
    }
    const unsigned my_bytes = (lane < n_r && in_ring) ? (unsigned)len * 8u : 0u;
    const unsigned ring_bytes = __reduce_add_sync(0xffffffffu, my_bytes);
    // chunks actually written to the list: everything up to the first row that did not fit it
    const int listed_chunks = __reduce_max_sync(0xffffffffu, (lane < n_r && listed) ? (my_chunk + nch) : 0);
    const unsigned multi = __ballot_sync(0xffffffffu, lane < n_r && listed && nch > 1);
    if (lane == 31) mt.n_pairs = ps;
    if (lane == 0) {
      mt.n_rows = n_r;
      mt.n_chunks = listed_chunks;
      mt.n_multi = __popc(multi);
    }
    __syncwarp();  // every lane's metadata is written before lane 0 arrives on the full barrier
    if (lane == 0) {
      if (ring_bytes) mbar_expect_tx(&sm.full[st], ring_bytes);
      else mbar_arrive(&sm.full[st]);  // metadata only: complete the phase
    }
    __syncwarp();
    if (my_bytes) bulk_g2s(&sm.ring[st][my_pair], p.pairs + (size_t)b0 * 2, my_bytes, &sm.full[st]);
    // advance the register pipeline
    b0 = b1; e0 = e1; y0 = y1;
    load_win(id_next, b1, e1, y1);
    id_next = load_id(t + 3);
  }
}

// acc_read for up to 32 accumulators at once: every lane requests 16 bytes of up to 4 of them before any is looked at
// (one L2 round trip instead of one per model); lane k returns model k's two sums (the conversion of acc_read).
__device__ __forceinline__ void acc_read_models(const unsigned long long *acc, int M, int lane, double &sd, double &sn) {
  unsigned long long q0[4], q1[4];
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    q0[g] = 0ull; q1[g] = 0ull;
    const int k = g * 8 + (lane >> 2);
    if (k < M)
      asm volatile("ld.relaxed.gpu.global.v2.u64 {%0, %1}, [%2];"
                   : "=l"(q0[g]), "=l"(q1[g]) : "l"(acc + (size_t)k * kAccStride + 2 * (lane & 3)) : "memory");
  }
  long long l[7];
#pragma unroll
  for (int i = 0; i < 7; ++i) {
    const int src = (lane & 7) * 4 + (i >> 1);
    long long v = 0;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      const long long x = (long long)__shfl_sync(0xffffffffu, (i & 1) ? q1[g] : q0[g], src);
      if (g == (lane >> 3)) v = x;
    }
    l[i] = v;
  }
  const double nan = __longlong_as_double(0x7ff8000000000000ll);
  sd = ((double)l[0] * 0x1p-80 + (double)l[1] * 0x1p-40) + (double)l[2];
  sn = ((double)l[3] * 0x1p-80 + (double)l[4] * 0x1p-40) + (double)l[5];
  if (l[6] != 0) { sd = nan; sn = nan; }
}

// The consumer warps' work on one stage for every model of the set: consume_stage (dsgd_persistent.cuh) with the
// (chunk, model) pair as the unit of work.  recp(k) / recc(k): records of slot k for steps t-1 / t.
template <int kCons, int kMaxChunks, class Smem, class RecPrev, class RecCur>
__device__ __forceinline__ void consume_stage_models(Smem &sm, StageMeta<kMaxChunks> &mt, const uint2 *ring, const ModelsParams &p,
                                                     const int M, RecPrev recp, RecCur recc, uint64_t *cbar, unsigned cpar,
                                                     const double *cval, int warp, int lane) {
  const int n_ch = mt.n_chunks;
  auto fetch_of = [&](int k) {
    return FetchLocal{recp(k), cbar, cpar, cval + k, p.abort_flag, p.timeout_cycles, 1.0, p.lr[k]};
  };
  auto add_hinge = [&](int k, unsigned h) {
    if (lane == 0 && h) atomicAdd(&sm.hinge_acc[k], h);
  };
  // ---- pass 1: dots of this warp's (chunk, model) units; rows of one chunk are finished here ----
  for (int u = warp; u < n_ch * M; u += kCons) {
    const int c = u / M, k = u - c * M;
    const uint32_t off = mt.ch_off[c];
    const int n = mt.ch_n[c];
    const uint2 *src = (off & kChunkGlobal) ? (p.pairs + (off & ~kChunkGlobal)) : (ring + off);
    uint2 pr[4];
    double wv[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int i = q * 32 + lane;
      pr[q] = (i < n) ? src[i] : make_uint2(0u, 0u);  // val 0: inert
    }
    FetchLocal fetch = fetch_of(k);
    fetch.get4(pr, wv);
    double acc = 0.0;
#pragma unroll
    for (int q = 0; q < 4; ++q) acc += filt(filt((double)__uint_as_float(pr[q].y)) * wv[q]);  // (x * w).sum
    acc = warp_sum(acc);
    const int row = mt.ch_row[c];
    if (mt.row_nch[row] == 1) {
      const int yi = mt.row_y[row];
      const double y = (double)yi;
      add_hinge(k, (unsigned)(1 - yi * pred_of(acc)));
      if (!(y * acc < 0.0)) {  // SparseSVM.scala:28
        double2 *R = recc(k);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const double gvv = filt(filt((double)__uint_as_float(pr[q].y)) * y);
          if (gvv != 0.0) red_add_f64(&R[pr[q].x].y, gvv);
        }
      }
      continue;
    }
    if (lane == 0) sm.part[c][k] = acc;
  }
  // ---- pass 2 (rows of several chunks): row dot = chunk partials in order, prediction, gate, scatter ----
  if (mt.n_multi > 0) {
    named_bar_sync(2, kCons * 32);
    for (int u = warp; u < n_ch * M; u += kCons) {
      const int c = u / M, k = u - c * M;
      const int row = mt.ch_row[c];
      const int first = mt.row_first[row], nch = mt.row_nch[row];
      if (nch == 1) continue;
      double dot = 0.0;
      for (int i = 0; i < nch; ++i) dot += sm.part[first + i][k];
      const int yi = mt.row_y[row];
      const double y = (double)yi;
      if (c == first) add_hinge(k, (unsigned)(1 - yi * pred_of(dot)));
      if (!(y * dot < 0.0)) {
        const uint32_t off = mt.ch_off[c];
        const int n = mt.ch_n[c];
        const uint2 *src = (off & kChunkGlobal) ? (p.pairs + (off & ~kChunkGlobal)) : (ring + off);
        double2 *R = recc(k);
        for (int i = lane; i < n; i += 32) {
          const uint2 pr = src[i];
          const double gvv = filt(filt((double)__uint_as_float(pr.y)) * y);
          if (gvv != 0.0) red_add_f64(&R[pr.x].y, gvv);
        }
      }
    }
  }
  // rows outside the chunk list: empty rows (hinge 1, nothing to scatter) and, if a step ever overflows the chunk list,
  // whole rows straight from global memory, one warp per (row, model)
  for (int u = warp; u < mt.n_rows * M; u += kCons) {
    const int m = u / M, k = u - m * M;
    const int nch = mt.row_nch[m];
    if (nch == 0) {
      add_hinge(k, 1u);
    } else if (nch < 0) {
      FetchLocal fetch = fetch_of(k);
      const uint2 *grow = p.pairs + (size_t)mt.row_b[m] * 2;
      const int len = mt.row_len[m];
      double acc = 0.0;
      for (int i = lane; i < len; i += 32) {
        const uint2 pr = __ldg(&grow[i]);
        acc += filt(filt((double)__uint_as_float(pr.y)) * fetch.get1(pr.x));
      }
      const double dot = warp_sum(acc);
      const int yi = mt.row_y[m];
      const double y = (double)yi;
      add_hinge(k, (unsigned)(1 - yi * pred_of(dot)));
      if (!(y * dot < 0.0)) {
        double2 *R = recc(k);
        for (int i = lane; i < len; i += 32) {
          const uint2 pr = __ldg(&grow[i]);
          const double gvv = filt(filt((double)__uint_as_float(pr.y)) * y);
          if (gvv != 0.0) red_add_f64(&R[pr.x].y, gvv);
        }
      }
    }
  }
}

template <int kCons, int kUpd, int kStages, int kStagePairs, int kMaxChunks>
__global__ void __launch_bounds__((kCons + kUpd + 1) * 32, 1) k_models_persistent(const ModelsParams p) {
  using Smem = ModelsSmem<kCons, kUpd, kStages, kStagePairs, kMaxChunks>;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  Smem &sm = *reinterpret_cast<Smem *>(smem_raw);

  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const bool is_cons = warp < kCons;
  const bool is_upd = warp >= kCons && warp < kCons + kUpd;
  const int G = gridDim.x;
  const int B = p.batch;
  const int64_t S = p.n_steps;
  const int M = p.n_act;
  constexpr int kSyncThreads = (kCons + kUpd) * 32;
  const int n_r = (B > (int)blockIdx.x) ? (B - 1 - (int)blockIdx.x) / G + 1 : 0;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&sm.full[s], 1u);
      mbar_init(&sm.empty[s], (unsigned)kCons);
    }
    mbar_init(&sm.c_bar[0], 1u);
    mbar_init(&sm.c_bar[1], 1u);
    mbar_init(&sm.u_bar, (unsigned)kUpd);
    for (int k = 0; k < kMaxModels; ++k) { sm.c_val[0][k] = 0.0; sm.hinge_acc[k] = 0u; }   // interval 0: nothing pending
    sm.ok = 1;
  }
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  __syncthreads();
  if (threadIdx.x == 0) mbar_arrive(&sm.c_bar[0]);

  if (!is_cons && !is_upd) {
    produce_stages<kStages, kStagePairs, kMaxChunks>(p, sm, S, B, G, n_r, lane);
    return;
  }

  const int64_t rs = p.rec_stride;
  const int n_upd = G * kUpd * 32;
  const int u0 = blockIdx.x * kUpd * 32 + ((int)threadIdx.x - kCons * 32);
  constexpr int kUpdCols = 2;   // columns an update thread keeps d of in registers (47 236 columns: <= 2 on 148 SMs)
  constexpr int kUB = 4;        // models whose records an update thread requests together
  double dreg[kUpdCols];
#pragma unroll
  for (int i = 0; i < kUpdCols; ++i) {
    const int j = u0 + i * n_upd;
    dreg[i] = (is_upd && j < p.dim) ? __ldg(&p.d[j]) : 0.0;
  }

  unsigned phase = 0;
  int ti_prev = 2, ti_cur = 0, ti_next = 1;
  for (int64_t t = 0; t <= S; ++t) {
    const bool first = (t == 0), last = (t == S);
    const unsigned long long *acc_prev = p.acc + (size_t)ti_prev * M * kAccStride;
    unsigned long long *acc_cur = p.acc + (size_t)ti_cur * M * kAccStride;
    unsigned long long *acc_next = p.acc + (size_t)ti_next * M * kAccStride;
    const int bp = ti_prev, bc = ti_cur, bn = ti_next;
    auto recp = [&](int k) -> const double2 * { return p.rec + (3 * (int64_t)k + bp) * rs; };
    auto recc = [&](int k) -> double2 * { return p.rec + (3 * (int64_t)k + bc) * rs; };
    auto recn = [&](int k) -> double2 * { return p.rec + (3 * (int64_t)k + bn) * rs; };
    const unsigned c_par = (unsigned)((t >> 1) & 1);

    // ---- update warp 0, first thing: c_{t-1} and ||W_{t-1}||^2 of every model from the partials the last barrier delivered ----
    if (warp == kCons && !first) {
      double sd, sn;
      acc_read_models(acc_prev, M, lane, sd, sn);
      if (lane < M) {
        sm.c_val[t & 1][lane] = p.lambda[lane] * 2.0 * sd;
        // loss of step t-1 = lambda*||W_{t-1}||^2 + hinge_{t-1}/batch  (SparseSVM.scala:20-23)
        if (p.losses && blockIdx.x == 0)
          p.losses[(t - 1) * M + lane] = p.lambda[lane] * sn + (double)__ldcg(&p.hinge[(t - 1) * M + lane]) / (double)B;
      }
      if (blockIdx.x == 0)
        for (int i = lane; i < M * 8; i += 32) acc_next[(size_t)(i >> 3) * kAccStride + (i & 7)] = 0ull;
      __syncwarp();
      if (lane == 0) mbar_arrive(&sm.c_bar[t & 1]);
    }

    if (is_cons) {
      if (!last) {
        const int st = (int)t & (kStages - 1);
        auto &mt = sm.meta[st];
        mbar_wait(&sm.full[st], (unsigned)(((unsigned)t / kStages) & 1u), p.abort_flag, p.timeout_cycles);
        consume_stage_models<kCons, kMaxChunks>(sm, mt, &sm.ring[st][0], p, M, recp, recc, &sm.c_bar[t & 1], c_par,
                                                &sm.c_val[t & 1][0], warp, lane);
        __syncwarp();
        if (lane == 0) mbar_arrive(&sm.empty[st]);
      }
    } else {
      // ---- update warps: every model, every column this thread owns ----
      const int uw = warp - kCons;
      bool have_c = false;
      for (int k0 = 0; k0 < M; k0 += kUB) {
        double2 r[kUB][kUpdCols];
#pragma unroll
        for (int q = 0; q < kUB; ++q)
#pragma unroll
          for (int i = 0; i < kUpdCols; ++i) {
            const int j = u0 + i * n_upd;
            r[q][i] = (k0 + q < M && j < p.dim) ? __ldcg(&recp(k0 + q)[j]) : make_double2(0.0, 0.0);
          }
        if (!have_c) {
          mbar_wait(&sm.c_bar[t & 1], c_par, p.abort_flag, p.timeout_cycles);
          have_c = true;
        }
#pragma unroll
        for (int q = 0; q < kUB; ++q) {
          const int k = k0 + q;
          if (k >= M) break;   // uniform: every thread has the same M
          const double c_prev = *(volatile double *)&sm.c_val[t & 1][k];
          const bool add_c = (c_prev != 0.0) && (fabs(c_prev) > kEps);
          const double lr = p.lr[k];
          double2 *Rc = recc(k), *Rn = recn(k);
          double *wres = p.w_res + (size_t)p.id[k] * p.dim;
          double pd = 0.0, pn = 0.0;
          auto column = [&](int j, double2 rv, double dj) {
            const double wn = apply_update(rv.x, rv.y, c_prev, add_c, 1.0, lr);
            if (rv.y != 0.0) Rc[j].x = wn;        // elsewhere buffer t already holds W_{t-1} == W_t
            Rn[j] = make_double2(wn, 0.0);        // W_t and a clean g for step t+1
            if (last) wres[j] = wn;
            pd += filt(wn * dj);
            pn += wn * wn;
          };
#pragma unroll
          for (int i = 0; i < kUpdCols; ++i) {
            const int j = u0 + i * n_upd;
            if (j < p.dim) column(j, r[q][i], dreg[i]);
          }
          for (int j = u0 + kUpdCols * n_upd; j < p.dim; j += n_upd)   // more columns than kUpdCols per update thread
            column(j, __ldcg(&recp(k)[j]), __ldg(&p.d[j]));
          pd = warp_sum(pd);
          pn = warp_sum(pn);
          if (lane == 0) { sm.red[k][uw][0] = pd; sm.red[k][uw][1] = pn; }
        }
      }
      if (!have_c) mbar_wait(&sm.c_bar[t & 1], c_par, p.abort_flag, p.timeout_cycles);
      __syncwarp();
      if (lane == 0) mbar_arrive(&sm.u_bar);
      // update warp 0: the CTA's partial of model `lane`, summed in warp order, into that model's accumulator
      if (uw == 0) {
        mbar_wait(&sm.u_bar, (unsigned)(t & 1), p.abort_flag, p.timeout_cycles);
        if (lane < M) {
          double sd = 0.0, sn = 0.0;
#pragma unroll
          for (int i = 0; i < kUpd; ++i) { sd += sm.red[lane][i][0]; sn += sm.red[lane][i][1]; }
          if (sd != 0.0 || sn != 0.0) acc_push(acc_cur + (size_t)lane * kAccStride, sd, sn);
        }
        __syncwarp();
      }
    }

    // the CTA's hinge totals ahead of the arrival (warp 0; thread 0 arrives after its warp's REDs)
    named_bar_sync(3, kSyncThreads);
    ++phase;
    if (warp == 0) {
      if (!last && lane < M) {
        const unsigned h = sm.hinge_acc[lane];
        if (h) atomicAdd(&p.hinge[t * M + lane], h);
        sm.hinge_acc[lane] = 0u;
      }
      __syncwarp();
      if (lane == 0) {
        bool bar_ok = grid_barrier_arrive_wait(p.bar, phase * (unsigned)G, p.abort_flag, p.timeout_cycles);
        if (*(volatile int *)&sm.ok == 0) { *(volatile int *)p.abort_flag = 1; bar_ok = false; }
        sm.ok = bar_ok ? 1 : 0;
      }
    }
    named_bar_sync(3, kSyncThreads);
    if (*(volatile int *)&sm.ok == 0) return;
    { const int a = ti_prev; ti_prev = ti_cur; ti_cur = ti_next; ti_next = a; }
  }
}

// Records a launch starts from: slot k's three buffers = {W of model id[k], 0}.  Grid (columns / 256, n_act).
__global__ void __launch_bounds__(256) k_models_rec_init(const ModelsParams p) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const int k = blockIdx.y;
  if (j < p.dim) {
    const double2 r = make_double2(p.w_res[(size_t)p.id[k] * p.dim + j], 0.0);
#pragma unroll
    for (int i = 0; i < 3; ++i) p.rec[(3 * (int64_t)k + i) * p.rec_stride + j] = r;
  }
}

}  // namespace dsgd
