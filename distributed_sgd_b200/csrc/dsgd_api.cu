// dsgd_api.cu -- the C ABI declared in include/dsgd.h over the sm_100a kernels in dsgd_kernels.cuh.
// There is no CPU path in this library: without a usable GPU dsgd_create fails with DSGD_ERR_CUDA.
#include "../../include/dsgd.h"

#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>  // types only: the library itself is bound at run time (see nccl_api)

#include <algorithm>
#include <cmath>
#include <limits>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "dsgd_kernels.cuh"
#include "dsgd_persistent.cuh"
#include "dsgd_stream.cuh"
#include "dsgd_async.cuh"
#include "dsgd_models.cuh"
#include <cstdlib>

using namespace dsgd;

struct dsgd_ctx {
  int device = 0;
  int32_t dim = 0;
  double lambda = 0.0;
  int rank = 0, world = 1;
  uint32_t flags = 0;
  int sm_count = 0;
  std::string dev_name;

  cudaStream_t own_stream = nullptr;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  int64_t launches = 0;

  // rows
  int64_t n_rows = 0, nnz = 0, n_pairs = 0;
  bool rows_unique = false;   // every row's columns are strictly increasing (no duplicate keys: the reference's rows are Maps)
  uint32_t *rp16 = nullptr;
  uint2 *pairs = nullptr;
  int8_t *label = nullptr;
  float *yabs = nullptr;   // label * sum_j |x_j| per row (dsgd_kernels.cuh: k_repack)

  // state (fp64, L2 resident) -- g has dim + 2 slots (hinge sum and batch size ride in the allreduce)
  double *w = nullptr, *g = nullptr, *d = nullptr, *w_req = nullptr;
  float *w32 = nullptr, *w32_req = nullptr;
  unsigned long long *n_exact = nullptr;  // rows that took the exact fallback in streaming passes (diagnostic)
  bool stream_ready = false;
  double *scal = nullptr;
  unsigned long long *cnt = nullptr;
  double *partial = nullptr;  // 2 doubles per k_update block
  double *out2 = nullptr;     // loss, acc, hinge sum, correct count, ||w||^2
  double *gsum = nullptr;     // master-side running sum of worker replies (dim + 2)
  std::vector<int32_t> worker_counts;  // logical workers on this ctx (empty: one worker, whole slice)
  int32_t n_local = 1, k_total = 0;    // k_total == 0: world
  bool have_d = false;

  // staged sample indices / per-step losses
  int32_t *samples = nullptr;
  int64_t samples_cap = 0, samples_n = 0;
  double *losses = nullptr;
  int64_t losses_cap = 0;
  double *preds = nullptr;
  int64_t preds_cap = 0;

  ncclComm_t comm = nullptr;

  // persistent sync kernel resources (allocated on first use)
  double *p_wbuf[2] = {nullptr, nullptr};            // K GPUs
  double *p_gbuf[3] = {nullptr, nullptr, nullptr};   // K GPUs
  double2 *p_rec[3] = {nullptr, nullptr, nullptr};   // one GPU: rotating {W, g} records
  unsigned long long *p_acc = nullptr;   // fixed-point accumulators of the per-CTA partials [3][kAccStride]
  unsigned *p_hinge = nullptr;
  int64_t p_hinge_cap = 0;
  unsigned *p_bar = nullptr;   // [0]: grid barrier counter, [1]: abort flag
  bool p_ready = false;
  long long *p_tl = nullptr;   // debug timeline (DSGD_PERSIST_TIMELINE)

  // async (Hogwild) mode
  cudaStream_t astream = nullptr;   // the worker loop
  cudaStream_t stream2 = nullptr;   // service calls that must not queue behind anything
  double *m_w = nullptr;            // master replica hosted by this ctx (dsgd_async_host_master)
  double *outbox = nullptr;         // dsgd_async_outbox_enable: running sum of -delta of THIS worker (a replica-shaped block)
  double *peer_w[kMaxReplicas] = {};  // [r] = replica of rank r, [world] = master replica; nullptr: not attached
  bool peer_ipc[kMaxReplicas] = {};
  int *a_stop = nullptr;
  unsigned long long *a_cnt = nullptr;   // [0] claimed, [1] done
  double *a_scratch = nullptr;
  int64_t a_scratch_lanes = 0;
  int32_t *a_rows = nullptr, *a_assigned = nullptr, *a_replay = nullptr;
  int64_t a_rows_cap = 0, a_assigned_cap = 0, a_replay_cap = 0;
  int32_t *u_idx = nullptr; double *u_val = nullptr; int64_t u_cap = 0;  // update_grad staging
  bool a_running = false;
  cudaEvent_t a_ev0 = nullptr, a_ev1 = nullptr;

  // sync-mode receive area shared with peers over NVLink: value words [sender][parity][dim + 8] x 16 B, then bitmap
  // words [sender][parity][ceil((dim + 1) / 32)] x 8 B (dsgd_persistent.cuh)
  double *xblk = nullptr;
  double *peer_x[kMaxWorld] = {};
  bool peer_x_ipc[kMaxWorld] = {};
  int grid_limit = 0;   // dsgd_set_grid_limit: CTAs of the persistent sync kernel (0: one per SM)
  int64_t x_step = 0;   // global step counter of the fused multi-GPU kernel (identical on every rank)
  int64_t x_steps_run = 0;  // SGD steps run by the fused kernel so far (dsgd_xchg_stats)
  unsigned long long *x_llw = nullptr;  // this rank's weights in LL form, two parities
  unsigned long long *x_stats = nullptr;  // [0] value words, [1] bitmap words pushed to each peer so far; [2] SGD steps of those launches

  // model set (dsgd_models_*): resident weights of every model and the model-set kernel's buffers
  int32_t ms_n = 0;
  std::vector<double> ms_lambda, ms_lr;
  double *ms_w = nullptr;               // [ms_n][dim]
  double2 *ms_rec = nullptr;            // [ms_n][3][dim]: rotating {W, g} records
  unsigned long long *ms_acc = nullptr; // [3][ms_n][kAccStride]
  unsigned *ms_hinge = nullptr;         // [n_steps][active models]
  double *ms_losses = nullptr;
  int64_t ms_hinge_cap = 0, ms_losses_cap = 0;
  unsigned *ms_bar = nullptr;           // [0]: grid barrier counter, [1]: abort flag
  bool ms_ready = false;

  // sampled per-launch timing of the gradient kernel
  int32_t prof_every = 0;
  int64_t prof_seen = 0;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> prof_events;
  size_t prof_used = 0;

  mutable std::string err;
  mutable std::string info;
};

static thread_local std::string g_create_err;

// NCCL is bound lazily with dlopen instead of at link time: a host process may already carry its own libnccl.so.2
// (PyTorch bundles a newer one than the system's), and two different libraries under one SONAME cannot coexist.
// Order: a copy already loaded in the process, then $DSGD_NCCL_PATH, then the default search path.
struct nccl_api {
  ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  const char *(*GetErrorString)(ncclResult_t) = nullptr;
  bool ok = false;
  std::string why;
};
static nccl_api &nccl() {
  static nccl_api api = [] {
    nccl_api a;
    void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);
    if (!h)
      if (const char *p = getenv("DSGD_NCCL_PATH")) h = dlopen(p, RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) { a.why = std::string("cannot load libnccl.so.2: ") + dlerror(); return a; }
    a.GetUniqueId = (decltype(a.GetUniqueId))dlsym(h, "ncclGetUniqueId");
    a.CommInitRank = (decltype(a.CommInitRank))dlsym(h, "ncclCommInitRank");
    a.AllReduce = (decltype(a.AllReduce))dlsym(h, "ncclAllReduce");
    a.CommDestroy = (decltype(a.CommDestroy))dlsym(h, "ncclCommDestroy");
    a.GetErrorString = (decltype(a.GetErrorString))dlsym(h, "ncclGetErrorString");
    a.ok = a.GetUniqueId && a.CommInitRank && a.AllReduce && a.CommDestroy && a.GetErrorString;
    if (!a.ok) a.why = "libnccl.so.2 lacks a required symbol";
    return a;
  }();
  return api;
}

static int fail(const dsgd_ctx *ctx, int code, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (ctx) ctx->err = buf; else g_create_err = buf;
  return code;
}

#define CU(call)                                                                                        \
  do {                                                                                                  \
    cudaError_t e_ = (call);                                                                            \
    if (e_ != cudaSuccess)                                                                              \
      return fail(ctx, DSGD_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, \
                  __LINE__);                                                                            \
  } while (0)
#define NC(call)                                                                                         \
  do {                                                                                                   \
    ncclResult_t r_ = (call);                                                                            \
    if (r_ != ncclSuccess)                                                                               \
      return fail(ctx, DSGD_ERR_NCCL, "%s failed: %s (%s:%d)", #call, nccl().GetErrorString(r_), __FILE__, \
                  __LINE__);                                                                             \
  } while (0)
#define NEED(cond, code, ...) \
  do {                        \
    if (!(cond)) return fail(ctx, code, __VA_ARGS__); \
  } while (0)
#define LAUNCHED() (++ctx->launches)

// returns the event pair to bracket this gradient launch with, or nullptr
static std::pair<cudaEvent_t, cudaEvent_t> *prof_slot(dsgd_ctx *ctx) {
  if (ctx->prof_every <= 0) return nullptr;
  if ((ctx->prof_seen++ % ctx->prof_every) != 0) return nullptr;
  if (ctx->prof_used == ctx->prof_events.size()) {
    if (ctx->prof_events.size() >= 16384) return nullptr;
    cudaEvent_t a, b;
    if (cudaEventCreate(&a) != cudaSuccess || cudaEventCreate(&b) != cudaSuccess) return nullptr;
    ctx->prof_events.emplace_back(a, b);
  }
  return &ctx->prof_events[ctx->prof_used++];
}

static inline int cdiv(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// ---- lifecycle ---------------------------------------------------------------------------------------

extern "C" int dsgd_create(dsgd_ctx **out, int device, int32_t dim, double lambda, int rank, int world, uint32_t flags) {
  dsgd_ctx *ctx = nullptr;
  if (!out) return fail(nullptr, DSGD_ERR_INVALID, "dsgd_create: out is NULL");
  *out = nullptr;
  if (dim <= 0) return fail(nullptr, DSGD_ERR_INVALID, "dsgd_create: dim must be positive (got %d)", dim);
  if (world <= 0 || rank < 0 || rank >= world)
    return fail(nullptr, DSGD_ERR_INVALID, "dsgd_create: bad rank/world %d/%d", rank, world);
  int n_dev = 0;
  cudaError_t e = cudaGetDeviceCount(&n_dev);
  if (e != cudaSuccess || n_dev == 0)
    return fail(nullptr, DSGD_ERR_CUDA, "dsgd_create: no usable CUDA device (%s); this library has no CPU path",
                e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
  if (device < 0 || device >= n_dev)
    return fail(nullptr, DSGD_ERR_INVALID, "dsgd_create: device %d out of range [0,%d)", device, n_dev);
  ctx = new dsgd_ctx();
  ctx->device = device; ctx->dim = dim; ctx->lambda = lambda; ctx->rank = rank; ctx->world = world; ctx->flags = flags;
  auto bail = [&](const char *what, cudaError_t err) {
    int rc = fail(nullptr, DSGD_ERR_CUDA, "dsgd_create: %s: %s", what, cudaGetErrorString(err));
    delete ctx;
    return rc;
  };
  if ((e = cudaSetDevice(device)) != cudaSuccess) return bail("cudaSetDevice", e);
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return bail("cudaGetDeviceProperties", e);
  ctx->sm_count = prop.multiProcessorCount;
  ctx->dev_name = prop.name;
  if (prop.major != 10)
    { int rc = fail(nullptr, DSGD_ERR_CUDA, "dsgd_create: device %d is sm_%d%d; this library is built for sm_100a only",
                    device, prop.major, prop.minor); delete ctx; return rc; }
  if ((e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking)) != cudaSuccess) return bail("stream", e);
  if (flags & DSGD_FLAG_ASYNC) {   // the worker loop's stream and the service stream exist in async mode only: streams
                                   // beyond the device's hardware queues (8 by default) alias and serialise each other
    if ((e = cudaStreamCreateWithFlags(&ctx->astream, cudaStreamNonBlocking)) != cudaSuccess) return bail("stream", e);
    if ((e = cudaStreamCreateWithFlags(&ctx->stream2, cudaStreamNonBlocking)) != cudaSuccess) return bail("stream", e);
  }
  if ((e = cudaMalloc(&ctx->a_stop, sizeof(int))) != cudaSuccess) return bail("cudaMalloc a_stop", e);
  if ((e = cudaMalloc(&ctx->a_cnt, sizeof(unsigned long long) * 2)) != cudaSuccess) return bail("cudaMalloc a_cnt", e);
  cudaMemsetAsync(ctx->a_stop, 0, sizeof(int), ctx->own_stream);
  cudaMemsetAsync(ctx->a_cnt, 0, sizeof(unsigned long long) * 2, ctx->own_stream);
  ctx->stream = ctx->own_stream;
  if ((e = cudaEventCreate(&ctx->ev0)) != cudaSuccess) return bail("event", e);
  if ((e = cudaEventCreate(&ctx->ev1)) != cudaSuccess) return bail("event", e);
  const size_t vd = sizeof(double) * (size_t)(dim + kReplicaPad);
  const int upd_blocks = cdiv(dim, 256);
  if ((e = cudaMalloc(&ctx->w, vd)) != cudaSuccess) return bail("cudaMalloc w", e);
  if ((e = cudaMalloc(&ctx->g, vd)) != cudaSuccess) return bail("cudaMalloc g", e);
  if ((e = cudaMalloc(&ctx->d, vd)) != cudaSuccess) return bail("cudaMalloc d", e);
  if ((e = cudaMalloc(&ctx->w_req, vd)) != cudaSuccess) return bail("cudaMalloc w_req", e);
  if ((e = cudaMalloc(&ctx->w32, sizeof(float) * (size_t)(dim + 4))) != cudaSuccess) return bail("cudaMalloc w32", e);
  if ((e = cudaMalloc(&ctx->w32_req, sizeof(float) * (size_t)(dim + 4))) != cudaSuccess) return bail("cudaMalloc w32_req", e);
  if ((e = cudaMalloc(&ctx->n_exact, sizeof(unsigned long long) * 2)) != cudaSuccess) return bail("cudaMalloc n_exact", e);
  cudaMemsetAsync(ctx->n_exact, 0, sizeof(unsigned long long) * 2, ctx->stream);
  if ((e = cudaMalloc(&ctx->scal, sizeof(double) * kNumScal)) != cudaSuccess) return bail("cudaMalloc scal", e);
  if ((e = cudaMalloc(&ctx->cnt, sizeof(unsigned long long) * kNumCnt)) != cudaSuccess) return bail("cudaMalloc cnt", e);
  if ((e = cudaMalloc(&ctx->partial, sizeof(double) * 2 * (size_t)upd_blocks)) != cudaSuccess) return bail("cudaMalloc partial", e);
  if ((e = cudaMalloc(&ctx->out2, sizeof(double) * 8)) != cudaSuccess) return bail("cudaMalloc out2", e);
  if ((e = cudaMalloc(&ctx->gsum, vd)) != cudaSuccess) return bail("cudaMalloc gsum", e);
  cudaMemsetAsync(ctx->gsum, 0, vd, ctx->stream);
  cudaMemsetAsync(ctx->w, 0, vd, ctx->stream);
  cudaMemsetAsync(ctx->g, 0, vd, ctx->stream);
  cudaMemsetAsync(ctx->d, 0, vd, ctx->stream);
  cudaMemsetAsync(ctx->w_req, 0, vd, ctx->stream);
  cudaMemsetAsync(ctx->w32, 0, sizeof(float) * (size_t)(dim + 2), ctx->stream);
  cudaMemsetAsync(ctx->scal, 0, sizeof(double) * kNumScal, ctx->stream);
  cudaMemsetAsync(ctx->cnt, 0, sizeof(unsigned long long) * kNumCnt, ctx->stream);
  if ((e = cudaStreamSynchronize(ctx->stream)) != cudaSuccess) return bail("init memset", e);
  *out = ctx;
  return DSGD_OK;
}

extern "C" int dsgd_destroy(dsgd_ctx *ctx) {
  if (!ctx) return DSGD_OK;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  if (ctx->comm) nccl().CommDestroy(ctx->comm);
  for (int r = 0; r < kMaxReplicas; ++r)
    if (ctx->peer_w[r] && ctx->peer_ipc[r]) cudaIpcCloseMemHandle(ctx->peer_w[r]);
  for (int r = 0; r < kMaxWorld; ++r)
    if (ctx->peer_x[r] && ctx->peer_x_ipc[r]) cudaIpcCloseMemHandle(ctx->peer_x[r]);
  if (ctx->xblk) cudaFree(ctx->xblk);
  if (ctx->x_llw) cudaFree(ctx->x_llw);
  void *aptrs[] = {ctx->m_w, ctx->outbox, ctx->a_stop, ctx->a_cnt, ctx->a_scratch, ctx->a_rows, ctx->a_assigned, ctx->a_replay, ctx->u_idx, ctx->u_val};
  for (void *q : aptrs) if (q) cudaFree(q);
  if (ctx->a_ev0) { cudaEventDestroy(ctx->a_ev0); cudaEventDestroy(ctx->a_ev1); }
  if (ctx->astream) cudaStreamDestroy(ctx->astream);
  if (ctx->stream2) cudaStreamDestroy(ctx->stream2);
  void *ptrs[] = {ctx->rp16, ctx->pairs, ctx->label, ctx->yabs, ctx->w, ctx->g, ctx->d, ctx->w_req, ctx->w32, ctx->w32_req, ctx->n_exact, ctx->scal,
                  ctx->cnt, ctx->partial, ctx->out2, ctx->gsum, ctx->p_wbuf[0], ctx->p_wbuf[1], ctx->p_gbuf[0],
                  ctx->p_gbuf[1], ctx->p_gbuf[2], ctx->p_rec[0], ctx->p_rec[1], ctx->p_rec[2], ctx->p_acc, ctx->p_hinge, ctx->p_bar, ctx->x_stats, ctx->samples,
                  ctx->losses, ctx->preds, ctx->ms_w, ctx->ms_rec, ctx->ms_acc, ctx->ms_hinge, ctx->ms_losses, ctx->ms_bar};
  for (void *p : ptrs) if (p) cudaFree(p);
  if (ctx->ev0) cudaEventDestroy(ctx->ev0);
  if (ctx->ev1) cudaEventDestroy(ctx->ev1);
  for (auto &pe : ctx->prof_events) { cudaEventDestroy(pe.first); cudaEventDestroy(pe.second); }
  if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
  delete ctx;
  return DSGD_OK;
}

extern "C" const char *dsgd_last_error(const dsgd_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

extern "C" const char *dsgd_info(const dsgd_ctx *ctx) {
  if (!ctx) return "{}";
  char buf[512];
  snprintf(buf, sizeof buf,
           "{\"device\": %d, \"name\": \"%s\", \"sm_count\": %d, \"arch\": \"sm_100a\", \"dim\": %d, \"rank\": %d, "
           "\"world\": %d, \"n_rows\": %lld, \"nnz\": %lld, \"state_dtype\": \"f64\", \"value_dtype\": \"f32\"}",
           ctx->device, ctx->dev_name.c_str(), ctx->sm_count, ctx->dim, ctx->rank, ctx->world, (long long)ctx->n_rows,
           (long long)ctx->nnz);
  ctx->info = buf;
  return ctx->info.c_str();
}

extern "C" int dsgd_set_stream(dsgd_ctx *ctx, void *cuda_stream) {
  if (!ctx) return DSGD_ERR_INVALID;
  CU(cudaSetDevice(ctx->device));
  CU(cudaStreamSynchronize(ctx->stream));
  ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
  return DSGD_OK;
}

extern "C" int dsgd_synchronize(dsgd_ctx *ctx) {
  if (!ctx) return DSGD_ERR_INVALID;
  CU(cudaSetDevice(ctx->device));
  CU(cudaStreamSynchronize(ctx->stream));
  return DSGD_OK;
}

extern "C" int dsgd_timer_start(dsgd_ctx *ctx) {
  if (!ctx) return DSGD_ERR_INVALID;
  CU(cudaSetDevice(ctx->device));
  CU(cudaEventRecord(ctx->ev0, ctx->stream));
  return DSGD_OK;
}

extern "C" int dsgd_timer_stop(dsgd_ctx *ctx, float *elapsed_ms) {
  if (!ctx || !elapsed_ms) return DSGD_ERR_INVALID;
  CU(cudaSetDevice(ctx->device));
  CU(cudaEventRecord(ctx->ev1, ctx->stream));
  CU(cudaEventSynchronize(ctx->ev1));
  CU(cudaEventElapsedTime(elapsed_ms, ctx->ev0, ctx->ev1));
  return DSGD_OK;
}

extern "C" int dsgd_launch_count(const dsgd_ctx *ctx, int64_t *count) {
  if (!ctx || !count) return DSGD_ERR_INVALID;
  *count = ctx->launches;
  return DSGD_OK;
}

extern "C" int dsgd_profile_begin(dsgd_ctx *ctx, int32_t sample_every) {
  if (!ctx) return DSGD_ERR_INVALID;
  NEED(sample_every > 0, DSGD_ERR_INVALID, "dsgd_profile_begin: sample_every must be positive");
  ctx->prof_every = sample_every;
  ctx->prof_seen = 0;
  ctx->prof_used = 0;
  return DSGD_OK;
}

extern "C" int dsgd_profile_end(dsgd_ctx *ctx, float *mean_ms, int64_t *n_sampled) {
  if (!ctx) return DSGD_ERR_INVALID;
  CU(cudaSetDevice(ctx->device));
  CU(cudaStreamSynchronize(ctx->stream));
  double tot = 0.0;
  for (size_t i = 0; i < ctx->prof_used; ++i) {
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, ctx->prof_events[i].first, ctx->prof_events[i].second));
    tot += ms;
  }
  if (mean_ms) *mean_ms = ctx->prof_used ? (float)(tot / (double)ctx->prof_used) : 0.f;
  if (n_sampled) *n_sampled = (int64_t)ctx->prof_used;
  ctx->prof_every = 0;
  ctx->prof_used = 0;
  return DSGD_OK;
}

// ---- data --------------------------------------------------------------------------------------------

extern "C" int dsgd_load_csr(dsgd_ctx *ctx, int64_t n_rows, int64_t nnz, const int64_t *row_ptr, const int32_t *col,
                             const float *val, const int8_t *label) {
  if (!ctx) return DSGD_ERR_INVALID;
  NEED(n_rows > 0 && nnz >= 0 && row_ptr && label && (nnz == 0 || (col && val)), DSGD_ERR_INVALID,
       "dsgd_load_csr: bad arguments (n_rows=%lld nnz=%lld)", (long long)n_rows, (long long)nnz);
  NEED(n_rows < (int64_t)INT32_MAX, DSGD_ERR_INVALID, "dsgd_load_csr: sample ids are int32; n_rows too large");
  NEED(row_ptr[0] == 0 && row_ptr[n_rows] == nnz, DSGD_ERR_INVALID, "dsgd_load_csr: row_ptr[0] != 0 or row_ptr[n] != nnz");
  // validate + build 16-byte window offsets (host side of the data load, like Dataset.rcv1 building the Map per row)
  std::vector<uint32_t> rp16((size_t)n_rows + 1);
  uint64_t acc = 0;
  for (int64_t r = 0; r < n_rows; ++r) {
    const int64_t len = row_ptr[r + 1] - row_ptr[r];
    NEED(len >= 0, DSGD_ERR_INVALID, "dsgd_load_csr: row_ptr not monotone at row %lld", (long long)r);
    NEED(label[r] == 1 || label[r] == -1, DSGD_ERR_INVALID, "dsgd_load_csr: label of row %lld is %d, expected +1/-1",
         (long long)r, (int)label[r]);
    rp16[(size_t)r] = (uint32_t)acc;
    acc += (uint64_t)((len + 1) / 2);
    NEED(acc < (1ull << 32), DSGD_ERR_INVALID, "dsgd_load_csr: too many non-zeros for 32-bit window offsets");
  }
  rp16[(size_t)n_rows] = (uint32_t)acc;
  for (int64_t k = 0; k < nnz; ++k)
    NEED(col[k] >= 0 && col[k] < ctx->dim, DSGD_ERR_RANGE, "dsgd_load_csr: column %d at position %lld outside [0,%d)",
         col[k], (long long)k, ctx->dim);
  bool unique = true;
  for (int64_t r = 0; r < n_rows && unique; ++r)
    for (int64_t k = row_ptr[r] + 1; k < row_ptr[r + 1]; ++k)
      if (col[k] <= col[k - 1]) { unique = false; break; }
  CU(cudaSetDevice(ctx->device));
  for (void *p : {(void *)ctx->rp16, (void *)ctx->pairs, (void *)ctx->label, (void *)ctx->yabs}) if (p) CU(cudaFree(p));
  ctx->rp16 = nullptr; ctx->pairs = nullptr; ctx->label = nullptr; ctx->yabs = nullptr;
  const int64_t n_pairs = (int64_t)acc * 2;
  CU(cudaMalloc(&ctx->rp16, sizeof(uint32_t) * ((size_t)n_rows + 1)));
  CU(cudaMalloc(&ctx->pairs, sizeof(uint2) * (size_t)std::max<int64_t>(n_pairs, 1)));
  CU(cudaMalloc(&ctx->label, (size_t)n_rows));
  CU(cudaMalloc(&ctx->yabs, sizeof(float) * (size_t)n_rows));
  int64_t *d_rp = nullptr; int32_t *d_col = nullptr; float *d_val = nullptr;
  CU(cudaMalloc(&d_rp, sizeof(int64_t) * ((size_t)n_rows + 1)));
  CU(cudaMalloc(&d_col, sizeof(int32_t) * (size_t)std::max<int64_t>(nnz, 1)));
  CU(cudaMalloc(&d_val, sizeof(float) * (size_t)std::max<int64_t>(nnz, 1)));
  CU(cudaMemcpyAsync(d_rp, row_ptr, sizeof(int64_t) * ((size_t)n_rows + 1), cudaMemcpyHostToDevice, ctx->stream));
  if (nnz) {
    CU(cudaMemcpyAsync(d_col, col, sizeof(int32_t) * (size_t)nnz, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(d_val, val, sizeof(float) * (size_t)nnz, cudaMemcpyHostToDevice, ctx->stream));
  }
  CU(cudaMemcpyAsync(ctx->rp16, rp16.data(), sizeof(uint32_t) * ((size_t)n_rows + 1), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(ctx->label, label, (size_t)n_rows, cudaMemcpyHostToDevice, ctx->stream));
  const int blocks = std::min<int64_t>(cdiv(n_rows, 8), (int64_t)ctx->sm_count * 16);
  k_repack<<<blocks, 256, 0, ctx->stream>>>(d_rp, d_col, d_val, ctx->rp16, ctx->label, n_rows, ctx->pairs, ctx->yabs);
  LAUNCHED();
  CU(cudaGetLastError());
  CU(cudaStreamSynchronize(ctx->stream));
  CU(cudaFree(d_rp)); CU(cudaFree(d_col)); CU(cudaFree(d_val));
  ctx->n_rows = n_rows; ctx->nnz = nnz; ctx->n_pairs = n_pairs; ctx->rows_unique = unique;
  return DSGD_OK;
}

// recompute c and ||w||^2 of the resident weights, refresh the fp32 shadow
static int refresh_resident(dsgd_ctx *ctx) {
  k_prepare<1024><<<1, 1024, 0, ctx->stream>>>(ctx->w, ctx->d, ctx->dim, ctx->lambda, ctx->scal + kScalC,
                                                ctx->scal + kScalNrm2);
  LAUNCHED();
  k_to_f32<<<cdiv(ctx->dim, 256), 256, 0, ctx->stream>>>(ctx->w, ctx->w32, ctx->dim);
  LAUNCHED();
  if (ctx->flags & DSGD_FLAG_ASYNC) {
    k_async_init_ctl<1024><<<1, 1024, 0, ctx->stream>>>(ctx->w, ctx->d, ctx->dim);
    LAUNCHED();
  }
  CU(cudaGetLastError());
  return DSGD_OK;
}

extern "C" int dsgd_set_dim_sparsity(dsgd_ctx *ctx, const double *d) {
  if (!ctx) return DSGD_ERR_INVALID;
  NEED(d, DSGD_ERR_INVALID, "dsgd_set_dim_sparsity: d is NULL");
  CU(cudaSetDevice(ctx->device));
  CU(cudaMemcpyAsync(ctx->d, d, sizeof(double) * (size_t)ctx->dim, cudaMemcpyHostToDevice, ctx->stream));
  ctx->have_d = true;
  int rc = refresh_resident(ctx);
  if (rc) return rc;
  CU(cudaStreamSynchronize(ctx->stream));
  return DSGD_OK;
}

extern "C" int dsgd_compute_dim_sparsity(dsgd_ctx *ctx, int64_t n_train, double *d_out) {
  if (!ctx) return DSGD_ERR_INVALID;
  NEED(ctx->pairs, DSGD_ERR_STATE, "dsgd_compute_dim_sparsity: no rows loaded");
  NEED(n_train >= 0 && n_train <= ctx->n_rows, DSGD_ERR_RANGE, "dsgd_compute_dim_sparsity: n_train %lld outside [0,%lld]",
       (long long)n_train, (long long)ctx->n_rows);
  CU(cudaSetDevice(ctx->device));
  unsigned *df = nullptr;
  CU(cudaMalloc(&df, sizeof(unsigned) * (size_t)ctx->dim));
  CU(cudaMemsetAsync(df, 0, sizeof(unsigned) * (size_t)ctx->dim, ctx->stream));
  uint32_t end16 = 0;
  CU(cudaMemcpyAsync(&end16, ctx->rp16 + n_train, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  const int64_t n_pairs = (int64_t)end16 * 2;
  if (n_pairs > 0) {
    const int blocks = std::min<int64_t>(cdiv(n_pairs, 256), (int64_t)ctx->sm_count * 16);
    k_col_hist<<<blocks, 256, 0, ctx->stream>>>(ctx->pairs, n_pairs, df);
    LAUNCHED();
  }
  k_dim_sparsity<<<cdiv(ctx->dim, 256), 256, 0, ctx->stream>>>(df, ctx->dim, ctx->d);
  LAUNCHED();
  CU(cudaGetLastError());
  ctx->have_d = true;
  int rc = refresh_resident(ctx);
  if (rc) return rc;
  if (d_out) CU(cudaMemcpyAsync(d_out, ctx->d, sizeof(double) * (size_t)ctx->dim, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  CU(cudaFree(df));
  return DSGD_OK;
}

extern "C" int dsgd_set_weights(dsgd_ctx *ctx, const double *w) {
  if (!ctx) return DSGD_ERR_INVALID;
  NEED(w, DSGD_ERR_INVALID, "dsgd_set_weights: w is NULL");
  CU(cudaSetDevice(ctx->device));
  CU(cudaMemcpyAsync(ctx->w, w, sizeof(double) * (size_t)ctx->dim, cudaMemcpyHostToDevice, ctx->stream));
  int rc = refresh_resident(ctx);
  if (rc) return rc;
  CU(cudaStreamSynchronize(ctx->stream));
  return DSGD_OK;
}

extern "C" int dsgd_get_weights(dsgd_ctx *ctx, double *w) {
  if (!ctx) return DSGD_ERR_INVALID;
  NEED(w, DSGD_ERR_INVALID, "dsgd_get_weights: w is NULL");
  CU(cudaSetDevice(ctx->device));
  CU(cudaMemcpyAsync(w, ctx->w, sizeof(double) * (size_t)ctx->dim, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return DSGD_OK;
}

// ---- sample staging ----------------------------------------------------------------------------------

static int ensure_i32(dsgd_ctx *ctx, int32_t **buf, int64_t *cap, int64_t n) {
  if (*cap >= n) return DSGD_OK;
  if (*buf) CU(cudaFree(*buf));
  *buf = nullptr; *cap = 0;
  const int64_t want = std::max<int64_t>(n, 1024);
  CU(cudaMalloc(buf, sizeof(int32_t) * (size_t)want));
  *cap = want;
  return DSGD_OK;
}
static int ensure_f64(dsgd_ctx *ctx, double **buf, int64_t *cap, int64_t n) {
  if (*cap >= n) return DSGD_OK;
  if (*buf) CU(cudaFree(*buf));
  *buf = nullptr; *cap = 0;
  const int64_t want = std::max<int64_t>(n, 1024);
  CU(cudaMalloc(buf, sizeof(double) * (size_t)want));
  *cap = want;
  return DSGD_OK;
}

extern "C" int dsgd_stage_samples(dsgd_ctx *ctx, const int32_t *samples, int64_t n) {
  if (!ctx) return DSGD_ERR_INVALID;
  NEED(ctx->pairs, DSGD_ERR_STATE, "dsgd_stage_samples: no rows loaded");
  NEED(n >= 0 && (n == 0 || samples), DSGD_ERR_INVALID, "dsgd_stage_samples: bad arguments");
  for (int64_t i = 0; i < n; ++i)
    NEED(samples[i] >= 0 && samples[i] < ctx->n_rows, DSGD_ERR_RANGE, "sample index %d at position %lld outside [0,%lld)",
         samples[i], (long long)i, (long long)ctx->n_rows);
  CU(cudaSetDevice(ctx->device));
  int rc = ensure_i32(ctx, &ctx->samples, &ctx->samples_cap, n);
  if (rc) return rc;
  if (n) CU(cudaMemcpyAsync(ctx->samples, samples, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
  ctx->samples_n = n;
  return DSGD_OK;
}

// weights to use for a request: NULL -> resident; else copy into w_req and compute its scalars
// (w_on_device: w is a device pointer, e.g. a model of the set)
static int request_weights(dsgd_ctx *ctx, const double *w, const double **w_dev, const double **c_dev,
                           const double **nrm_dev, const float **w32_dev = nullptr, bool w_on_device = false) {
  CU(cudaSetDevice(ctx->device));  // every request path passes here: a caller thread may have another device current
  if (!w) {
    *w_dev = ctx->w; *c_dev = ctx->scal + kScalC; *nrm_dev = ctx->scal + kScalNrm2;
    if (w32_dev) *w32_dev = ctx->w32;
    return DSGD_OK;
  }
  if (w32_dev) *w32_dev = ctx->w32_req;
  CU(cudaMemcpyAsync(ctx->w_req, w, sizeof(double) * (size_t)ctx->dim,
                     w_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, ctx->stream));
  k_prepare<1024><<<1, 1024, 0, ctx->stream>>>(ctx->w_req, ctx->d, ctx->dim, ctx->lambda, ctx->scal + kScalReqC,
                                                ctx->scal + kScalReqNrm2);
  LAUNCHED();
  k_to_f32<<<cdiv(ctx->dim, 256), 256, 0, ctx->stream>>>(ctx->w_req, ctx->w32_req, ctx->dim);
  LAUNCHED();
  CU(cudaGetLastError());
  *w_dev = ctx->w_req; *c_dev = ctx->scal + kScalReqC; *nrm_dev = ctx->scal + kScalReqNrm2;
  return DSGD_OK;
}

static inline int rows_grid(const dsgd_ctx *ctx, int64_t n) {
  return (int)std::min<int64_t>(std::max<int64_t>(cdiv(n, 8), 1), (int64_t)ctx->sm_count * 8);
}

// ---- streaming pass (large n): fp32 weights staged in shared memory, one persistent CTA per SM (dsgd_stream.cuh) ----
constexpr int64_t kStreamMinRows = 2048;

static bool stream_eligible(const dsgd_ctx *ctx, int64_t n) {
  return n >= kStreamMinRows && stream_smem_bytes(ctx->dim) + 1024 <= 227u * 1024u;
}

template <bool kScatter, bool kPreds, bool kContig>
static int stream_launch(dsgd_ctx *ctx, const int32_t *samples_dev, int64_t row_begin, int64_t n, const double *w_dev,
                         const float *w32_dev, double *g, double *preds) {
  const size_t smem = stream_smem_bytes(ctx->dim);
  if (!ctx->stream_ready) {
    CU(cudaFuncSetAttribute(k_stream_rows<false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CU(cudaFuncSetAttribute(k_stream_rows<false, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CU(cudaFuncSetAttribute(k_stream_rows<true, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ctx->stream_ready = true;
  }
  NEED(kContig == (samples_dev == nullptr), DSGD_ERR_INVALID, "stream_launch: sample list / row range mismatch");
  StreamParams sp;
  memset(&sp, 0, sizeof sp);
  sp.rp16 = ctx->rp16; sp.units = reinterpret_cast<const uint4 *>(ctx->pairs); sp.yabs = ctx->yabs;
  sp.samples = samples_dev; sp.row_begin = row_begin; sp.n = n;
  sp.w = w_dev; sp.w32 = w32_dev; sp.dim = ctx->dim;
  sp.g = g; sp.preds = preds; sp.cnt = ctx->cnt; sp.n_exact = ctx->n_exact; sp.next_block = ctx->n_exact + 1;
  CU(cudaMemsetAsync(ctx->n_exact + 1, 0, sizeof(unsigned long long), ctx->stream));
  // rows per block (the unit of the dynamic work distribution): 32, or fewer when that leaves a warp fewer than ~6 blocks
  const int64_t n_warps_all = (int64_t)ctx->sm_count * (kStreamThreads / 32);
  sp.rows_log2 = 5;
  while (sp.rows_log2 > 3 && ((n + (1 << sp.rows_log2) - 1) >> sp.rows_log2) < 6 * n_warps_all) --sp.rows_log2;
  // the last fifth of the pass goes out in blocks of half the size (not below 8 rows): warps end closer together.
  // (Measured r2q: 2 to 6 blocks per warp and a tail of 0 to 35 % all land within 1 % of each other, profiles/r2_streaming.md.)
  sp.tail_log2 = std::max(3, sp.rows_log2 - 1);
  sp.n_big = sp.tail_log2 < sp.rows_log2 ? ((n - n / 5) >> sp.rows_log2) : ((n + (1 << sp.rows_log2) - 1) >> sp.rows_log2);
  const int64_t n_blk = sp.n_big + cdiv(std::max<int64_t>(0, n - (sp.n_big << sp.rows_log2)), (int64_t)1 << sp.tail_log2);
  const int grid = (int)std::min<int64_t>(ctx->sm_count, std::max<int64_t>(1, cdiv(n_blk, kStreamThreads / 32)));
  auto *pe = prof_slot(ctx);
  if (pe) cudaEventRecord(pe->first, ctx->stream);
  k_stream_rows<kScatter, kPreds, kContig><<<grid, kStreamThreads, smem, ctx->stream>>>(sp);
  if (pe) cudaEventRecord(pe->second, ctx->stream);
  LAUNCHED();
  CU(cudaGetLastError());
  return DSGD_OK;
}

// ---- forward / gradient / eval -------------------------------------------------------------------------

extern "C" int dsgd_forward(dsgd_ctx *ctx, const double *w, const int32_t *samples, int64_t n, double *preds_out) {
  if (!ctx) return DSGD_ERR_INVALID;
  NEED(n >= 0 && (n == 0 || (samples && preds_out)), DSGD_ERR_INVALID, "dsgd_forward: bad arguments");
  if (n == 0) return DSGD_OK;
  int rc = dsgd_stage_samples(ctx, samples, n);
  if (rc) return rc;
  rc = ensure_f64(ctx, &ctx->preds, &ctx->preds_cap, n);
  if (rc) return rc;
  const double *wd, *cd, *nd;
  const float *w32d;
  if ((rc = request_weights(ctx, w, &wd, &cd, &nd, &w32d))) return rc;
  if (stream_eligible(ctx, n)) {
    if ((rc = stream_launch<false, true, false>(ctx, ctx->samples, 0, n, wd, w32d, nullptr, ctx->preds))) return rc;
  } else {
    k_rows<false, true><<<rows_grid(ctx, n), 256, 0, ctx->stream>>>(ctx->rp16, ctx->pairs, ctx->label, ctx->samples, 0, n,
                                                                    wd, nullptr, ctx->preds, ctx->cnt);
    LAUNCHED();
  }
  CU(cudaGetLastError());
  CU(cudaMemsetAsync(ctx->cnt, 0, sizeof(unsigned long long) * 2, ctx->stream));
  CU(cudaMemcpyAsync(preds_out, ctx->preds, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return DSGD_OK;
}

extern "C" int dsgd_gradient(dsgd_ctx *ctx, const double *w, const int32_t *samples, int64_t n, double *grad_out,
                             double *loss_out) {
  if (!ctx) return DSGD_ERR_INVALID;
  NEED(n >= 0 && grad_out, DSGD_ERR_INVALID, "dsgd_gradient: bad arguments");
  NEED(n > 0, DSGD_ERR_EMPTY, "dsgd_gradient: empty batch (Vec.sum of an empty list throws in the reference)");
  NEED(samples, DSGD_ERR_INVALID, "dsgd_gradient: samples is NULL");
  NEED(ctx->have_d, DSGD_ERR_STATE, "dsgd_gradient: dimSparsity not set");
  int rc = dsgd_stage_samples(ctx, samples, n);
  if (rc) return rc;
  const double *wd, *cd, *nd;
  const float *w32d;
  if ((rc = request_weights(ctx, w, &wd, &cd, &nd, &w32d))) return rc;
  if (stream_eligible(ctx, n)) {
    if ((rc = stream_launch<true, false, false>(ctx, ctx->samples, 0, n, wd, w32d, ctx->g, nullptr))) return rc;
  } else {
    k_rows<true, false><<<rows_grid(ctx, n), 256, 0, ctx->stream>>>(ctx->rp16, ctx->pairs, ctx->label, ctx->samples, 0, n,
                                                                    wd, ctx->g, nullptr, ctx->cnt);
    LAUNCHED();
  }
  k_finish<<<cdiv(ctx->dim + 1, 256), 256, 0, ctx->stream>>>(ctx->g, ctx->dim, cd, ctx->cnt, (double)n);
  LAUNCHED();
  k_loss_scalar<<<1, 1, 0, ctx->stream>>>(nd, ctx->cnt, ctx->lambda, (double)n, ctx->out2);
  LAUNCHED();
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(grad_out, ctx->g, sizeof(double) * (size_t)ctx->dim, cudaMemcpyDeviceToHost, ctx->stream));
  double out2[2];
  CU(cudaMemcpyAsync(out2, ctx->out2, sizeof out2, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaMemsetAsync(ctx->g, 0, sizeof(double) * (size_t)(ctx->dim + 2), ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  if (loss_out) *loss_out = out2[0];
  return DSGD_OK;
}

static int eval_impl(dsgd_ctx *ctx, const double *w, int64_t row_begin, int64_t row_end, double out[5],
                     bool w_on_device = false) {
  NEED(ctx->pairs, DSGD_ERR_STATE, "dsgd_eval: no rows loaded");
  NEED(row_begin >= 0 && row_end <= ctx->n_rows && row_begin <= row_end, DSGD_ERR_RANGE,
       "dsgd_eval: rows [%lld,%lld) outside [0,%lld)", (long long)row_begin, (long long)row_end, (long long)ctx->n_rows);
  NEED(row_end > row_begin, DSGD_ERR_EMPTY, "dsgd_eval: empty range (reduce on an empty collection throws in the reference)");
  CU(cudaSetDevice(ctx->device));
  const int64_t n = row_end - row_begin;
  const double *wd, *cd, *nd;
  const float *w32d;
  int rc;
  if ((rc = request_weights(ctx, w, &wd, &cd, &nd, &w32d, w_on_device))) return rc;
  if (stream_eligible(ctx, n)) {
    if ((rc = stream_launch<false, false, true>(ctx, nullptr, row_begin, n, wd, w32d, nullptr, nullptr))) return rc;
  } else {
    k_rows<false, false><<<rows_grid(ctx, n), 256, 0, ctx->stream>>>(ctx->rp16, ctx->pairs, ctx->label, nullptr, row_begin, n,
                                                                     wd, nullptr, nullptr, ctx->cnt);
    LAUNCHED();
  }
  k_loss_scalar<<<1, 1, 0, ctx->stream>>>(nd, ctx->cnt, ctx->lambda, (double)n, ctx->out2);
  LAUNCHED();
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(out, ctx->out2, sizeof(double) * 5, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return DSGD_OK;
}

extern "C" int dsgd_eval(dsgd_ctx *ctx, const double *w, int64_t row_begin, int64_t row_end, double *loss_out,
                         double *acc_out) {
  if (!ctx) return DSGD_ERR_INVALID;
  double out[5];
  int rc = eval_impl(ctx, w, row_begin, row_end, out);
  if (rc) return rc;
  if (loss_out) *loss_out = out[0];
  if (acc_out) *acc_out = out[1];
  return DSGD_OK;
}

extern "C" int dsgd_eval_counts(dsgd_ctx *ctx, const double *w, int64_t row_begin, int64_t row_end, int64_t *hinge_sum,
                                int64_t *correct, double *norm_squared) {
  if (!ctx) return DSGD_ERR_INVALID;
  double out[5];
  int rc = eval_impl(ctx, w, row_begin, row_end, out);
  if (rc) return rc;
  if (hinge_sum) *hinge_sum = (int64_t)out[2];
  if (correct) *correct = (int64_t)out[3];
  if (norm_squared) *norm_squared = out[4];
  return DSGD_OK;
}

// ---- sync mode -------------------------------------------------------------------------------------------

extern "C" int dsgd_comm_unique_id(uint8_t id[DSGD_UNIQUE_ID_BYTES]) {
  static_assert(sizeof(ncclUniqueId) == DSGD_UNIQUE_ID_BYTES, "ncclUniqueId size");
  if (!id) return DSGD_ERR_INVALID;
  if (!nccl().ok) return fail(nullptr, DSGD_ERR_NCCL, "%s", nccl().why.c_str());
  ncclUniqueId u;
  ncclResult_t r = nccl().GetUniqueId(&u);
  if (r != ncclSuccess) return fail(nullptr, DSGD_ERR_NCCL, "ncclGetUniqueId: %s", nccl().GetErrorString(r));
  memcpy(id, &u, sizeof u);
  return DSGD_OK;
}

extern "C" int dsgd_comm_init(dsgd_ctx *ctx, const uint8_t id[DSGD_UNIQUE_ID_BYTES]) {
  if (!ctx) return DSGD_ERR_INVALID;
  NEED(id, DSGD_ERR_INVALID, "dsgd_comm_init: id is NULL");
  NEED(!ctx->comm, DSGD_ERR_STATE, "dsgd_comm_init: communicator already initialised");
  CU(cudaSetDevice(ctx->device));
  ncclUniqueId u;
  memcpy(&u, id, sizeof u);
  NEED(nccl().ok, DSGD_ERR_NCCL, "%s", nccl().why.c_str());
  NC(nccl().CommInitRank(&ctx->comm, ctx->world, u, ctx->rank));
  return DSGD_OK;
}

// ---- persistent sync loop (dsgd_persistent.cuh) ----------------------------------------------------------------
constexpr int kPCons = 8, kPUpd = 6, kPStages = 8, kPStagePairs = 2560, kPMaxChunks = 128;
using PSmem = PersistSmem<kPCons, kPUpd, kPStages, kPStagePairs, kPMaxChunks>;
#define DSGD_PERSIST_KERNEL(multi) k_sync_persistent<kPCons, kPUpd, kPStages, kPStagePairs, kPMaxChunks, multi>
static bool persist_timeline() { static const bool v = getenv("DSGD_PERSIST_TIMELINE") != nullptr; return v; }

static int persist_prepare(dsgd_ctx *ctx, int64_t n_steps) {
  if (!ctx->p_ready) {
    const size_t vd = sizeof(double) * (size_t)(ctx->dim + 2);
    for (int i = 0; i < 2; ++i) CU(cudaMalloc(&ctx->p_wbuf[i], vd));
    for (int i = 0; i < 3; ++i) {
      CU(cudaMalloc(&ctx->p_gbuf[i], vd));
      CU(cudaMemsetAsync(ctx->p_gbuf[i], 0, vd, ctx->stream));
      CU(cudaMalloc(&ctx->p_rec[i], 2 * vd));
      CU(cudaMemsetAsync(ctx->p_rec[i], 0, 2 * vd, ctx->stream));
    }
    CU(cudaMalloc(&ctx->p_acc, sizeof(unsigned long long) * 3 * kAccStride));
    CU(cudaMalloc(&ctx->p_bar, sizeof(unsigned) * 4));
    CU(cudaFuncSetAttribute((const void *)DSGD_PERSIST_KERNEL(false), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(PSmem)));
    CU(cudaFuncSetAttribute((const void *)DSGD_PERSIST_KERNEL(true), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(PSmem)));
    ctx->p_ready = true;
  }
  if (ctx->p_hinge_cap < n_steps) {
    if (ctx->p_hinge) CU(cudaFree(ctx->p_hinge));
    ctx->p_hinge = nullptr;
    const int64_t want = std::max<int64_t>(n_steps, 4096);
    CU(cudaMalloc(&ctx->p_hinge, sizeof(unsigned) * (size_t)want));
    ctx->p_hinge_cap = want;
  }
  return DSGD_OK;
}

// CTAs of the persistent kernel: one per SM (measured in round 1 with tools/sweep_persist.py: fastest at batch 64, 256
// and 1024); every CTA owns at most kMaxRowsPerCta rows of a step.  0: the batch is too large for this kernel.
static int persist_grid(const dsgd_ctx *ctx, int64_t batch) {
  const int g = ctx->grid_limit > 0 ? std::min(ctx->grid_limit, ctx->sm_count) : ctx->sm_count;
  if (cdiv(batch, kMaxRowsPerCta) > g) return 0;
  if (ctx->n_pairs >= (1ll << 31)) return 0;  // chunk descriptors carry a 31-bit global pair index
  return g;
}
// K GPUs: one column of the CTA's slice per barrier-synchronised thread
static bool persist_multi_fits(const dsgd_ctx *ctx, int G) {
  const int slice = (cdiv(ctx->dim + 1, G) + 31) & ~31;
  return slice <= (kPCons + kPUpd) * 32;
}

// The kernel synchronises its CTAs itself, so all of them must be resident: a cooperative launch guarantees that.  With a
// grid limit (several contexts sharing one GPU: the K-rank tests on one device) the kernels of the ranks must also run
// CONCURRENTLY, which cooperative launches of different contexts do not (measured: they serialise and the ranks time
// out waiting for each other); a plain launch of at most one CTA per SM on an otherwise idle GPU is resident in full too.
static cudaError_t persist_launch(dsgd_ctx *ctx, void *fn, int G, void **args) {
  if (ctx->grid_limit > 0) return cudaLaunchKernel(fn, dim3(G), dim3((kPCons + kPUpd + 1) * 32), args, sizeof(PSmem), ctx->stream);
  return cudaLaunchCooperativeKernel(fn, dim3(G), dim3((kPCons + kPUpd + 1) * 32), args, sizeof(PSmem), ctx->stream);
}

// fields shared by the one-GPU and the K-GPU launch
static int persist_params(dsgd_ctx *ctx, PersistParams &pp, const int32_t *samples_dev, int64_t n_per_step, int64_t n_steps,
                          double lr, double *losses_dev, int G) {
  (void)G;
  memset(&pp, 0, sizeof pp);
  pp.rp16 = ctx->rp16; pp.pairs = ctx->pairs; pp.label = ctx->label; pp.samples = samples_dev;
  pp.n_steps = n_steps; pp.batch = (int32_t)n_per_step; pp.dim = ctx->dim;
  pp.wbuf[0] = ctx->p_wbuf[0]; pp.wbuf[1] = ctx->p_wbuf[1];
  for (int i = 0; i < 3; ++i) { pp.gbuf[i] = ctx->p_gbuf[i]; pp.rec[i] = ctx->p_rec[i]; }
  pp.d = ctx->d; pp.acc = ctx->p_acc; pp.bar = ctx->p_bar; pp.hinge = ctx->p_hinge; pp.losses = losses_dev;
  pp.w_out = ctx->w; pp.w32_out = ctx->w32; pp.scal = ctx->scal;
  pp.abort_flag = reinterpret_cast<int *>(ctx->p_bar + 1);
  CU(cudaMemsetAsync(ctx->p_acc, 0, sizeof(unsigned long long) * 3 * kAccStride, ctx->stream));
  pp.lambda = ctx->lambda; pp.lr = lr; pp.world = 1;
  CU(cudaMemsetAsync(ctx->p_hinge, 0, sizeof(unsigned) * (size_t)n_steps, ctx->stream));
  CU(cudaMemsetAsync(ctx->p_bar, 0, sizeof(unsigned) * 4, ctx->stream));
  if (persist_timeline()) {
    if (!ctx->p_tl) CU(cudaMalloc(&ctx->p_tl, sizeof(long long) * kTlWords));
    CU(cudaMemsetAsync(ctx->p_tl, 0, sizeof(long long) * kTlWords, ctx->stream));
    pp.tl = ctx->p_tl;
  }
  return DSGD_OK;
}

static int persist_run(dsgd_ctx *ctx, const int32_t *samples_dev, int64_t n_per_step, int64_t n_steps, double lr,
                       double *losses_dev) {
  int rc = persist_prepare(ctx, n_steps);
  if (rc) return rc;
  const int G = persist_grid(ctx, n_per_step);
  NEED((uint64_t)G * (uint64_t)(n_steps + 2) < (1ull << 32), DSGD_ERR_INVALID, "dsgd_sync_steps: too many steps for one launch");
  PersistParams pp;
  if ((rc = persist_params(ctx, pp, samples_dev, n_per_step, n_steps, lr, losses_dev, G))) return rc;
  k_rec_init<<<cdiv(ctx->dim, 256), 256, 0, ctx->stream>>>(ctx->w, ctx->dim, ctx->p_rec[0], ctx->p_rec[1], ctx->p_rec[2]);
  LAUNCHED();
  pp.k_den = 1.0;
  pp.timeout_cycles = 4000000000ll;  // ~2 s at 1.9 GHz: a healthy barrier takes well under a microsecond
  void *args[] = {&pp};
  auto *pe = prof_slot(ctx);
  if (pe) cudaEventRecord(pe->first, ctx->stream);
  CU(persist_launch(ctx, (void *)DSGD_PERSIST_KERNEL(false), G, args));
  if (pe) cudaEventRecord(pe->second, ctx->stream);
  LAUNCHED();
  return DSGD_OK;
}

// ---- fused K-GPU loop: all ranks run the persistent kernel and exchange gradients through peer memory ----
// exported block of a rank (in 8-byte words): value words [sender][parity][dim + 8] x 2, then bitmap words
// [sender][parity][ceil((dim + 1) / 32)]
static size_t xblk_stride(const dsgd_ctx *ctx) { return (size_t)(ctx->dim + kReplicaPad); }
static size_t xblk_words(const dsgd_ctx *ctx) { return ((size_t)ctx->dim + 1 + 31) / 32; }
static size_t xblk_bm_offset(const dsgd_ctx *ctx) { return 2 * (size_t)kMaxWorld * 2 * xblk_stride(ctx); }
static size_t xblk_doubles(const dsgd_ctx *ctx) { return xblk_bm_offset(ctx) + (size_t)kMaxWorld * 2 * xblk_words(ctx); }

static int xblk_ensure(dsgd_ctx *ctx) {
  if (ctx->xblk) return DSGD_OK;
  CU(cudaSetDevice(ctx->device));
  CU(cudaMalloc(&ctx->xblk, sizeof(double) * xblk_doubles(ctx)));
  CU(cudaMemset(ctx->xblk, 0, sizeof(double) * xblk_doubles(ctx)));
  CU(cudaMalloc(&ctx->x_stats, sizeof(unsigned long long) * 4));
  CU(cudaMemset(ctx->x_stats, 0, sizeof(unsigned long long) * 4));
  return DSGD_OK;
}

static int xllw_ensure(dsgd_ctx *ctx) {
  if (ctx->x_llw) return DSGD_OK;
  CU(cudaMalloc(&ctx->x_llw, 2 * 2 * sizeof(unsigned long long) * xblk_stride(ctx)));
  CU(cudaMemsetAsync(ctx->x_llw, 0, 2 * 2 * sizeof(unsigned long long) * xblk_stride(ctx), ctx->stream));
  return DSGD_OK;
}

static bool xchg_complete(const dsgd_ctx *ctx) {
  if (ctx->world <= 1 || ctx->world > kMaxWorld || !ctx->xblk) return false;
  for (int r = 0; r < ctx->world; ++r)
    if (r != ctx->rank && !ctx->peer_x[r]) return false;
  return true;
}

static int persist_run_multi(dsgd_ctx *ctx, const int32_t *samples_dev, int64_t n_per_step, int64_t n_steps, double lr,
                             double *losses_dev) {
  int rc = persist_prepare(ctx, n_steps);
  if (rc) return rc;
  const int G = persist_grid(ctx, n_per_step);
  NEED((uint64_t)G * (uint64_t)(n_steps + 2) < (1ull << 32), DSGD_ERR_INVALID, "dsgd_sync_steps: too many steps for one launch");
  PersistParams pp;
  if ((rc = persist_params(ctx, pp, samples_dev, n_per_step, n_steps, lr, losses_dev, G))) return rc;
  // the kernel's first interval reads the host-provided weights from wbuf[0] and publishes them in LL form
  CU(cudaMemcpyAsync(ctx->p_wbuf[0], ctx->w, sizeof(double) * (size_t)ctx->dim, cudaMemcpyDeviceToDevice, ctx->stream));
  pp.k_den = (double)ctx->world;
  pp.timeout_cycles = 20000000000ll;  // ~10 s: covers a peer that launches late
  pp.world = ctx->world; pp.rank = ctx->rank; pp.step_base = ctx->x_step;
  pp.xstride = (int)xblk_stride(ctx);
  pp.xwords = (int)xblk_words(ctx);
  for (int r = 0; r < ctx->world; ++r) {
    unsigned long long *blk = reinterpret_cast<unsigned long long *>((r == ctx->rank) ? ctx->xblk : ctx->peer_x[r]);
    pp.xval[r] = blk;
    pp.xbm[r] = blk + xblk_bm_offset(ctx);
  }
  if ((rc = xllw_ensure(ctx))) return rc;
  pp.llw[0] = ctx->x_llw;
  pp.llw[1] = ctx->x_llw + 2 * xblk_stride(ctx);
  pp.xstats = ctx->x_stats;
  void *args[] = {&pp};
  auto *pe = prof_slot(ctx);
  if (pe) cudaEventRecord(pe->first, ctx->stream);
  CU(persist_launch(ctx, (void *)DSGD_PERSIST_KERNEL(true), G, args));
  if (pe) cudaEventRecord(pe->second, ctx->stream);
  LAUNCHED();
  // The next launch must not meet LL words carrying tags this one used (the host may install new weights in between): the
  // step counter jumps.  By 6: a multiple of 3 keeps the rotation of the three gradient buffers (the dirty one is re-zeroed
  // before use), and an EVEN jump makes the first push of launch n+1 (its second interval) land in the receive parity that
  // a slow peer is NOT reading in launch n's last interval (+3 put them on the same one: ADVICE.md round 1).
  ctx->x_step += n_steps + 6;
  ctx->x_steps_run += n_steps;
  return DSGD_OK;
}

extern "C" int dsgd_reserve(dsgd_ctx *ctx, int64_t n_samples, int64_t n_steps) {
  if (!ctx) return DSGD_ERR_INVALID;
  NEED(n_samples >= 0 && n_steps >= 0, DSGD_ERR_INVALID, "dsgd_reserve: negative size");
  CU(cudaSetDevice(ctx->device));
  int rc = ensure_i32(ctx, &ctx->samples, &ctx->samples_cap, n_samples);
  if (rc) return rc;
  if ((rc = ensure_f64(ctx, &ctx->losses, &ctx->losses_cap, n_steps))) return rc;
  if ((rc = persist_prepare(ctx, n_steps))) return rc;
  if (persist_timeline() && !ctx->p_tl) CU(cudaMalloc(&ctx->p_tl, sizeof(long long) * kTlWords));
  if (ctx->world > 1 && !(ctx->flags & DSGD_FLAG_ASYNC)) {
    if ((rc = xblk_ensure(ctx))) return rc;
    if ((rc = xllw_ensure(ctx))) return rc;
  }
  CU(cudaStreamSynchronize(ctx->stream));
  return DSGD_OK;
}

extern "C" int dsgd_set_grid_limit(dsgd_ctx *ctx, int32_t n_ctas) {
  if (!ctx) return DSGD_ERR_INVALID;
  NEED(n_ctas >= 0, DSGD_ERR_INVALID, "dsgd_set_grid_limit: negative");
  ctx->grid_limit = n_ctas;
  return DSGD_OK;
}

// Diagnostic for the bandwidth figures of the fused K-GPU step: words this rank has pushed to EACH peer so far (a value word
// is 16 bytes on the wire, a bitmap word 8) and the SGD steps of those launches.
extern "C" int dsgd_xchg_stats(dsgd_ctx *ctx, int64_t *value_words, int64_t *bitmap_words, int64_t *steps) {
  if (!ctx) return DSGD_ERR_INVALID;
  unsigned long long host[2] = {0, 0};
  if (ctx->x_stats) {
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(ctx->stream));
    CU(cudaMemcpy(host, ctx->x_stats, sizeof host, cudaMemcpyDeviceToHost));
  }
  if (value_words) *value_words = (int64_t)host[0];
  if (bitmap_words) *bitmap_words = (int64_t)host[1];
  if (steps) *steps = ctx->x_steps_run;
  return DSGD_OK;
}

extern "C" int dsgd_xchg_export(dsgd_ctx *ctx, uint8_t handle[DSGD_IPC_HANDLE_BYTES]) {
  if (!ctx || !handle) return DSGD_ERR_INVALID;
  NEED(!(ctx->flags & DSGD_FLAG_ASYNC), DSGD_ERR_STATE, "dsgd_xchg_export: ctx is in async mode");
  int rc = xblk_ensure(ctx);
  if (rc) return rc;
  cudaIpcMemHandle_t h;
  CU(cudaIpcGetMemHandle(&h, ctx->xblk));
  memcpy(handle, &h, sizeof h);
  return DSGD_OK;
}

extern "C" int dsgd_xchg_import(dsgd_ctx *ctx, int peer_rank, const uint8_t handle[DSGD_IPC_HANDLE_BYTES]) {
  if (!ctx || !handle) return DSGD_ERR_INVALID;
  NEED(peer_rank >= 0 && peer_rank < ctx->world && peer_rank < kMaxWorld && peer_rank != ctx->rank, DSGD_ERR_INVALID,
       "dsgd_xchg_import: bad peer rank %d", peer_rank);
  int rc = xblk_ensure(ctx);
  if (rc) return rc;
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof h);
  void *ptr = nullptr;
  CU(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
  if (ctx->peer_x[peer_rank] && ctx->peer_x_ipc[peer_rank]) cudaIpcCloseMemHandle(ctx->peer_x[peer_rank]);
  ctx->peer_x[peer_rank] = static_cast<double *>(ptr);
  ctx->peer_x_ipc[peer_rank] = true;
  return DSGD_OK;
}

extern "C" int dsgd_xchg_attach(dsgd_ctx *ctx, int peer_rank, dsgd_ctx *peer) {
  if (!ctx || !peer) return DSGD_ERR_INVALID;
  NEED(peer_rank >= 0 && peer_rank < ctx->world && peer_rank < kMaxWorld && peer_rank != ctx->rank, DSGD_ERR_INVALID,
       "dsgd_xchg_attach: bad peer rank %d", peer_rank);
  NEED(peer->dim == ctx->dim, DSGD_ERR_INVALID, "dsgd_xchg_attach: dimension mismatch");
  int rc = xblk_ensure(ctx);
  if (rc) return rc;
  if ((rc = xblk_ensure(peer))) { ctx->err = peer->err; return rc; }
  CU(cudaSetDevice(ctx->device));
  if (peer->device != ctx->device) {
    int can = 0;
    CU(cudaDeviceCanAccessPeer(&can, ctx->device, peer->device));
    NEED(can, DSGD_ERR_CUDA, "dsgd_xchg_attach: device %d cannot access device %d", ctx->device, peer->device);
    cudaError_t e = cudaDeviceEnablePeerAccess(peer->device, 0);
    if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) CU(e);
    (void)cudaGetLastError();
  }
  ctx->peer_x[peer_rank] = peer->xblk;
  ctx->peer_x_ipc[peer_rank] = false;
  return DSGD_OK;
}

static int persist_check(dsgd_ctx *ctx) {  // after a stream sync: did a device-side wait hit its watchdog?
  if (!ctx->p_ready) return DSGD_OK;
  unsigned host[2] = {0, 0};
  CU(cudaMemcpy(host, ctx->p_bar, sizeof host, cudaMemcpyDeviceToHost));
  NEED(host[1] == 0, DSGD_ERR_TIMEOUT, "persistent sync kernel: a device-side wait (grid barrier, peer word) hit its watchdog");
  return DSGD_OK;
}

// Debug: copies the last persistent run's timeline out (include/dsgd.h); needs DSGD_PERSIST_TIMELINE.
static_assert(kTlWords == DSGD_TIMELINE_WORDS, "timeline layout");
extern "C" int dsgd_debug_timeline(dsgd_ctx *ctx, long long *out) {
  if (!ctx || !out) return DSGD_ERR_INVALID;
  NEED(ctx->p_tl, DSGD_ERR_STATE, "no timeline recorded (set DSGD_PERSIST_TIMELINE=1)");
  CU(cudaStreamSynchronize(ctx->stream));
  CU(cudaMemcpy(out, ctx->p_tl, sizeof(long long) * kTlWords, cudaMemcpyDeviceToHost));
  return DSGD_OK;
}

extern "C" int dsgd_set_workers(dsgd_ctx *ctx, int32_t n_local, const int32_t *counts, int32_t k_total) {
  if (!ctx) return DSGD_ERR_INVALID;
  NEED(n_local >= 0 && k_total >= 0, DSGD_ERR_INVALID, "dsgd_set_workers: negative count");
  NEED(n_local <= 1 || counts, DSGD_ERR_INVALID, "dsgd_set_workers: counts is NULL");
  std::vector<int32_t> c;
  if (counts)
    for (int32_t v = 0; v < n_local; ++v) {
      NEED(counts[v] > 0, DSGD_ERR_EMPTY, "dsgd_set_workers: worker %d has an empty batch (Vec.sum of an empty list throws)", v);
      c.push_back(counts[v]);
    }
  ctx->worker_counts = c;
  ctx->n_local = n_local;
  ctx->k_total = k_total;
  return DSGD_OK;
}

extern "C" int dsgd_sync_steps_staged(dsgd_ctx *ctx, int64_t first, int64_t n_per_step, int64_t n_steps, double lr,
                                      int want_losses) {
  if (!ctx) return DSGD_ERR_INVALID;
  NEED(!(ctx->flags & DSGD_FLAG_ASYNC), DSGD_ERR_STATE, "sync step on a ctx created in async mode");
  NEED(ctx->have_d, DSGD_ERR_STATE, "dsgd_sync_steps: dimSparsity not set");
  NEED(n_steps >= 0 && first >= 0, DSGD_ERR_INVALID, "dsgd_sync_steps: bad arguments");
  NEED(n_per_step >= 0, DSGD_ERR_INVALID, "dsgd_sync_steps: bad arguments");
  NEED(first + n_per_step * n_steps <= ctx->samples_n, DSGD_ERR_RANGE, "dsgd_sync_steps: staged samples exhausted");
  NEED(ctx->world == 1 || ctx->comm || xchg_complete(ctx), DSGD_ERR_STATE,
       "dsgd_sync_steps: world > 1 but neither dsgd_comm_init nor the peer exchange (dsgd_xchg_*) was set up");
  if (ctx->n_local == 0) {
    NEED(n_per_step == 0, DSGD_ERR_INVALID, "dsgd_sync_steps: a bystander rank (n_local == 0) takes no samples");
  } else {
    NEED(n_per_step > 0, DSGD_ERR_EMPTY, "dsgd_sync_steps: empty batch (Vec.sum of an empty list throws in the reference)");
    if (!ctx->worker_counts.empty()) {
      int64_t tot = 0;
      for (int32_t c : ctx->worker_counts) tot += c;
      NEED(tot == n_per_step, DSGD_ERR_INVALID, "dsgd_sync_steps: n_per_step %lld != sum of worker counts %lld",
           (long long)n_per_step, (long long)tot);
    }
  }
  CU(cudaSetDevice(ctx->device));
  if (want_losses) {
    int rc = ensure_f64(ctx, &ctx->losses, &ctx->losses_cap, n_steps);
    if (rc) return rc;
  }
  const int upd_blocks = cdiv(ctx->dim, 256);
  const int fin_blocks = cdiv(ctx->dim + 1, 256);
  const int32_t k_total = ctx->k_total > 0 ? ctx->k_total : ctx->world;
  const bool single = (ctx->world == 1 && ctx->n_local == 1 && k_total == 1);
  if (single && n_steps > 0 && persist_grid(ctx, n_per_step) > 0) {
    // one worker on one GPU: the whole run of steps is one persistent cooperative kernel
    return persist_run(ctx, ctx->samples + first, n_per_step, n_steps, lr, want_losses ? ctx->losses : nullptr);
  }
  if (ctx->world > 1 && ctx->n_local == 1 && k_total == ctx->world && n_steps > 0 && xchg_complete(ctx) &&
      persist_grid(ctx, n_per_step) > 0 && persist_multi_fits(ctx, persist_grid(ctx, n_per_step))) {
    // one worker per GPU, every peer's exchange block mapped: aggregate inside the persistent kernel over NVLink
    return persist_run_multi(ctx, ctx->samples + first, n_per_step, n_steps, lr, want_losses ? ctx->losses : nullptr);
  }
  for (int64_t s = 0; s < n_steps; ++s) {
    const int32_t *smp = ctx->samples + first + s * n_per_step;
    double *loss_dev = want_losses ? ctx->losses + s : nullptr;
    if (single) {
      // one worker, one GPU: gradient -> (regularize + update) fused, two launches per step
      auto *pe = prof_slot(ctx);
      if (pe) cudaEventRecord(pe->first, ctx->stream);
      k_rows<true, false><<<rows_grid(ctx, n_per_step), 256, 0, ctx->stream>>>(ctx->rp16, ctx->pairs, ctx->label, smp, 0,
                                                                               n_per_step, ctx->w, ctx->g, nullptr, ctx->cnt);
      if (pe) cudaEventRecord(pe->second, ctx->stream);
      LAUNCHED();
      k_update<true><<<upd_blocks, 256, 0, ctx->stream>>>(ctx->w, ctx->w32, ctx->g, ctx->d, ctx->dim, ctx->lambda, lr, 1.0,
                                                          ctx->scal, ctx->cnt, ctx->partial, (double)n_per_step, loss_dev);
      LAUNCHED();
      continue;
    }
    int64_t off = 0;
    for (int32_t v = 0; v < ctx->n_local; ++v) {
      const int64_t nv = ctx->worker_counts.empty() ? n_per_step : ctx->worker_counts[(size_t)v];
      auto *pe = prof_slot(ctx);
      if (pe) cudaEventRecord(pe->first, ctx->stream);
      k_rows<true, false><<<rows_grid(ctx, nv), 256, 0, ctx->stream>>>(ctx->rp16, ctx->pairs, ctx->label, smp + off, 0, nv,
                                                                       ctx->w, ctx->g, nullptr, ctx->cnt);
      if (pe) cudaEventRecord(pe->second, ctx->stream);
      LAUNCHED();
      k_finish_acc<<<fin_blocks, 256, 0, ctx->stream>>>(ctx->g, ctx->gsum, ctx->dim, ctx->scal + kScalC, ctx->cnt, (double)nv,
                                                        v == 0 ? 1 : 0);
      LAUNCHED();
      off += nv;
    }
    if (ctx->n_local == 0) CU(cudaMemsetAsync(ctx->gsum, 0, sizeof(double) * (size_t)(ctx->dim + 2), ctx->stream));
    if (ctx->world > 1)
      NC(nccl().AllReduce(ctx->gsum, ctx->gsum, (size_t)ctx->dim + 2, ncclDouble, ncclSum, ctx->comm, ctx->stream));
    k_update<false><<<upd_blocks, 256, 0, ctx->stream>>>(ctx->w, ctx->w32, ctx->gsum, ctx->d, ctx->dim, ctx->lambda, lr,
                                                         (double)k_total, ctx->scal, ctx->cnt, ctx->partial, 0.0, loss_dev);
    LAUNCHED();
  }
  CU(cudaGetLastError());
  return DSGD_OK;
}

extern "C" int dsgd_read_losses(dsgd_ctx *ctx, double *losses_out, int64_t n_steps) {
  if (!ctx) return DSGD_ERR_INVALID;
  NEED(losses_out && n_steps >= 0 && n_steps <= ctx->losses_cap, DSGD_ERR_INVALID, "dsgd_read_losses: bad arguments");
  CU(cudaSetDevice(ctx->device));
  if (n_steps)
    CU(cudaMemcpyAsync(losses_out, ctx->losses, sizeof(double) * (size_t)n_steps, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return persist_check(ctx);
}

extern "C" int dsgd_sync_steps(dsgd_ctx *ctx, const int32_t *samples, int64_t n_per_step, int64_t n_steps, double lr,
                               double *losses_out) {
  if (!ctx) return DSGD_ERR_INVALID;
  NEED(n_steps >= 0 && n_per_step >= 0, DSGD_ERR_INVALID, "dsgd_sync_steps: bad arguments");
  NEED(n_per_step > 0 || ctx->n_local == 0, DSGD_ERR_EMPTY,
       "dsgd_sync_steps: empty batch (Vec.sum of an empty list throws in the reference)");
  int rc = dsgd_stage_samples(ctx, samples, n_per_step * n_steps);
  if (rc) return rc;
  if ((rc = dsgd_sync_steps_staged(ctx, 0, n_per_step, n_steps, lr, losses_out != nullptr))) return rc;
  if (losses_out) return dsgd_read_losses(ctx, losses_out, n_steps);
  CU(cudaStreamSynchronize(ctx->stream));
  return persist_check(ctx);
}

extern "C" int dsgd_sync_step(dsgd_ctx *ctx, const int32_t *samples, int64_t n, double lr, double *loss_out) {
  return dsgd_sync_steps(ctx, samples, n, 1, lr, loss_out);
}

// ---- async (Hogwild) mode -------------------------------------------------------------------------------------

static int ensure_dev(dsgd_ctx *ctx, void **buf, int64_t *cap, int64_t n, size_t elt) {
  if (*cap >= n) return DSGD_OK;
  if (*buf) CU(cudaFree(*buf));
  *buf = nullptr; *cap = 0;
  const int64_t want = std::max<int64_t>(n, 1024);
  CU(cudaMalloc(buf, elt * (size_t)want));
  *cap = want;
  return DSGD_OK;
}

extern "C" int dsgd_async_host_master(dsgd_ctx *ctx, const double *w0) {
  if (!ctx) return DSGD_ERR_INVALID;
  NEED(ctx->flags & DSGD_FLAG_ASYNC, DSGD_ERR_STATE, "Cannot host the async master replica: ctx is in synchronous mode.");
  NEED(w0, DSGD_ERR_INVALID, "dsgd_async_host_master: w0 is NULL");
  NEED(ctx->have_d, DSGD_ERR_STATE, "dsgd_async_host_master: dimSparsity not set");
  CU(cudaSetDevice(ctx->device));
  if (!ctx->m_w) CU(cudaMalloc(&ctx->m_w, sizeof(double) * (size_t)(ctx->dim + kReplicaPad)));
  CU(cudaMemsetAsync(ctx->m_w, 0, sizeof(double) * (size_t)(ctx->dim + kReplicaPad), ctx->stream));
  CU(cudaMemcpyAsync(ctx->m_w, w0, sizeof(double) * (size_t)ctx->dim, cudaMemcpyHostToDevice, ctx->stream));
  k_async_init_ctl<1024><<<1, 1024, 0, ctx->stream>>>(ctx->m_w, ctx->d, ctx->dim);
  LAUNCHED();
  CU(cudaGetLastError());
  CU(cudaStreamSynchronize(ctx->stream));
  return DSGD_OK;
}

extern "C" int dsgd_ipc_export(dsgd_ctx *ctx, int which, uint8_t handle[DSGD_IPC_HANDLE_BYTES]) {
  if (!ctx || !handle) return DSGD_ERR_INVALID;
  static_assert(sizeof(cudaIpcMemHandle_t) == DSGD_IPC_HANDLE_BYTES, "cudaIpcMemHandle_t size");
  NEED(which == DSGD_REPLICA_SELF || which == DSGD_REPLICA_MASTER, DSGD_ERR_INVALID, "dsgd_ipc_export: bad `which`");
  NEED(which == DSGD_REPLICA_SELF || ctx->m_w, DSGD_ERR_STATE, "dsgd_ipc_export: this ctx does not host the master replica");
  CU(cudaSetDevice(ctx->device));
  cudaIpcMemHandle_t h;
  CU(cudaIpcGetMemHandle(&h, which == DSGD_REPLICA_SELF ? ctx->w : ctx->m_w));
  memcpy(handle, &h, sizeof h);
  return DSGD_OK;
}

extern "C" int dsgd_ipc_import(dsgd_ctx *ctx, int peer_rank, const uint8_t handle[DSGD_IPC_HANDLE_BYTES]) {
  if (!ctx || !handle) return DSGD_ERR_INVALID;
  NEED(peer_rank >= 0 && peer_rank <= ctx->world && peer_rank < kMaxReplicas, DSGD_ERR_INVALID,
       "dsgd_ipc_import: peer_rank %d outside [0,%d]", peer_rank, ctx->world);
  NEED(peer_rank != ctx->rank, DSGD_ERR_INVALID, "dsgd_ipc_import: a worker does not import its own replica");
  NEED(!ctx->a_running, DSGD_ERR_STATE, "dsgd_ipc_import: async computation is running");
  CU(cudaSetDevice(ctx->device));
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof h);
  void *ptr = nullptr;
  CU(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
  if (ctx->peer_w[peer_rank] && ctx->peer_ipc[peer_rank]) cudaIpcCloseMemHandle(ctx->peer_w[peer_rank]);
  ctx->peer_w[peer_rank] = static_cast<double *>(ptr);
  ctx->peer_ipc[peer_rank] = true;
  return DSGD_OK;
}

extern "C" int dsgd_peer_attach(dsgd_ctx *ctx, int peer_rank, dsgd_ctx *peer, int which) {
  if (!ctx || !peer) return DSGD_ERR_INVALID;
  NEED(peer_rank >= 0 && peer_rank <= ctx->world && peer_rank < kMaxReplicas, DSGD_ERR_INVALID,
       "dsgd_peer_attach: peer_rank %d outside [0,%d]", peer_rank, ctx->world);
  NEED(which == DSGD_REPLICA_SELF || peer->m_w, DSGD_ERR_STATE, "dsgd_peer_attach: peer does not host the master replica");
  NEED(peer->dim == ctx->dim, DSGD_ERR_INVALID, "dsgd_peer_attach: dimension mismatch");
  CU(cudaSetDevice(ctx->device));
  if (peer->device != ctx->device) {
    int can = 0;
    CU(cudaDeviceCanAccessPeer(&can, ctx->device, peer->device));
    NEED(can, DSGD_ERR_CUDA, "dsgd_peer_attach: device %d cannot access device %d", ctx->device, peer->device);
    cudaError_t e = cudaDeviceEnablePeerAccess(peer->device, 0);
    if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) CU(e);
    (void)cudaGetLastError();
  }
  ctx->peer_w[peer_rank] = which == DSGD_REPLICA_SELF ? peer->w : peer->m_w;
  ctx->peer_ipc[peer_rank] = false;
  return DSGD_OK;
}

static int async_launch(dsgd_ctx *ctx, const double *w0, const int32_t *assigned, int64_t n_assigned, const int32_t *replay,
                        int32_t batch, double lr, int32_t lanes, int64_t max_updates, uint64_t seed, cudaStream_t st) {
  NEED(ctx->flags & DSGD_FLAG_ASYNC, DSGD_ERR_STATE, "Cannot initialize async computation: slave is in synchronous mode.");
  NEED(!ctx->a_running, DSGD_ERR_STATE,
       "Async computation already running, can't be initialized unless stopped first");
  NEED(ctx->pairs && ctx->have_d, DSGD_ERR_STATE, "dsgd_start_async: rows or dimSparsity missing");
  NEED(batch >= 1 && lanes >= 1 && lanes <= 4096, DSGD_ERR_INVALID, "dsgd_start_async: bad arguments");
  CU(cudaSetDevice(ctx->device));
  int rc = DSGD_OK;
  if (w0) {  // weights() = request.weights
    CU(cudaMemcpyAsync(ctx->w, w0, sizeof(double) * (size_t)ctx->dim, cudaMemcpyHostToDevice, ctx->stream));
    rc = refresh_resident(ctx);  // also S = w . d and the control slots of the replica
    if (rc) return rc;
  }  // else: keep the resident replica (already initialised; deltas peers pushed since then must survive)
  if (ctx->a_scratch_lanes < lanes) {
    if (ctx->a_scratch) CU(cudaFree(ctx->a_scratch));
    ctx->a_scratch = nullptr; ctx->a_scratch_lanes = 0;
    CU(cudaMalloc(&ctx->a_scratch, sizeof(double) * (size_t)lanes * (size_t)ctx->dim));
    CU(cudaMemsetAsync(ctx->a_scratch, 0, sizeof(double) * (size_t)lanes * (size_t)ctx->dim, ctx->stream));
    ctx->a_scratch_lanes = lanes;
  }
  if ((rc = ensure_dev(ctx, (void **)&ctx->a_rows, &ctx->a_rows_cap, (int64_t)lanes * batch, sizeof(int32_t)))) return rc;
  CU(cudaMemsetAsync(ctx->a_stop, 0, sizeof(int), ctx->stream));
  CU(cudaMemsetAsync(ctx->a_cnt, 0, sizeof(unsigned long long) * 2, ctx->stream));
  AsyncParams ap;
  ap.rp16 = ctx->rp16; ap.pairs = ctx->pairs; ap.label = ctx->label; ap.d = ctx->d; ap.dim = ctx->dim;
  ap.assigned = assigned; ap.n_assigned = n_assigned; ap.replay = replay; ap.batch = batch; ap.lr = lr; ap.lambda = ctx->lambda;
  ap.rows_unique = ctx->rows_unique ? 1 : 0;
  int nr = 0;
  ap.replica[nr++] = ctx->w;
  for (int r = 0; r < ctx->world && r < kMaxReplicas - 1; ++r)
    if (r != ctx->rank && ctx->peer_w[r]) ap.replica[nr++] = ctx->peer_w[r];
  ap.master_slot = -1;
  double *master = ctx->m_w ? ctx->m_w : (ctx->world < kMaxReplicas ? ctx->peer_w[ctx->world] : nullptr);
  if (master) { ap.master_slot = nr; ap.replica[nr++] = master; }
  if (ctx->outbox) {   // colleagues reached over the host: one more target of every delta, relayed by the host in batches
    NEED(nr < kMaxReplicas, DSGD_ERR_INVALID, "dsgd_start_async: no replica slot left for the outbox");
    ap.replica[nr++] = ctx->outbox;
  }
  for (int q = nr; q < kMaxReplicas; ++q) ap.replica[q] = nullptr;
  ap.n_replicas = nr;
  ap.scratch = ctx->a_scratch; ap.batch_rows = ctx->a_rows; ap.n_lanes = lanes; ap.max_updates = max_updates; ap.seed = seed;
  ap.stop = ctx->a_stop; ap.claimed = ctx->a_cnt; ap.done = ctx->a_cnt + 1;
  CU(cudaStreamSynchronize(ctx->stream));  // inputs in place before the loop's own stream starts
  if (!ctx->a_ev0) { CU(cudaEventCreate(&ctx->a_ev0)); CU(cudaEventCreate(&ctx->a_ev1)); }
  CU(cudaEventRecord(ctx->a_ev0, st));
  // batch 1 on rows with unique columns (what the reference's Map rows are): the delta of every non-zero is formed straight
  // from the pair, without the per-lane scratch vector
  if (batch == 1 && ctx->rows_unique) k_async_worker_b1<<<cdiv(lanes, 4), 128, 0, st>>>(ap);
  else k_async_worker<<<cdiv(lanes, 4), 128, 0, st>>>(ap);
  CU(cudaEventRecord(ctx->a_ev1, st));
  LAUNCHED();
  CU(cudaGetLastError());
  return DSGD_OK;
}

extern "C" int dsgd_start_async(dsgd_ctx *ctx, const double *w0, const int32_t *assigned, int64_t n_assigned, int32_t batch,
                                double lr, int32_t concurrency, int64_t max_updates, uint64_t seed) {
  if (!ctx) return DSGD_ERR_INVALID;
  NEED(ctx->flags & DSGD_FLAG_ASYNC, DSGD_ERR_STATE, "Cannot initialize async computation: slave is in synchronous mode.");
  NEED(assigned && n_assigned >= 1, DSGD_ERR_EMPTY, "dsgd_start_async: no samples assigned (Random.nextInt(0) throws)");
  NEED(n_assigned <= ctx->n_rows, DSGD_ERR_RANGE, "dsgd_start_async: more assigned samples than rows");
  for (int64_t i = 0; i < n_assigned; ++i)
    NEED(assigned[i] >= 0 && assigned[i] < ctx->n_rows, DSGD_ERR_RANGE, "assigned sample %d at position %lld outside [0,%lld)",
         assigned[i], (long long)i, (long long)ctx->n_rows);
  CU(cudaSetDevice(ctx->device));
  int rc = ensure_dev(ctx, (void **)&ctx->a_assigned, &ctx->a_assigned_cap, n_assigned, sizeof(int32_t));
  if (rc) return rc;
  CU(cudaMemcpyAsync(ctx->a_assigned, assigned, sizeof(int32_t) * (size_t)n_assigned, cudaMemcpyHostToDevice, ctx->stream));
  if (batch > n_assigned) batch = (int32_t)n_assigned;  // `take batchSize` of a shorter shuffle
  rc = async_launch(ctx, w0, ctx->a_assigned, n_assigned, nullptr, batch, lr, concurrency, max_updates, seed, ctx->astream);
  if (rc) return rc;
  ctx->a_running = true;
  return DSGD_OK;
}

extern "C" int dsgd_async_replay(dsgd_ctx *ctx, const double *w0, const int32_t *samples, int32_t batch, int64_t n_updates,
                                 double lr) {
  if (!ctx) return DSGD_ERR_INVALID;
  NEED(ctx->flags & DSGD_FLAG_ASYNC, DSGD_ERR_STATE, "Cannot initialize async computation: slave is in synchronous mode.");
  NEED(samples && batch >= 1 && n_updates >= 1, DSGD_ERR_EMPTY, "dsgd_async_replay: empty sequence");
  const int64_t n = (int64_t)batch * n_updates;
  for (int64_t i = 0; i < n; ++i)
    NEED(samples[i] >= 0 && samples[i] < ctx->n_rows, DSGD_ERR_RANGE, "sample index %d at position %lld outside [0,%lld)",
         samples[i], (long long)i, (long long)ctx->n_rows);
  CU(cudaSetDevice(ctx->device));
  int rc = ensure_dev(ctx, (void **)&ctx->a_replay, &ctx->a_replay_cap, n, sizeof(int32_t));
  if (rc) return rc;
  CU(cudaMemcpyAsync(ctx->a_replay, samples, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
  rc = async_launch(ctx, w0, nullptr, 1, ctx->a_replay, batch, lr, 1, n_updates, 0, ctx->stream);
  if (rc) return rc;
  CU(cudaStreamSynchronize(ctx->stream));
  rc = refresh_resident(ctx);
  // refresh_resident re-derives S from the weights; the loop's running S is what the NEXT replay would start from anyway
  if (rc) return rc;
  CU(cudaStreamSynchronize(ctx->stream));
  return DSGD_OK;
}

extern "C" int dsgd_async_running(dsgd_ctx *ctx, int *running) {
  if (!ctx || !running) return DSGD_ERR_INVALID;
  CU(cudaSetDevice(ctx->device));
  *running = 0;
  if (ctx->a_running) {
    cudaError_t e = cudaStreamQuery(ctx->astream);
    if (e == cudaErrorNotReady) *running = 1;
    else if (e != cudaSuccess) CU(e);
  }
  return DSGD_OK;
}

extern "C" int dsgd_stop_async(dsgd_ctx *ctx) {
  if (!ctx) return DSGD_ERR_INVALID;
  NEED(ctx->flags & DSGD_FLAG_ASYNC, DSGD_ERR_STATE, "Cannot stop async computation: slave is in synchronous mode.");
  CU(cudaSetDevice(ctx->device));
  if (!ctx->a_running) return DSGD_OK;  // runningAsync() = false on an idle slave is a no-op in the reference too
  static const int one = 1;
  CU(cudaMemcpyAsync(ctx->a_stop, &one, sizeof(int), cudaMemcpyHostToDevice, ctx->stream2));
  CU(cudaStreamSynchronize(ctx->stream2));
  CU(cudaStreamSynchronize(ctx->astream));
  ctx->a_running = false;
  k_prepare<1024><<<1, 1024, 0, ctx->stream>>>(ctx->w, ctx->d, ctx->dim, ctx->lambda, ctx->scal + kScalC, ctx->scal + kScalNrm2);
  LAUNCHED();
  k_to_f32<<<cdiv(ctx->dim, 256), 256, 0, ctx->stream>>>(ctx->w, ctx->w32, ctx->dim);
  LAUNCHED();
  CU(cudaGetLastError());
  CU(cudaStreamSynchronize(ctx->stream));
  return DSGD_OK;
}

extern "C" int dsgd_async_elapsed_ms(dsgd_ctx *ctx, float *elapsed_ms) {
  if (!ctx || !elapsed_ms) return DSGD_ERR_INVALID;
  NEED(ctx->a_ev0 && !ctx->a_running, DSGD_ERR_STATE, "dsgd_async_elapsed_ms: no finished async loop (stop it first)");
  CU(cudaSetDevice(ctx->device));
  CU(cudaEventSynchronize(ctx->a_ev1));
  CU(cudaEventElapsedTime(elapsed_ms, ctx->a_ev0, ctx->a_ev1));
  return DSGD_OK;
}

extern "C" int dsgd_update_grad(dsgd_ctx *ctx, const int32_t *idx, const double *val, int64_t nnz) {
  if (!ctx) return DSGD_ERR_INVALID;
  NEED(ctx->flags & DSGD_FLAG_ASYNC, DSGD_ERR_STATE, "Cannot update gradient: slave is in synchronous mode.");
  NEED(nnz >= 0 && (nnz == 0 || (idx && val)), DSGD_ERR_INVALID, "dsgd_update_grad: bad arguments");
  for (int64_t k = 0; k < nnz; ++k)
    NEED(idx[k] >= 0 && idx[k] < ctx->dim, DSGD_ERR_RANGE, "dsgd_update_grad: key %d outside [0,%d)", idx[k], ctx->dim);
  if (nnz == 0) return DSGD_OK;
  CU(cudaSetDevice(ctx->device));
  if (ctx->u_cap < nnz) {
    if (ctx->u_idx) CU(cudaFree(ctx->u_idx));
    if (ctx->u_val) CU(cudaFree(ctx->u_val));
    ctx->u_idx = nullptr; ctx->u_val = nullptr; ctx->u_cap = 0;
    const int64_t want = std::max<int64_t>(nnz, 4096);
    CU(cudaMalloc(&ctx->u_idx, sizeof(int32_t) * (size_t)want));
    CU(cudaMalloc(&ctx->u_val, sizeof(double) * (size_t)want));
    ctx->u_cap = want;
  }
  CU(cudaMemcpyAsync(ctx->u_idx, idx, sizeof(int32_t) * (size_t)nnz, cudaMemcpyHostToDevice, ctx->stream2));
  CU(cudaMemcpyAsync(ctx->u_val, val, sizeof(double) * (size_t)nnz, cudaMemcpyHostToDevice, ctx->stream2));
  k_async_apply_delta<<<std::min(cdiv(nnz, 256), 64), 256, 0, ctx->stream2>>>(ctx->w, ctx->dim, ctx->d, ctx->u_idx, ctx->u_val, nnz, 0);
  LAUNCHED();
  CU(cudaGetLastError());
  CU(cudaStreamSynchronize(ctx->stream2));
  return DSGD_OK;
}

static double *master_replica(dsgd_ctx *ctx) {
  return ctx->m_w ? ctx->m_w : (ctx->world < kMaxReplicas ? ctx->peer_w[ctx->world] : nullptr);
}

extern "C" int dsgd_async_updates(dsgd_ctx *ctx, int64_t *count) {
  if (!ctx || !count) return DSGD_ERR_INVALID;
  NEED(ctx->flags & DSGD_FLAG_ASYNC, DSGD_ERR_STATE, "dsgd_async_updates: ctx is in synchronous mode");
  CU(cudaSetDevice(ctx->device));
  unsigned long long v = 0;
  double *m = master_replica(ctx);
  const void *src = m ? (const void *)(reinterpret_cast<unsigned long long *>(m) + ctx->dim + kCtlUpdates) : (const void *)(ctx->a_cnt + 1);
  CU(cudaMemcpyAsync(&v, src, sizeof v, cudaMemcpyDeviceToHost, ctx->stream2));
  CU(cudaStreamSynchronize(ctx->stream2));
  *count = (int64_t)v;
  return DSGD_OK;
}

extern "C" int dsgd_async_outbox_enable(dsgd_ctx *ctx) {
  if (!ctx) return DSGD_ERR_INVALID;
  NEED(ctx->flags & DSGD_FLAG_ASYNC, DSGD_ERR_STATE, "dsgd_async_outbox_enable: ctx is in synchronous mode");
  NEED(!ctx->a_running, DSGD_ERR_STATE, "dsgd_async_outbox_enable: async computation is running");
  CU(cudaSetDevice(ctx->device));
  if (!ctx->outbox) CU(cudaMalloc(&ctx->outbox, sizeof(double) * (size_t)(ctx->dim + kReplicaPad)));
  CU(cudaMemsetAsync(ctx->outbox, 0, sizeof(double) * (size_t)(ctx->dim + kReplicaPad), ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return DSGD_OK;
}

extern "C" int dsgd_async_outbox_read(dsgd_ctx *ctx, double *acc_out) {
  if (!ctx || !acc_out) return DSGD_ERR_INVALID;
  NEED(ctx->outbox, DSGD_ERR_STATE, "dsgd_async_outbox_read: the outbox is not enabled");
  CU(cudaSetDevice(ctx->device));
  CU(cudaMemcpyAsync(acc_out, ctx->outbox, sizeof(double) * (size_t)ctx->dim, cudaMemcpyDeviceToHost, ctx->stream2));
  CU(cudaStreamSynchronize(ctx->stream2));
  return DSGD_OK;
}

extern "C" int dsgd_async_master_weights(dsgd_ctx *ctx, double *w_out) {
  if (!ctx || !w_out) return DSGD_ERR_INVALID;
  NEED(ctx->flags & DSGD_FLAG_ASYNC, DSGD_ERR_STATE, "dsgd_async_master_weights: ctx is in synchronous mode");
  double *m = master_replica(ctx);
  NEED(m, DSGD_ERR_STATE, "dsgd_async_master_weights: no master replica hosted or imported");
  CU(cudaSetDevice(ctx->device));
  CU(cudaMemcpyAsync(w_out, m, sizeof(double) * (size_t)ctx->dim, cudaMemcpyDeviceToHost, ctx->stream2));
  CU(cudaStreamSynchronize(ctx->stream2));
  return DSGD_OK;
}

// ---- model sets (dsgd_models.cuh): M SparseSVMs, each with its own lambda and learning rate, on the same draws ---------
// Main.scala:68 builds ONE `new SparseSVM(config.lambda, ...)` per run and Master.fit (core/Master.scala:179-198) trains it;
// a model set trains up to DSGD_MAX_MODELS of them in one persistent kernel per call.  One GPU, one worker per step.
static_assert(kMaxModels == DSGD_MAX_MODELS, "model-set cap");
constexpr int kMCons = 8, kMUpd = 8, kMStages = 4, kMStagePairs = 2560, kMMaxChunks = 128;
using MSmem = ModelsSmem<kMCons, kMUpd, kMStages, kMStagePairs, kMMaxChunks>;
#define DSGD_MODELS_KERNEL k_models_persistent<kMCons, kMUpd, kMStages, kMStagePairs, kMMaxChunks>

static int models_shape_ok(dsgd_ctx *ctx, const char *who) {
  NEED(!(ctx->flags & DSGD_FLAG_ASYNC), DSGD_ERR_STATE, "%s: ctx is in async mode", who);
  NEED(ctx->world == 1, DSGD_ERR_STATE, "%s: model sets run on one GPU (world is %d)", who, ctx->world);
  const int32_t k_total = ctx->k_total > 0 ? ctx->k_total : ctx->world;
  NEED(ctx->n_local == 1 && k_total == 1, DSGD_ERR_STATE, "%s: model sets take one worker per step (n_local %d, k_total %d)",
       who, ctx->n_local, k_total);
  return DSGD_OK;
}

static void models_free(dsgd_ctx *ctx) {
  void *ptrs[] = {ctx->ms_w, ctx->ms_rec, ctx->ms_acc};
  for (void *q : ptrs) if (q) cudaFree(q);
  ctx->ms_w = nullptr; ctx->ms_rec = nullptr; ctx->ms_acc = nullptr;
  ctx->ms_n = 0;
  ctx->ms_lambda.clear(); ctx->ms_lr.clear();
}

extern "C" int dsgd_models_set(dsgd_ctx *ctx, int32_t n_models, const double *lambda, const double *lr, const double *w0) {
  if (!ctx) return DSGD_ERR_INVALID;
  int rc = models_shape_ok(ctx, "dsgd_models_set");
  if (rc) return rc;
  NEED(n_models >= 0 && n_models <= DSGD_MAX_MODELS, DSGD_ERR_INVALID, "dsgd_models_set: n_models %d outside [0,%d]", n_models,
       DSGD_MAX_MODELS);
  NEED(n_models == 0 || (lambda && lr), DSGD_ERR_INVALID, "dsgd_models_set: lambda / lr is NULL");
  for (int32_t m = 0; m < n_models; ++m) {
    NEED(std::isfinite(lambda[m]) && lambda[m] >= 0.0, DSGD_ERR_INVALID, "dsgd_models_set: lambda[%d] = %g is not a finite non-negative number", m, lambda[m]);
    NEED(std::isfinite(lr[m]), DSGD_ERR_INVALID, "dsgd_models_set: lr[%d] = %g is not finite", m, lr[m]);
  }
  CU(cudaSetDevice(ctx->device));
  CU(cudaStreamSynchronize(ctx->stream));
  models_free(ctx);
  if (n_models == 0) return DSGD_OK;
  const size_t dim = (size_t)ctx->dim;
  CU(cudaMalloc(&ctx->ms_w, sizeof(double) * dim * (size_t)n_models));
  CU(cudaMalloc(&ctx->ms_rec, sizeof(double2) * 3 * dim * (size_t)n_models));
  CU(cudaMalloc(&ctx->ms_acc, sizeof(unsigned long long) * 3 * kAccStride * (size_t)n_models));
  if (!ctx->ms_bar) CU(cudaMalloc(&ctx->ms_bar, sizeof(unsigned) * 4));
  if (w0) CU(cudaMemcpyAsync(ctx->ms_w, w0, sizeof(double) * dim * (size_t)n_models, cudaMemcpyHostToDevice, ctx->stream));
  else CU(cudaMemsetAsync(ctx->ms_w, 0, sizeof(double) * dim * (size_t)n_models, ctx->stream));
  if (!ctx->ms_ready) {
    CU(cudaFuncSetAttribute((const void *)DSGD_MODELS_KERNEL, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(MSmem)));
    ctx->ms_ready = true;
  }
  CU(cudaStreamSynchronize(ctx->stream));
  ctx->ms_n = n_models;
  ctx->ms_lambda.assign(lambda, lambda + n_models);
  ctx->ms_lr.assign(lr, lr + n_models);
  return DSGD_OK;
}

extern "C" int dsgd_models_shape(const dsgd_ctx *ctx, int32_t *n_models, int32_t *dim) {
  if (!ctx) return DSGD_ERR_INVALID;
  if (n_models) *n_models = ctx->ms_n;
  if (dim) *dim = ctx->dim;
  return DSGD_OK;
}

extern "C" int dsgd_models_get_weights(dsgd_ctx *ctx, double *w_out) {
  if (!ctx) return DSGD_ERR_INVALID;
  NEED(ctx->ms_n > 0, DSGD_ERR_STATE, "dsgd_models_get_weights: no model set (dsgd_models_set)");
  NEED(w_out, DSGD_ERR_INVALID, "dsgd_models_get_weights: w_out is NULL");
  CU(cudaSetDevice(ctx->device));
  CU(cudaMemcpyAsync(w_out, ctx->ms_w, sizeof(double) * (size_t)ctx->dim * (size_t)ctx->ms_n, cudaMemcpyDeviceToHost,
                     ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return DSGD_OK;
}

extern "C" int dsgd_models_steps(dsgd_ctx *ctx, const int32_t *samples, int64_t n_per_step, int64_t n_steps,
                                 const uint8_t *active, double *losses_out) {
  if (!ctx) return DSGD_ERR_INVALID;
  int rc = models_shape_ok(ctx, "dsgd_models_steps");
  if (rc) return rc;
  NEED(ctx->have_d, DSGD_ERR_STATE, "dsgd_models_steps: dimSparsity not set");
  NEED(ctx->ms_n > 0, DSGD_ERR_STATE, "dsgd_models_steps: no model set (dsgd_models_set)");
  NEED(n_steps >= 0 && n_per_step >= 0, DSGD_ERR_INVALID, "dsgd_models_steps: bad arguments");
  NEED(n_per_step > 0, DSGD_ERR_EMPTY, "dsgd_models_steps: empty batch (Vec.sum of an empty list throws in the reference)");
  NEED(n_steps == 0 || samples, DSGD_ERR_INVALID, "dsgd_models_steps: samples is NULL");
  NEED(n_steps <= INT64_MAX / n_per_step, DSGD_ERR_INVALID, "dsgd_models_steps: too many samples");
  const int G = persist_grid(ctx, n_per_step);
  NEED(G > 0, DSGD_ERR_INVALID, "dsgd_models_steps: %lld samples per step exceed the kernel's %d rows per SM",
       (long long)n_per_step, kMaxRowsPerCta);
  NEED((uint64_t)G * (uint64_t)(n_steps + 2) < (1ull << 32), DSGD_ERR_INVALID, "dsgd_models_steps: too many steps for one launch");
  const int M = ctx->ms_n;
  ModelsParams pp;
  memset(&pp, 0, sizeof pp);
  int n_act = 0;
  for (int m = 0; m < M; ++m)
    if (!active || active[m]) {
      pp.id[n_act] = m;
      pp.lambda[n_act] = ctx->ms_lambda[(size_t)m];
      pp.lr[n_act] = ctx->ms_lr[(size_t)m];
      ++n_act;
    }
  if ((rc = dsgd_stage_samples(ctx, samples, n_per_step * n_steps))) return rc;
  if (n_steps == 0 || n_act == 0) {
    if (losses_out)
      for (int64_t i = 0; i < n_steps * M; ++i) losses_out[i] = std::numeric_limits<double>::quiet_NaN();
    CU(cudaStreamSynchronize(ctx->stream));
    return DSGD_OK;
  }
  if ((rc = ensure_dev(ctx, (void **)&ctx->ms_hinge, &ctx->ms_hinge_cap, n_steps * n_act, sizeof(unsigned)))) return rc;
  if (losses_out && (rc = ensure_f64(ctx, &ctx->ms_losses, &ctx->ms_losses_cap, n_steps * n_act))) return rc;
  pp.rp16 = ctx->rp16; pp.pairs = ctx->pairs; pp.label = ctx->label; pp.samples = ctx->samples;
  pp.n_steps = n_steps; pp.batch = (int32_t)n_per_step; pp.dim = ctx->dim; pp.n_act = n_act;
  pp.rec_stride = ctx->dim; pp.rec = ctx->ms_rec; pp.d = ctx->d; pp.acc = ctx->ms_acc;
  pp.hinge = ctx->ms_hinge; pp.losses = losses_out ? ctx->ms_losses : nullptr; pp.w_res = ctx->ms_w;
  pp.bar = ctx->ms_bar; pp.abort_flag = reinterpret_cast<int *>(ctx->ms_bar + 1);
  pp.timeout_cycles = 4000000000ll;  // ~2 s at 1.9 GHz, as for the single-model kernel
  CU(cudaMemsetAsync(ctx->ms_acc, 0, sizeof(unsigned long long) * 3 * kAccStride * (size_t)n_act, ctx->stream));
  CU(cudaMemsetAsync(ctx->ms_hinge, 0, sizeof(unsigned) * (size_t)(n_steps * n_act), ctx->stream));
  CU(cudaMemsetAsync(ctx->ms_bar, 0, sizeof(unsigned) * 4, ctx->stream));
  // every launch starts from the resident weights of its models: several calls continue one trajectory
  k_models_rec_init<<<dim3(cdiv(ctx->dim, 256), n_act), 256, 0, ctx->stream>>>(pp);
  LAUNCHED();
  void *args[] = {&pp};
  const dim3 block((kMCons + kMUpd + 1) * 32);
  auto *pe = prof_slot(ctx);
  if (pe) cudaEventRecord(pe->first, ctx->stream);
  if (ctx->grid_limit > 0) CU(cudaLaunchKernel((void *)DSGD_MODELS_KERNEL, dim3(G), block, args, sizeof(MSmem), ctx->stream));
  else CU(cudaLaunchCooperativeKernel((void *)DSGD_MODELS_KERNEL, dim3(G), block, args, sizeof(MSmem), ctx->stream));
  if (pe) cudaEventRecord(pe->second, ctx->stream);
  LAUNCHED();
  if (losses_out) {
    std::vector<double> compact((size_t)(n_steps * n_act));
    CU(cudaMemcpyAsync(compact.data(), ctx->ms_losses, sizeof(double) * compact.size(), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    for (int64_t s = 0; s < n_steps; ++s) {
      int k = 0;
      for (int m = 0; m < M; ++m)
        losses_out[s * M + m] = (!active || active[m]) ? compact[(size_t)(s * n_act + k++)] : std::numeric_limits<double>::quiet_NaN();
    }
  }
  CU(cudaStreamSynchronize(ctx->stream));
  unsigned host[2] = {0, 0};
  CU(cudaMemcpy(host, ctx->ms_bar, sizeof host, cudaMemcpyDeviceToHost));
  NEED(host[1] == 0, DSGD_ERR_TIMEOUT, "model-set kernel: a device-side wait (grid barrier, stage) hit its watchdog");
  return DSGD_OK;
}

extern "C" int dsgd_models_eval_counts(dsgd_ctx *ctx, int32_t m, int64_t row_begin, int64_t row_end, int64_t *hinge_sum,
                                       int64_t *correct, double *norm_squared) {
  if (!ctx) return DSGD_ERR_INVALID;
  NEED(ctx->ms_n > 0, DSGD_ERR_STATE, "dsgd_models_eval_counts: no model set (dsgd_models_set)");
  NEED(m >= 0 && m < ctx->ms_n, DSGD_ERR_INVALID, "dsgd_models_eval_counts: model %d outside [0,%d)", m, ctx->ms_n);
  double out[5];
  int rc = eval_impl(ctx, ctx->ms_w + (size_t)m * (size_t)ctx->dim, row_begin, row_end, out, true);
  if (rc) return rc;
  if (hinge_sum) *hinge_sum = (int64_t)out[2];
  if (correct) *correct = (int64_t)out[3];
  if (norm_squared) *norm_squared = out[4];
  return DSGD_OK;
}
