/*
 * dsgd.h -- C ABI of the B200-native data-parallel SGD hot path (libdsgd.so).
 *
 * This is the drop-in boundary for zifeo/distributed-sgd's hot path.  The reference has no FFI of its
 * own (it is 100 % Scala over gRPC, SURVEY.md F1/F2); the seams this ABI sits behind are the handlers of
 * its gRPC `Slave` service and the step body of `Master.fit`.  Every entry point names the reference
 * interface it replaces (path:line under /root/reference/src/main/).  INTEGRATION.md shows the JNI /
 * Scala binding a maintainer would add; distributed_sgd_b200/ is the Python host that mirrors the
 * reference's Slave / Master / SparseSVM surface over this ABI.
 *
 * Conventions
 *  - One opaque dsgd_ctx per GPU == one reference Slave (+ its SparseSVM).  In sync mode every ctx also
 *    carries the Master's weight vector (weights stay resident on the device; the reference's per-request
 *    weight broadcast, core/Master.scala:186-188, disappears).
 *  - Every call returns 0 (DSGD_OK) or a negative DSGD_ERR_*; dsgd_last_error() gives the message.  No
 *    exception crosses the ABI.  The caller owns all host buffers; they are consumed before the call
 *    returns.  The ctx owns all device memory.
 *  - Vectors (weights, gradients, dimSparsity) are dense double[dim]; 0.0 stands for "key absent from the
 *    reference's Map[Int, Number]".  The reference's wire type is double (protobuf/proto.proto:28-31).
 *  - Rows are CSR with 0-based int32 columns and fp32 values; CSR column c stands for the reference's
 *    1-based feature key c+1 (utils/Dataset.scala:30).  Sample indices are row ids into what
 *    dsgd_load_csr received (the reference addresses a slave by global row id, core/Slave.scala:149).
 *  - Arithmetic: values fp32 (exactly promoted), every accumulation and all state in fp64, like the
 *    reference's spire.math.Number over Double.
 *  - Threading: calls on one ctx are serialised by the caller, except dsgd_update_grad,
 *    dsgd_get_weights, dsgd_async_updates and dsgd_stop_async, which are safe while the async loop runs
 *    (the reference serves them from its 8-thread pool concurrently with asyncTask, core/Slave.scala:24-30).
 */
#ifndef DSGD_H
#define DSGD_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DSGD_OK 0
#define DSGD_ERR_INVALID (-1) /* bad argument; the reference's require(...) / IllegalArgumentException        */
#define DSGD_ERR_STATE (-2)   /* wrong mode or state: "slave is in synchronous mode", "already running"        */
#define DSGD_ERR_EMPTY (-3)   /* empty batch: Vec.sum on an empty list throws (math/Vec.scala:129, quirk Q7)   */
#define DSGD_ERR_RANGE (-4)   /* sample index outside the loaded rows (ArrayIndexOutOfBounds in the reference)  */
#define DSGD_ERR_CUDA (-5)    /* CUDA runtime error, or no usable GPU (there is no CPU fallback)                */
#define DSGD_ERR_NCCL (-6)    /* NCCL error                                                                     */
#define DSGD_ERR_NOMEM (-7)
#define DSGD_ERR_TIMEOUT (-8) /* a device-side wait (peer flag, grid barrier) hit its watchdog                  */

#define DSGD_UNIQUE_ID_BYTES 128
#define DSGD_IPC_HANDLE_BYTES 64

/* dsgd_create flags */
#define DSGD_FLAG_ASYNC 1u /* the `async` constructor argument of Slave / Master (core/Slave.scala:20) */

typedef struct dsgd_ctx dsgd_ctx;

/* ---- lifecycle: `new Slave(node, master, data, model, async)` + `new SparseSVM(lambda, dimSparsity)`
 *      (Main.scala:68,138,149; core/Slave.scala:20; core/ml/SparseSVM.scala:11) ------------------------ */
int dsgd_create(dsgd_ctx **out, int device, int32_t dim, double lambda, int rank, int world, uint32_t flags);
int dsgd_destroy(dsgd_ctx *ctx);
/* Message of the last failing call on ctx (ctx == NULL: last failing dsgd_create on this thread). */
const char *dsgd_last_error(const dsgd_ctx *ctx);
/* Build / device facts as a JSON string (SM count, arch, kernels compiled). */
const char *dsgd_info(const dsgd_ctx *ctx);
/* Use the caller's CUDA stream (a cudaStream_t) for everything the ctx launches; NULL restores the
 * ctx's own stream.  Lets a host time the ctx's kernels with its own events. */
int dsgd_set_stream(dsgd_ctx *ctx, void *cuda_stream);
int dsgd_synchronize(dsgd_ctx *ctx);
/* CUDA-event stopwatch on the ctx's launch stream (what bench.py times kernels with). */
int dsgd_timer_start(dsgd_ctx *ctx);
int dsgd_timer_stop(dsgd_ctx *ctx, float *elapsed_ms);
/* Number of kernels this ctx has launched so far (bench.py's gpu_launches). */
int dsgd_launch_count(const dsgd_ctx *ctx, int64_t *count);

/* Kernel stopwatch for the roofline figure: between begin and end, every sample_every-th launch of the
 * gradient kernel (the dominant kernel of a step) is bracketed by CUDA events on the launch stream; end
 * returns their mean duration and how many launches were sampled. */
int dsgd_profile_begin(dsgd_ctx *ctx, int32_t sample_every);
int dsgd_profile_end(dsgd_ctx *ctx, float *mean_ms, int64_t *n_sampled);
/* Optional: allocate every device buffer the sync path needs for calls of up to n_samples sample ids and n_steps steps
 * now (staging, per-step losses, the persistent kernel's buffers, the exchange's weight words) instead of on first
 * use.  cudaMalloc synchronises the whole device: a host that drives several contexts on ONE GPU from several threads
 * must reserve before the first fused step, or a rank allocating late waits for a rank that already runs and waits for
 * it.  (One context per GPU never needs this.) */
int dsgd_reserve(dsgd_ctx *ctx, int64_t n_samples, int64_t n_steps);
/* CTAs of the persistent sync kernel (0 = one per SM, the default and the fastest).  The kernel is cooperative and its
 * ranks wait for each other, so K contexts that share ONE GPU (the K-rank tests on a single-GPU box: tests/
 * test_gpu_fused_one_gpu.py) must each take at most 1/K of the SMs. */
int dsgd_set_grid_limit(dsgd_ctx *ctx, int32_t n_ctas);
/* Developer aid (tools/timeline.py): with the environment variable DSGD_PERSIST_TIMELINE set, the persistent sync kernel
 * stamps clock64 per phase (CTA 0, 256 steps x 16 slots) and, for steps 100..103, {barrier arrival ns, barrier exit ns,
 * pairs of the CTA's rows, spare} per CTA; this copies the last launch's DSGD_TIMELINE_WORDS int64 words out. */
#define DSGD_TIMELINE_WORDS (256 * 16 + 4 * 160 * 4)
int dsgd_debug_timeline(dsgd_ctx *ctx, long long *out);

/* ---- data: the `data: Array[(Vec, Int)]` constructor argument (core/Slave.scala:20; Main.scala:138,149).
 *      Rows are repacked on the device into 16-byte aligned (col, val) windows.  label in {-1, +1}. ------ */
int dsgd_load_csr(dsgd_ctx *ctx, int64_t n_rows, int64_t nnz, const int64_t *row_ptr, const int32_t *col,
                  const float *val, const int8_t *label);

/* ---- model: SparseSVM.dimSparsity (core/ml/SparseSVM.scala:11).  d is given in the WEIGHT index space. */
int dsgd_set_dim_sparsity(dsgd_ctx *ctx, const double *d);
/* Main.scala:54-65 on the device: inverse (document frequency + 1) over rows [0, n_train), including the
 * reference's off-by-one key shift (quirk Q3).  Installs the result; d_out (optional) receives a copy. */
int dsgd_compute_dim_sparsity(dsgd_ctx *ctx, int64_t n_train, double *d_out);

/* ---- resident weights: GradState.grad on the master (core/ml/GradState.scala:6), `weights` Ref on an
 *      async slave (core/Slave.scala:30) ---------------------------------------------------------------- */
int dsgd_set_weights(dsgd_ctx *ctx, const double *w);
int dsgd_get_weights(dsgd_ctx *ctx, double *w);

/* ---- SlaveImpl.forward (core/Slave.scala:129-140; SparseSVM.scala:14): preds[i] = -signum(x_i . w).
 *      w == NULL: use the resident weights. ----------------------------------------------------------------- */
int dsgd_forward(dsgd_ctx *ctx, const double *w, const int32_t *samples, int64_t n, double *preds_out);

/* ---- SlaveImpl.gradient (core/Slave.scala:142-157; SparseSVM.scala:26-31): grad_out[dim] =
 *      regularize(sum_i backward(w, x_i, y_i), w).  loss_out (optional) = SparseSVM.loss(w, these samples)
 *      (SparseSVM.scala:20-23).  w == NULL: resident weights.  n == 0 -> DSGD_ERR_EMPTY. -------------------- */
int dsgd_gradient(dsgd_ctx *ctx, const double *w, const int32_t *samples, int64_t n, double *grad_out,
                  double *loss_out);

/* ---- Master.localLoss / localAccuracy over rows [row_begin, row_end) (core/Master.scala:100-107): one
 *      streaming pass; loss = lambda*||w||^2 + mean hinge, acc = #{pred == y} / n. ------------------------- */
int dsgd_eval(dsgd_ctx *ctx, const double *w, int64_t row_begin, int64_t row_end, double *loss_out,
              double *acc_out);

/* Sharded form of the same pass: the exact integer sums (hinge losses are 0, 1 or 2 per sample) and
 * ||w||^2, so that a host can combine row shards evaluated on different GPUs without rounding. */
int dsgd_eval_counts(dsgd_ctx *ctx, const double *w, int64_t row_begin, int64_t row_end, int64_t *hinge_sum,
                     int64_t *correct, double *norm_squared);

/* ---- communicator for sync mode: replaces the gRPC channels between master and slaves
 *      (core/package.scala:16-21; core/Master.scala:222-243).  Rank 0 makes an id, the host transports it
 *      (its own RPC), every rank calls dsgd_comm_init.  world == 1 needs neither. -------------------------- */
int dsgd_comm_unique_id(uint8_t id[DSGD_UNIQUE_ID_BYTES]);
int dsgd_comm_init(dsgd_ctx *ctx, const uint8_t id[DSGD_UNIQUE_ID_BYTES]);

/* Peer exchange for the FUSED multi-GPU step: each rank exports its receive area, the host transports the handles, every rank imports every other rank's.  Once all world-1 peers
 * are attached, sync steps with one worker per GPU run as one persistent kernel per call that sums the workers'
 * replies directly out of peer memory over NVLink (no NCCL call, no launch per step; only the non-zero entries of a
 * reply travel); otherwise the NCCL allreduce path is used.  Up to 8 ranks (one NVSwitch box).  dsgd_xchg_attach is
 * the same-process form. */
int dsgd_xchg_export(dsgd_ctx *ctx, uint8_t handle[DSGD_IPC_HANDLE_BYTES]);
int dsgd_xchg_import(dsgd_ctx *ctx, int peer_rank, const uint8_t handle[DSGD_IPC_HANDLE_BYTES]);
int dsgd_xchg_attach(dsgd_ctx *ctx, int peer_rank, dsgd_ctx *peer);
/* Traffic of the fused step so far, for the NVLink figures of the bench: words this rank has stored into EACH peer's
 * receive area (a value word is 16 bytes on the wire -- one non-zero gradient entry --, a bitmap word 8 bytes -- which of
 * 32 columns were sent) and the SGD steps of those launches.  Any pointer may be NULL. */
int dsgd_xchg_stats(dsgd_ctx *ctx, int64_t *value_words, int64_t *bitmap_words, int64_t *steps);

/* ---- logical workers of a sync step.  Default: this ctx is ONE worker (its whole slice is one
 *      GradientRequest) and the master averages over `world` results.  With n_local > 1 the slice of every
 *      following step is cut into n_local consecutive requests of counts[v] samples, each with its own batch
 *      sum and its own regularize() support, exactly as if n_local slaves had answered (core/Slave.scala:
 *      147-155); k_total is the number of results the master averages (Vec.mean divisor, core/Master.scala:194
 *      -- the reference zips workers with split groups, so it can be smaller than the node count).
 *      n_local == 0: this rank only joins the exchange (a slave without a split group). ---------------- */
int dsgd_set_workers(dsgd_ctx *ctx, int32_t n_local, const int32_t *counts, int32_t k_total);

/* ---- one synchronous step of Master.fit (core/Master.scala:184-197): this rank's worker computes its
 *      regularized batch-sum gradient on `samples`, gradients are summed over ranks (allreduce over NVLink
 *      instead of K gRPC replies), and every rank applies w <- w - lr * (sum / world).  All ranks call it with
 *      their own slice.  loss_out (optional) = SparseSVM.loss(w_before, all samples of the step). ------------ */
int dsgd_sync_step(dsgd_ctx *ctx, const int32_t *samples, int64_t n, double lr, double *loss_out);
/* n_steps consecutive steps (the inner loop of an epoch, core/Master.scala:179): samples holds
 * n_steps * n_per_step indices, step-major.  losses_out (optional) holds n_steps values. */
int dsgd_sync_steps(dsgd_ctx *ctx, const int32_t *samples, int64_t n_per_step, int64_t n_steps, double lr,
                    double *losses_out);
/* The same split in three, so a host can keep the index stream resident: stage = H2D of the sample slices
 * (the `samples` field of GradientRequest, protobuf/proto.proto:60-63); run = device only; read = D2H. */
int dsgd_stage_samples(dsgd_ctx *ctx, const int32_t *samples, int64_t n);
int dsgd_sync_steps_staged(dsgd_ctx *ctx, int64_t first, int64_t n_per_step, int64_t n_steps, double lr,
                           int want_losses);
int dsgd_read_losses(dsgd_ctx *ctx, double *losses_out, int64_t n_steps);

/* ---- model sets: several SparseSVMs, each with its own lambda and learning rate, trained on the SAME batch draws.
 *      The reference trains one `new SparseSVM(config.lambda, ...)` per run (Main.scala:68) with the batch loop of
 *      Master.fit (core/Master.scala:179-198); a lambda / learning-rate sweep reruns everything.  A model set runs the
 *      steps of all its models in one persistent kernel per call: they share the sample ids, the row loads, the launch
 *      and one grid barrier per step.  One GPU and one worker per step (world == 1, the default dsgd_set_workers);
 *      at most 32 samples per SM and step.  Each model follows exactly the arithmetic of dsgd_sync_steps with its own
 *      lambda and lr.  Model-set calls leave the ctx's resident weights (dsgd_get_weights) untouched. */
#define DSGD_MAX_MODELS 32
/* Replace the ctx's model set (n_models == 0 frees it).  lambda, lr: [n_models]; lambda finite and >= 0, lr finite.
 * w0: [n_models * dim] initial weights, model-major, or NULL (zeros). */
int dsgd_models_set(dsgd_ctx *ctx, int32_t n_models, const double *lambda, const double *lr, const double *w0);
/* n_models of the current set (0: none) and dim, so that a binding can size its buffers. */
int dsgd_models_shape(const dsgd_ctx *ctx, int32_t *n_models, int32_t *dim);
/* w_out: [n_models * dim], model-major. */
int dsgd_models_get_weights(dsgd_ctx *ctx, double *w_out);
/* n_steps steps of every active model on the same samples (n_steps * n_per_step ids, step-major, like dsgd_sync_steps).
 * active: [n_models], non-zero = takes part, or NULL (all); a frozen model keeps its weights bit for bit.
 * losses_out: [n_steps * n_models] step-major (SparseSVM.loss at the pre-step weights; NaN for frozen models) or NULL.
 * Several calls in a row continue one trajectory per model. */
int dsgd_models_steps(dsgd_ctx *ctx, const int32_t *samples, int64_t n_per_step, int64_t n_steps, const uint8_t *active,
                      double *losses_out);
/* dsgd_eval_counts over rows [row_begin, row_end) for model m's resident weights. */
int dsgd_models_eval_counts(dsgd_ctx *ctx, int32_t m, int64_t row_begin, int64_t row_end, int64_t *hinge_sum,
                            int64_t *correct, double *norm_squared);

/* ---- async (Hogwild) mode.  Every worker keeps its own weight replica (core/Slave.scala:30) and pushes each
 *      delta to every peer replica and to the master's replica (core/Slave.scala:101-105).  Here replicas are
 *      reached by ADDRESS over NVLink: a rank exports its replica, the host transports the handle, peers import
 *      it and the device loop issues system-scope fp64 reductions (red.add) straight into peer memory.
 *      Replaces the slave<->slave and slave->master channels (core/Slave.scala:23,26; core/Master.scala:
 *      229-233).  `which`: DSGD_REPLICA_SELF = this worker's replica; DSGD_REPLICA_MASTER = the master's replica
 *      (GradState.grad + the update counter, core/MasterAsync.scala:66,164-177), hosted by the ctx that calls
 *      dsgd_async_host_master.  peer_rank in dsgd_ipc_import: 0..world-1, or `world` for the master replica. */
#define DSGD_REPLICA_SELF 0
#define DSGD_REPLICA_MASTER 1
int dsgd_async_host_master(dsgd_ctx *ctx, const double *w0);
int dsgd_ipc_export(dsgd_ctx *ctx, int which, uint8_t handle[DSGD_IPC_HANDLE_BYTES]);
int dsgd_ipc_import(dsgd_ctx *ctx, int peer_rank, const uint8_t handle[DSGD_IPC_HANDLE_BYTES]);
/* Same-process peers (several ctxs in one host process, e.g. a JVM driving all GPUs of a box): attach by ctx. */
int dsgd_peer_attach(dsgd_ctx *ctx, int peer_rank, dsgd_ctx *peer, int which);
/* SlaveImpl.startAsync (core/Slave.scala:159-175): weights := w0, then the worker loop (asyncTask,
 * core/Slave.scala:79-111) runs on the device until dsgd_stop_async or until this worker has made max_updates
 * updates (0: unbounded).  concurrency = Hogwild lanes on this GPU (warps running the loop body concurrently on
 * the shared replica; 1 = the reference's strictly sequential loop).  seed drives the device-side sampling of
 * `assigned` (core/Slave.scala:84,87; batch > 1 indexes rows by POSITION like the reference, quirk Q6).
 * w0 == NULL keeps the resident replica: initialise every replica with dsgd_set_weights first, then start the
 * loops, and no delta a faster peer pushes early is overwritten (the reference has that start-up race).
 * Returns immediately; the loop runs on its own stream. */
int dsgd_start_async(dsgd_ctx *ctx, const double *w0, const int32_t *assigned, int64_t n_assigned, int32_t batch,
                     double lr, int32_t concurrency, int64_t max_updates, uint64_t seed);
/* The same loop body over a RECORDED sampling sequence (n_updates * batch row ids), one lane, blocking: the
 * deterministic K = 1 case of core/Slave.scala:79-111, used to replay a reference run and by the parity tests. */
int dsgd_async_replay(dsgd_ctx *ctx, const double *w0, const int32_t *samples, int32_t batch, int64_t n_updates,
                      double lr);
/* SlaveImpl.stopAsync (core/Slave.scala:187-195): raises the stop flag and waits for the loop to drain. */
int dsgd_stop_async(dsgd_ctx *ctx);
/* 1 while the device loop is running (it also ends by itself after max_updates). */
int dsgd_async_running(dsgd_ctx *ctx, int *running);
/* Device time of the last finished async loop (CUDA events on the loop's stream), for benchmarks. */
int dsgd_async_elapsed_ms(dsgd_ctx *ctx, float *elapsed_ms);
/* SlaveImpl.updateGrad / AsyncMasterGrpcImpl.updateGrad (core/Slave.scala:177-185; core/MasterAsync.scala:
 * 164-177): weights -= delta for a sparse delta given as (idx, val) pairs, applied to this context's own replica (a host-side
 * sender -- e.g. a gRPC colleague -- uses it; GPU peers write the replica directly over NVLink). */
int dsgd_update_grad(dsgd_ctx *ctx, const int32_t *idx, const double *val, int64_t nnz);
/* GradState.updates (core/ml/GradState.scala:8; core/MasterAsync.scala:165): updates the master replica has
 * received if this ctx hosts or has imported it, else the updates this worker has made. */
int dsgd_async_updates(dsgd_ctx *ctx, int64_t *count);
/* Snapshot of the master replica (gradState.single().grad, core/MasterAsync.scala:109). */
int dsgd_async_master_weights(dsgd_ctx *ctx, double *w_out);
/* Colleagues that are NOT GPU peers (reference JVM slaves or a JVM master reached over gRPC, core/Slave.scala:104-105): the
 * worker loop adds every -delta it applies to one more replica-shaped accumulator, the OUTBOX.  The host reads it while the
 * loop runs and forwards the difference since its last read as ONE updateGrad message (w -= sum of the deltas of the period:
 * the reference sends one message per iteration; Hogwild's additions commute).  Enable before dsgd_start_async (zeroes the
 * accumulator); acc_out[dim] = sum of -delta since then.  dsgd_async_outbox_read is safe while the loop runs. */
int dsgd_async_outbox_enable(dsgd_ctx *ctx);
int dsgd_async_outbox_read(dsgd_ctx *ctx, double *acc_out);

#ifdef __cplusplus
}
#endif
#endif /* DSGD_H */
