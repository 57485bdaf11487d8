/* JNI shim between epfl.distributed.nativ.DsgdNative (Scala, see DsgdNative.scala) and the C ABI of
 * include/dsgd.h.  Compile-gated: the build image has no JDK (no jni.h); on a box with one:
 *   gcc -shared -fPIC -I$JAVA_HOME/include -I$JAVA_HOME/include/linux -I../../include \
 *       -o libdsgd_jni.so dsgd_jni.c -L.. -ldsgd
 *
 * Every C-ABI call that touches the GPU BLOCKS (it synchronises a CUDA stream; a fused multi-GPU step even waits for
 * the other ranks' threads to launch), so no array is ever pinned across one: inputs are copied out with
 * Get<Type>ArrayRegion before the call and outputs copied back with Set<Type>ArrayRegion after it.  (JNI forbids
 * blocking inside a GetPrimitiveArrayCritical region -- it stalls the collector for the whole JVM, and with several
 * contexts driven from several JVM threads it can deadlock: rank A's kernel waits for rank B's launch while B's thread
 * waits for the collector that A's critical region holds off.)  A NULL array is passed on as NULL / length 0.
 *
 * tests/test_abi_surface.py compiles this file against a minimal stand-in jni.h (tests/jni_mock/) -- a syntax and type
 * check against include/dsgd.h, not a run under a JVM -- and checks that the facade covers the header. */
#ifdef DSGD_HAVE_JNI
#include <jni.h>
#include <stddef.h>
#include <stdint.h>
#include <stdlib.h>
#include "dsgd.h"

#define CTX(h) ((dsgd_ctx *)(intptr_t)(h))
#define FN(name) JNIEXPORT jint JNICALL Java_epfl_distributed_nativ_DsgdNative_00024_##name

/* copy of a Java array in C memory (in), or a C buffer of the array's length to be copied back (out) */
typedef struct { void *p; jsize n; int bad; } buf_t;
#define DEF_BUF(Name, JT, CT)                                                                                  \
  static __attribute__((unused)) buf_t in_##Name(JNIEnv *env, JT##Array a) {                                                             \
    buf_t b = {NULL, 0, 0};                                                                                      \
    if (!a) return b;                                                                                            \
    b.n = (*env)->GetArrayLength(env, a);                                                                        \
    b.p = malloc(sizeof(CT) * (size_t)(b.n > 0 ? b.n : 1));                                                      \
    if (!b.p) { b.bad = 1; return b; }                                                                           \
    if (b.n > 0) (*env)->Get##Name##ArrayRegion(env, a, 0, b.n, (JT *)b.p);                                      \
    return b;                                                                                                    \
  }                                                                                                              \
  static __attribute__((unused)) buf_t out_##Name(JNIEnv *env, JT##Array a) {                                                            \
    buf_t b = {NULL, 0, 0};                                                                                      \
    if (!a) return b;                                                                                            \
    b.n = (*env)->GetArrayLength(env, a);                                                                        \
    b.p = calloc((size_t)(b.n > 0 ? b.n : 1), sizeof(CT));                                                       \
    if (!b.p) b.bad = 1;                                                                                         \
    return b;                                                                                                    \
  }                                                                                                              \
  static __attribute__((unused)) void back_##Name(JNIEnv *env, JT##Array a, buf_t b, int rc) {                                           \
    if (a && b.p && rc == DSGD_OK && b.n > 0) (*env)->Set##Name##ArrayRegion(env, a, 0, b.n, (const JT *)b.p);   \
    free(b.p);                                                                                                   \
  }
DEF_BUF(Int, jint, int32_t)
DEF_BUF(Long, jlong, int64_t)
DEF_BUF(Float, jfloat, float)
DEF_BUF(Double, jdouble, double)
DEF_BUF(Byte, jbyte, int8_t)

/* ---- lifecycle ---- */
JNIEXPORT jlong JNICALL Java_epfl_distributed_nativ_DsgdNative_00024_create(JNIEnv *env, jobject self, jint device, jint dim,
                                                                          jdouble lambda, jint rank, jint world, jint flags) {
  dsgd_ctx *ctx = NULL;
  int rc = dsgd_create(&ctx, device, dim, lambda, rank, world, (uint32_t)flags);   /* new Slave(...) + SparseSVM(lambda, .) */
  return rc == DSGD_OK ? (jlong)(intptr_t)ctx : (jlong)rc; /* negative = error code */
}
FN(destroy)(JNIEnv *env, jobject self, jlong h) { return dsgd_destroy(CTX(h)); }
JNIEXPORT jstring JNICALL Java_epfl_distributed_nativ_DsgdNative_00024_lastError(JNIEnv *env, jobject self, jlong h) {
  return (*env)->NewStringUTF(env, dsgd_last_error(CTX(h)));
}

/* ---- data / model ---- */
FN(loadCsr)(JNIEnv *env, jobject self, jlong h, jlongArray rowPtr, jintArray col, jfloatArray value, jbyteArray label) {
  buf_t rp = in_Long(env, rowPtr), c = in_Int(env, col), v = in_Float(env, value), l = in_Byte(env, label);
  int rc = DSGD_ERR_NOMEM;                               /* Dataset.rcv1 rows as CSR (utils/Dataset.scala:23-47) */
  if (!(rp.bad | c.bad | v.bad | l.bad))
    rc = rp.n < 1 ? DSGD_ERR_INVALID : dsgd_load_csr(CTX(h), rp.n - 1, c.n, rp.p, c.p, v.p, l.p);
  free(rp.p); free(c.p); free(v.p); free(l.p);
  return rc;
}
FN(setDimSparsity)(JNIEnv *env, jobject self, jlong h, jdoubleArray d) {
  buf_t b = in_Double(env, d);
  int rc = b.bad ? DSGD_ERR_NOMEM : dsgd_set_dim_sparsity(CTX(h), b.p);            /* SparseSVM.dimSparsity */
  free(b.p);
  return rc;
}
FN(computeDimSparsity)(JNIEnv *env, jobject self, jlong h, jlong nTrain, jdoubleArray out) {
  buf_t o = out_Double(env, out);
  int rc = o.bad ? DSGD_ERR_NOMEM : dsgd_compute_dim_sparsity(CTX(h), nTrain, o.p); /* Main.scala:54-65 */
  back_Double(env, out, o, rc);
  return rc;
}
FN(setWeights)(JNIEnv *env, jobject self, jlong h, jdoubleArray w) {
  buf_t b = in_Double(env, w);
  int rc = b.bad ? DSGD_ERR_NOMEM : dsgd_set_weights(CTX(h), b.p);
  free(b.p);
  return rc;
}
FN(getWeights)(JNIEnv *env, jobject self, jlong h, jdoubleArray w) {
  buf_t o = out_Double(env, w);
  int rc = o.bad ? DSGD_ERR_NOMEM : dsgd_get_weights(CTX(h), o.p);
  back_Double(env, w, o, rc);
  return rc;
}

/* ---- requests ---- */
FN(gradient)(JNIEnv *env, jobject self, jlong h, jdoubleArray w, jintArray samples, jdoubleArray grad) {
  buf_t bw = in_Double(env, w), bs = in_Int(env, samples), bg = out_Double(env, grad);
  int rc = DSGD_ERR_NOMEM;
  if (!(bw.bad | bs.bad | bg.bad)) rc = dsgd_gradient(CTX(h), bw.p, bs.p, bs.n, bg.p, NULL);  /* core/Slave.scala:142-157 */
  back_Double(env, grad, bg, rc);
  free(bw.p); free(bs.p);
  return rc;
}
FN(forward)(JNIEnv *env, jobject self, jlong h, jdoubleArray w, jintArray samples, jdoubleArray preds) {
  buf_t bw = in_Double(env, w), bs = in_Int(env, samples), bp = out_Double(env, preds);
  int rc = DSGD_ERR_NOMEM;
  if (!(bw.bad | bs.bad | bp.bad)) rc = dsgd_forward(CTX(h), bw.p, bs.p, bs.n, bp.p);          /* core/Slave.scala:129-140 */
  back_Double(env, preds, bp, rc);
  free(bw.p); free(bs.p);
  return rc;
}
FN(eval)(JNIEnv *env, jobject self, jlong h, jdoubleArray w, jlong rowBegin, jlong rowEnd, jdoubleArray lossAcc) {
  buf_t bw = in_Double(env, w), bo = out_Double(env, lossAcc);          /* lossAcc(0) = loss, lossAcc(1) = accuracy */
  int rc = DSGD_ERR_NOMEM;
  if (!(bw.bad | bo.bad))
    rc = bo.n < 2 ? DSGD_ERR_INVALID
                  : dsgd_eval(CTX(h), bw.p, rowBegin, rowEnd, (double *)bo.p, (double *)bo.p + 1);  /* core/Master.scala:100-107 */
  back_Double(env, lossAcc, bo, rc);
  free(bw.p);
  return rc;
}
FN(evalCounts)(JNIEnv *env, jobject self, jlong h, jdoubleArray w, jlong rowBegin, jlong rowEnd, jlongArray hingeCorrect,
               jdoubleArray normSquared) {
  buf_t bw = in_Double(env, w), bc = out_Long(env, hingeCorrect), bn = out_Double(env, normSquared);
  int rc = DSGD_ERR_NOMEM;               /* exact shardable form: hingeCorrect(0) = hinge sum, (1) = #correct */
  if (!(bw.bad | bc.bad | bn.bad))
    rc = (bc.n < 2 || bn.n < 1) ? DSGD_ERR_INVALID
                                : dsgd_eval_counts(CTX(h), bw.p, rowBegin, rowEnd, (int64_t *)bc.p, (int64_t *)bc.p + 1, bn.p);
  back_Long(env, hingeCorrect, bc, rc);
  back_Double(env, normSquared, bn, rc);
  free(bw.p);
  return rc;
}

/* ---- sync mode ---- */
FN(commUniqueId)(JNIEnv *env, jobject self, jbyteArray id) {
  buf_t b = out_Byte(env, id);
  int rc = b.bad ? DSGD_ERR_NOMEM : (b.n < DSGD_UNIQUE_ID_BYTES ? DSGD_ERR_INVALID : dsgd_comm_unique_id((uint8_t *)b.p));
  back_Byte(env, id, b, rc);
  return rc;
}
FN(commInit)(JNIEnv *env, jobject self, jlong h, jbyteArray id) {
  buf_t b = in_Byte(env, id);
  int rc = b.bad ? DSGD_ERR_NOMEM : (b.n < DSGD_UNIQUE_ID_BYTES ? DSGD_ERR_INVALID : dsgd_comm_init(CTX(h), (const uint8_t *)b.p));
  free(b.p);
  return rc;
}
FN(xchgExport)(JNIEnv *env, jobject self, jlong h, jbyteArray handle) {
  buf_t b = out_Byte(env, handle);
  int rc = b.bad ? DSGD_ERR_NOMEM : (b.n < DSGD_IPC_HANDLE_BYTES ? DSGD_ERR_INVALID : dsgd_xchg_export(CTX(h), (uint8_t *)b.p));
  back_Byte(env, handle, b, rc);
  return rc;
}
FN(xchgImport)(JNIEnv *env, jobject self, jlong h, jint peerRank, jbyteArray handle) {
  buf_t b = in_Byte(env, handle);
  int rc = b.bad ? DSGD_ERR_NOMEM
                 : (b.n < DSGD_IPC_HANDLE_BYTES ? DSGD_ERR_INVALID : dsgd_xchg_import(CTX(h), peerRank, (const uint8_t *)b.p));
  free(b.p);
  return rc;
}
/* one JVM driving all GPUs of the box: the Master's slave list (core/Master.scala:222-243) becomes attach calls */
FN(xchgAttach)(JNIEnv *env, jobject self, jlong h, jint peerRank, jlong peer) { return dsgd_xchg_attach(CTX(h), peerRank, CTX(peer)); }
FN(xchgStats)(JNIEnv *env, jobject self, jlong h, jlongArray out) {   /* out(0) value words, (1) bitmap words, (2) steps */
  buf_t b = out_Long(env, out);
  int rc = b.bad ? DSGD_ERR_NOMEM
                 : (b.n < 3 ? DSGD_ERR_INVALID : dsgd_xchg_stats(CTX(h), (int64_t *)b.p, (int64_t *)b.p + 1, (int64_t *)b.p + 2));
  back_Long(env, out, b, rc);
  return rc;
}
FN(setWorkers)(JNIEnv *env, jobject self, jlong h, jintArray counts, jint kTotal) {
  buf_t b = in_Int(env, counts);
  int rc = b.bad ? DSGD_ERR_NOMEM : dsgd_set_workers(CTX(h), b.n, b.p, kTotal);
  free(b.p);
  return rc;
}
FN(syncSteps)(JNIEnv *env, jobject self, jlong h, jintArray samples, jlong n_per_step, jlong n_steps, jdouble lr,
              jdoubleArray losses) {
  buf_t bs = in_Int(env, samples), bl = out_Double(env, losses);
  int rc = DSGD_ERR_NOMEM;
  if (!(bs.bad | bl.bad)) {
    if ((jlong)bs.n < n_per_step * n_steps || (bl.p && (jlong)bl.n < n_steps)) rc = DSGD_ERR_INVALID;
    else rc = dsgd_sync_steps(CTX(h), bs.p, n_per_step, n_steps, lr, bl.p);   /* Master.fit's batch loop, core/Master.scala:179-198 */
  }
  back_Double(env, losses, bl, rc);
  free(bs.p);
  return rc;
}

/* ---- model sets: one SparseSVM per (lambda, lr) setting on the same draws (Main.scala:68; core/Master.scala:179-198).
 *      Every Java array is checked against the set's n_models, dim and n_steps * n_models before the ABI sees it; the
 *      products are formed in 64 bits after their factors are bounded. */
static int models_shape(jlong h, int64_t *n_models, int64_t *dim) {
  int32_t n = 0, d = 0;
  int rc = dsgd_models_shape(CTX(h), &n, &d);
  *n_models = n; *dim = d;
  return rc;
}
FN(modelsShape)(JNIEnv *env, jobject self, jlong h, jintArray out) {   /* out(0) n_models, (1) dim */
  buf_t b = out_Int(env, out);
  int rc = b.bad ? DSGD_ERR_NOMEM : (b.n < 2 ? DSGD_ERR_INVALID : dsgd_models_shape(CTX(h), (int32_t *)b.p, (int32_t *)b.p + 1));
  back_Int(env, out, b, rc);
  return rc;
}
FN(modelsSet)(JNIEnv *env, jobject self, jlong h, jdoubleArray lambda, jdoubleArray lr, jdoubleArray w0) {
  int64_t n_old = 0, dim = 0;
  int rc = models_shape(h, &n_old, &dim);
  if (rc != DSGD_OK) return rc;
  const jsize n = lambda ? (*env)->GetArrayLength(env, lambda) : 0;
  const jsize n_lr = lr ? (*env)->GetArrayLength(env, lr) : 0;
  if (n > DSGD_MAX_MODELS || n_lr != n) return DSGD_ERR_INVALID;
  if (w0 && (int64_t)(*env)->GetArrayLength(env, w0) != (int64_t)n * dim) return DSGD_ERR_INVALID;
  buf_t bl = in_Double(env, lambda), br = in_Double(env, lr), bw = in_Double(env, w0);
  rc = DSGD_ERR_NOMEM;
  if (!(bl.bad | br.bad | bw.bad)) rc = dsgd_models_set(CTX(h), (int32_t)n, bl.p, br.p, bw.p);
  free(bl.p); free(br.p); free(bw.p);
  return rc;
}
FN(modelsGetWeights)(JNIEnv *env, jobject self, jlong h, jdoubleArray out) {   /* out: n_models * dim, model-major */
  int64_t n = 0, dim = 0;
  int rc = models_shape(h, &n, &dim);
  if (rc != DSGD_OK) return rc;
  if (!out || (int64_t)(*env)->GetArrayLength(env, out) != n * dim) return DSGD_ERR_INVALID;
  buf_t b = out_Double(env, out);
  rc = b.bad ? DSGD_ERR_NOMEM : dsgd_models_get_weights(CTX(h), b.p);
  back_Double(env, out, b, rc);
  return rc;
}
FN(modelsSteps)(JNIEnv *env, jobject self, jlong h, jintArray samples, jlong n_per_step, jlong n_steps, jbyteArray active,
                jdoubleArray losses) {
  int64_t n = 0, dim = 0;
  int rc = models_shape(h, &n, &dim);
  if (rc != DSGD_OK) return rc;
  if (n_per_step < 0 || n_steps < 0) return DSGD_ERR_INVALID;
  if (n_steps > 0 && n_per_step > INT64_MAX / n_steps) return DSGD_ERR_INVALID;
  const int64_t n_ids = n_per_step * n_steps;   /* n <= DSGD_MAX_MODELS: n_steps * n overflows only for absurd n_steps */
  if (n > 0 && n_steps > INT64_MAX / n) return DSGD_ERR_INVALID;
  if ((int64_t)(samples ? (*env)->GetArrayLength(env, samples) : 0) < n_ids) return DSGD_ERR_INVALID;
  if (active && (int64_t)(*env)->GetArrayLength(env, active) != n) return DSGD_ERR_INVALID;
  if (losses && (int64_t)(*env)->GetArrayLength(env, losses) < n_steps * n) return DSGD_ERR_INVALID;
  buf_t bs = in_Int(env, samples), ba = in_Byte(env, active), bl = out_Double(env, losses);
  rc = DSGD_ERR_NOMEM;
  if (!(bs.bad | ba.bad | bl.bad))
    rc = dsgd_models_steps(CTX(h), bs.p, n_per_step, n_steps, (const uint8_t *)ba.p, bl.p);  /* losses: step-major */
  back_Double(env, losses, bl, rc);
  free(bs.p); free(ba.p);
  return rc;
}
FN(modelsEvalCounts)(JNIEnv *env, jobject self, jlong h, jint m, jlong rowBegin, jlong rowEnd, jlongArray hingeCorrect,
                     jdoubleArray normSquared) {
  buf_t bc = out_Long(env, hingeCorrect), bn = out_Double(env, normSquared);
  int rc = DSGD_ERR_NOMEM;               /* hingeCorrect(0) = hinge sum, (1) = #correct of model m */
  if (!(bc.bad | bn.bad))
    rc = (bc.n < 2 || bn.n < 1) ? DSGD_ERR_INVALID
                                : dsgd_models_eval_counts(CTX(h), m, rowBegin, rowEnd, (int64_t *)bc.p, (int64_t *)bc.p + 1, bn.p);
  back_Long(env, hingeCorrect, bc, rc);
  back_Double(env, normSquared, bn, rc);
  return rc;
}

/* ---- async (Hogwild) mode ---- */
FN(asyncHostMaster)(JNIEnv *env, jobject self, jlong h, jdoubleArray w0) {
  buf_t b = in_Double(env, w0);
  int rc = b.bad ? DSGD_ERR_NOMEM : dsgd_async_host_master(CTX(h), b.p);   /* GradState of MasterAsync, core/MasterAsync.scala:66 */
  free(b.p);
  return rc;
}
FN(ipcExport)(JNIEnv *env, jobject self, jlong h, jint which, jbyteArray handle) {
  buf_t b = out_Byte(env, handle);
  int rc = b.bad ? DSGD_ERR_NOMEM : (b.n < DSGD_IPC_HANDLE_BYTES ? DSGD_ERR_INVALID : dsgd_ipc_export(CTX(h), which, (uint8_t *)b.p));
  back_Byte(env, handle, b, rc);
  return rc;
}
FN(ipcImport)(JNIEnv *env, jobject self, jlong h, jint peerRank, jbyteArray handle) {
  buf_t b = in_Byte(env, handle);
  int rc = b.bad ? DSGD_ERR_NOMEM
                 : (b.n < DSGD_IPC_HANDLE_BYTES ? DSGD_ERR_INVALID : dsgd_ipc_import(CTX(h), peerRank, (const uint8_t *)b.p));
  free(b.p);
  return rc;
}
FN(peerAttach)(JNIEnv *env, jobject self, jlong h, jint peerRank, jlong peer, jint which) {
  return dsgd_peer_attach(CTX(h), peerRank, CTX(peer), which);             /* the slave<->slave channels, core/Slave.scala:23,26 */
}
FN(startAsync)(JNIEnv *env, jobject self, jlong h, jdoubleArray w0, jintArray assigned, jint batch, jdouble lr,
               jint concurrency, jlong maxUpdates, jlong seed) {
  buf_t bw = in_Double(env, w0), ba = in_Int(env, assigned);
  int rc = DSGD_ERR_NOMEM;
  if (!(bw.bad | ba.bad))
    rc = dsgd_start_async(CTX(h), bw.p, ba.p, ba.n, batch, lr, concurrency, maxUpdates, (uint64_t)seed);  /* core/Slave.scala:159-175 */
  free(bw.p); free(ba.p);
  return rc;
}
FN(stopAsync)(JNIEnv *env, jobject self, jlong h) { return dsgd_stop_async(CTX(h)); }   /* core/Slave.scala:187-195 */
FN(asyncRunning)(JNIEnv *env, jobject self, jlong h, jintArray out) {
  buf_t b = out_Int(env, out);
  int rc = b.bad ? DSGD_ERR_NOMEM : (b.n < 1 ? DSGD_ERR_INVALID : dsgd_async_running(CTX(h), (int *)b.p));
  back_Int(env, out, b, rc);
  return rc;
}
FN(updateGrad)(JNIEnv *env, jobject self, jlong h, jintArray idx, jdoubleArray value) {
  buf_t bi = in_Int(env, idx), bv = in_Double(env, value);
  int rc = DSGD_ERR_NOMEM;
  if (!(bi.bad | bv.bad)) rc = bi.n != bv.n ? DSGD_ERR_INVALID : dsgd_update_grad(CTX(h), bi.p, bv.p, bi.n);  /* core/Slave.scala:177-185 */
  free(bi.p); free(bv.p);
  return rc;
}
FN(asyncUpdates)(JNIEnv *env, jobject self, jlong h, jlongArray out) {
  buf_t b = out_Long(env, out);
  int rc = b.bad ? DSGD_ERR_NOMEM : (b.n < 1 ? DSGD_ERR_INVALID : dsgd_async_updates(CTX(h), (int64_t *)b.p));  /* GradState.updates */
  back_Long(env, out, b, rc);
  return rc;
}
FN(asyncMasterWeights)(JNIEnv *env, jobject self, jlong h, jdoubleArray out) {
  buf_t b = out_Double(env, out);
  int rc = b.bad ? DSGD_ERR_NOMEM : dsgd_async_master_weights(CTX(h), b.p);   /* gradState.single().grad, core/MasterAsync.scala:109 */
  back_Double(env, out, b, rc);
  return rc;
}
FN(asyncOutboxEnable)(JNIEnv *env, jobject self, jlong h) {
  (void)env; (void)self;
  return dsgd_async_outbox_enable(CTX(h));            /* deltas for colleagues reached over gRPC, core/Slave.scala:104-105 */
}
FN(asyncOutboxRead)(JNIEnv *env, jobject self, jlong h, jdoubleArray out) {
  buf_t b = out_Double(env, out);
  int rc = b.bad ? DSGD_ERR_NOMEM : (b.n < 1 ? DSGD_ERR_INVALID : dsgd_async_outbox_read(CTX(h), b.p));
  back_Double(env, out, b, rc);
  return rc;
}
#endif /* DSGD_HAVE_JNI */
