// Scala facade over libdsgd_jni.so -> libdsgd.so (include/dsgd.h).  NOT compiled in this repository: the build
// image has no JVM toolchain (no javac / scalac / sbt / jni.h).  It is the binding a maintainer of
// zifeo/distributed-sgd would add under src/main/scala/epfl/distributed/nativ/.
package epfl.distributed.nativ

import epfl.distributed.math.Vec

object DsgdNative {
  System.loadLibrary("dsgd_jni") // links against libdsgd.so

  // every native returns the C ABI's status code; 0 = OK, negative = DSGD_ERR_*  (include/dsgd.h).  Arrays are copied in
  // before and out after the call (Get/Set<Type>ArrayRegion): nothing is pinned while a call blocks on the GPU.
  @native def create(device: Int, dim: Int, lambda: Double, rank: Int, world: Int, flags: Int): Long
  @native def destroy(ctx: Long): Int
  @native def lastError(ctx: Long): String
  // data / model
  @native def loadCsr(ctx: Long, rowPtr: Array[Long], col: Array[Int], value: Array[Float], label: Array[Byte]): Int
  @native def setDimSparsity(ctx: Long, d: Array[Double]): Int
  @native def computeDimSparsity(ctx: Long, nTrain: Long, out: Array[Double]): Int
  @native def setWeights(ctx: Long, w: Array[Double]): Int
  @native def getWeights(ctx: Long, w: Array[Double]): Int
  // SlaveImpl.forward / gradient, Master.localLoss / localAccuracy (w == null: the resident weights)
  @native def forward(ctx: Long, w: Array[Double], samples: Array[Int], preds: Array[Double]): Int
  @native def gradient(ctx: Long, w: Array[Double], samples: Array[Int], grad: Array[Double]): Int
  @native def eval(ctx: Long, w: Array[Double], rowBegin: Long, rowEnd: Long, lossAcc: Array[Double]): Int
  @native def evalCounts(ctx: Long, w: Array[Double], rowBegin: Long, rowEnd: Long, hingeCorrect: Array[Long],
                         normSquared: Array[Double]): Int
  // sync mode: cluster membership (core/Master.scala:222-243) becomes attach / import calls; the step loop one call
  @native def commUniqueId(id: Array[Byte]): Int                       // 128 bytes; rank 0 makes it, every rank commInit()s it
  @native def commInit(ctx: Long, id: Array[Byte]): Int
  @native def xchgExport(ctx: Long, handle: Array[Byte]): Int          // 64 bytes; one JVM per GPU: ship it over the node's gRPC
  @native def xchgImport(ctx: Long, peerRank: Int, handle: Array[Byte]): Int
  @native def xchgAttach(ctx: Long, peerRank: Int, peerCtx: Long): Int // one JVM driving all GPUs of the box
  @native def xchgStats(ctx: Long, out: Array[Long]): Int
  @native def setWorkers(ctx: Long, counts: Array[Int], kTotal: Int): Int
  @native def syncSteps(ctx: Long, samples: Array[Int], nPerStep: Long, nSteps: Long, lr: Double, losses: Array[Double]): Int
  // model sets: one SparseSVM per (lambda(m), lr(m)) on the same draws; weights / losses are model-major / step-major
  @native def modelsSet(ctx: Long, lambda: Array[Double], lr: Array[Double], w0: Array[Double]): Int  // w0 == null: zeros
  @native def modelsShape(ctx: Long, out: Array[Int]): Int             // out(0) models, out(1) dim
  @native def modelsGetWeights(ctx: Long, out: Array[Double]): Int     // models * dim
  @native def modelsSteps(ctx: Long, samples: Array[Int], nPerStep: Long, nSteps: Long, active: Array[Byte],
                          losses: Array[Double]): Int                  // active == null: all; losses: nSteps * models
  @native def modelsEvalCounts(ctx: Long, m: Int, rowBegin: Long, rowEnd: Long, hingeCorrect: Array[Long],
                               normSquared: Array[Double]): Int
  // async (Hogwild) mode
  @native def asyncHostMaster(ctx: Long, w0: Array[Double]): Int
  @native def ipcExport(ctx: Long, which: Int, handle: Array[Byte]): Int
  @native def ipcImport(ctx: Long, peerRank: Int, handle: Array[Byte]): Int
  @native def peerAttach(ctx: Long, peerRank: Int, peerCtx: Long, which: Int): Int
  @native def startAsync(ctx: Long, w0: Array[Double], assigned: Array[Int], batch: Int, lr: Double,
                         concurrency: Int, maxUpdates: Long, seed: Long): Int
  @native def stopAsync(ctx: Long): Int
  @native def asyncRunning(ctx: Long, out: Array[Int]): Int
  @native def updateGrad(ctx: Long, idx: Array[Int], value: Array[Double]): Int
  @native def asyncUpdates(ctx: Long, out: Array[Long]): Int
  @native def asyncMasterWeights(ctx: Long, out: Array[Double]): Int
  @native def asyncOutboxEnable(ctx: Long): Int
  @native def asyncOutboxRead(ctx: Long, out: Array[Double]): Int

  /** Vec (keys are the reference's 1-based feature ids) -> dense array in the ABI's 0-based column space. */
  def densify(v: Vec, dim: Int): Array[Double] = {
    val a = new Array[Double](dim)
    v.map.foreach { case (k, x) => a(k - 1) = x.toDouble }
    a
  }

  def sparsify(a: Array[Double], dim: Int): Vec =
    Vec(a.iterator.zipWithIndex.collect { case (x, i) if x != 0.0 => (i + 1) -> spire.math.Number(x) }.toMap, dim)

  def check(ctx: Long, rc: Int): Unit = rc match {
    case 0            => ()
    case -1 | -3      => throw new IllegalArgumentException(lastError(ctx)) // require(...) / Vec.sum(empty)
    case -4           => throw new IndexOutOfBoundsException(lastError(ctx))
    case _            => throw new IllegalStateException(lastError(ctx))
  }
}
