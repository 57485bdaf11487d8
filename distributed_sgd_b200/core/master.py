"""core/Master.scala, MasterSync.scala, MasterAsync.scala -- the coordination loop.

The reference master is a separate process that shuffles index ranges, fans `gradient` RPCs out to K
slaves, averages the replies and updates the weights (core/Master.scala:120-218).  Here the master
logic runs SPMD: every rank executes the same loop with the same seed, so all ranks draw the same
batches; each rank feeds ITS slice to its GPU and the replies are summed on the devices (NCCL over
NVLink inside libdsgd.so).  Weights never leave the GPUs during `fit`.  What remains on the host is
control flow over a handful of scalars per epoch (losses, accuracies, the stopping rule).
"""
from __future__ import annotations

from typing import Callable, List, Optional, Sequence

import numpy as np

from ..ml import split_strategy as SplitStrategy  # noqa: N812
from ..ml.grad_state import GradState
from ..ml.sparse_svm import SparseSVM
from ..native import NativeCtx
from ..utils.dataset import Data
from .group import Group
from .slave import Slave

EarlyStopping = Callable[[Sequence[float]], bool]
Split = Callable[[int, int], List[range]]


class EpochDraw(list):
    """The batch draws of one epoch: `self[s][k]` = row ids of worker k at step s (a list of lists of int32 arrays, the
    shape the tests and the oracle replay), backed by ONE array `ids[steps, K, batch]` (-1 beyond a short slice) and
    `counts[steps, K]` so that `fit` can hand whole runs of steps to the device without per-step Python work."""

    ids: np.ndarray
    counts: np.ndarray

    @classmethod
    def _wrap(cls, ids: np.ndarray, counts: np.ndarray) -> "EpochDraw":
        self = cls([[ids[s, k, :counts[s, k]] for k in range(ids.shape[1])] for s in range(ids.shape[0])])
        self.ids, self.counts = ids, counts
        return self

    @classmethod
    def draw(cls, seed: int, epoch: int, groups: List[range], batch_size: int) -> "EpochDraw":
        import ctypes as C
        from .. import native
        K = len(groups)
        g_start = np.array([g.start for g in groups], dtype=np.int64)
        g_len = np.array([len(g) for g in groups], dtype=np.int64)
        steps = -(-int(g_len.max()) // batch_size) if K else 0
        ids = np.empty((steps, K, batch_size), dtype=np.int32)
        counts = np.empty((steps, K), dtype=np.int32)
        h = native.host_lib()
        rc = h.dsgd_draw_epoch(C.c_uint64(seed & 0xFFFFFFFFFFFFFFFF), epoch, K, g_start.ctypes.data_as(C.c_void_p),
                               g_len.ctypes.data_as(C.c_void_p), batch_size, ids.ctypes.data_as(C.c_void_p),
                               counts.ctypes.data_as(C.c_void_p), ids.size)
        if rc != steps:
            raise ValueError(f"draw_epoch failed ({rc})")
        return cls._wrap(ids, counts)

    @classmethod
    def from_steps(cls, steps_list) -> "EpochDraw":
        steps, K = len(steps_list), len(steps_list[0]) if steps_list else 0
        B = max((len(b) for st in steps_list for b in st), default=0)
        ids = np.full((steps, K, B), -1, dtype=np.int32)
        counts = np.zeros((steps, K), dtype=np.int32)
        for s, st in enumerate(steps_list):
            for k, b in enumerate(st):
                ids[s, k, :len(b)] = b
                counts[s, k] = len(b)
        return cls._wrap(ids, counts)


class Master:
    """core/Master.scala:19-255 (abstract).  `Master.apply` (Master.scala:259-271) is `Master.create`."""

    def __init__(self, node: int, data: Data, test_data: Data, model: SparseSVM, expected_node_count: int, *,
                 slave: Slave, group: Optional[Group] = None, seed: int = 0, log: Optional[Callable[[str], None]] = None,
                 jvm_exact: bool = False, attach: bool = True):
        self.node, self.model, self.expected_node_count = node, model, expected_node_count
        self.n_train, self.n_test = data.n_rows, test_data.n_rows
        self.dim = data.dim
        self.slave = slave
        self.ctx: NativeCtx = slave.ctx
        self.group = group or Group()
        if self.group.world != slave.world:
            raise ValueError("process group size and Slave world size differ")
        if slave.n_test != self.n_test or slave.n_train != self.n_train:
            raise ValueError("the Slave must hold the same train/test rows as the Master")
        # Random.setSeed(0) (Main.scala:32): one stream, identical on every rank
        self.seed = int(seed)
        self.rng = np.random.default_rng(seed)
        self._epochs_drawn = 0
        # jvm_exact: draw the batches with java.util.Random(seed) + Scala 2.12's Random.shuffle, the stream a reference
        # run consumes (SURVEY.md 8f N4); default: numpy's generator (statistically the same draws, much faster)
        self.jvm = None
        if jvm_exact:
            from ..utils.jvm_random import JvmRandom
            self.jvm = JvmRandom(seed)
        self.log = log or (lambda s: None)
        # attach=False: the Slave's device context already carries its communicator / peer exchange
        if attach and self.group.world > 1 and not slave.is_async:
            # NCCL communicator (general path: several logical workers per GPU) ...
            uid = NativeCtx.comm_unique_id() if self.group.rank == 0 else b""
            self.ctx.comm_init(self.group.broadcast_bytes(uid, 0))
            # ... and the peer-memory exchange of the fused persistent kernel (one worker per GPU)
            if hasattr(self.ctx, "setup_peer_exchange"):
                self.ctx.setup_peer_exchange(self.group)

    @staticmethod
    def create(node, data, test_data, model, is_async, node_count, **kw) -> "Master":
        """Master.apply (core/Master.scala:259-271)."""
        return (MasterAsync if is_async else MasterSync)(node, data, test_data, model, node_count, **kw)

    # ---- evaluation ------------------------------------------------------------------------------------
    def _eval_rows(self, weights, begin: int, end: int):
        """Row-sharded pass: each rank evaluates a contiguous share, integer counters are summed."""
        W, r = self.group.world, self.group.rank
        n = end - begin
        lo, hi = begin + (n * r) // W, begin + (n * (r + 1)) // W
        if hi > lo:
            h, c, n2 = self.ctx.eval_counts(lo, hi, weights)
        else:
            h, c, n2 = 0, 0, 0.0
        hs, cs = self.group.all_reduce_sum([h, c])
        n2 = self.group.all_reduce_max(n2)  # identical on every rank that evaluated; 0 on idle ranks
        return self.model.lam * n2 + hs / n, cs / n

    def local_loss(self, weights=None, test_data: bool = False) -> float:
        """Master.localLoss (core/Master.scala:105-107)."""
        b, e = (self.n_train, self.n_train + self.n_test) if test_data else (0, self.n_train)
        return self._eval_rows(weights, b, e)[0]

    def local_accuracy(self, weights=None, test_data: bool = False) -> float:
        """Master.localAccuracy (core/Master.scala:100-103)."""
        b, e = (self.n_train, self.n_train + self.n_test) if test_data else (0, self.n_train)
        return self._eval_rows(weights, b, e)[1]

    def local_loss_accuracy(self, weights=None, test_data: bool = False):
        b, e = (self.n_train, self.n_train + self.n_test) if test_data else (0, self.n_train)
        return self._eval_rows(weights, b, e)

    def predict(self, weights, split_strategy: Split = SplitStrategy.vanilla) -> dict:
        """Master.predict (core/Master.scala:61-75): idx -> prediction over the training rows; each worker
        answers for its split group."""
        groups = split_strategy(self.n_train, self.group.world)
        mine = groups[self.group.rank] if self.group.rank < len(groups) else range(0)
        idx = np.fromiter(mine, dtype=np.int32, count=len(mine))
        preds = self.slave.forward(idx, weights) if len(idx) else np.zeros(0)
        import pickle
        parts = self.group.all_gather_bytes(pickle.dumps((idx, preds)))
        out = {}
        for blob in parts:
            i, p = pickle.loads(blob)
            out.update(zip(i.tolist(), p.tolist()))
        return out

    def distributed_accuracy(self, weights, split_strategy: Split = SplitStrategy.vanilla) -> float:
        """Master.distributedAccuracy (core/Master.scala:77-85)."""
        return self._distributed(weights, split_strategy)[1]

    def distributed_loss(self, weights, split_strategy: Split = SplitStrategy.vanilla) -> float:
        """Master.distributedLoss (core/Master.scala:87-98)."""
        return self._distributed(weights, split_strategy)[0]

    def _distributed(self, weights, split_strategy: Split):
        # same numbers as predict + host-side counting, without shipping N predictions around
        groups = split_strategy(self.n_train, self.group.world)
        mine = groups[self.group.rank] if self.group.rank < len(groups) else range(0)
        if len(mine):
            h, c, n2 = self.ctx.eval_counts(mine.start, mine.stop, weights)
        else:
            h, c, n2 = 0, 0, 0.0
        hs, cs, ns = self.group.all_reduce_sum([h, c, len(mine)])
        n2 = self.group.all_reduce_max(n2)
        return self.model.lam * n2 + hs / ns, cs / ns


class MasterSync(Master):
    """core/MasterSync.scala + the sync `fit` of core/Master.scala:120-218."""

    def update_grad(self, grad_update):  # MasterSync.scala:16-17
        raise NotImplementedError("Synchronous master cannot perform async operation update grad")

    def draw_epoch(self, groups: List[range], batch_size: int, epoch: Optional[int] = None):
        """Sample ids of one epoch: for every step (`0 until maxSamples by batchSize`, Master.scala:179) and
        every worker a fresh shuffle of its range, sliced at [batch, batch + batchSize) (Master.scala:
        184-187, quirk Q5).  A slice of a fresh permutation is a uniform draw without replacement of
        min(batchSize, len - batch) elements -- drawn directly (csrc/dsgd_host.c: dsgd_draw_epoch) from a counter-based
        generator keyed by (seed, epoch, step, worker), identical on every rank.  Returns an EpochDraw: a list of steps,
        each a list of per-worker arrays (what the oracle replays), plus the same ids as one array for the device."""
        if epoch is None:
            epoch = self._epochs_drawn
        self._epochs_drawn = epoch + 1
        if self.jvm is not None:
            n, size = groups[-1].stop, len(groups[0])
            if [(g.start, g.stop) for g in groups] != [(a, min(a + size, n)) for a in range(0, n, size)]:
                raise ValueError("jvm_exact draws are defined for SplitStrategy.vanilla groups")
            return EpochDraw.from_steps(self.jvm.sync_epoch(n, len(groups), batch_size, group_size=size))
        return EpochDraw.draw(self.seed, epoch, groups, batch_size)

    def fit(self, initial_weights: np.ndarray, max_epochs: int, batch_size: int, learning_rate: float,
            stopping_criterion: EarlyStopping, split_strategy: Split = SplitStrategy.vanilla, *,
            virtual_workers: int = 1, on_epoch: Optional[Callable[[int, dict], None]] = None) -> GradState:
        """Master.fit (core/Master.scala:120-218).

        virtual_workers (extension): logical reference workers per GPU, so that `node-count` can exceed the
        number of GPUs (K = world * virtual_workers).
        """
        W, r, V = self.group.world, self.group.rank, virtual_workers
        K = W * V
        groups = split_strategy(self.n_train, K)             # Master.scala:136 (may hold fewer than K groups)
        k_total = len(groups)                                 # workers.zip(split): extra workers get no request
        my_groups = [k for k in range(r * V, (r + 1) * V) if k < k_total]
        self.ctx.set_weights(initial_weights)
        state = GradState.start_state(np.asarray(initial_weights, dtype=np.float64))
        losses: List[float] = []
        accs: List[float] = []
        test_losses: List[float] = []
        test_accs: List[float] = []
        self.step_losses: List[np.ndarray] = []
        epoch = 0
        # a one-thread pool overlaps the next epoch's draw with the current epoch's kernel (not with jvm_exact: that
        # stream is sequential and must not run ahead of an early stop)
        from concurrent.futures import ThreadPoolExecutor
        prefetch = ThreadPoolExecutor(1) if self.jvm is None else None
        pending = None
        while True:
            if losses:
                self.log(f"loss after epoch {epoch}: {losses[0]}")
                self.log(f"acc after epoch {epoch}: {accs[0]}")
            if epoch >= max_epochs or stopping_criterion(test_losses):   # Master.scala:154,166
                self.log("Reached max number of epochs: stopping computation" if epoch >= max_epochs
                         else "Converged to target: stopping computation")
                self.history = {"losses": losses[::-1], "test_losses": test_losses[::-1], "accs": accs[::-1],
                                "test_accs": test_accs[::-1]}
                if prefetch is not None:
                    prefetch.shutdown(wait=True)
                # `losses.head` throws on an empty list in the reference (max_epochs == 0)
                return state.finish(losses[0])
            steps = pending.result() if pending is not None else self.draw_epoch(groups, batch_size)
            pending = None
            if not isinstance(steps, EpochDraw):
                steps = EpochDraw.from_steps(steps)
            if prefetch is not None and epoch + 1 < max_epochs:
                # the draws of epoch e + 1 do not depend on epoch e: make them while the GPU runs epoch e
                pending = prefetch.submit(self.draw_epoch, groups, batch_size, self._epochs_drawn)
            counts = steps.counts                                                 # [steps, k_total]
            if counts.size and (counts[:, :k_total] == 0).any():
                raise ValueError("Cannot sum an empty list of vectors")  # Vec.scala:129 via Master.scala:187 (Q7)
            # consecutive steps with identical counts for ALL workers go to the device in one call; the boundaries come
            # from the global shape so that every rank issues the same sequence of calls (the fused multi-GPU kernel
            # numbers its exchange tags by call)
            n_steps = counts.shape[0]
            change = np.flatnonzero((counts[1:] != counts[:-1]).any(axis=1)) + 1 if n_steps > 1 else np.zeros(0, dtype=np.int64)
            bounds = [0, *change.tolist(), n_steps]
            for i, j in zip(bounds[:-1], bounds[1:]):
                if j == i:
                    continue
                shape = [int(counts[i, k]) for k in my_groups]
                if my_groups:
                    g0, g1 = my_groups[0], my_groups[-1] + 1
                    if all(c == steps.ids.shape[2] for c in shape):
                        flat = np.ascontiguousarray(steps.ids[i:j, g0:g1, :]).reshape(-1)
                    else:
                        flat = np.concatenate([steps.ids[s, k, :counts[s, k]] for s in range(i, j) for k in my_groups])
                else:
                    flat = np.zeros(0, dtype=np.int32)
                self.ctx.set_workers(shape, k_total)
                ls = self.ctx.sync_steps(flat, int(sum(shape)), j - i, learning_rate, want_losses=True)
                self.step_losses.append(ls)
            w = None  # evaluate the resident weights
            tl, ta = self.local_loss_accuracy(w, test_data=False)        # Master.scala:206-207
            vl, va = self.local_loss_accuracy(w, test_data=True)         # Master.scala:208-209
            losses.insert(0, tl); accs.insert(0, ta); test_losses.insert(0, vl); test_accs.insert(0, va)
            epoch += 1
            state = state.replace_grad(self.ctx.get_weights())          # Master.scala:205
            if on_epoch:
                on_epoch(epoch, {"loss": tl, "acc": ta, "test_loss": vl, "test_acc": va})

    def fit_models(self, initial_weights: np.ndarray, max_epochs: int, batch_size: int, lambdas: Sequence[float],
                   learning_rates: Sequence[float], stopping_criterion: EarlyStopping,
                   split_strategy: Split = SplitStrategy.vanilla, *,
                   on_epoch: Optional[Callable[[int, List[Optional[dict]]], None]] = None) -> List[GradState]:
        """`fit` for several (lambda, learning rate) settings at once: one SparseSVM(lambdas[m]) trained with
        learning_rates[m] per setting, all on the same batch draws, as a model set on the device (one kernel per run of
        equal-count steps for all models).  Model m's GradState and history are what `fit(initial_weights, max_epochs,
        batch_size, learning_rates[m], stopping_criterion, split_strategy)` returns on a master whose model is
        SparseSVM(lambdas[m]) with the same seed: each model stops (is frozen) at the epoch its own test losses stop it.
        One GPU, one worker per step.  Sets `self.histories` (one dict per model, the keys of `fit`'s `self.history`)."""
        from ..native import MAX_MODELS
        lambdas = [float(x) for x in lambdas]
        learning_rates = [float(x) for x in learning_rates]
        M = len(lambdas)
        if len(learning_rates) != M or not 1 <= M <= MAX_MODELS:
            raise ValueError(f"fit_models: need 1 to {MAX_MODELS} (lambda, learning rate) pairs, got {M} and "
                             f"{len(learning_rates)}")
        if self.group.world != 1:
            raise ValueError("fit_models: model sets run on one GPU (process group of size 1)")
        groups = split_strategy(self.n_train, 1)
        if len(groups) != 1:
            raise ValueError("fit_models: model sets take one worker per step")
        w0 = np.asarray(initial_weights, dtype=np.float64)
        self.ctx.models_set(lambdas, learning_rates, w0)
        states = [GradState.start_state(w0) for _ in range(M)]
        hist = [{"losses": [], "test_losses": [], "accs": [], "test_accs": []} for _ in range(M)]  # newest first
        done: List[Optional[GradState]] = [None] * M
        self.step_losses: List[np.ndarray] = []
        n_train, n_test = self.n_train, self.n_test
        epoch = 0
        from concurrent.futures import ThreadPoolExecutor
        prefetch = ThreadPoolExecutor(1) if self.jvm is None else None
        pending = None
        try:
            while True:
                for m in range(M):                                                    # Master.scala:154,166, per model
                    if done[m] is None and (epoch >= max_epochs or stopping_criterion(hist[m]["test_losses"])):
                        done[m] = states[m].finish(hist[m]["losses"][0])
                active = np.array([d is None for d in done])
                if not active.any():
                    break
                steps = pending.result() if pending is not None else self.draw_epoch(groups, batch_size)
                pending = None
                if not isinstance(steps, EpochDraw):
                    steps = EpochDraw.from_steps(steps)
                if prefetch is not None and epoch + 1 < max_epochs:
                    pending = prefetch.submit(self.draw_epoch, groups, batch_size, self._epochs_drawn)
                counts = steps.counts[:, 0]
                if counts.size and (counts == 0).any():
                    raise ValueError("Cannot sum an empty list of vectors")       # Vec.scala:129 via Master.scala:187 (Q7)
                n_steps = counts.shape[0]
                bounds = [0, *(np.flatnonzero(counts[1:] != counts[:-1]) + 1).tolist(), n_steps]
                for i, j in zip(bounds[:-1], bounds[1:]):
                    if j == i:
                        continue
                    c = int(counts[i])
                    flat = np.ascontiguousarray(steps.ids[i:j, 0, :c]).reshape(-1)
                    self.step_losses.append(self.ctx.models_steps(flat, c, j - i, active=active))
                epoch += 1
                weights = self.ctx.models_get_weights()
                report: List[Optional[dict]] = [None] * M
                for m in np.flatnonzero(active).tolist():
                    h, cr, n2 = self.ctx.models_eval_counts(m, 0, n_train)                     # Master.scala:206-207
                    th, tc, _ = self.ctx.models_eval_counts(m, n_train, n_train + n_test)      # Master.scala:208-209
                    tl, ta = lambdas[m] * n2 + h / n_train, cr / n_train
                    vl, va = lambdas[m] * n2 + th / n_test, tc / n_test
                    for k, v in (("losses", tl), ("accs", ta), ("test_losses", vl), ("test_accs", va)):
                        hist[m][k].insert(0, v)
                    states[m] = states[m].replace_grad(weights[m].copy())                  # Master.scala:205
                    report[m] = {"loss": tl, "acc": ta, "test_loss": vl, "test_acc": va}
                if on_epoch:
                    on_epoch(epoch, report)
        finally:
            if prefetch is not None:
                prefetch.shutdown(wait=True)
        self.histories = [{k: v[::-1] for k, v in h.items()} for h in hist]
        return done


class MasterAsync(Master):
    """core/MasterAsync.scala -- Hogwild: every worker runs its loop on its GPU and pushes deltas into every peer
    replica and into the master replica (hosted on rank 0's GPU) over NVLink; the master logic polls the update
    counter, evaluates the master replica on the test rows every `check_every` updates with a leaky average, keeps
    the best weights, and stops on `n_train * max_epoch` updates or the early-stopping rule."""

    def _attach_replicas(self):
        from ..native import REPLICA_MASTER, REPLICA_SELF
        W, r = self.group.world, self.group.rank
        mine = self.ctx.ipc_export(REPLICA_SELF)
        master = self.ctx.ipc_export(REPLICA_MASTER) if r == 0 else b""
        handles = self.group.all_gather_bytes(mine)
        master = self.group.broadcast_bytes(master, 0)
        for k, h in enumerate(handles):
            if k != r:
                self.ctx.ipc_import(k, h)
        if r != 0:
            self.ctx.ipc_import(W, master)
        self.group.barrier()

    def fit(self, initial_weights: np.ndarray, max_epoch: int, batch_size: int, learning_rate: float,
            stopping_criterion: EarlyStopping, split_strategy: Split = SplitStrategy.vanilla, check_every: int = 100,
            leak_loss_coef: float = 0.9, *, concurrency: int = 1, poll_seconds: float = 0.05, seed: int = 0,
            on_check: Optional[Callable[[int, dict], None]] = None) -> GradState:
        """MasterAsync.fit (core/MasterAsync.scala:32-62) + startLossChecking (96-162) + updateGrad's stop rule
        (164-177) + endComputation (87-94).  concurrency (extension): Hogwild lanes per GPU."""
        import time
        if not (0 <= leak_loss_coef <= 1):
            raise ValueError("leaking coefficient must be between 0 and 1")      # MasterAsync.scala:97
        if getattr(self, "_running", False):
            raise RuntimeError("Cannot start async computation: a computation is already running")
        W, r = self.group.world, self.group.rank
        w0 = np.asarray(initial_weights, dtype=np.float64)
        groups = split_strategy(self.n_train, W)
        max_steps = self.n_train * max_epoch                                      # MasterAsync.scala:83
        self.ctx.set_weights(w0)                     # every replica first, then the loops (no start-up race)
        if r == 0:
            self.ctx.async_host_master(w0)
        if W > 1:
            self._attach_replicas()
        self._running = True
        mine = groups[r] if r < len(groups) else range(0)
        if len(mine):
            self.slave.start_async(None, np.fromiter(mine, dtype=np.int32, count=len(mine)), batch_size, learning_rate,
                                   concurrency=concurrency, max_updates=0, seed=seed + 1000 * r)
        state = GradState.start_state(w0)
        test_losses: List[float] = []
        test_accs: List[float] = []
        best_loss, best_w = float("inf"), None
        last_step = -check_every                                                  # MasterAsync.scala:161
        # polls: every look at the update counter (updates, computed?); raw_*: the unsmoothed numbers of the computed polls --
        # what a replay of core/MasterAsync.scala:96-162 over the same stream needs (tests/test_host_logic.py)
        self.history = {"test_losses": test_losses, "test_accs": test_accs, "checks_at": [], "polls": [],
                        "raw_test_losses": [], "raw_test_accs": [], "best_check": None, "ended_by": None}
        try:
            while True:
                updates = self.ctx.async_updates() if r == 0 else 0
                updates = int(self.group.all_reduce_max(float(updates)))
                if updates >= max_steps:                                          # MasterAsync.scala:171-174
                    self.log("max number of steps reached: stopping computation")
                    self.history["polls"].append((updates, False))
                    self.history["ended_by"] = "max_steps"
                    break
                if updates - last_step < check_every:                             # latest computation was too close
                    self.history["polls"].append((updates, False))
                    time.sleep(poll_seconds)                                      # (the reference waits 2.5 s)
                    continue
                # innerGradState.grad: ONE snapshot (rank 0 hosts the master replica), evaluated row-sharded by everybody
                blob = self.ctx.async_master_weights().tobytes() if r == 0 else b""
                w = np.frombuffer(self.group.broadcast_bytes(blob, 0), dtype=np.float64).copy()
                loss, acc = self.local_loss_accuracy(w, test_data=True)           # MasterAsync.scala:118-120
                loss_s = leak_loss_coef * loss + (1 - leak_loss_coef) * (test_losses[0] if test_losses else loss)
                acc_s = leak_loss_coef * acc + (1 - leak_loss_coef) * (test_accs[0] if test_accs else acc)
                if best_loss > loss_s:                                            # MasterAsync.scala:130-139
                    best_loss, best_w = loss_s, w
                    self.history["best_check"] = len(self.history["checks_at"])
                test_losses.insert(0, loss_s)
                test_accs.insert(0, acc_s)
                self.history["checks_at"].append(updates)
                self.history["polls"].append((updates, True))
                self.history["raw_test_losses"].append(loss)
                self.history["raw_test_accs"].append(acc)
                if on_check:
                    on_check(updates, {"test_loss": loss_s, "test_acc": acc_s, "weights": w})
                if stopping_criterion(test_losses):                               # MasterAsync.scala:146-152
                    self.log("converged to target: stopping computation")
                    self.history["ended_by"] = "converged"
                    break
                last_step = updates
        finally:
            if len(mine):
                self.slave.stop_async()                                           # endComputation: stopAsync to all
            self._running = False
            self.group.barrier()
        if best_w is None:
            # the reference would hand back its initial bestGrad (Vec.zeros(1)) here; we return what the master holds
            blob = self.ctx.async_master_weights().tobytes() if r == 0 else b""
            best_w = np.frombuffer(self.group.broadcast_bytes(blob, 0), dtype=np.float64).copy()
            best_loss = self.local_loss_accuracy(best_w, test_data=True)[0]
        return state.replace_grad(best_w).finish(best_loss)                       # MasterAsync.scala:91
