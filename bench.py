#!/usr/bin/env python
"""bench.py -- SGD samples/sec on RCV1-shaped synthetic sparse data (BASELINE.json's metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--batch 256] [--mode sync]
                  [--dump-outputs DIR]

--dump-outputs DIR writes, after the timed steps, what the timed leg computed in its last bench step: sync mode
weights.npy (the final weights) and losses.npy (the loss of each SGD step); async mode master_weights.npy.  The inputs
depend only on the arguments (seeded synthetic rows and batch draws), so sync outputs of two builds compare one to one.

Workload (BASELINE.json configs[1]/[2]): sync mode, RCV1-shaped synthetic rows (47 236 features, 700 000
rows of which the first 80 % train -- Main.scala:52 --, ~0.2 % non-zeros), batch 256 per GPU, lambda 1e-5,
lr 0.5 (resources/application.conf).  One bench "step" is one pass of the hot path over one epoch-sized
slice of the reference's fit loop (core/Master.scala:179): SGD_STEPS consecutive mini-batch steps
(gradient -> aggregate -> update), every one on weights produced by the previous one.  samples/sec counts
the samples all GPUs consumed.

Keys of the JSON line (one line on stdout, rank 0):
  value        device-resident: sample ids staged in HBM before the timed region; CUDA events on the
               launch stream; max over ranks.
  e2e          the same work through the public C-ABI call with HOST buffers (dsgd_sync_steps): per bench
               step the sample ids go host->device from pinned memory and the per-batch losses come back.
  e2e_fit      the same metric through the reference-shaped driver MasterSync.fit (core/Master.scala:120-218):
               per-epoch batch draws on the host, the step loop, the four per-epoch evaluations, the weight read-back.
  roofline     the dominant kernel: algorithmic bytes (8*nnz + 16 per sample, SURVEY.md 8d) per launch /
               its mean duration (CUDA events around its launches), against MEASURED_PEAKS.json.
  roofline_streaming  the bandwidth-bound forms of the same row kernels (full-shard evaluation, large-batch gradient).
  sweep        BASELINE.json configs[4] at this GPU count: sync batch {64, 256, 1024} (device-resident).
  async        BASELINE.json configs[3] at this GPU count: Hogwild, batch 1, one worker per GPU (lanes = 1, the
               reference's sequential loop) and the many-lanes extension, with the master replica's test accuracy.
  parity       a fresh 300-step trajectory at this GPU count checked against the CPU oracle IN THIS RUN.
  rpc_seam     the literal per-request seam of SlaveImpl.gradient / forward (host weights in, dense result out).
  nvlink       N > 1: bytes this rank stored into its peers per SGD step (counted by the kernel) and, where NVML
               exposes them, the hardware NVLink tx/rx counters over the timed region.
  cpu_baseline the fp64 CPU oracle (array restatement of the Scala path -- the reference itself needs a
               JVM, which this image lacks) timed on this host on a bounded sample of the same workload.
               `cores` = 1: one thread per worker, like the reference (core/Slave.scala:142).  `all_cores` beside it is
               CONTEXT: one worker's batch split over the best of 4-64 host threads (not how the reference runs).
--impl reference times that CPU restatement as the reference arm.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

DIM = 47236
N_ROWS = 700_000
TRAIN_FRAC = 0.8
LAMBDA = 1e-5
LR = 0.5
METRIC = "sgd_samples_per_sec"
UNIT = "samples/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=None, help="samples per GPU per step (default: 256 sync, 1 async)")
    ap.add_argument("--mode", default="sync", choices=["sync", "async"])
    ap.add_argument("--lanes", type=int, default=256, help="async: Hogwild lanes (warps) per GPU")
    ap.add_argument("--async-updates", type=int, default=400000, help="async: updates per GPU per bench step")
    ap.add_argument("--rows", type=int, default=N_ROWS)
    ap.add_argument("--sgd-steps", type=int, default=0, help="SGD steps per bench step (0: one epoch at 1 worker)")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--no-extras", action="store_true", help="skip sweep / async / parity / rpc_seam / e2e_fit sub-records")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path computed in its last bench step to DIR/<name>.npy (fp64)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs: the reference arm sizes its sample by elapsed time, its outputs are not reproducible")
    if a.batch is None:
        a.batch = 256 if a.mode == "sync" else 1        # BASELINE.json configs[1]/[2] and configs[3]
    return a


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel_key: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per SGD step of the persistent kernel from this round's `ncu --set full`
    capture (profiles/ncu_traffic.json), valid only while the kernel source is the one that was captured."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            rec = json.load(f)[kernel_key]
        src = os.path.join(ROOT, "distributed_sgd_b200", "csrc", rec["source"])
        if hashlib.sha256(open(src, "rb").read()).hexdigest()[:16] != rec["source_sha16"]:
            return None, "profiles/ncu_traffic.json is from an older kernel source: not reported"
        return rec, rec.get("capture", "profiles/ncu_traffic.json")
    except Exception:
        return None, "no ncu capture recorded for this kernel source"


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md's clocks line), read every 25 ms from NVML
    in this process -- the same counters `nvidia-smi --query-gpu=clocks.sm,clocks_event_reasons.*` prints, without a
    looping nvidia-smi process next to the launching rank (whose peers spin for it inside the fused multi-GPU kernel).
    `nvidia-smi -lms 20` remains the fallback when NVML cannot be loaded."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device, self.rows, self.proc, self.first = device, [], None, 0
        self.nvml, self.handle, self.run, self.thread = None, None, False, None

    def mark(self):
        """Samples before this call (GPU idle while the sampler starts) are not used."""
        self.first = len(self.rows)

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.device)
            pynvml.nvmlDeviceGetClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
            self.nvml, self.run = pynvml, True
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.device)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _poll(self):
        n = self.nvml
        names = (("hw_slowdown", n.nvmlClocksEventReasonHwSlowdown), ("hw_thermal_slowdown", n.nvmlClocksEventReasonHwThermalSlowdown),
                 ("sw_thermal_slowdown", n.nvmlClocksEventReasonSwThermalSlowdown), ("sw_power_cap", n.nvmlClocksEventReasonSwPowerCap))
        try:
            mx = n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)
        except Exception:
            mx = None
        while self.run:
            try:
                sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
                mask = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                self.rows.append([str(self.device), str(sm), str(mx), ""] + ["Active" if mask & bit else "Not Active" for _, bit in names])
            except Exception:
                pass
            time.sleep(0.025)

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.nvml is not None:
            time.sleep(0.03)
            self.run = False
            self.thread.join(timeout=1.0)
        elif self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
        else:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no clock source: NVML and nvidia-smi unavailable"]}
        sm, mx, reasons = [], [], set()
        for r in self.rows[self.first:]:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm),
                "source": "NVML, every 25 ms during warm-up + timed region" if self.nvml is not None else "nvidia-smi -lms 20"}


def nvlink_counters(device: int):
    """(tx_bytes, rx_bytes) summed over the GPU's NVLinks from NVML's throughput counters (KiB), or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(device)
        ids = [pynvml.NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_TX, pynvml.NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_RX]
        out = []
        for fid in ids:
            fv = pynvml.nvmlDeviceGetFieldValues(h, [(fid, 0xFFFFFFFF)])[0]     # scope UINT_MAX: all links
            if fv.nvmlReturn != 0:
                return None
            out.append(int(fv.value.ullVal) * 1024)
        return tuple(out)
    except Exception:
        return None


def sync_config(args, world, n_train, B, S):
    """The `config` object of a sync line -- shared by the GPU arm and the reference arm so that they name the same
    workload."""
    return {"workload": f"sync SGD (configs[{1 if world == 1 else 2}]): RCV1-shaped synthetic, {DIM} feats, "
                        f"{args.rows} rows ({n_train} train), ~0.2% nnz, batch {B} per GPU",
            "mode": "sync", "batch_per_gpu": B, "sgd_steps_per_bench_step": S, "lambda": LAMBDA, "lr": LR,
            "parallelism": f"dp{world}", "l2": "inputs (train CSR 0.43 GB) larger than the 126 MB L2; rows drawn at random",
            "values": "fp32", "state": "fp64"}


def make_data(args):
    from distributed_sgd_b200.utils import synthetic_rcv1
    data = synthetic_rcv1(n_rows=args.rows, dim=DIM, seed=args.seed)
    n_train = int(data.n_rows * TRAIN_FRAC)  # Main.scala:52
    return data, n_train


def draw_batches(rng, lo: int, hi: int, batch: int, n_steps: int) -> np.ndarray:
    """n_steps uniform draws without replacement of `batch` rows from [lo, hi) -- what a slice of a freshly
    shuffled worker range is (core/Master.scala:184-187)."""
    out = np.empty((n_steps, batch), dtype=np.int32)
    for s in range(n_steps):
        out[s] = lo + rng.choice(hi - lo, size=batch, replace=False)
    return out


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """--dump-outputs: one DIR/<name>.npy per array, fp64, so that two builds run with the same arguments (hence the same
    seeded inputs) can be compared output for output."""
    arrays = {k: np.ascontiguousarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed {DUMP_MAX_BYTES}; use fewer --sgd-steps")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def make_oracle(data, d):
    from oracle.oracle import Oracle
    orc = Oracle(data.row_ptr, data.col, data.val, data.label, data.dim, LAMBDA)
    orc.set_dim_sparsity(d)
    return orc


def cpu_leg(data, n_train, d, batch, workers, budget_s, threads, seed):
    """Times the oracle's sync steps (K logical workers) on a bounded sample; returns (samples/s, description)."""
    orc = make_oracle(data, d)
    rng = np.random.default_rng(seed + 17)
    per = n_train // workers
    probe = 40
    def run(n_steps, w):
        idx = np.concatenate([draw_batches(rng, k * per, (k + 1) * per, batch, n_steps)[:, None, :] for k in range(workers)],
                             axis=1).reshape(-1)
        t = time.perf_counter()
        w, _ = orc.sync_steps(w, idx, [batch] * workers, LR, n_steps=n_steps, threads=threads)
        return time.perf_counter() - t, w
    dt, w = run(probe, np.zeros(data.dim))
    n_steps = int(max(probe, min(20000, budget_s / max(dt / probe, 1e-9))))
    dt, w = run(n_steps, w)
    cpu_leg.last_seconds = dt
    return n_steps * batch * workers / dt, f"{n_steps} sync SGD steps x {workers} worker(s) x batch {batch}, {dt:.1f} s"


def cpu_all_cores(data, n_train, d, batch, seed, budget_s=1.5):
    """CONTEXT, not the reference's parallelism: ONE worker's batch split over T threads (rows in parallel, shared accumulator;
    oracle/dsgd_oracle.c: dsgd_oracle_sync_steps_allcores), best T of a few -- what the same arithmetic reaches when every
    core of the host works on a single worker's step.  The reference runs a gradient request on one thread
    (core/Slave.scala:142), which is what `cpu_baseline.value` times."""
    orc = make_oracle(data, d)
    rng = np.random.default_rng(seed + 29)
    try:
        cores = len(os.sched_getaffinity(0))
    except Exception:
        cores = os.cpu_count() or 1
    best = None
    for T in sorted({t for t in (4, 8, 16, 32, 64) if t <= cores} | {min(cores, 2)}):
        probe = 20     # short: the threads spin at their barriers, an oversubscribed T would crawl
        idx = draw_batches(rng, 0, n_train, batch, probe).reshape(-1)
        t0 = time.perf_counter()
        w, _ = orc.sync_steps_allcores(np.zeros(data.dim), idx, batch, LR, probe, T)
        dt = time.perf_counter() - t0
        if best is not None and probe * batch / dt < 0.5 * best["value"]:
            break      # more threads only lose from here on
        n_steps = int(max(probe, min(20000, budget_s / max(dt / probe, 1e-9))))
        idx = draw_batches(rng, 0, n_train, batch, n_steps).reshape(-1)
        t0 = time.perf_counter()
        orc.sync_steps_allcores(w, idx, batch, LR, n_steps, T)
        dt = time.perf_counter() - t0
        v = n_steps * batch / dt
        if best is None or v > best["value"]:
            best = {"value": v, "unit": UNIT, "threads": T, "sample": f"{n_steps} steps of batch {batch}, {dt:.1f} s"}
    best["note"] = ("one worker's batch split over T threads (rows in parallel) -- NOT how the reference runs (one thread per "
                    "gradient request); best T of those tried; host has %d cores" % cores)
    return best


# ---------------------------------------------------------------------------------------------------------------------
# sub-records
# ---------------------------------------------------------------------------------------------------------------------

def parity_record(ctx, group, data, n_train, d, B, rank, world, steps=300):
    """A fresh trajectory from w = 0 (recorded batch draws, K = world workers) on the GPUs, replayed by the fp64 CPU oracle
    on rank 0: per-step losses and final weights must agree; replicas must be bit-identical."""
    per = n_train // world
    rng = np.random.default_rng(4242)                              # same stream on every rank
    idx = np.stack([np.concatenate([k * per + rng.choice(per, size=B, replace=False) for k in range(world)])
                    for _ in range(steps)]).astype(np.int32)       # [steps, world * B]
    mine = idx.reshape(steps, world, B)[:, rank, :].reshape(-1)
    ctx.set_weights(np.zeros(data.dim))
    group.barrier()
    losses = ctx.sync_steps(mine, B, steps, LR, want_losses=True)
    w = ctx.get_weights()
    digests = group.all_gather_bytes(hashlib.sha256(w.tobytes()).digest())
    rec = None
    if rank == 0:
        orc = make_oracle(data, d)
        w_ref, l_ref = orc.sync_steps(np.zeros(data.dim), idx.reshape(-1), [B] * world, LR, n_steps=steps)
        nz = w_ref != 0
        rec = {"steps": steps, "workers": world, "batch_per_worker": B,
               "max_rel_err_loss": float(np.max(np.abs(losses - l_ref) / np.abs(l_ref))),
               "max_rel_err_weights": float(np.max(np.abs(w[nz] - w_ref[nz]) / np.abs(w_ref[nz]))) if nz.any() else 0.0,
               "support_equal": bool(np.array_equal(w != 0, nz)),
               "replicas_identical": all(b == digests[0] for b in digests),
               "checker": "oracle/dsgd_oracle.c (fp64 CPU restatement of core/Master.scala:184-197), same batch draws"}
    group.barrier()
    return rec


def sweep_record(ctx, group, data, n_train, rank, world, hbm_peak, batches=(64, 256, 1024), s_steps=600, reps=3):
    """configs[4], sync side: device-resident samples/s for batch 64 / 256 / 1024 per GPU at this GPU count."""
    per = n_train // world
    out = []
    for B in batches:
        rng = np.random.default_rng(900 + rank)
        idx = draw_batches(rng, rank * per, (rank + 1) * per, B, s_steps)
        ctx.set_weights(np.zeros(data.dim))
        ctx.stage_samples(idx.reshape(-1))
        group.barrier()
        ctx.sync_steps_staged(0, B, s_steps, LR, want_losses=False)        # warm-up
        ctx.synchronize()
        group.barrier()
        ctx.timer_start()
        for _ in range(reps):
            ctx.sync_steps_staged(0, B, s_steps, LR, want_losses=False)
        ms = group.all_reduce_max(ctx.timer_stop())
        by = data.algorithmic_bytes(idx.reshape(-1)) * reps
        out.append({"mode": "sync", "batch_per_gpu": B, "n_gpus": world, "value": reps * s_steps * B * world / (ms * 1e-3),
                    "unit": UNIT, "us_per_step": ms * 1e3 / (reps * s_steps),
                    "roofline_frac": by / (ms * 1e-3) / 1e9 / hbm_peak, "sgd_steps_timed": reps * s_steps})
    return out


def async_record(args, group, data, n_train, rank, local_rank, world, hbm_peak):
    """configs[3]: async Hogwild, batch 1, one worker per GPU, lock-free peer replica writes over NVLink.  lanes = 1 is the
    reference's loop (one sequential asyncTask per slave, core/Slave.scala:79-111); lanes = 256 is this build's extension
    (256 Hogwild lanes share the GPU's replica).  lr from application.conf."""
    from distributed_sgd_b200.native import REPLICA_MASTER, REPLICA_SELF, NativeCtx
    actx = NativeCtx(local_rank, data.dim, LAMBDA, rank=rank, world=world, is_async=True)
    actx.load_csr(data.row_ptr, data.col, data.val, data.label)
    actx.compute_dim_sparsity(n_train)
    w0 = np.zeros(data.dim)
    per = n_train // world
    assigned = np.arange(rank * per, (rank + 1) * per, dtype=np.int32)
    actx.set_weights(w0)
    if rank == 0:
        actx.async_host_master(w0)
    if world > 1:
        handles = group.all_gather_bytes(actx.ipc_export(REPLICA_SELF))
        master = group.broadcast_bytes(actx.ipc_export(REPLICA_MASTER) if rank == 0 else b"", 0)
        for k, h in enumerate(handles):
            if k != rank:
                actx.ipc_import(k, h)
        if rank != 0:
            actx.ipc_import(world, master)
    group.barrier()
    mean_bytes = data.algorithmic_bytes() / data.n_rows
    out = []
    # (batch, lanes, updates per GPU): configs[3] = batch 1; configs[4] sweeps batch 64 / 256 / 1024 in async mode too
    for B_a, lanes, U in ((1, 1, 60000), (1, 256, 1500000), (64, 64, 12000), (256, 64, 4000), (1024, 64, 1200)):
        actx.set_weights(w0)
        if rank == 0:
            actx.async_host_master(w0)
        group.barrier()

        def run(seed, n_upd):
            actx.start_async(None, assigned, B_a, LR, concurrency=lanes, max_updates=n_upd, seed=seed)
            while actx.async_running():
                time.sleep(0.0002)
            actx.stop_async()
            return actx.async_elapsed_ms()

        run(7, U // 10)
        group.barrier()
        t0 = time.perf_counter()
        ms = run(11, U)
        wall = group.all_reduce_max(time.perf_counter() - t0)
        ms = group.all_reduce_max(ms)
        group.barrier()
        w_self = actx.get_weights()
        blobs = group.all_gather_bytes(w_self.tobytes())
        rec = {"mode": "async", "batch": B_a, "lanes_per_gpu": lanes, "n_gpus": world, "updates_per_gpu": U, "lr": LR,
               "value": U * B_a * world / (ms * 1e-3), "e2e_value": U * B_a * world / wall, "unit": UNIT,
               "us_per_update_per_lane": ms * 1e3 * lanes / U,
               "roofline_frac": U * B_a * mean_bytes / (ms * 1e-3) / 1e9 / hbm_peak,
               "label": ("one worker per GPU, sequential loop: the reference's Slave.asyncTask" if lanes == 1 else
                         f"EXTENSION: {lanes} Hogwild lanes per GPU on the GPU's replica (the reference runs one loop per slave)")}
        if rank == 0:
            ws = [np.frombuffer(b, dtype=np.float64) for b in blobs]
            w_master = actx.async_master_weights()
            loss, acc = actx.eval(n_train, data.n_rows, w_master)
            rec.update({"master_test_loss": loss, "master_test_acc": acc, "master_updates": int(actx.async_updates()),
                        "replica_max_abs_diff": float(max(np.max(np.abs(w - ws[0])) for w in ws)),
                        "replica_vs_master_max_abs_diff": float(np.max(np.abs(ws[0] - w_master)))})
        out.append(rec)
    actx.close()
    return out


def rpc_seam_record(ctx, data, n_train, d, B=256, reps=200):
    """The literal drop-in seam of SlaveImpl.gradient / SlaveImpl.forward (core/Slave.scala:129-157): weights arrive with the
    request (host buffer, 378 KB), the dense gradient / the predictions go back to the host, one blocking C-ABI call each;
    next to it the CPU port's time for the same request."""
    rng = np.random.default_rng(77)
    w = rng.standard_normal(data.dim) * 0.05
    idx = [rng.choice(n_train, size=B, replace=False).astype(np.int32) for _ in range(reps)]
    for i in range(10):
        ctx.gradient(idx[i], w); ctx.forward(idx[i], w)
    t = time.perf_counter()
    for i in range(reps):
        ctx.gradient(idx[i], w)
    g_us = (time.perf_counter() - t) / reps * 1e6
    t = time.perf_counter()
    for i in range(reps):
        ctx.forward(idx[i], w)
    f_us = (time.perf_counter() - t) / reps * 1e6
    t = time.perf_counter()
    for i in range(reps):
        ctx.gradient(idx[i], None)
    gr_us = (time.perf_counter() - t) / reps * 1e6
    orc = make_oracle(data, d)
    n_cpu = 50
    t = time.perf_counter()
    for i in range(n_cpu):
        orc.gradient(w, idx[i])
    cg_us = (time.perf_counter() - t) / n_cpu * 1e6
    t = time.perf_counter()
    for i in range(n_cpu):
        orc.forward(w, idx[i])
    cf_us = (time.perf_counter() - t) / n_cpu * 1e6
    return {"batch": B, "requests_timed": reps, "gradient_us_per_request": g_us, "forward_us_per_request": f_us,
            "gradient_resident_weights_us_per_request": gr_us,
            "h2d_bytes_per_request": data.dim * 8 + B * 4, "d2h_bytes_gradient": data.dim * 8, "d2h_bytes_forward": B * 8,
            "cpu_port_gradient_us_per_request": cg_us, "cpu_port_forward_us_per_request": cf_us,
            "samples_per_s_gradient": B / (g_us * 1e-6), "cpu_port_samples_per_s_gradient": B / (cg_us * 1e-6),
            "api": "dsgd_gradient / dsgd_forward (C ABI), weights passed with the request like GradientRequest.weights"}


def fit_record(ctx, group, data, n_train, rank, world, B, epochs=8):
    """samples/s through MasterSync.fit (the reference's public API for this path, core/Master.scala:120-218), everything
    inside the timed region: per-epoch batch draws on the host, H2D of the ids, the step loop, train/test loss and accuracy
    after every epoch, the weight read-back.  (8 epochs: the first epoch's draw cannot overlap anything -- the draw of epoch
    e + 1 runs on a host thread during epoch e -- and a real fit has tens of epochs; application.conf's default is 100.)"""
    from distributed_sgd_b200 import MasterSync, Slave, SparseSVM
    train, test = data.split_at(n_train)
    model = SparseSVM(LAMBDA)
    slave = Slave(rank, 0, train, model, world=world, test_data=test, ctx=ctx)
    # the ctx already carries its peer exchange: build the master around it without re-initialising it
    master = MasterSync(rank, train, test, model, world, slave=slave, group=group, seed=5, attach=False)
    never = lambda losses: False
    master.fit(np.zeros(data.dim), 1, B, LR, never)                 # warm-up epoch
    group.barrier()
    t0 = time.perf_counter()
    state = master.fit(np.zeros(data.dim), epochs, B, LR, never)
    dt = group.all_reduce_max(time.perf_counter() - t0)
    steps_per_epoch = -(-(n_train // world) // B)
    samples = sum(int(min(B, n_train // world - s * B)) for s in range(steps_per_epoch)) * world * epochs
    return {"value": samples / dt, "unit": UNIT, "epochs": epochs, "sgd_steps_per_epoch": steps_per_epoch,
            "seconds": dt, "final_train_loss": float(state.loss), "final_test_acc": float(master.history["test_accs"][-1]),
            "api": "MasterSync.fit (Python mirror of core/Master.scala:120-218 over the C ABI), epoch evaluations included"}


def bench_async(args, ctx, data, n_train, d, group, rank, local_rank, world):
    """`--mode async`: BASELINE.json configs[3] as the headline line.  A bench step = `--async-updates` worker iterations per
    GPU (device-side sampling), lr from application.conf."""
    from distributed_sgd_b200.native import REPLICA_MASTER, REPLICA_SELF
    B = args.batch
    U = args.async_updates
    w0 = np.zeros(data.dim)
    per = n_train // world
    assigned = np.arange(rank * per, (rank + 1) * per, dtype=np.int32)
    ctx.set_weights(w0)
    if rank == 0:
        ctx.async_host_master(w0)
    if world > 1:
        handles = group.all_gather_bytes(ctx.ipc_export(REPLICA_SELF))
        master = group.broadcast_bytes(ctx.ipc_export(REPLICA_MASTER) if rank == 0 else b"", 0)
        for k, h in enumerate(handles):
            if k != rank:
                ctx.ipc_import(k, h)
        if rank != 0:
            ctx.ipc_import(world, master)
    group.barrier()

    def run(seed):
        ctx.start_async(None, assigned, B, LR, concurrency=args.lanes, max_updates=U, seed=seed)
        while ctx.async_running():
            time.sleep(0.0002)
        ctx.stop_async()
        return ctx.async_elapsed_ms()

    for i in range(args.warmup):
        run(100 + i); group.barrier()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    launches0 = ctx.launch_count()
    ms_dev, t0 = 0.0, time.perf_counter()
    for i in range(args.steps):
        ms_dev += run(200 + i)
        group.barrier()
    wall = time.perf_counter() - t0
    launches = ctx.launch_count() - launches0
    clock_info = clocks.stop() if rank == 0 else None
    ms_dev = group.all_reduce_max(ms_dev)
    wall = group.all_reduce_max(wall)
    samples_total = args.steps * U * B * world
    value = samples_total / (ms_dev * 1e-3)
    e2e_value = samples_total / wall
    w_master = ctx.async_master_weights() if rank == 0 else None
    if rank == 0 and args.dump_outputs:      # Hogwild: the update order, hence the weights, differ from run to run
        dump_outputs(args.dump_outputs, {"master_weights": w_master})
    hbm_peak, peak_src = peaks()
    mean_bytes = data.algorithmic_bytes() / data.n_rows
    achieved = (args.steps * U * B * mean_bytes) / (ms_dev * 1e-3) / 1e9     # per GPU
    if rank == 0:
        orc = make_oracle(data, d)
        n_cpu = 20000
        idx = np.random.default_rng(3).integers(0, n_train, size=n_cpu * B).astype(np.int32)
        t = time.perf_counter(); orc.async_run(w0, idx, B, LR); dt = time.perf_counter() - t
        cpu = {"value": n_cpu * B / dt, "unit": UNIT, "cores": 1, "kind": "port",
               "sample": f"{n_cpu} sequential async iterations of batch {B} (one worker), {dt:.1f} s; the reference recomputes "
                         "w.dimSparsity (47 236 products) every iteration (core/ml/SparseSVM.scala:31) and so does this port"}
        loss, acc = ctx.eval(n_train, data.n_rows, w_master)
        print(json.dumps({
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"async Hogwild (configs[3]): RCV1-shaped synthetic, {DIM} feats, {args.rows} rows, batch {B}, "
                                   f"one worker per GPU, {args.lanes} Hogwild lanes per GPU, peer replica writes over NVLink",
                       "mode": "async", "batch": B, "lr": LR, "updates_per_gpu_per_step": U, "lanes": args.lanes,
                       "parallelism": f"dp{world}", "l2": "rows drawn at random from 0.43 GB of CSR (larger than the 126 MB L2)"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(assigned.nbytes), "d2h_bytes_per_step": 0,
                    "api": "dsgd_start_async ... dsgd_stop_async (C ABI)"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": "k_async_worker", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                         "frac": achieved / hbm_peak, "traffic": None, "peak_source": peak_src,
                         "note": "latency-bound by construction: each iteration is a dependent chain on one replica"},
            "cpu_baseline": cpu, "clocks": clock_info,
            "final_test_loss": loss, "final_test_acc": acc,
        }))
    ctx.close()
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus and "WORLD_SIZE" in os.environ:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")

    if args.impl == "reference":
        if rank != 0:
            return
        data, n_train = make_data(args)
        from oracle.oracle import Oracle
        d = Oracle(data.row_ptr, data.col, data.val, data.label, data.dim, LAMBDA).dim_sparsity(n_train)
        workers = args.gpus
        threads = min(workers, os.cpu_count() or 1)
        vals, secs = [], []
        desc = ""
        for i in range(args.warmup + args.steps):
            v, desc = cpu_leg(data, n_train, d, args.batch, workers, max(2.0, 60.0 / (args.warmup + args.steps)), threads,
                              args.seed + i)
            if i >= args.warmup:
                vals.append(v)
                secs.append(cpu_leg.last_seconds)
        value = float(np.mean(vals))
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": float(np.mean(secs)) * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": sync_config(args, workers, n_train, args.batch, args.sgd_steps or -(-n_train // args.batch)),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                             "sample": desc + " per step; fp64 array restatement of the Scala path (no JVM in this image)",
                             "all_cores": cpu_all_cores(data, n_train, d, args.batch, args.seed) if workers == 1 else None},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
        return

    import torch
    import torch.distributed as dist
    from distributed_sgd_b200.core import Group
    from distributed_sgd_b200.native import NativeCtx

    torch.cuda.set_device(local_rank)
    # stdout carries exactly ONE JSON line: keep NCCL's banner out of it, and use gloo for the control plane (a few
    # small host-side exchanges; the data path is the kernels' own peer-memory exchange)
    os.environ["NCCL_DEBUG"] = "WARN"
    if world > 1:
        dist.init_process_group(backend="gloo", rank=rank, world_size=world)
    group = Group()

    data, n_train = make_data(args)
    ctx = NativeCtx(local_rank, data.dim, LAMBDA, rank=rank, world=world, is_async=(args.mode == "async"))
    ctx.load_csr(data.row_ptr, data.col, data.val, data.label)   # every slave holds every row (quirk Q13)
    d = ctx.compute_dim_sparsity(n_train)
    use_nccl = bool(os.environ.get("BENCH_NCCL_PATH"))           # A/B: NCCL allreduce between the kernels of a step
    if world > 1 and args.mode == "sync":
        if use_nccl:
            uid = NativeCtx.comm_unique_id() if rank == 0 else b""
            ctx.comm_init(group.broadcast_bytes(uid, 0))
        else:
            ctx.setup_peer_exchange(group)   # fused step: gradients summed out of peer memory over NVLink

    if args.mode == "async":
        return bench_async(args, ctx, data, n_train, d, group, rank, local_rank, world)

    B = args.batch
    S = args.sgd_steps or -(-n_train // B)            # one epoch of the 1-worker fit loop: ceil(560000 / 256) = 2188
    per = n_train // world                             # SplitStrategy.vanilla: contiguous range per worker
    lo, hi = rank * per, (rank + 1) * per
    rng = np.random.default_rng(args.seed * 1000 + rank)
    total_steps = args.warmup + args.steps
    samples_np = draw_batches(rng, lo, hi, B, S * total_steps).reshape(total_steps, S * B)
    pinned = torch.empty((total_steps, S * B), dtype=torch.int32).pin_memory()
    pinned.numpy()[:] = samples_np
    alg_bytes_per_step = [data.algorithmic_bytes(samples_np[i]) for i in range(total_steps)]
    hbm_peak, peak_src = peaks()

    def barrier():
        ctx.synchronize()
        torch.cuda.synchronize()
        group.barrier()

    # ---- leg 1: device-resident (value) ---------------------------------------------------------------
    ctx.set_weights(np.zeros(data.dim))
    ctx.stage_samples(samples_np.reshape(-1))
    clocks = ClockSampler(local_rank)   # sampled every 20 ms over the warm-up (same workload) and the timed region
    if rank == 0:
        clocks.start()
        time.sleep(0.25)                # nvidia-smi needs a moment to start reporting
        clocks.mark()
    for i in range(args.warmup):
        ctx.sync_steps_staged(i * S * B, B, S, LR, want_losses=True)
    ctx.synchronize()
    # (read BEFORE the barrier: the first NVML query takes tens of ms on rank 0 alone, and a rank that starts its timed
    #  launches late keeps its peers spinning inside theirs -- with the query after the barrier `value` fell below `e2e`)
    nvl0 = nvlink_counters(local_rank) if (rank == 0 and world > 1) else None
    xs0 = ctx.xchg_stats() if world > 1 else None
    launches0 = ctx.launch_count()
    barrier()
    ctx.timer_start()
    for i in range(args.warmup, total_steps):
        ctx.sync_steps_staged(i * S * B, B, S, LR, want_losses=True)
    ms = ctx.timer_stop()
    launches = ctx.launch_count() - launches0
    barrier()
    nvl1 = nvlink_counters(local_rank) if (rank == 0 and world > 1) else None
    xs1 = ctx.xchg_stats() if world > 1 else None
    clock_info = clocks.stop() if rank == 0 else None
    ms = group.all_reduce_max(ms)
    samples_total = args.steps * S * B * world
    value = samples_total / (ms * 1e-3)
    w_after = ctx.get_weights()
    last_losses = ctx.read_losses(S)
    if rank == 0 and args.dump_outputs:      # replicas are bit-identical and the losses cover every worker's samples
        dump_outputs(args.dump_outputs, {"weights": w_after, "losses": last_losses})

    # ---- leg 2: end to end through the C-ABI call with host buffers (e2e) --------------------------------
    ctx.set_weights(np.zeros(data.dim))
    for i in range(args.warmup):
        ctx.sync_steps(pinned[i].numpy(), B, S, LR, want_losses=True)
    barrier()
    t0 = time.perf_counter()
    for i in range(args.warmup, total_steps):
        losses_host = ctx.sync_steps(pinned[i].numpy(), B, S, LR, want_losses=True)
    ctx.synchronize()
    e2e_s = group.all_reduce_max(time.perf_counter() - t0)
    barrier()
    e2e_value = samples_total / e2e_s
    # both legs walked the same batches from the same start: identical results expected
    same = bool(np.array_equal(ctx.get_weights(), w_after)) if world == 1 else None

    # ---- leg 3: mean duration of the dominant kernel over the same work -----------------------
    ctx.set_weights(np.zeros(data.dim))
    ctx.stage_samples(samples_np.reshape(-1))   # leg 2 re-staged one bench step at a time
    ctx.profile_begin(sample_every=1)
    for i in range(args.warmup, total_steps):
        ctx.sync_steps_staged(i * S * B, B, S, LR, want_losses=False)
    k_ms, k_n = ctx.profile_end()
    barrier()
    # every launch of the dominant kernel was bracketed: algorithmic bytes of the region / launches
    alg_per_launch = float(np.sum(alg_bytes_per_step[args.warmup:])) / max(k_n, 1)
    achieved = alg_per_launch / (k_ms * 1e-3) / 1e9 if k_ms > 0 else 0.0
    persistent = (k_n == args.steps)
    kernel_name = ("k_sync_persistent (whole run of %d SGD steps per launch)" % S) if persistent \
        else "k_rows<scatter> (gradient, one launch per SGD step)"
    step_frac = (float(np.mean(alg_bytes_per_step[args.warmup:])) * args.steps / (ms * 1e-3) / 1e9) / hbm_peak
    traffic_rec, traffic_src = ncu_traffic("k_sync_persistent_multi" if world > 1 else "k_sync_persistent") if persistent else (None, "n/a")
    traffic = float(traffic_rec["dram_bytes_per_sgd_step_batch256"]) * (B / 256.0) * S if traffic_rec else None

    # ---- leg 3b: the same row kernels where they are bandwidth- rather than latency-bound -----------------------
    # (batch 256 moves 197 KB per step; the HBM roofline of the path shows on the full-shard evaluation pass,
    #  Master.localLoss/localAccuracy, and on the gradient of a very large batch -- SURVEY.md 8d "Expected regime")
    streaming = None
    if rank == 0:
        def best_ms(fn, reps=5):
            fn(); ctx.synchronize()
            ts = []
            for _ in range(reps):
                ctx.profile_begin(1); fn(); t_ms, _n = ctx.profile_end(); ts.append(t_ms)
            return min(ts)
        ev_bytes = data.algorithmic_bytes(np.arange(n_train))
        ev_ms = best_ms(lambda: ctx.eval(0, n_train))
        big = np.random.default_rng(1).choice(n_train, size=min(262144, n_train), replace=False).astype(np.int32)
        gr_bytes = data.algorithmic_bytes(big)
        gr_ms = best_ms(lambda: ctx.gradient(big))
        w_trained = ctx.get_weights()
        gr0_ms = best_ms(lambda: ctx.gradient(big, np.zeros(data.dim)))
        tr_e, tr_e_src = ncu_traffic("k_stream_rows_eval")
        tr_g, _ = ncu_traffic("k_stream_rows_scatter")
        streaming = {
            "eval_full_train_pass": {"kernel": "k_stream_rows<eval>", "rows": int(n_train), "ms": ev_ms,
                                     "achieved": ev_bytes / ev_ms / 1e6, "unit": "GB/s", "frac": ev_bytes / ev_ms / 1e6 / hbm_peak,
                                     "algorithmic_bytes": ev_bytes, "traffic": tr_e["dram_bytes"] if tr_e else None},
            "gradient_batch_%d" % len(big): {"kernel": "k_stream_rows<scatter>", "rows": int(len(big)), "ms": gr_ms,
                                             "achieved": gr_bytes / gr_ms / 1e6, "unit": "GB/s",
                                             "frac": gr_bytes / gr_ms / 1e6 / hbm_peak, "algorithmic_bytes": gr_bytes,
                                             "traffic": tr_g["dram_bytes"] if tr_g else None,
                                             "weights": "trained (the resident weights after the timed legs): the rows that pass "
                                                        "the gate are the misclassified ones"},
            "gradient_batch_%d_untrained" % len(big): {
                "kernel": "k_stream_rows<scatter>", "rows": int(len(big)), "ms": gr0_ms, "achieved": gr_bytes / gr0_ms / 1e6,
                "unit": "GB/s", "frac": gr_bytes / gr0_ms / 1e6 / hbm_peak,
                "weights": "w = 0: EVERY row passes the gate (SparseSVM.scala:28), the scatter is bound by the fp64 RED rate at "
                           "L2, not by HBM"},
        }
        ctx.set_weights(w_trained)
    barrier()

    extras = {}
    if not args.no_extras:
        # ---- configs[4] sweep, sync side ----
        extras["sweep"] = sweep_record(ctx, group, data, n_train, rank, world, hbm_peak)
        # ---- parity of a fresh trajectory against the oracle, in this run ----
        extras["parity"] = parity_record(ctx, group, data, n_train, d, B, rank, world)
        # ---- e2e through MasterSync.fit ----
        try:
            extras["e2e_fit"] = fit_record(ctx, group, data, n_train, rank, world, B)
        except Exception as e:  # the headline line must not die on a sub-record
            extras["e2e_fit"] = {"error": repr(e)}
        # ---- configs[3] async Hogwild ----
        try:
            extras["async"] = async_record(args, group, data, n_train, rank, local_rank, world, hbm_peak)
        except Exception as e:
            extras["async"] = {"error": repr(e)}
        if rank == 0 and world == 1:
            extras["rpc_seam"] = rpc_seam_record(ctx, data, n_train, d)
    barrier()

    # ---- CPU baseline on this host (rank 0, N = 1 only) -------------------------------------------
    cpu = None
    if rank == 0 and world == 1:
        v, desc = cpu_leg(data, n_train, d, B, 1, args.cpu_seconds, 1, args.seed)
        cpu = {"value": v, "unit": UNIT, "cores": 1, "kind": "port",
               "sample": desc + "; fp64 array restatement of the Scala path, one thread per worker like the reference "
                                "(core/Slave.scala:142); host has %d cores" % (os.cpu_count() or 0),
               "all_cores": cpu_all_cores(data, n_train, d, B, args.seed)}

    if rank == 0:
        nvlink = None
        if world > 1 and xs0 and xs1:
            dv, db, dn = (xs1[0] - xs0[0]), (xs1[1] - xs0[1]), max(xs1[2] - xs0[2], 1)
            nvlink = {"stored_bytes_per_sgd_step_rank0": (16 * dv + 8 * db) * (world - 1) / dn,
                      "value_words_per_peer_per_step": dv / dn, "bitmap_words_per_peer_per_step": db / dn,
                      "dense_exchange_bytes_per_sgd_step": (world - 1) * (data.dim + 1) * 16,
                      "source": "counted by the kernel (dsgd_xchg_stats): 16-byte value words + 8-byte bitmap words x (N - 1) peers"}
            if nvl0 and nvl1:
                nvlink["nvml_tx_bytes_per_sgd_step_rank0"] = (nvl1[0] - nvl0[0]) / (args.steps * S)
                nvlink["nvml_rx_bytes_per_sgd_step_rank0"] = (nvl1[1] - nvl0[1]) / (args.steps * S)
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": sync_config(args, world, n_train, B, S),
            "us_per_sgd_step": ms * 1e3 / (args.steps * S),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(S * B * 4), "d2h_bytes_per_step": int(S * 8),
                    "api": "dsgd_sync_steps (C ABI, pinned host buffers)", "matches_device_leg": same},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": kernel_name, "achieved": achieved, "peak": hbm_peak,
                         "unit": "GB/s", "frac": achieved / hbm_peak,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_per_launch, "kernel_ms": k_ms,
                         "launches_sampled": int(k_n), "whole_step_frac": step_frac},
            "roofline_streaming": streaming,
            "cpu_baseline": cpu,
            "clocks": clock_info,
            "exchange": ("nccl allreduce between kernels" if use_nccl else "fused: sparse LL words over peer memory") if world > 1 else None,
            "nvlink": nvlink,
            "final_batch_loss": float(last_losses[-1]),
            # fingerprints of the device-resident leg, for tools/verify_bench_loss.py (oracle replay of the same run)
            "final_weights_l1": float(np.abs(w_after).sum()), "final_weights_nnz": int(np.count_nonzero(w_after)),
        }
        out.update(extras)
        print(json.dumps(out))
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
