#!/usr/bin/env python
"""models_bench.py -- throughput of a model set (dsgd_models_steps) against the same settings run one after the other.

  python tools/models_bench.py [--models 1,2,4,8,16,32] [--repeats 5] [--out profiles/models/NAME.json]

Workload: bench.py's sync workload -- RCV1-shaped synthetic rows (47 236 features, 700 000 rows, seed as bench.py), batch
256 -- over one epoch-sized slice of the fit loop (ceil(560 000 / 256) = 2 188 steps).  For every M, M distinct
(lambda, lr) settings:
  model_set   ONE dsgd_models_steps call training all M settings on the slice;
  sequential  M dsgd_sync_steps calls on the same slice, one per learning rate, each from w = 0 (the ctx has one lambda;
              lambda does not change the work of a step).
Both arms are timed with the ctx's CUDA events (dsgd_timer_start / dsgd_timer_stop) around the public calls, so the host
gaps between calls count; every shape is warmed up first; the arms alternate over the repeats; median and spread are
reported.  `model_samples_per_s` counts samples x models.  `parity`: a 300-step prefix of the M = 8 set against the fp64
oracle run once per setting (the fields of bench.py's parity record, worst over the models).  The card's name and power
limit are read in the same run (query only).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bench  # noqa: E402  (the workload: make_data, draw_batches, LAMBDA, LR)


def settings(M):
    """M distinct (lambda, lr): lambdas around the reference's 1e-5, learning rates around its 0.5."""
    lams = [bench.LAMBDA * 10.0 ** ((m % 4) - 1) for m in range(M)]
    lrs = [bench.LR * (0.25 + 0.125 * (m // 4 + m % 4)) for m in range(M)]
    return lams, lrs


def card():
    q = "name,power.limit,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=30)
        name, power, clk = [x.strip() for x in r.stdout.strip().split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clk, "source": "nvidia-smi --query-gpu (query only)"}
    except Exception as e:   # the measurement stands without it, but says so
        return {"name": None, "error": str(e)}


def parity(ctx, data, d, samples, B, lams, lrs, steps=300):
    from oracle.oracle import Oracle
    idx = samples[:steps * B]
    ctx.models_set(lams, lrs)
    losses = ctx.models_steps(idx, B, steps)
    W = ctx.models_get_weights()
    worst = {"max_rel_err_loss": 0.0, "max_rel_err_weights": 0.0, "support_equal": True}
    for m, (lam, lr) in enumerate(zip(lams, lrs)):
        orc = Oracle(data.row_ptr, data.col, data.val, data.label, data.dim, lam)
        orc.set_dim_sparsity(d)
        w_ref, l_ref = orc.sync_steps(np.zeros(data.dim), idx, [B], lr, n_steps=steps)
        nz = w_ref != 0
        worst["max_rel_err_loss"] = max(worst["max_rel_err_loss"], float(np.max(np.abs(losses[:, m] - l_ref) / np.abs(l_ref))))
        if nz.any():
            worst["max_rel_err_weights"] = max(worst["max_rel_err_weights"],
                                               float(np.max(np.abs(W[m][nz] - w_ref[nz]) / np.abs(w_ref[nz]))))
        worst["support_equal"] = worst["support_equal"] and bool(np.array_equal(W[m] != 0, nz))
    return {"steps": steps, "models": len(lams), "batch": B, **worst,
            "checker": "oracle/dsgd_oracle.c (fp64 CPU restatement of core/Master.scala:184-197), once per setting, "
                       "same batch draws"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--models", default="1,2,4,8,16,32")
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--rows", type=int, default=bench.N_ROWS)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--sgd-steps", type=int, default=0, help="steps of the slice (0: one epoch, ceil(n_train / batch))")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default=None, help="also write the JSON record to this file")
    args = ap.parse_args()
    from distributed_sgd_b200.native import NativeCtx

    data, n_train = bench.make_data(argparse.Namespace(rows=args.rows, seed=args.seed))
    B = args.batch
    S = args.sgd_steps or -(-n_train // B)
    samples = bench.draw_batches(np.random.default_rng(args.seed * 1000), 0, n_train, B, S).reshape(-1)
    ctx = NativeCtx(0, data.dim, bench.LAMBDA)
    ctx.load_csr(data.row_ptr, data.col, data.val, data.label)
    d = ctx.compute_dim_sparsity(n_train)
    w0 = np.zeros(data.dim)
    Ms = [int(x) for x in args.models.split(",")]

    def run_set(lams, lrs):
        ctx.models_set(lams, lrs)                   # allocation and initial weights: outside the timed window
        ctx.timer_start()
        ctx.models_steps(samples, B, S, want_losses=False)
        return ctx.timer_stop()

    def run_seq(lrs):
        ctx.timer_start()
        for lr in lrs:
            ctx.set_weights(w0)
            ctx.sync_steps(samples, B, S, lr, want_losses=False)
        return ctx.timer_stop()

    for M in Ms:                                     # warm-up of every shape
        lams, lrs = settings(M)
        run_set(lams, lrs)
        run_seq(lrs[:1])
    times = {M: {"set": [], "seq": []} for M in Ms}
    for _ in range(args.repeats):                    # alternate the arms
        for M in Ms:
            lams, lrs = settings(M)
            times[M]["set"].append(run_set(lams, lrs))
            times[M]["seq"].append(run_seq(lrs))

    def stats(ms, M):
        a = np.array(ms)
        med = float(np.median(a))
        return {"ms_median": med, "ms_min": float(a.min()), "ms_max": float(a.max()),
                "spread_pct": float((a.max() - a.min()) / med * 100.0),
                "us_per_step": med * 1e3 / S, "model_samples_per_s": M * S * B / (med * 1e-3)}

    rows = []
    for M in Ms:
        st, sq = stats(times[M]["set"], M), stats(times[M]["seq"], M)
        rows.append({"models": M, "model_set": st, "sequential": sq,
                     "speedup_vs_sequential": st["model_samples_per_s"] / sq["model_samples_per_s"]})
    single = next((r["sequential"] for r in rows if r["models"] == 1), None)
    base_set = next((r["model_set"] for r in rows if r["models"] == 1), None)
    for r in rows:
        if single:
            r["vs_single_model_sync_steps"] = r["model_set"]["model_samples_per_s"] / single["model_samples_per_s"]
        if base_set and r["models"] > 1:
            r["us_per_step_per_extra_model"] = (r["model_set"]["us_per_step"] - base_set["us_per_step"]) / (r["models"] - 1)
    lams8, lrs8 = settings(8)
    rec = {"tool": "tools/models_bench.py", "card": card(), "device": ctx.info(),
           "workload": f"RCV1-shaped synthetic, {data.dim} feats, {args.rows} rows ({n_train} train), batch {B}, "
                       f"{S} steps per call (one epoch-sized slice), seed {args.seed}",
           "timing": f"CUDA events around the public calls, median of {args.repeats} alternated repeats after a warm-up",
           "settings": "lambda = 1e-5 * 10^((m % 4) - 1), lr = 0.5 * (0.25 + 0.125 * (m // 4 + m % 4))",
           "rows": rows, "parity": parity(ctx, data, d, samples, B, lams8, lrs8)}
    ctx.close()
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(rec, indent=1) + "\n")


if __name__ == "__main__":
    main()
