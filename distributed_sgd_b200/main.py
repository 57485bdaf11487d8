"""Main.scala -- the reference's entry point, as a calling sequence over this package.

    python -m distributed_sgd_b200.main [--conf application.conf] [--synthetic-rows N]
    torchrun --nproc-per-node K -m distributed_sgd_b200.main ...

Mirrors `Main.scenario` (Main.scala:70-120): load the `dsgd` configuration (file and/or DSGD_* variables,
Main.scala:36), load the data (Main.scala:47-49; RCV1 text files from `data-path`, or RCV1-shaped synthetic rows when
`--synthetic-rows` is given because no RCV1 copy ships here), 80/20 split by position (:52), dimSparsity (:54-65, on
the device), model (:68), initial distributed loss / accuracy (:75-78), fit (:80-112), final test loss / accuracy
(:115-118).  One process per GPU; `node-count` reference workers are spread over the GPUs as logical workers
(node-count must be a multiple of the number of processes).  Prints one JSON report (the reference logs text).
"""
from __future__ import annotations

import argparse
import json
import os
import time
from typing import Optional, Sequence

import numpy as np


def scenario(cfg, data, *, rank: int = 0, world: int = 1, device: Optional[int] = None, seed: int = 0, log=print,
             async_concurrency: int = 64, jvm_exact: bool = False, inspect=None,
             lambdas: Optional[Sequence[float]] = None, learning_rates: Optional[Sequence[float]] = None) -> dict:
    """Main.scenario (Main.scala:70-120).  inspect (tests): called as inspect("master", master) once the master exists
    and as inspect("done", (master, state)) before the device context is released.

    lambdas / learning_rates (sync mode, one GPU, node-count 1): train every (lambda, learning rate) of their Cartesian
    product (missing list: the configured value) as one model set (MasterSync.fit_models); the report then has one entry
    per setting under "settings" and the index of the lowest final test loss under "best"."""
    from . import EarlyStopping, Master, Slave, SparseSVM
    from .core import Group
    from .native import MAX_MODELS

    sweep = None
    if lambdas is not None or learning_rates is not None:
        sweep = [(float(a), float(b)) for a in (lambdas if lambdas is not None else [cfg.lam])
                 for b in (learning_rates if learning_rates is not None else [cfg.learning_rate])]
        if cfg.is_async:
            raise ValueError("--lambdas / --learning-rates train a model set in sync mode; async is set")
        if cfg.node_count != 1 or world != 1:
            raise ValueError(f"--lambdas / --learning-rates train a model set on one GPU with one worker: node-count is "
                             f"{cfg.node_count} and the run has {world} processes (both must be 1)")
        if not 1 <= len(sweep) <= MAX_MODELS:
            raise ValueError(f"--lambdas x --learning-rates makes {len(sweep)} settings; a model set holds 1 to {MAX_MODELS}")

    train, test = data.split_at(int(data.n_rows * 0.8))                       # Main.scala:52
    model = SparseSVM(cfg.lam)                                                 # dimSparsity: computed by the Slave on the device
    slave = Slave(rank, 0, train, model, cfg.is_async, world=world, device=device, test_data=test)
    master = Master.create(rank, train, test, model, cfg.is_async, cfg.node_count, slave=slave, group=Group(), seed=seed,
                           log=(log if rank == 0 else None), jvm_exact=jvm_exact)
    if inspect:
        inspect("master", master)
    w0 = np.zeros(data.dim)                                                    # data(0)._1.zerosLike (Main.scala:74)
    report = {"config": {k: getattr(cfg, k) for k in ("batch_size", "learning_rate", "lam", "node_count", "is_async",
                                                      "max_epochs", "check_every", "leaky_loss", "patience", "conv_delta")},
              "rows": {"train": train.n_rows, "test": test.n_rows}, "world": world}
    report["initial_loss"] = master.distributed_loss(w0)                      # Main.scala:75-76
    report["initial_accuracy"] = master.distributed_accuracy(w0)              # Main.scala:77-78
    stop = EarlyStopping.no_improvement(patience=cfg.patience, min_delta=cfg.conv_delta, min_steps=None)
    t0 = time.perf_counter()
    if sweep is not None:
        states = master.fit_models(w0, cfg.max_epochs, cfg.batch_size, [a for a, _ in sweep], [b for _, b in sweep], stop)
        report["fit_seconds"] = time.perf_counter() - t0
        n_tr, n_te = train.n_rows, test.n_rows
        settings = []
        for (lam, lr), st, hist in zip(sweep, states, master.histories):
            h, c, n2 = master.ctx.eval_counts(n_tr, n_tr + n_te, st.grad)                  # Main.scala:115-118
            settings.append({"config": {"lam": lam, "learning_rate": lr},
                             "history": {k: [float(x) for x in v] for k, v in hist.items()},
                             "final_test_loss": lam * n2 + h / n_te, "final_test_accuracy": c / n_te,
                             "final_weights_nonzero": int(np.count_nonzero(st.grad)), "updates": st.updates})
        report["settings"] = settings
        report["best"] = int(np.argmin([s["final_test_loss"] for s in settings]))
        if inspect:
            inspect("done", (master, states))
        slave.stop()
        return report
    if cfg.is_async:                                                          # Main.scala:82-96
        state = master.fit(w0, cfg.max_epochs, cfg.batch_size, cfg.learning_rate, stop, check_every=cfg.check_every,
                           leak_loss_coef=cfg.leaky_loss, concurrency=async_concurrency, seed=seed)
    else:                                                                      # Main.scala:97-109
        if cfg.node_count % world:
            raise ValueError(f"node-count {cfg.node_count} is not a multiple of the {world} GPU processes")
        state = master.fit(w0, cfg.max_epochs, cfg.batch_size, cfg.learning_rate, stop,
                           virtual_workers=cfg.node_count // world)
    report["fit_seconds"] = time.perf_counter() - t0                          # Measure.durationLog(log, "fit") (Main.scala:80)
    w1 = state.grad
    report["history"] = {k: [float(x) for x in v] for k, v in getattr(master, "history", {}).items()
                         if isinstance(v, list) and all(isinstance(x, (int, float)) for x in v)}
    report["final_test_loss"], report["final_test_accuracy"] = master.local_loss_accuracy(w1, test_data=True)  # :115-118
    report["final_weights_nonzero"] = int(np.count_nonzero(w1))
    report["updates"] = state.updates
    if inspect:
        inspect("done", (master, state))
    slave.stop()
    return report


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--conf", default=None, help="application.conf (HOCON `dsgd { }` block); DSGD_* variables override")
    ap.add_argument("--synthetic-rows", type=int, default=0, help="use RCV1-shaped synthetic rows instead of data-path")
    ap.add_argument("--seed", type=int, default=0)                            # Random.setSeed(0) (Main.scala:32)
    ap.add_argument("--jvm-exact", action="store_true",
                    help="sync mode: draw the batches from java.util.Random(seed) + Scala's Random.shuffle like the reference")
    ap.add_argument("--lambdas", default=None,
                    help="sync, one GPU: comma-separated lambdas; with --learning-rates, train their Cartesian product as a "
                         "model set (at most 32 settings) and report every setting")
    ap.add_argument("--learning-rates", default=None, help="comma-separated learning rates (see --lambdas)")
    args = ap.parse_args(argv)
    lambdas = [float(x) for x in args.lambdas.split(",")] if args.lambdas else None
    learning_rates = [float(x) for x in args.learning_rates.split(",")] if args.learning_rates else None
    from .utils import load_config, rcv1, synthetic_rcv1

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group(backend="gloo", rank=rank, world_size=world)
    cfg = load_config(args.conf)
    data = synthetic_rcv1(n_rows=args.synthetic_rows, seed=args.seed) if args.synthetic_rows else rcv1(cfg.data_path, full=cfg.full)
    report = scenario(cfg, data, rank=rank, world=world, device=local_rank, seed=args.seed,
                      log=lambda s: print(s, flush=True), jvm_exact=args.jvm_exact, lambdas=lambdas,
                      learning_rates=learning_rates)
    if rank == 0:
        print(json.dumps(report))
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    raise SystemExit(main())
