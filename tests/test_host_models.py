"""MasterSync.fit_models and the --lambdas / --learning-rates sweep on the host, over a stand-in device context that
records what would go to the GPU (no arithmetic): the epoch loop runs once for all settings, each setting is frozen at
the epoch its own test losses stop it, and the shapes a model set cannot take are refused."""
import numpy as np
import pytest


class _ModelsCtx:
    """Model-set calls of NativeCtx; model m's test loss after epoch e is losses[m][e - 1]."""

    def __init__(self, dim, losses):
        self.dim, self.losses, self.calls = dim, losses, []

    def set_weights(self, w):
        pass

    def models_set(self, lambdas, learning_rates, w0=None):
        self.M, self.epoch = len(lambdas), 0
        self.calls.append(("set", list(lambdas), list(learning_rates)))

    def models_steps(self, samples, n_per_step, n_steps, active=None, want_losses=True):
        self.calls.append(("steps", n_per_step, n_steps, np.asarray(active).tolist()))
        return np.zeros((n_steps, self.M))

    def models_get_weights(self):
        self.epoch += 1
        return np.zeros((self.M, self.dim))

    def models_eval_counts(self, m, lo, hi):
        n = hi - lo
        return int(round(self.losses[m][self.epoch - 1] * n)), 0, 0.0


def _master(losses, n_train=9, n_test=5, dim=8, world=1):
    from types import SimpleNamespace
    from distributed_sgd_b200.core.master import MasterSync
    from distributed_sgd_b200.ml import SparseSVM
    from distributed_sgd_b200.utils.dataset import Data
    stub = lambda n: Data(np.arange(n + 1, dtype=np.int64), np.zeros(n, np.int32), np.ones(n, np.float32), np.ones(n, np.int8), dim)
    slave = SimpleNamespace(ctx=_ModelsCtx(dim, losses), world=1, is_async=False, n_train=n_train, n_test=n_test, dim=dim)
    m = MasterSync(0, stub(n_train), stub(n_test), SparseSVM(0.1), 1, slave=slave, seed=0)
    return m, slave.ctx


def test_fit_models_freezes_each_setting_where_fit_would_return():
    from distributed_sgd_b200.ml import EarlyStopping
    # model 0 improves every epoch; model 1 stops improving after epoch 1; model 2 after epoch 2
    losses = [[0.8, 0.6, 0.4, 0.2], [0.4, 0.6, 0.6, 0.6], [0.8, 0.2, 0.6, 0.6]]
    m, ctx = _master(losses, n_test=5)
    stop = EarlyStopping.no_improvement(patience=1, min_delta=0.0)
    states = m.fit_models(np.zeros(8), 4, 4, [0.0, 1e-5, 1e-3], [0.5, 0.5, 0.1], stop)
    assert [s.updates for s in states] == [4, 2, 3]
    steps = [c for c in ctx.calls if c[0] == "steps"]
    # 9 train rows, batch 4: steps of 4, 4 and 1 rows -> two calls per epoch (counts 4 then 1)
    assert [(c[1], c[2]) for c in steps[:2]] == [(4, 2), (1, 1)]
    assert [c[3] for c in steps[::2]] == [[True, True, True], [True, True, True], [True, False, True], [True, False, False]]
    assert [h["test_losses"] for h in m.histories] == [losses[0], losses[1][:2], losses[2][:3]]
    assert states[1].loss == m.histories[1]["losses"][-1]


def test_fit_models_refuses_shapes_a_model_set_cannot_take():
    m, _ = _master([[1.0]])
    with pytest.raises(ValueError, match="1 to 32"):
        m.fit_models(np.zeros(8), 1, 4, [1e-5] * 33, [0.5] * 33, lambda l: False)
    with pytest.raises(ValueError, match="1 to 32"):
        m.fit_models(np.zeros(8), 1, 4, [1e-5, 1e-4], [0.5], lambda l: False)
    with pytest.raises(ValueError, match="one worker"):
        m.fit_models(np.zeros(8), 1, 4, [1e-5], [0.5], lambda l: False, split_strategy=lambda n, k: [range(0, 4), range(4, n)])
    m.group.world = 2
    with pytest.raises(ValueError, match="one GPU"):
        m.fit_models(np.zeros(8), 1, 4, [1e-5], [0.5], lambda l: False)


def test_sweep_refuses_several_workers_or_processes():
    from types import SimpleNamespace
    from distributed_sgd_b200.main import scenario
    cfg = SimpleNamespace(lam=1e-5, learning_rate=0.5, is_async=False, node_count=2)
    with pytest.raises(ValueError, match="node-count is 2"):
        scenario(cfg, None, lambdas=[1e-5, 1e-4])
    cfg.node_count = 1
    with pytest.raises(ValueError, match="2 processes"):
        scenario(cfg, None, world=2, learning_rates=[0.1, 0.5])
    with pytest.raises(ValueError, match="makes 36 settings"):
        scenario(cfg, None, lambdas=[1e-5 * i for i in range(1, 7)], learning_rates=[0.1 * i for i in range(1, 7)])
