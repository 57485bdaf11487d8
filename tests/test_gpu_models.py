"""Model sets (dsgd_models_*, MasterSync.fit_models): several (lambda, learning rate) settings trained on the same batch
draws in one persistent kernel, against the fp64 oracle run once per setting.  Tolerances as in test_gpu_parity.py:
losses rtol 1e-12, weight supports equal, weights rtol 1e-11 / atol 1e-15, integer counters exact."""
import numpy as np
import pytest

from helpers import data_from_csr, make_pair

pytestmark = pytest.mark.gpu

RTOL = 1e-12
LAMS = [0.0, 1e-5, 1e-4, 1e-3, 1e-5]
LRS = [0.1, 0.5, 1.0, 0.3, 0.7]


@pytest.fixture(scope="module")
def synth():
    from distributed_sgd_b200.utils import synthetic_rcv1
    return synthetic_rcv1(n_rows=6000, seed=3)


def oracle_for(orc, lam):
    """An oracle over the same rows and dimSparsity with another lambda."""
    from oracle.oracle import Oracle
    o = Oracle(orc.row_ptr, orc.col, orc.val, orc.label, orc.dim, lam)
    o.set_dim_sparsity(orc.d)
    return o


def draws(rng, n_rows, batch, steps):
    return np.stack([rng.choice(n_rows, size=batch, replace=False) for _ in range(steps)]).astype(np.int32)


def start_weights(rng, dim, M):
    """Zeros for the even models, sparse random weights for the odd ones (c != 0 from the first step)."""
    w0 = np.zeros((M, dim))
    for m in range(1, M, 2):
        w0[m] = np.where(rng.random(dim) < 0.3, rng.standard_normal(dim) * 0.05, 0.0)
    return w0


def check_against_oracle(orc, w0, idx, batch, losses, W, lams=LAMS, lrs=LRS, atol=1e-15):
    """atol None: 1e-13 * max|w| -- fp64 sums in another order whose result cancels to far below the summands keep an
    absolute error at the summands' scale (as in smoke()); needed once weights reach O(1) or c is large."""
    steps = idx.shape[0]
    for m, (lam, lr) in enumerate(zip(lams, lrs)):
        w_ref, l_ref = oracle_for(orc, lam).sync_steps(w0[m], idx.reshape(-1), [batch], lr, n_steps=steps)
        np.testing.assert_allclose(losses[:, m], l_ref, rtol=RTOL, err_msg=f"model {m}")
        assert (W[m] == 0).tolist() == (w_ref == 0).tolist(), f"model {m}: weight supports differ"
        np.testing.assert_allclose(W[m], w_ref, rtol=1e-11, err_msg=f"model {m}",
                                   atol=1e-13 * float(np.abs(w_ref).max()) if atol is None else atol)


def settings_for(M):
    """M (lambda, learning rate) settings: the five above for M = 5, else lambda 0 then 1e-6 .. 1e-2 geometrically with
    learning rates 1 .. 0.05 evenly (the largest lambda with the smallest rate: lambda 1e-2 at rate 1 diverges)."""
    if M == len(LAMS):
        return LAMS, LRS
    return [0.0] + list(np.geomspace(1e-6, 1e-2, M - 1)), list(np.linspace(1.0, 0.05, M))


@pytest.mark.parametrize("batch,steps,M", [
    pytest.param(1, 40, 5, id="1-40"), pytest.param(16, 60, 5, id="16-60"), pytest.param(256, 30, 5, id="256-30"),
    # models 8-31 are read through the shuffle groups 1-3 of acc_read_models and use the per-model slots k >= 8
    pytest.param(256, 20, 8, id="256-20-M8"), pytest.param(256, 20, 9, id="256-20-M9"),
    pytest.param(256, 20, 16, id="256-20-M16"), pytest.param(256, 20, 32, id="256-20-M32"),
    pytest.param(1, 20, 32, id="1-20-M32")])
def test_model_set_trajectories(synth, batch, steps, M):
    rng = np.random.default_rng(100 + batch + (M if M != len(LAMS) else 0))
    lams, lrs = settings_for(M)
    ctx, orc = make_pair(synth, lam=1e-5, n_train=4800)
    idx = draws(rng, 4800, batch, steps)
    w0 = start_weights(rng, synth.dim, M)
    ctx.models_set(lams, lrs, w0)
    losses = ctx.models_steps(idx.reshape(-1), batch, steps)
    assert losses.shape == (steps, M)
    check_against_oracle(orc, w0, idx, batch, losses, ctx.models_get_weights(), lams, lrs,
                         atol=1e-15 if M == len(LAMS) else None)
    ctx.close()


def test_several_calls_continue_one_trajectory(synth):
    rng = np.random.default_rng(7)
    batch = 64
    ctx, orc = make_pair(synth, lam=1e-5, n_train=4800)
    idx = draws(rng, 4800, batch, 30)
    w0 = start_weights(rng, synth.dim, len(LAMS))
    ctx.models_set(LAMS, LRS, w0)
    losses = np.concatenate([ctx.models_steps(idx[s:s + 10].reshape(-1), batch, 10) for s in (0, 10, 20)])
    W3 = ctx.models_get_weights()
    check_against_oracle(orc, w0, idx, batch, losses, W3)
    ctx.models_set(LAMS, LRS, w0)                                          # one call of 30 steps
    np.testing.assert_allclose(ctx.models_steps(idx.reshape(-1), batch, 30), losses, rtol=RTOL)
    np.testing.assert_allclose(ctx.models_get_weights(), W3, rtol=1e-11, atol=1e-15)
    ctx.close()


def test_known_answer_ka4_through_a_one_model_set():
    # KA4 (SURVEY 8c): x = {key 1 -> 1.0}, y = +1, w0 = 0, lr = 0.5
    data = data_from_csr([0, 1], [0], [1.0], [1], 4)
    ctx, _ = make_pair(data, lam=1e-5)
    ctx.models_set([1e-5], [0.5])
    assert ctx.models_steps([0], 1, 1)[0, 0] == 1.0
    np.testing.assert_array_equal(ctx.models_get_weights()[0], [-0.5, 0, 0, 0])
    assert ctx.models_eval_counts(0, 0, 1)[:2] == (0, 1)                   # pred == y: hinge 0, one correct
    ctx.models_steps([0], 1, 1)                                            # activity < 0: empty support, no change
    np.testing.assert_array_equal(ctx.models_get_weights()[0], [-0.5, 0, 0, 0])
    ctx.close()


@pytest.mark.parametrize("batch", [16, 256])
def test_one_model_set_equals_sync_steps(synth, batch):
    rng = np.random.default_rng(11)
    lam, lr, steps = 1e-4, 0.5, 40
    ctx, _ = make_pair(synth, lam=lam, n_train=4800)
    idx = draws(rng, 4800, batch, steps)
    ctx.set_weights(np.zeros(synth.dim))
    l_ref = ctx.sync_steps(idx.reshape(-1), batch, steps, lr)
    w_ref = ctx.get_weights()
    ctx.models_set([lam], [lr])
    losses = ctx.models_steps(idx.reshape(-1), batch, steps)
    np.testing.assert_allclose(losses[:, 0], l_ref, rtol=1e-11)
    np.testing.assert_allclose(ctx.models_get_weights()[0], w_ref, rtol=1e-11, atol=1e-15)
    ctx.close()


def test_model_set_leaves_the_resident_weights_alone(synth):
    rng = np.random.default_rng(12)
    ctx, _ = make_pair(synth, lam=1e-5, n_train=4800)
    w = np.where(rng.random(synth.dim) < 0.3, rng.standard_normal(synth.dim), 0.0)
    ctx.set_weights(w)
    before = ctx.get_weights()
    ctx.models_set(LAMS, LRS)
    ctx.models_steps(draws(rng, 4800, 256, 20).reshape(-1), 256, 20)
    ctx.models_eval_counts(2, 0, 6000)
    assert ctx.get_weights().view(np.uint64).tolist() == before.view(np.uint64).tolist()
    assert ctx.eval_counts(0, 6000) == ctx.eval_counts(0, 6000, w)
    ctx.close()


def test_frozen_model_keeps_its_bits(synth):
    rng = np.random.default_rng(13)
    batch = 32
    ctx, orc = make_pair(synth, lam=1e-5, n_train=4800)
    idx = draws(rng, 4800, batch, 40)
    w0 = start_weights(rng, synth.dim, len(LAMS))
    ctx.models_set(LAMS, LRS, w0)
    l1 = ctx.models_steps(idx[:20].reshape(-1), batch, 20)
    W1 = ctx.models_get_weights()
    active = np.array([1, 0, 1, 1, 0], dtype=bool)
    l2 = ctx.models_steps(idx[20:].reshape(-1), batch, 20, active=active)
    W2 = ctx.models_get_weights()
    for m in np.flatnonzero(~active):
        assert W2[m].view(np.uint64).tolist() == W1[m].view(np.uint64).tolist()
        assert np.isnan(l2[:, m]).all()
    keep = np.flatnonzero(active)
    losses = np.concatenate([l1, l2])
    check_against_oracle(orc, w0[keep], idx, batch, losses[:, keep], W2[keep], [LAMS[m] for m in keep],
                         [LRS[m] for m in keep])
    ctx.close()


def test_models_eval_counts_equals_eval_counts(synth):
    rng = np.random.default_rng(14)
    ctx, _ = make_pair(synth, lam=1e-5, n_train=4800)
    ctx.models_set(LAMS, LRS)
    ctx.models_steps(draws(rng, 4800, 256, 30).reshape(-1), 256, 30)
    W = ctx.models_get_weights()
    for m in range(len(LAMS)):
        for b, e in ((0, 4800), (4800, 6000), (17, 18), (0, 6000)):          # streaming pass and the small-range kernel
            assert ctx.models_eval_counts(m, b, e) == ctx.eval_counts(b, e, W[m])
    ctx.close()


def test_model_set_errors(synth):
    from distributed_sgd_b200 import native
    from distributed_sgd_b200.native import NativeCtx
    dim = synth.dim

    def code(fn, *a, **kw):
        with pytest.raises(native.DsgdError) as e:
            fn(*a, **kw)
        return e.value.code

    ctx, _ = make_pair(synth, lam=1e-5, n_train=4800)
    # no model set yet
    assert code(ctx.models_steps, [0], 1, 1) == native.ERR_STATE
    assert code(ctx.models_get_weights) == native.ERR_STATE
    assert code(ctx.models_eval_counts, 0, 0, 10) == native.ERR_STATE
    # bad sets
    assert code(ctx.models_set, [1e-5] * 33, [0.5] * 33) == native.ERR_INVALID
    assert ctx._l.dsgd_models_set(ctx._h, -1, None, None, None) == native.ERR_INVALID
    for lam, lr in ((-1e-5, 0.5), (float("nan"), 0.5), (float("inf"), 0.5), (1e-5, float("nan")), (1e-5, float("inf"))):
        assert code(ctx.models_set, [1e-5, lam], [0.5, lr]) == native.ERR_INVALID
    ctx.models_set([1e-5, 1e-4], [0.5, 0.1])
    assert code(ctx.models_eval_counts, 2, 0, 10) == native.ERR_INVALID
    assert code(ctx.models_eval_counts, -1, 0, 10) == native.ERR_INVALID
    assert code(ctx.models_steps, [0, 6000], 2, 1) == native.ERR_RANGE
    assert code(ctx.models_steps, [], 0, 3) == native.ERR_EMPTY
    ctx.set_workers([2, 2], 2)                                            # two logical workers per step
    assert code(ctx.models_steps, [0, 1, 2, 3], 4, 1) == native.ERR_STATE
    ctx.set_workers([4], 1)
    ctx.models_steps([0, 1, 2, 3], 4, 1)
    ctx.models_set([], [])                                                 # n_models == 0 frees the set
    assert code(ctx.models_get_weights) == native.ERR_STATE
    ctx.close()
    bare = NativeCtx(0, dim, 1e-5)                                         # no dimSparsity
    bare.load_csr(synth.row_ptr, synth.col, synth.val, synth.label)
    bare.models_set([1e-5], [0.5])
    assert code(bare.models_steps, [0], 1, 1) == native.ERR_STATE
    bare.close()
    for kw in ({"is_async": True}, {"rank": 0, "world": 2}):
        other = NativeCtx(0, dim, 1e-5, **kw)
        assert code(other.models_set, [1e-5], [0.5]) == native.ERR_STATE
        other.close()


def test_fit_models_matches_per_setting_fits(synth):
    """MasterSync.fit_models against one MasterSync.fit per setting with the same seed: stop epochs, per-epoch loss and
    accuracy lists, final weights.  The learning-rate-0 setting never moves (test loss 1.0 every epoch) and stops after
    three epochs; the others stop on their own test losses or at max_epochs."""
    from distributed_sgd_b200 import MasterSync, Slave, SparseSVM
    from distributed_sgd_b200.ml import EarlyStopping
    settings = [(1e-3, 0.5), (1e-4, 0.1), (0.0, 1.0), (1e-3, 0.0)]
    batch, epochs = 100, 5
    stop = EarlyStopping.no_improvement(patience=2, min_delta=0.0)
    train, test = synth.split_at(4800)
    train, _ = train.split_at(1200)
    w0 = np.zeros(synth.dim)

    def master_for(lam):
        model = SparseSVM(lam)
        slave = Slave(0, 0, train, model, world=1, device=0, test_data=test)
        return MasterSync(0, train, test, model, 1, slave=slave, seed=0), slave

    master, slave = master_for(1e-5)
    states = master.fit_models(w0, epochs, batch, [s[0] for s in settings], [s[1] for s in settings], stop)
    histories = master.histories
    slave.stop()
    stop_epochs = [st.updates for st in states]
    assert len(set(stop_epochs)) >= 2, stop_epochs
    assert stop_epochs[3] == 3
    for m, (lam, lr) in enumerate(settings):
        ref_master, ref_slave = master_for(lam)
        ref = ref_master.fit(w0, epochs, batch, lr, stop)
        h, hr = histories[m], ref_master.history
        assert states[m].updates == ref.updates, f"setting {m}"
        np.testing.assert_allclose(h["losses"], hr["losses"], rtol=RTOL)
        np.testing.assert_allclose(h["test_losses"], hr["test_losses"], rtol=RTOL)
        assert h["accs"] == hr["accs"] and h["test_accs"] == hr["test_accs"]
        np.testing.assert_allclose(states[m].grad, ref.grad, rtol=1e-11, atol=1e-15)
        assert states[m].loss == pytest.approx(ref.loss, rel=RTOL)
        ref_slave.stop()
