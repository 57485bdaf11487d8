"""Shape-dependent branches of the kernels that the bench shapes never reach, each against the fp64 oracle: model sets
above 8 models, the model-set kernel's overflow paths and its 32-rows-per-CTA cap, update threads that own more than two
columns, the one-worker k_rows + k_update fallback of the sync loop, the streaming pass at and beyond its shared-memory
limit, from a row other than 0 and in all its block sizes, and the 1e-20 filter in the streaming pass's fp32 decisions.

Tolerances as in test_gpu_parity.py / test_gpu_models.py: predictions, supports and integer counters exact; losses
rtol 1e-12; weights rtol 1e-11 with atol 1e-13 * max|w| (as in smoke(): with weights of O(1) and large lambdas, entries that
cancel to ~1e-5 keep an fp64 reordering error at the summands' scale), long rows 1e-10 / 1e-14."""
import numpy as np
import pytest

from helpers import data_from_csr, make_pair
from test_gpu_models import check_against_oracle, draws, oracle_for, settings_for, start_weights

pytestmark = pytest.mark.gpu

RTOL = 1e-12


@pytest.fixture(scope="module")
def synth():
    from distributed_sgd_b200.utils import synthetic_rcv1
    return synthetic_rcv1(n_rows=6000, seed=3)


@pytest.fixture(scope="module")
def synth_100003():
    """dim 100 003 (odd): above 2 * 148 * 256 = 75 776 and 2 * 148 * 192 = 56 832 columns, and above the streaming
    pass's 57 856."""
    from distributed_sgd_b200.utils import synthetic_rcv1
    return synthetic_rcv1(n_rows=3000, dim=100_003, seed=17)


@pytest.fixture(scope="module")
def sm_count():
    from distributed_sgd_b200.native import NativeCtx
    with NativeCtx(0, 8, 0.0) as ctx:
        return ctx.info()["sm_count"]


@pytest.fixture(scope="module")
def long_rows():
    """The rows of test_persistent_loop_with_rows_that_overflow_the_tma_stage: 1 600 rows of 1 800-2 000 non-zeros."""
    rng = np.random.default_rng(256)
    dim, n = 47236, 1600
    lens = rng.integers(1800, 2001, size=n)
    rp = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    col = np.concatenate([np.sort(rng.choice(dim, size=int(l), replace=False)) for l in lens]).astype(np.int32)
    val = (np.abs(rng.standard_normal(len(col))) * 0.02 + 1e-3).astype(np.float32)
    lab = rng.choice(np.array([-1, 1], dtype=np.int8), size=n)
    return data_from_csr(rp, col, val, lab, dim)


def rand_w(rng, dim, density=0.5, scale=0.05):
    return np.where(rng.random(dim) < density, rng.standard_normal(dim) * scale, 0.0)


def counts_ref(orc, w, idx):
    """(hinge sum, correct count) from the oracle's predictions: hinge 1 - y * p, correct p == y (SparseSVM.scala:14-16)."""
    p = orc.forward(w, idx)
    y = orc.label[np.asarray(idx)].astype(np.float64)
    return int(np.sum(1.0 - y * p)), int(np.sum(p == y))


def check_weights(W, w_ref, rtol=1e-11, atol=None, what=""):
    atol = 1e-13 * float(np.abs(w_ref).max()) if atol is None else atol
    assert (W == 0).tolist() == (w_ref == 0).tolist(), f"{what}: weight supports differ"
    np.testing.assert_allclose(W, w_ref, rtol=rtol, atol=atol, err_msg=what)


def check_requests(ctx, orc, w, ids, what):
    """forward and gradient on the sample list `ids`, eval_counts / eval on rows [0, len(ids)) when ids == arange."""
    np.testing.assert_array_equal(ctx.forward(ids, w), orc.forward(w, ids), err_msg=f"{what}: forward")
    g_ref, _ = orc.gradient(w, ids)
    g, loss = ctx.gradient(ids, w, want_loss=True)
    assert (g == 0).tolist() == (g_ref == 0).tolist(), f"{what}: gradient supports differ"
    np.testing.assert_allclose(g, g_ref, rtol=RTOL, atol=1e-13, err_msg=f"{what}: gradient")
    assert loss == pytest.approx(orc.loss_acc(w, idx=ids)[0], rel=RTOL), what


def check_range(ctx, orc, w, b, e, what):
    h, c, n2 = ctx.eval_counts(b, e, w)
    assert (h, c) == counts_ref(orc, w, np.arange(b, e, dtype=np.int32)), f"{what}: eval_counts [{b},{e})"
    loss, acc = ctx.eval(b, e, w)
    loss_ref, acc_ref = orc.loss_acc(w, begin=b, n=e - b)
    assert acc == acc_ref, f"{what}: eval accuracy [{b},{e})"
    assert loss == pytest.approx(loss_ref, rel=RTOL), f"{what}: eval loss [{b},{e})"


# ---- A. model sets (dsgd_models.cuh) ---------------------------------------------------------------------------------

@pytest.mark.parametrize("active", [[31], [0, 9, 17, 31], list(range(1, 32, 2))], ids=["only31", "0-9-17-31", "odd"])
def test_frozen_masks_at_32_models(synth, active):
    """Active-model masks at M = 32: the kernel's slots 0 .. n_act-1 map to model ids above 8, and each slot's w_res
    offset is that id's.  Frozen models keep their bits and report NaN losses; active ones follow their oracle run."""
    rng = np.random.default_rng(31 + len(active))
    M, batch = 32, 64
    lams, lrs = settings_for(M)
    ctx, orc = make_pair(synth, lam=1e-5, n_train=4800)
    idx = draws(rng, 4800, batch, 20)
    w0 = start_weights(rng, synth.dim, M)
    ctx.models_set(lams, lrs, w0)
    l1 = ctx.models_steps(idx[:8].reshape(-1), batch, 8)
    W1 = ctx.models_get_weights()
    mask = np.zeros(M, dtype=bool)
    mask[active] = True
    l2 = ctx.models_steps(idx[8:].reshape(-1), batch, 12, active=mask)
    W2 = ctx.models_get_weights()
    for m in np.flatnonzero(~mask):
        assert W2[m].view(np.uint64).tolist() == W1[m].view(np.uint64).tolist(), f"frozen model {m} moved"
        assert np.isnan(l2[:, m]).all()
    assert not np.isnan(l2[:, mask]).any()
    keep = np.flatnonzero(mask)
    check_against_oracle(orc, w0[keep], idx, batch, np.concatenate([l1, l2])[:, keep], W2[keep],
                         [lams[m] for m in keep], [lrs[m] for m in keep], atol=None)
    ctx.close()


@pytest.mark.parametrize("batch", [256, 1500])
def test_model_set_with_rows_that_overflow_the_stage(long_rows, batch):
    """consume_stage_models on rows of 1 800-2 000 non-zeros: at batch 256 the stage ring overflows and chunks are read
    from global memory (kChunkGlobal); at batch 1 500 the chunk list overflows too and every (row, model) takes the
    whole-row path.  12 models against the oracle, and a one-model set against dsgd_sync_steps on the same draws."""
    data = long_rows
    rng = np.random.default_rng(batch + 1)
    M, steps = 12, 5
    lams, lrs = [0.0] + list(np.geomspace(1e-6, 1e-2, M - 1)), list(np.linspace(0.01, 0.2, M))
    ctx, orc = make_pair(data, lam=1e-3)
    idx = draws(rng, data.n_rows, batch, steps)
    w0 = start_weights(rng, data.dim, M)
    ctx.models_set(lams, lrs, w0)
    losses = ctx.models_steps(idx.reshape(-1), batch, steps)
    W = ctx.models_get_weights()
    for m in range(M):
        w_ref, l_ref = oracle_for(orc, lams[m]).sync_steps(w0[m], idx.reshape(-1), [batch], lrs[m], n_steps=steps)
        np.testing.assert_allclose(losses[:, m], l_ref, rtol=RTOL, err_msg=f"model {m}")
        check_weights(W[m], w_ref, 1e-10, 1e-14, f"model {m}")
    ctx.set_weights(w0[1])
    l_sync = ctx.sync_steps(idx.reshape(-1), batch, steps, lrs[1])
    w_sync = ctx.get_weights()
    ctx.models_set([1e-3], [lrs[1]], w0[1])
    l_one = ctx.models_steps(idx.reshape(-1), batch, steps)
    np.testing.assert_allclose(l_one[:, 0], l_sync, rtol=RTOL)
    check_weights(ctx.models_get_weights()[0], w_sync, 1e-10, 1e-14, "one-model set vs sync_steps")
    ctx.close()


def test_model_set_at_the_rows_per_cta_cap(synth, sm_count):
    """kMaxRowsPerCta = 32: with 4 CTAs a batch of 128 runs (about 3 000 pairs per CTA, so the 2 560-pair stage ring
    overflows as well) and 129 is refused with DSGD_ERR_INVALID; at full grid 32 * SMs runs and 32 * SMs + 1 is refused."""
    from distributed_sgd_b200 import native
    rng = np.random.default_rng(128)
    M, steps = 3, 4
    lams, lrs = [0.0, 1e-4, 1e-2], [1.0, 0.5, 0.05]
    ctx, orc = make_pair(synth, lam=1e-5, n_train=4800)
    w0 = start_weights(rng, synth.dim, M)
    for grid, batch in ((4, 128), (0, 32 * sm_count)):
        ctx.set_grid_limit(grid)
        idx = draws(rng, synth.n_rows, batch, steps)
        ctx.models_set(lams, lrs, w0)
        losses = ctx.models_steps(idx.reshape(-1), batch, steps)
        check_against_oracle(orc, w0, idx, batch, losses, ctx.models_get_weights(), lams, lrs, atol=None)
        with pytest.raises(native.DsgdInvalid):
            ctx.models_steps(np.arange(batch + 1, dtype=np.int32), batch + 1, 1)
    ctx.close()


@pytest.mark.parametrize("case", ["dim100003", "grid4"])
def test_model_set_update_threads_with_more_than_two_columns(synth, synth_100003, case):
    """The model-set update threads keep two columns each in registers; the columns beyond 2 * G * 256 go through the
    extra loop.  dim 100 003 at full grid (odd dim, 9 models), and dim 47 236 with 4 CTAs.  At dim 100 003 the
    evaluation of a model goes through k_rows also for n >= 2 048 (the streaming pass does not fit): models_eval_counts
    against the oracle there."""
    data, grid, batch = (synth_100003, 0, 256) if case == "dim100003" else (synth, 4, 100)
    rng = np.random.default_rng(9)
    M, steps = 9, 12
    lams, lrs = settings_for(M)
    n_train = data.n_rows * 4 // 5
    ctx, orc = make_pair(data, lam=1e-5, n_train=n_train)
    ctx.set_grid_limit(grid)
    idx = draws(rng, n_train, batch, steps)
    w0 = start_weights(rng, data.dim, M)
    ctx.models_set(lams, lrs, w0)
    losses = ctx.models_steps(idx.reshape(-1), batch, steps)
    W = ctx.models_get_weights()
    check_against_oracle(orc, w0, idx, batch, losses, W, lams, lrs, atol=None)
    if case == "dim100003":
        for m in (0, 4, 8):
            for b, e in ((0, data.n_rows), (0, 2048), (5, 6)):
                h, c, n2 = ctx.models_eval_counts(m, b, e)
                assert (h, c) == counts_ref(orc, W[m], np.arange(b, e, dtype=np.int32)), (m, b, e)
                assert n2 == pytest.approx(float(np.dot(W[m], W[m])), rel=RTOL)
    ctx.close()


# ---- B. single-model sync (dsgd_persistent.cuh, dsgd_api.cu) ---------------------------------------------------------

def _sync_run(ctx, w0, idx, batch, lr):
    ctx.set_weights(w0)
    n0 = ctx.launch_count()
    losses = ctx.sync_steps(idx.reshape(-1), batch, idx.shape[0], lr)
    return losses, ctx.get_weights(), ctx.launch_count() - n0


def test_one_trajectory_three_sync_routes(synth, sm_count):
    """dsgd_sync_steps routes a one-worker run to the persistent kernel when the batch fits 32 rows per CTA (2 launches
    per call: k_rec_init + the kernel) and to k_rows + k_update<true> otherwise (2 launches per step).  The same draws
    (batch 128) through the full-grid persistent kernel, the persistent kernel on 4 CTAs (exactly 32 rows per CTA) and the
    fallback on 3 CTAs; then the fallback at full grid with a batch of 32 * SMs + 64.  Every run against the oracle."""
    rng = np.random.default_rng(3)
    lam, lr, batch, steps = 1e-5, 0.5, 128, 8
    ctx, orc = make_pair(synth, lam=lam, n_train=4800)
    idx = draws(rng, 4800, batch, steps)
    w0 = np.zeros(synth.dim)
    w_ref, l_ref = orc.sync_steps(w0, idx.reshape(-1), [batch], lr, n_steps=steps)
    for grid, launches in ((0, 2), (4, 2), (3, 2 * steps)):
        ctx.set_grid_limit(grid)
        losses, w, n_launch = _sync_run(ctx, w0, idx, batch, lr)
        assert n_launch == launches, f"grid {grid}: {n_launch} launches"
        np.testing.assert_allclose(losses, l_ref, rtol=RTOL, err_msg=f"grid {grid}")
        check_weights(w, w_ref, what=f"grid {grid}")
    ctx.set_grid_limit(0)
    big, steps = 32 * sm_count + 64, 3
    idx = draws(rng, synth.n_rows, big, steps)
    w_ref, l_ref = orc.sync_steps(w0, idx.reshape(-1), [big], lr, n_steps=steps)
    losses, w, n_launch = _sync_run(ctx, w0, idx, big, lr)
    assert n_launch == 2 * steps
    np.testing.assert_allclose(losses, l_ref, rtol=RTOL)
    check_weights(w, w_ref)
    ctx.close()


@pytest.mark.parametrize("case", ["dim100003", "grid4"])
def test_sync_update_threads_with_more_than_two_columns(synth, synth_100003, case):
    """k_sync_persistent keeps two columns per update thread in registers; the columns beyond 2 * G * 192 go through the
    extra loop, and the epilogue writes them (weights, fp32 shadow, c and ||w||^2) from Rfin.  dim 100 003 at full grid and
    dim 47 236 with 4 CTAs: losses and final weights against the oracle, then the resident weights' c and ||w||^2 (what
    the epilogue published) against those computed for the same weights passed with the request."""
    data, grid, batch = (synth_100003, 0, 256) if case == "dim100003" else (synth, 4, 100)
    rng = np.random.default_rng(10)
    lam, lr, steps = 1e-5, 0.5, 12
    n_train = data.n_rows * 4 // 5
    ctx, orc = make_pair(data, lam=lam, n_train=n_train)
    ctx.set_grid_limit(grid)
    idx = draws(rng, n_train, batch, steps)
    w0 = np.zeros(data.dim)
    w_ref, l_ref = orc.sync_steps(w0, idx.reshape(-1), [batch], lr, n_steps=steps)
    losses, w, n_launch = _sync_run(ctx, w0, idx, batch, lr)
    assert n_launch == 2
    np.testing.assert_allclose(losses, l_ref, rtol=RTOL)
    check_weights(w, w_ref)
    loss, acc = ctx.eval(0, data.n_rows)
    loss_w, acc_w = ctx.eval(0, data.n_rows, w)
    assert acc == acc_w and loss == pytest.approx(loss_w, rel=RTOL)   # ||w||^2 reduced in two different fixed orders
    probe = idx[0]
    g, g_w = ctx.gradient(probe), ctx.gradient(probe, w)                 # c of the resident weights vs the request's
    assert (g == 0).tolist() == (g_w == 0).tolist()
    np.testing.assert_allclose(g, g_w, rtol=RTOL, atol=0)
    ctx.close()


# ---- C. streaming pass (dsgd_stream.cuh) -----------------------------------------------------------------------------

@pytest.mark.parametrize("dim", [57856, 57857, 4099])
def test_streaming_pass_at_its_dim_limit(dim):
    """The streaming pass stages the fp32 weights in shared memory: dim 57 856 is the largest that fits (231 424 bytes
    plus 256 of static shared memory), 57 857 falls back to k_rows, 4 099 is odd (the scalar tail of the staging loop).
    forward / gradient (sample lists) and eval / eval_counts (row ranges) at n = 2 048, 2 049 and 3 001."""
    from distributed_sgd_b200.utils import synthetic_rcv1
    data = synthetic_rcv1(n_rows=3001, dim=dim, seed=dim % 97)
    rng = np.random.default_rng(dim)
    ctx, orc = make_pair(data, lam=1e-3, n_train=2400)
    w = rand_w(rng, dim, 0.5, 0.2)
    for n in (2048, 2049, 3001):
        check_requests(ctx, orc, w, rng.integers(0, data.n_rows, size=n).astype(np.int32), f"dim {dim} n {n}")
        check_range(ctx, orc, w, 0, n, f"dim {dim}")
    ctx.close()


def test_contiguous_evaluation_from_another_row():
    """Evaluation over consecutive rows (kContig) that starts at a row other than 0: the ranges [1 237, 4 238) and
    [2 053, 9 998) of a 10 000-row set, both long enough for the streaming pass, n odd and not a multiple of 8."""
    from distributed_sgd_b200.utils import synthetic_rcv1
    data = synthetic_rcv1(n_rows=10_000, seed=23)
    rng = np.random.default_rng(23)
    ctx, orc = make_pair(data, lam=1e-4, n_train=8000)
    for w in (rand_w(rng, data.dim, 0.5, 0.05), rand_w(rng, data.dim, 0.1, 1.0)):
        for b, e in ((1237, 4238), (2053, 9998)):
            check_range(ctx, orc, w, b, e, "contiguous")
    ctx.close()


def test_streaming_block_sizes_on_a_million_rows():
    """Rows per block of the streaming pass: 32 (tail 16) when every warp gets at least 6 blocks of 32, i.e. above 909 281
    rows on 148 SMs; 16 (tail 8) below.  eval_counts over all 1 000 000 rows and over 500 000, and forward on 950 000
    sampled ids (32-row blocks through the sample-list path), against the oracle.  About 0.8 GB on the device."""
    from distributed_sgd_b200.utils import synthetic_rcv1
    data = synthetic_rcv1(n_rows=1_000_000, seed=29)
    rng = np.random.default_rng(29)
    ctx, orc = make_pair(data, lam=1e-5, n_train=800_000)
    w = rand_w(rng, data.dim, 0.5, 0.05)
    for b, e in ((0, 1_000_000), (250_000, 750_000)):
        h, c, _ = ctx.eval_counts(b, e, w)
        assert (h, c) == counts_ref(orc, w, np.arange(b, e, dtype=np.int32)), (b, e)
    loss, acc = ctx.eval(0, 1_000_000, w)
    loss_ref, acc_ref = orc.loss_acc(w, begin=0, n=1_000_000)
    assert acc == acc_ref and loss == pytest.approx(loss_ref, rel=RTOL)
    ids = rng.integers(0, data.n_rows, size=950_000).astype(np.int32)
    np.testing.assert_array_equal(ctx.forward(ids, w), orc.forward(w, ids))
    ctx.close()


# ---- C.4 the 1e-20 filter in the streaming pass's fp32 decisions ----

TINY = np.array([1e-21, 1e-25, -1e-30, 1e-40], dtype=np.float32)   # |x| <= 1e-20: absent keys for the fp64 arithmetic


def _tiny_value_rows(rng, n=3000, dim=2000):
    """Every third row mixes normal values with values <= 1e-20, every third holds only such values, the rest are
    normal."""
    rp, col, val = [0], [], []
    for r in range(n):
        kind = r % 3
        n_norm = 0 if kind == 1 else int(rng.integers(10, 60))
        n_tiny = 0 if kind == 2 else int(rng.integers(1, 9))
        c = np.sort(rng.choice(dim, size=n_norm + n_tiny, replace=False))
        v = np.concatenate([np.abs(rng.standard_normal(n_norm)) * 0.1 + 1e-3, rng.choice(TINY, size=n_tiny)])
        rng.shuffle(v)
        col += c.tolist(); val += v.tolist(); rp.append(len(col))
    lab = rng.choice([-1, 1], size=n)
    return data_from_csr(rp, col, np.asarray(val, np.float32), lab, dim), rng.standard_normal(dim)


def _subnormal_weight_rows(n=3000, dim=64):
    """x = +-1e20 on three columns, weights that are all fp32 subnormals: every product is above 1e-20, the fp64 dot is
    1e20 * (-0.19 * 2^-149) < 0, and rounding the weights to fp32 makes the fp32 dot 1e20 * 2^-149 > 0."""
    q = 2.0 ** -149
    w = np.zeros(dim)
    w[0], w[1], w[2] = 200_000.51 * q, -100_000.4 * q, -100_000.3 * q
    rp, col, val = [0], [], []
    for r in range(n):
        col += [0, 1, 2]; val += [(-1.0 if r % 2 else 1.0) * 1e20] * 3
        rp.append(len(col))
    lab = [1 if (r // 4) % 2 == 0 else -1 for r in range(n)]
    data = data_from_csr(rp, col, np.asarray(val, np.float32), lab, dim)
    x32 = np.float64(np.float32(1e20))
    assert float(np.sum(x32 * w[:3])) < 0 < float(np.sum(x32 * w[:3].astype(np.float32).astype(np.float64)))
    return data, w


def _filter_case(name):
    from distributed_sgd_b200.utils import synthetic_rcv1
    rng = np.random.default_rng(41)
    if name == "tiny_values":
        return _tiny_value_rows(rng)
    if name == "subnormal_weights":
        return _subnormal_weight_rows()
    data = synthetic_rcv1(n_rows=3000, seed=41)
    if name == "w_1e-21":                                                 # every product below the filter
        return data, 1e-21 * rng.standard_normal(data.dim)
    return data, 1e-19 * rng.standard_normal(data.dim)                    # |x w| spans 1e-21 .. 1e-19


@pytest.mark.parametrize("name", ["tiny_values", "w_1e-21", "w_1e-19", "subnormal_weights"])
def test_streaming_pass_applies_the_1e20_filter(name):
    """The fp64 arithmetic drops values and products of magnitude <= 1e-20; the streaming pass's fp32 dot must not decide
    a row on them.  Where the fp64 dot is 0 (prediction 0, hinge 1) or has the other sign, the row falls inside the
    rounding band and is recomputed in fp64.  forward, gradient and eval_counts through the streaming pass (n >= 2 048)
    and through k_rows (the first 2 047 rows) must both equal the oracle."""
    data, w = _filter_case(name)
    ctx, orc = make_pair(data, lam=1e-3)
    n = data.n_rows
    for m in (n, 2047):
        ids = np.arange(m, dtype=np.int32)
        check_requests(ctx, orc, w, ids, f"{name} n {m}")
        check_range(ctx, orc, w, 0, m, f"{name}")
    ctx.close()
