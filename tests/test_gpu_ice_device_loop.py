"""hc_ice_dense_balance with its loop control on the device: the iteration loop is one graph launch (a WHILE node ended
by the last update CTA), the live work list is compacted on the device when a chromosome converges, and the shape's
tables, buffers and graph are kept between calls.  Every case is checked against the oracle and against the int32
tiles (HC_ICE_PACKED=0)."""
import numpy as np
import pytest

from oracle import cooler_ice

pytestmark = pytest.mark.gpu

RTOL = 1e-6


def _matrix(n, seed, scale=30.0, heavy_diag=False):
    rng = np.random.default_rng(seed)
    bias = np.exp(rng.normal(0, 0.4, n))
    d = np.abs(np.subtract.outer(np.arange(n), np.arange(n))) + 1.0
    M = rng.poisson(scale * bias[:, None] * bias[None, :] / d)
    if heavy_diag:                      # counts far above 255 next to the diagonal: overflow cells of the packed encoding
        M = M + rng.poisson(3000.0 / d ** 2)
    M = np.triu(M) + np.triu(M, 1).T
    return M


def _run(mats, **kw):
    """weights, per-chromosome results and the run record of one balancing call"""
    from hichap_master_b200 import kernels
    from hichap_master_b200.device import DenseBatch
    b = DenseBatch.from_numpy(mats)
    params = kernels.ice_params(**kw)
    bias = kernels.ice_dense_filters(b, params)
    res, info = kernels.ice_dense_iterate(b, bias, params)
    return bias.cpu().numpy(), res, info


def _oracle(mats, **kw):
    off = np.concatenate([[0], np.cumsum([m.shape[0] for m in mats])])
    b1, b2, cnt = [], [], []
    for m, lo in zip(mats, off[:-1]):
        x, y = np.nonzero(np.triu(m)); b1.append(x + lo); b2.append(y + lo); cnt.append(m[x, y])
    return cooler_ice.balance(np.concatenate(b1), np.concatenate(b2), np.concatenate(cnt), int(off[-1]), off,
                              cis_only=True, **kw)


def _check(w, ref, what):
    assert np.array_equal(np.isnan(w), np.isnan(ref)), what
    ok = ~np.isnan(ref)
    if ok.any():
        err = np.max(np.abs(w[ok] - ref[ok]) / np.abs(ref[ok]))
        assert err < RTOL, "%s: max rel err %.3g" % (what, err)


def _int32(monkeypatch, mats, **kw):
    monkeypatch.setenv("HC_ICE_PACKED", "0")
    out = _run(mats, **kw)
    monkeypatch.delenv("HC_ICE_PACKED")
    return out


def _check_launches(info, res):
    """one stream + one update launch per iteration, at most 3 more past the last convergence (the loop checks its
    condition every 4 iterations), and the finalising launch"""
    it = int(res["iters"].max())
    assert 2 * it + 1 <= info.launches <= 2 * (it + 3) + 1, (it, info.launches)


@pytest.fixture(scope="module")
def dev(cuda_device):
    return cuda_device


def test_repeated_calls_reuse_the_shape_and_switch_shapes(dev, monkeypatch):
    """Same shape twice, another shape, the first again: every call gives the bits of the first call of its shape
    (the kept graph and tables are those of the right shape) and matches the oracle and the int32 tiles."""
    monkeypatch.delenv("HC_ICE_PACKED", raising=False)
    a = [_matrix(900, 1, heavy_diag=True), _matrix(400, 2, heavy_diag=True)]
    b = [_matrix(700, 3, heavy_diag=True), _matrix(1300, 4, heavy_diag=True), _matrix(90, 5)]
    first = {}
    for name in ("a", "a", "b", "a", "b"):
        mats = a if name == "a" else b
        w, res, info = _run(mats)
        if name not in first:
            first[name] = (w, res)
            ref, rst = _oracle(mats)
            _check(w, ref, "shape %s vs oracle" % name)
            assert [int(i) for i in res["iters"]] == rst["iters"], name
            w32, res32, _ = _int32(monkeypatch, mats)
            _check(w, w32, "shape %s vs int32 tiles" % name)
            assert np.array_equal(res["iters"], res32["iters"]), name
        else:
            assert np.array_equal(w, first[name][0], equal_nan=True), name
            assert np.array_equal(res, first[name][1]), name
        _check_launches(info, res)


def test_max_iters_stops_the_device_loop(dev, monkeypatch):
    """max_iters=5: exactly 5 iterations (no run past the limit), none converged."""
    monkeypatch.delenv("HC_ICE_PACKED", raising=False)
    mats = [_matrix(2100, 7, heavy_diag=True), _matrix(600, 8)]
    w, res, info = _run(mats, max_iters=5)
    assert [int(i) for i in res["iters"]] == [5, 5] and not res["converged"].any()
    assert info.launches == 11
    ref, rst = _oracle(mats, max_iters=5)
    assert rst["iters"] == [5, 5]
    _check(w, ref, "max_iters=5 vs oracle")
    w32, res32, _ = _int32(monkeypatch, mats, max_iters=5)
    _check(w, w32, "max_iters=5 vs int32 tiles")
    assert np.array_equal(res["iters"], res32["iters"])


def test_convergence_far_apart_empty_and_all_filtered(dev, monkeypatch):
    """Chromosomes that converge many iterations apart (the live work list is rewritten on the device after each
    convergence), next to an empty matrix and an all-zero one whose bins are all filtered out."""
    monkeypatch.delenv("HC_ICE_PACKED", raising=False)
    rng = np.random.default_rng(11)
    flat = rng.poisson(40.0, (300, 300)); flat = np.triu(flat) + np.triu(flat, 1).T          # nearly balanced already
    mats = [_matrix(1800, 9, scale=60.0, heavy_diag=True), flat, np.zeros((0, 0), np.int64),
            _matrix(500, 10, heavy_diag=True), np.zeros((200, 200), np.int64), _matrix(1000, 12)]
    kw = dict(mad_max=0)       # filters per bin: the oracle can balance the non-empty matrices on their own
    w, res, info = _run(mats, **kw)
    iters = [int(i) for i in res["iters"]]
    assert iters[2] == 0 and res["converged"][2] and np.isnan(res["scale"][2])     # empty: never iterated
    assert np.isnan(res["scale"][4]) and res["converged"][4]                        # all filtered
    live = [0, 1, 3, 5]
    assert max(iters[i] for i in live) - min(iters[i] for i in live) >= 10, iters
    off = np.concatenate([[0], np.cumsum([m.shape[0] for m in mats])])
    assert np.isnan(w[off[4]:off[5]]).all()
    ref, rst = _oracle([mats[i] for i in live], **kw)
    _check(np.concatenate([w[off[i]:off[i + 1]] for i in live]), ref, "live chromosomes vs oracle")
    assert [iters[i] for i in live] == rst["iters"]
    w32, res32, _ = _int32(monkeypatch, mats, **kw)
    _check(w, w32, "vs int32 tiles")
    assert np.array_equal(res["iters"], res32["iters"])
    _check_launches(info, res)


def test_overflow_arrays_grow_and_the_call_runs_again(dev, monkeypatch):
    """A call with far more overflow cells (weighted counts above 255) than any earlier call: the arrays kept between
    calls are too small, the call finds out on the device, grows them and runs again -- same weights as a repeated
    call (which fits) and as the oracle; the overflow count is exact."""
    from hichap_master_b200 import _abi
    monkeypatch.delenv("HC_ICE_PACKED", raising=False)
    n = 1500
    small = [_matrix(n, 13)]
    rng = np.random.default_rng(14)
    big = rng.poisson(400.0, (n, n)); big = np.triu(big) + np.triu(big, 1).T       # ~ every cell above 255
    _run(small)
    c0 = _abi.launch_count()
    w1, res1, info1 = _run([big])
    c1 = _abi.launch_count()
    w2, res2, info2 = _run([big])
    c2 = _abi.launch_count()
    d = np.abs(np.subtract.outer(np.arange(n), np.arange(n)))
    assert info1.overflow_cells == info2.overflow_cells == int(((big > 255) & (d >= 1)).sum())
    assert c1 - c0 > c2 - c1, (c1 - c0, c2 - c1)          # the first call ran its set-up twice
    assert np.array_equal(w1, w2, equal_nan=True) and np.array_equal(res1, res2)
    ref, rst = _oracle([big])
    _check(w1, ref, "grown overflow arrays vs oracle")
    assert [int(i) for i in res1["iters"]] == rst["iters"]
    w32, res32, _ = _int32(monkeypatch, [big])
    _check(w1, w32, "vs int32 tiles")
