"""GPU parity tests (run on the B200 box): the CUDA path, called through the C ABI via the
reference-named Python functions, against (i) the committed golden vectors produced by the
unmodified reference and (ii) the CPU oracle on larger seeded inputs.
Bar: integer / index work bit-exact; fp64 results within 1e-6 relative (BASELINE.json
north_star tolerance) -- in practice they agree to ~1e-12 and the tests also print the max."""
import io

import numpy as np
import pytest

from conftest import CHROMS, SMALL_GENOME, load_golden, unflatten
from hichap_master_b200 import synth
from oracle import cooler_ice
from oracle import hichap_oracle as ho

pytestmark = pytest.mark.gpu

RTOL = 1e-6   # north_star: "bias vectors and corrected matrices within 1e-6 relative (fp64)"


@pytest.fixture(scope="module")
def mb(cuda_device):
    from hichap_master_b200 import matrixBuilding
    return matrixBuilding


def records_equal(a, b):
    return (a.dtype == b.dtype and a.shape == b.shape and
            all(np.array_equal(a[f], b[f]) for f in ("bin1", "bin2", "IF")))


# ---------------------------------------------------------------------------------------
# (a) binning
# ---------------------------------------------------------------------------------------
def test_traditional_matrix_building_golden(mb, small_genome_file):
    g = load_golden("traditional_small.npz")
    names = [str(x) for x in g["names"]]
    text = "".join(synth.valid23_lines(names, g["c1"], g["p1"], g["c2"], g["p2"]))
    whole, local = mb.TraditionalMatrixBuilding(io.StringIO(text), small_genome_file, [500000], [40000], CHROMS)
    gw, gl = unflatten(g, "whole")["500000"], unflatten(g, "local")["40000"]
    assert set(whole[500000]) == set(gw) and set(local[40000]) == set(gl)
    for k in gw:
        assert records_equal(whole[500000][k], gw[k]), k
    for k in gl:
        assert records_equal(local[40000][k], gl[k]), k


def test_traditional_bytes_stream_and_empty_filter(mb, small_genome_file):
    """The reference is fed a subprocess pipe; chroms=[] keeps every chromosome."""
    genome = {c: l for c, l in SMALL_GENOME.items() if c != "M"}
    names = list(genome)
    c1, p1, c2, p2 = synth.genome_pairs(genome, names, 5000, 77, trans_frac=0.2)
    text = "".join(synth.valid23_lines(names, c1, p1, c2, p2))
    whole, local = mb.TraditionalMatrixBuilding(io.BytesIO(text.encode()), small_genome_file, [1000000], [100000], [])
    ow, ol = ho.traditional_matrix_building(text.splitlines(True), small_genome_file, [1000000], [100000], [])
    assert set(whole[1000000]) == set(ow[1000000]) and set(local[100000]) == set(ol[100000])
    for k in ow[1000000]:
        assert records_equal(whole[1000000][k], ow[1000000][k]), k
    for k in ol[100000]:
        assert records_equal(local[100000][k], ol[100000][k]), k


def test_binning_empty_and_ragged_inputs(mb, small_genome_file, cuda_device):
    from hichap_master_b200.device import PairColumns
    genome = mb.Load_Genome(small_genome_file, CHROMS)
    order = mb.Sort_Chromosomes(genome)
    # empty stream
    whole, local = mb.TraditionalMatrixBuilding(io.StringIO(""), small_genome_file, [500000], [40000], CHROMS)
    assert all(v.size == 0 for v in local[40000].values()) and set(local[40000]) == set(order)
    # 1..9 pairs: exercises the < 4 tail and the vector body together
    rng = np.random.default_rng(3)
    for n in (1, 2, 3, 4, 5, 7, 9):
        c = rng.integers(0, len(order), n).astype(np.int32)
        p1 = rng.integers(0, 3_000_000, n).astype(np.int32)
        p2 = rng.integers(0, 3_000_000, n).astype(np.int32)
        _, loc = mb.bin_traditional(PairColumns(c, p1, c, p2), genome, [], [40000])
        exp = ho.bin_local_dense(c, p1, c, p2, [genome[k] // 40000 + 1 for k in order], 40000)
        for i in range(len(order)):
            assert np.array_equal(loc[40000].to_numpy(i), exp[i])
    # a position beyond the chromosome end is an IndexError in the reference
    bad = PairColumns(np.array([0], np.int32), np.array([7_000_000], np.int32), np.array([0], np.int32),
                      np.array([10], np.int32))
    with pytest.raises(IndexError):
        mb.bin_traditional(bad, genome, [], [40000])


def test_chromosome_missing_from_genome_is_keyerror(mb, tmp_path):
    gs = synth.write_genome_size(str(tmp_path / "gs"), {"1": 1_000_000})
    line = next(synth.valid23_lines(["1", "2"], [0], [10], [1], [20]))
    with pytest.raises(KeyError):
        mb.TraditionalMatrixBuilding(io.StringIO(line), gs, [], [100000], ["#"])


def test_allelic_binning_golden(mb, small_genome_file, cuda_device):
    from hichap_master_b200 import _abi, kernels
    from hichap_master_b200.device import DenseBatch, PairColumns
    import torch
    g = load_golden("allelic_small.npz")
    names = [str(x) for x in g["names"]]
    genome = mb.Load_Genome(small_genome_file, CHROMS)
    order = mb.Sort_Chromosomes(genome)
    res, wres = 80000, 500000
    # TraditionalMatrixInAllelic on the concatenation of the five beds
    cls, mark = g["cls"], g["mark"]
    text = []
    for k in range(5):
        sel = cls == k
        mk = mark[sel] if k in (1, 2) else None
        text.extend(synth.allelic_lines(names, g["c1"][sel], g["p1"][sel], g["c2"][sel], g["p2"][sel], mk))
    W, L = mb.TraditionalMatrixInAllelic(io.StringIO("".join(text)), small_genome_file, [wres], [res], CHROMS)
    gt = unflatten(g, "Tradition_Local")[str(res)]
    for c in order:
        assert L[res][c].dtype == np.int64 and np.array_equal(L[res][c], gt[c])
    gtw = unflatten(g, "Tradition_Whole")[str(wres)]
    assert np.array_equal(W[wres]["Matrix"], gtw["Matrix"])
    assert {k: tuple(v) for k, v in W[wres]["Bins"].items()} == {k: tuple(int(x) for x in v) for k, v in gtw["Bins"].items()}
    # haplotype matrices: un-imputed (Both), imputed (+ one-sided R1/R2), whole-genome blocks
    remap = np.array([order.index(n) if n in order else -1 for n in names], np.int32)
    hb, htot = mb.Get_Chro_Bins_Haplotypes(small_genome_file, wres, CHROMS)
    H = DenseBatch([htot], cuda_device)
    sm = torch.tensor([hb["M" + c][0] for c in order], dtype=torch.int64, device=cuda_device)
    sp = torch.tensor([hb["P" + c][0] for c in order], dtype=torch.int64, device=cuda_device)
    gu = unflatten(g, "UnImputated_Local")[str(res)]
    gi = unflatten(g, "Imputated_Local")[str(res)]
    for tag, k, st in (("M", 1, sm), ("P", 2, sp)):
        sel = cls == k
        pc = PairColumns(remap[g["c1"][sel]], g["p1"][sel], remap[g["c2"][sel]], g["p2"][sel], mark[sel])
        Lb = mb.bin_haplotype_local(pc, genome, res, onesided=False)
        for i, c in enumerate(order):
            assert np.array_equal(Lb.to_numpy(i), gu[tag + c]), (tag, c)
        mb.bin_haplotype_local(pc, genome, res, onesided=True, out=Lb)
        for i, c in enumerate(order):
            assert np.array_equal(Lb.to_numpy(i), gi[tag + c]), (tag, c)
        kernels.bin_pairs_whole(pc, wres, st, st, H, _abi.HC_BIN_SYM_BOTH)
    for k, (s1, s2) in ((3, (sm, sp)), (4, (sp, sm))):
        sel = cls == k
        pc = PairColumns(remap[g["c1"][sel]], g["p1"][sel], remap[g["c2"][sel]], g["p2"][sel], mark[sel])
        kernels.bin_pairs_whole(pc, wres, s1, s2, H, _abi.HC_BIN_SYM_ALL)
    assert np.array_equal(H.to_numpy(0), unflatten(g, "UnImputated_Whole")[str(wres)]["Matrix"])
    # imputed whole matrix: cis one-sided contacts are added asymmetrically; with the default
    # 10 Mb imputation region nothing inter-chromosomal is imputable on this small genome
    for k, st in ((1, sm), (2, sp)):
        sel = cls == k
        pc = PairColumns(remap[g["c1"][sel]], g["p1"][sel], remap[g["c2"][sel]], g["p2"][sel], mark[sel])
        kernels.bin_pairs_whole(pc, wres, st, st, H, _abi.HC_BIN_ONESIDED)
    assert np.array_equal(H.to_numpy(0), unflatten(g, "Imputated_Whole")[str(wres)]["Matrix"])


def test_sparse_marshalling_float_and_rect(mb, cuda_device):
    rng = np.random.default_rng(9)
    M = rng.poisson(0.3, size=(37, 37)).astype(np.int64)
    rec = mb.IntraMatrixToSparseDict({"a": M, "b": M.astype(float) * 0.5})
    assert records_equal(rec["a"], ho.dense_to_triu_records(M))
    assert records_equal(rec["b"], ho.dense_to_triu_records(M.astype(float) * 0.5))
    bins = {"1": (0, 11), "2": (12, 30), "X": (31, 36)}
    S = M + M.T
    out = mb.WholeMatrixToSparseDict(bins, S)
    exp = ho.whole_matrix_to_sparse_dict(bins, S)
    assert set(out) == set(exp) == {"1", "2", "X", "1_2", "1_X", "2_X"}
    for k in exp:
        assert records_equal(out[k], exp[k]), k


# ---------------------------------------------------------------------------------------
# (b) ICE
# ---------------------------------------------------------------------------------------
def dense_from_pixels(b1, b2, cnt, lo, hi):
    n = hi - lo
    M = np.zeros((n, n), np.int64)
    sel = (b1 >= lo) & (b1 < hi) & (b2 >= lo) & (b2 < hi)
    M[b1[sel] - lo, b2[sel] - lo] = cnt[sel]
    return M + np.triu(M, 1).T


def check_weights(w, ref, what):
    assert np.array_equal(np.isnan(w), np.isnan(ref)), what + ": NaN mask differs"
    ok = ~np.isnan(ref)
    err = np.max(np.abs(w[ok] - ref[ok]) / np.abs(ref[ok])) if ok.any() else 0.0
    print("%s: max rel err %.3e over %d bins" % (what, err, int(ok.sum())))
    assert err < RTOL, what


def test_ice_cis_only_restated_golden(mb):
    g = load_golden("ice_restated.npz")
    off = g["chrom_offsets"]
    mats = [dense_from_pixels(g["bin1"], g["bin2"], g["count"], int(lo), int(hi)) for lo, hi in zip(off[:-1], off[1:])]
    w, st = mb.ice_balance_dense(mats)
    check_weights(w, g["weight_cis"], "cis-only")
    assert st["iters"] == [int(i) for i in g["iters_cis"]]
    np.testing.assert_allclose(st["scale"], g["scale_cis"], rtol=RTOL)
    assert st["cis_only"] and st["ignore_diags"] == 1


def test_ice_genome_wide_restated_golden(mb):
    g = load_golden("ice_restated.npz")
    off = g["chrom_offsets"]
    n = int(off[-1])
    M = dense_from_pixels(g["gw_bin1"], g["gw_bin2"], g["gw_count"], 0, n)
    w, st = mb.ice_balance_dense([M], chrom_offsets=off)
    check_weights(w, g["weight_gw"], "genome-wide")
    assert st["iters"] == int(g["iters_gw"]) and st["converged"]
    np.testing.assert_allclose(st["scale"], float(g["scale_gw"]), rtol=RTOL)
    np.testing.assert_allclose(st["var"], float(g["var_gw"]), rtol=1e-4)


@pytest.mark.parametrize("kw", [dict(), dict(ignore_diags=0), dict(ignore_diags=2), dict(mad_max=0, min_nnz=0),
                                dict(max_iters=5), dict(rescale_marginals=False), dict(min_count=400)])
def test_ice_parameters_vs_oracle(mb, kw):
    rng = np.random.default_rng(12)
    mats = []
    for n in (150, 61, 260):
        bias = np.exp(rng.normal(0, 0.4, n))
        d = np.abs(np.subtract.outer(np.arange(n), np.arange(n))) + 1.0
        M = rng.poisson(30.0 * bias[:, None] * bias[None, :] / d)
        M = np.triu(M) + np.triu(M, 1).T
        M[20:24, :] = 0; M[:, 20:24] = 0
        mats.append(M)
    w, st = mb.ice_balance_dense(mats, **kw)
    off = np.concatenate([[0], np.cumsum([m.shape[0] for m in mats])])
    b1, b2, cnt = [], [], []
    for m, lo in zip(mats, off[:-1]):
        x, y = np.nonzero(np.triu(m)); b1.append(x + lo); b2.append(y + lo); cnt.append(m[x, y])
    b1, b2, cnt = (np.concatenate(v) for v in (b1, b2, cnt))
    ref, rst = cooler_ice.balance(b1, b2, cnt, int(off[-1]), off, cis_only=True, **kw)
    check_weights(w, ref, "params %r" % (kw,))
    assert st["iters"] == rst["iters"]
    assert st["converged_per_chrom"] == rst["converged_per_chrom"]


def test_ice_degenerate_inputs(mb):
    # all-zero chromosome next to a normal one; 1x1 matrix; everything filtered
    rng = np.random.default_rng(4)
    A = rng.poisson(5.0, size=(64, 64)); A = np.triu(A) + np.triu(A, 1).T
    Z = np.zeros((33, 33), np.int64)
    one = np.array([[7]])
    w, st = mb.ice_balance_dense([A, Z, one])
    off = [0, 64, 97, 98]
    x, y = np.nonzero(np.triu(A))
    ref, rst = cooler_ice.balance(x, y, A[x, y], 98, off, cis_only=True)
    check_weights(w, ref, "degenerate")
    assert np.isnan(w[64:]).all()
    assert st["iters"] == rst["iters"]


def test_ice_chr21_sized_vs_oracle(mb, cuda_device):
    """Config 1 shape: chr21 at 40 kb (1204 bins), 2 M synthetic cis pairs."""
    L = synth.HG19["21"]
    p1, p2 = synth.cis_pairs("21", L, 2_000_000, seed=1)
    n = L // 40000 + 1
    M = ho.bin_local_dense(np.zeros(p1.size, np.int32), p1, np.zeros(p1.size, np.int32), p2, [n], 40000)[0]
    w, st = mb.ice_balance_dense([M])
    ref, rst = cooler_ice.balance_dense(M, cis_only=True)
    check_weights(w, ref, "chr21@40kb")
    assert st["iters"] == rst["iters"] and st["converged"]
    # property: balanced marginals are flat
    wz = np.nan_to_num(w)
    B = M * wz[:, None] * wz[None, :]
    np.fill_diagonal(B, 0)
    m = B.sum(1)[~np.isnan(w)]
    assert abs(m.mean() - 1) < 1e-3 and m.var() < 1e-4


def _ice_matrix(n, seed, scale=30.0, heavy_diag=False):
    rng = np.random.default_rng(seed)
    bias = np.exp(rng.normal(0, 0.4, n))
    d = np.abs(np.subtract.outer(np.arange(n), np.arange(n))) + 1.0
    M = rng.poisson(scale * bias[:, None] * bias[None, :] / d)
    if heavy_diag:                      # counts far above 255 next to the diagonal: the overflow list of the packed encoding
        M = M + rng.poisson(3000.0 / d ** 2)
    M = np.triu(M) + np.triu(M, 1).T
    M[n // 3:n // 3 + 5, :] = 0; M[:, n // 3:n // 3 + 5] = 0
    return M


def _ice_vs_oracle(mb, mats, what, **kw):
    w, st = mb.ice_balance_dense(mats, **kw)
    off = np.concatenate([[0], np.cumsum([m.shape[0] for m in mats])])
    b1, b2, cnt = [], [], []
    for m, lo in zip(mats, off[:-1]):
        x, y = np.nonzero(np.triu(m)); b1.append(x + lo); b2.append(y + lo); cnt.append(m[x, y])
    b1, b2, cnt = (np.concatenate(v) for v in (b1, b2, cnt))
    ref, rst = cooler_ice.balance(b1, b2, cnt, int(off[-1]), off, cis_only=True, **kw)
    check_weights(w, ref, what)
    assert st["iters"] == rst["iters"], what
    assert st["converged_per_chrom"] == rst["converged_per_chrom"], what


@pytest.mark.parametrize("env,sizes,kw", [
    ({}, (700, 333), dict()),                                        # packed encoding, cluster update kernel
    ({}, (700, 333), dict(ignore_diags=0)),                          # kept diagonal counts twice: values up to 2 x count
    # K segments of the packed kernel: kseg starts at 48 k-tiles and drops by 16 (floor 16) while the batch has fewer
    # than 4 x SMs x 2 x 8 items (9472 on 148 SMs); items = ceil(n / 16) x ceil(KT / kseg), KT = ceil(n / 128) x 4.
    # 5000 bins: KT = 160; 313 x 4 = 1252 items at kseg 48, 1565 at 32 -> kseg 16, 10 segments per row: more than
    # the unrolled 8 of the cluster update kernel
    ({}, (5000,), dict()),
    # 8200 bins have 8320 padded columns, more than the 8 x 256 x 4 of the cluster update: the single-CTA update
    # kernel runs for the whole batch (kseg 16), its general packed branch for 8200 and, for 5000, its
    # register-resident branch with 10 segments, so that branch's loop over segments beyond 8 runs too
    ({}, (8200, 5000), dict()),
    ({"HC_ICE_PACKED": "0"}, (700, 333), dict()),                    # int32 tiles, fp64 FMA kernel
    ({"HC_ICE_PACKED": "1"}, (700, 333), dict()),                    # full-matrix packed encoding, one launch pair per iteration
    ({}, (700, 333), dict(ignore_diags=3)),
    ({}, (256, 257, 40, 1), dict()),                                 # on and one past a tile edge, a 1-bin chromosome
    ({}, (2100,), dict(max_iters=7)),                                # stops at max_iters
    ({}, (1500, 900, 333, 90, 64), dict(mad_max=0, min_nnz=0)),      # five chromosomes in flight at once
    ({"HC_ICE_PACKED": "0"}, (256, 257, 40, 1), dict()),             # the same shapes on the int32 tiles
    ({"HC_ICE_PACKED": "0"}, (1500, 900, 333, 90, 64), dict(mad_max=0, min_nnz=0)),
])
def test_ice_encodings_and_kernel_variants(mb, monkeypatch, env, sizes, kw):
    """Every stream / update kernel variant of hc_ice_dense_balance against the oracle, with counts far above 255
    (overflow cells of the packed encoding) and masked rows."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    mats = [_ice_matrix(n, 40 + i, heavy_diag=True) for i, n in enumerate(sizes)]
    assert max(int(m.max()) for m in mats) > 1000
    _ice_vs_oracle(mb, mats, "variant %r %r" % (env, kw), **kw)


def test_ice_packed_wide_bias_range_matches_int32_path(mb, monkeypatch):
    """Biases spread over more than 2^20 within one chromosome: the fixed-point byte planes of the packed kernel
    lose low mantissa bits of the small biases (rounded to nearest).  NaN mask and iteration count must equal
    the int32 / fp64 path and the oracle; weights stay within the tolerance."""
    n, rng = 640, np.random.default_rng(5)
    expo = np.linspace(0.0, 21.0, n)                        # row scales 2^-21 .. 1  ->  weights spread over > 2^20
    s = 2.0 ** (-expo)
    rng.shuffle(s)
    d = np.abs(np.subtract.outer(np.arange(n), np.arange(n))) + 1.0
    lam = 4.0e7 * s[:, None] * s[None, :] / d
    M = rng.poisson(np.minimum(lam, 2.0e9 / n)).astype(np.int64)
    M = np.triu(M) + np.triu(M, 1).T
    kw = dict(mad_max=0, min_nnz=1, max_iters=300)
    monkeypatch.setenv("HC_ICE_PACKED", "1")
    w_packed, st_packed = mb.ice_balance_dense([M], **kw)
    monkeypatch.setenv("HC_ICE_PACKED", "0")
    w_i32, st_i32 = mb.ice_balance_dense([M], **kw)
    x, y = np.nonzero(np.triu(M))
    ref, rst = cooler_ice.balance(x, y, M[x, y], n, [0, n], cis_only=True, **kw)
    ok = ~np.isnan(ref)
    print("bias range 2^%.1f; iters packed %r int32 %r oracle %r" % (np.log2(np.nanmax(ref) / np.nanmin(ref)), st_packed["iters"], st_i32["iters"], rst["iters"]))
    assert np.nanmax(ref) / np.nanmin(ref) > 2.0 ** 20
    assert np.array_equal(np.isnan(w_packed), np.isnan(w_i32)) and np.array_equal(np.isnan(w_packed), np.isnan(ref))
    assert st_packed["iters"] == st_i32["iters"] == rst["iters"]
    check_weights(w_packed, ref, "packed, wide bias range")
    check_weights(w_i32, ref, "int32, wide bias range")


def test_ice_chr21_and_chr22_sized_packed_and_int32_vs_oracle(mb, monkeypatch):
    """chr21- and chr22-sized matrices at 40 kb (1.5 M contacts each): the packed encoding (default) and the int32
    tiles against the oracle."""
    mats = []
    for c, seed in (("21", 1), ("22", 2)):
        L = synth.HG19[c]
        p1, p2 = synth.cis_pairs(c, L, 1_500_000, seed=seed)
        n = L // 40000 + 1
        z = np.zeros(p1.size, np.int32)
        mats.append(ho.bin_local_dense(z, p1, z, p2, [n], 40000)[0])
    out = {}
    for mode in ("1", "0"):
        monkeypatch.setenv("HC_ICE_PACKED", mode)
        out[mode] = mb.ice_balance_dense(mats)
    off = np.concatenate([[0], np.cumsum([m.shape[0] for m in mats])])
    b1, b2, cnt = [], [], []
    for m, lo in zip(mats, off[:-1]):
        x, y = np.nonzero(np.triu(m)); b1.append(x + lo); b2.append(y + lo); cnt.append(m[x, y])
    ref, rst = cooler_ice.balance(np.concatenate(b1), np.concatenate(b2), np.concatenate(cnt), int(off[-1]), off, cis_only=True)
    for mode, (w, st) in out.items():
        check_weights(w, ref, "HC_ICE_PACKED=%s" % mode)
        assert st["iters"] == rst["iters"], mode
        np.testing.assert_allclose(st["scale"], rst["scale"], rtol=RTOL)


def test_ice_degenerate_chromosomes(mb):
    """A 300 x 300 chromosome batched with an all-zero one (nothing to balance: NaN weights, converged after one
    pass) and a 1 x 1 one."""
    rng = np.random.default_rng(4)
    A = rng.poisson(5.0, size=(300, 300)); A = np.triu(A) + np.triu(A, 1).T
    Z = np.zeros((33, 33), np.int64)
    one = np.array([[7]])
    w, st = mb.ice_balance_dense([A, Z, one])
    x, y = np.nonzero(np.triu(A))
    ref, rst = cooler_ice.balance(x, y, A[x, y], 334, [0, 300, 333, 334], cis_only=True)
    check_weights(w, ref, "degenerate chromosomes")
    assert np.isnan(w[300:]).all()
    assert st["iters"] == rst["iters"]


def test_ice_more_than_8192_columns(mb):
    """A matrix wider than the cluster update kernel covers (8 x 256 x 4 columns): generic update path on the
    packed encoding, several K-segments."""
    n, rng = 8300, np.random.default_rng(77)
    bias = np.exp(rng.normal(0, 0.3, n))
    M = np.zeros((n, n), np.int64)
    for k in range(0, 400):                 # banded counts, built diagonal by diagonal (cheap to generate)
        lam = (3000.0 / (k + 1) ** 2 + 40.0 / (k + 1)) * bias[:n - k] * bias[k:]
        v = rng.poisson(lam)
        M[np.arange(n - k), np.arange(k, n)] = v
        M[np.arange(k, n), np.arange(n - k)] = v
    M[2000:2010, :] = 0; M[:, 2000:2010] = 0
    assert M.max() > 1000
    _ice_vs_oracle(mb, [M], "n=8300", max_iters=60)


# ---------------------------------------------------------------------------------------
# (c) two-step correction
# ---------------------------------------------------------------------------------------
def check_matrix(a, ref, what):
    assert a.shape == ref.shape and a.dtype == np.float64
    denom = np.maximum(np.abs(ref), 1e-300)
    err = float(np.max(np.abs(a - ref) / denom))
    print("%s: max rel err %.3e" % (what, err))
    assert np.array_equal(a == 0, ref == 0), what + ": zero pattern differs"
    assert err < RTOL, what


def gaps_equal(a, b):
    return a.size == b.size and np.array_equal(np.asarray(a, np.int64), np.asarray(b, np.int64))


def test_two_step_golden_cases(mb):
    g = load_golden("twostep_cases.npz")
    for tag in ("nogap", "gappy"):
        nm, npm, gm, gp = mb.TwoStepCorrection(g[tag + "|TM"], g[tag + "|MM"], g[tag + "|PM"])
        assert gaps_equal(gm, g[tag + "|Gap_M"]) and gaps_equal(gp, g[tag + "|Gap_P"]), tag
        check_matrix(nm, g[tag + "|Nor_MM"], tag + " Nor_MM")
        check_matrix(npm, g[tag + "|Nor_PM"], tag + " Nor_PM")


def test_standalone_building_blocks_golden(mb):
    """Correct_VC, Coverage_M, Gap_defined(+LowRes), Non_Gap_Defined, Trans2symmetry(+LowRes) with the
    reference's signatures, against outputs of the reference functions themselves."""
    g = load_golden("building_blocks.npz")
    for tag in ("nogap", "gappy"):
        M = g[tag + "|M"]
        for mat in (M, M.astype(np.float64)):                       # integer tiles and the float64 kernel
            assert np.array_equal(mb.Coverage_M(mat), g[tag + "|Coverage"]), tag
            assert gaps_equal(mb.Gap_defined(mat), g[tag + "|Gap"]), tag
            assert gaps_equal(mb.Gap_definedLowRes(mat), g[tag + "|GapLowRes"]), tag
        assert gaps_equal(mb.Non_Gap_Defined(M.shape[0], g[tag + "|Gap"]), g[tag + "|NonGap"])
        assert gaps_equal(mb.Non_Gap_DefinedLowRes(M.shape[0], g[tag + "|Gap"]), g[tag + "|NonGap"])
        sym = mb.Trans2symmetry(g[tag + "|S"], g[tag + "|Gap"])
        check_matrix(sym, g[tag + "|Sym"], tag + " Trans2symmetry")
        check_matrix(mb.Trans2symmetryLowRes(g[tag + "|S"]), g[tag + "|SymLowRes"], tag + " Trans2symmetryLowRes")
        check_matrix(mb.Correct_VC(g[tag + "|Sym"], 2.0 / 3), g[tag + "|VC"], tag + " Correct_VC")
    check_matrix(mb.Trans2symmetry(g["forced|S"], g["forced|Gap"]), g["forced|Sym"], "forced gap pairs (max rule)")
    check_matrix(mb.Correct_VC(g["rect|X"], 0.5), g["rect|VC"], "rectangular Correct_VC")
    with pytest.raises(IndexError):
        mb.Gap_defined(np.zeros((5, 5), dtype=np.int64))            # no covered row: np.percentile([]) in the reference


def test_intra_chrom_correction_golden(mb):
    g = load_golden("allelic_small.npz")
    res = "80000"
    tra = unflatten(g, "Tradition_Local")[res]
    hap = unflatten(g, "Imputated_Local")[res]
    nor, gaps = mb.IntraChromMatrixCorrection(tra, hap)
    gn, gg = unflatten(g, "Nor_Local")[res], unflatten(g, "Gap")[res]
    assert set(nor) == set(gn)
    for k in gn:
        assert gaps_equal(gaps[k], gg[k]), k
        check_matrix(nor[k], gn[k], k)
    gb = unflatten(g, "Balanced_Local")[res]
    sp = mb.IntraMatrixToSparseDict(nor)
    for k in gb:
        assert np.array_equal(sp[k]["bin1"], gb[k]["bin1"]) and np.array_equal(sp[k]["bin2"], gb[k]["bin2"])
        np.testing.assert_allclose(sp[k]["IF"], gb[k]["IF"], rtol=RTOL)


def test_genome_wide_correction_golden(mb):
    g = load_golden("allelic_small.npz")
    tw = unflatten(g, "Tradition_Whole")["500000"]
    iw = unflatten(g, "Imputated_Whole")["500000"]
    bins = {k: tuple(int(x) for x in v) for k, v in tw["Bins"].items()}
    hbins = {k: tuple(int(x) for x in v) for k, v in iw["Bins"].items()}
    out = mb.GenomeWideMatrixCorrection(bins, hbins, tw["Matrix"], iw["Matrix"])
    check_matrix(out, g["GenomeWide|500000"], "GenomeWideMatrixCorrection")


@pytest.mark.parametrize("n,seed", [(1, 1), (63, 2), (64, 3), (65, 4), (129, 5), (700, 6)])
def test_two_step_sizes_vs_oracle(mb, n, seed):
    """Tile edges (T = 64) and a multi-tile case against the vectorised oracle."""
    rng = np.random.default_rng(seed)
    dens = np.clip(rng.gamma(2.0, 0.3, size=n), 0, 1)
    if n > 10:
        dens[3:6] = 0
    lam = 4.0 * dens[:, None] * dens[None, :] + (0.5 if n == 1 else 0.0)
    mm, pm = rng.poisson(lam), rng.poisson(0.7 * lam)
    tm = rng.poisson(6 * lam); tm = tm + tm.T + mm + pm
    if n == 1:
        mm[:] = 3; pm[:] = 2; tm[:] = 9
    ref = ho.two_step_correction(tm, mm, pm)
    out = mb.TwoStepCorrection(tm, mm, pm)
    assert gaps_equal(out[2], ref[2]) and gaps_equal(out[3], ref[3])
    check_matrix(out[0], ref[0], "n=%d MM" % n)
    check_matrix(out[1], ref[1], "n=%d PM" % n)
    np.testing.assert_allclose(out[0], out[0].T, rtol=1e-12)   # symmetric
    np.testing.assert_allclose(out[0].mean(), mm.mean(), rtol=1e-9)  # rescaled to the raw mean
    # M and P not next to each other in the batch: the per-matrix entry points (hc_twostep_alpha / hc_twostep_correct)
    # instead of the batched driver
    from hichap_master_b200.device import DenseBatch
    b = DenseBatch.from_numpy([tm, mm, tm, pm])
    nm, npm, gm, gp = mb.two_step_device(b, 0, b, 1, b, 3)
    assert gaps_equal(gm, ref[2]) and gaps_equal(gp, ref[3])
    check_matrix(nm.cpu().numpy(), ref[0], "n=%d MM (per-matrix path)" % n)
    check_matrix(npm.cpu().numpy(), ref[1], "n=%d PM (per-matrix path)" % n)


# ---------------------------------------------------------------------------------------
# banded binning (upper-only updates, L2-resident near-diagonal band, merge, mirror)
# ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,res,mode", [(0, 40000, 0), (3, 40000, 0), (2049, 40000, 0), (300_000, 40000, 0),
                                        (300_000, 7919, 0), (100_000, 40000, 1)])
def test_banded_binning_equals_direct_and_oracle(mb, cuda_device, n, res, mode):
    from hichap_master_b200 import kernels
    from hichap_master_b200.device import DenseBatch, PairColumns
    genome = {c: l for c, l in SMALL_GENOME.items() if c != "M"}
    order = list(genome)
    c1, p1, c2, p2 = synth.genome_pairs(genome, order, max(n, 1), 31, trans_frac=0.2)
    c1, p1, c2, p2 = c1[:n].copy(), p1[:n], c2[:n].copy(), p2[:n]
    if n > 10:
        c1[::17] = -1                                  # filtered chromosome
    rng = np.random.default_rng(2)
    mark = rng.integers(0, 4, size=n).astype(np.uint8)
    sizes = [genome[c] // res + 1 for c in order]
    pc = PairColumns(c1, p1, c2, p2, mark)
    A = DenseBatch(sizes, cuda_device); B = DenseBatch(sizes, cuda_device)
    kernels.bin_pairs_local(pc, res, A, mode)
    kernels.bin_pairs_local_banded(pc, res, B, mode)
    keep = (c1 >= 0) & (c2 >= 0) & ((mark == 0) | (mode == 0))
    exp = ho.bin_local_dense(c1[keep], p1[keep], c2[keep], p2[keep], sizes, res)
    for i in range(len(sizes)):
        a, b = A.to_numpy(i), B.to_numpy(i)
        assert np.array_equal(a, exp[i]) and np.array_equal(b, exp[i]), (i, sizes[i])
    assert int(B.buf.sum().item()) == int(A.buf.sum().item())   # nothing landed in the row padding
    # out-of-range positions raise like the direct kernel
    bad = PairColumns(np.array([0], np.int32), np.array([2_000_000_000], np.int32), np.array([0], np.int32),
                      np.array([5], np.int32))
    with pytest.raises(IndexError):
        kernels.bin_pairs_local_banded(bad, res, DenseBatch(sizes, cuda_device))


@pytest.mark.parametrize("pile", [True, False])
def test_hot_diagonal_binning_equals_direct(mb, cuda_device, pile):
    """1.4 M pairs (>= 2^20): every CTA counts the hottest diagonals in 16-bit shared-memory counters, drained into the
    band when they reach 0x8000.  `pile`: 200 000 pairs in ONE cell, several times the 16-bit drain threshold."""
    import torch
    from hichap_master_b200 import kernels
    from hichap_master_b200.device import DenseBatch, PairColumns
    genome = {c: l for c, l in SMALL_GENOME.items() if c != "M"}
    order = list(genome)
    res = 40000
    c1, p1, c2, p2 = synth.genome_pairs(genome, order, 1_400_000, 91, trans_frac=0.1)
    if pile:
        c1[:200_000] = 1; c2[:200_000] = 1; p1[:200_000] = 1_234_567; p2[:200_000] = 1_240_000
        c1[200_000:260_000] = 2; c2[200_000:260_000] = 2; p1[200_000:260_000] = 40_000 * 7; p2[200_000:260_000] = 40_000 * 8 + 5
    sizes = [genome[c] // res + 1 for c in order]
    pc = PairColumns(c1, p1, c2, p2)
    A = DenseBatch(sizes, cuda_device); B = DenseBatch(sizes, cuda_device)
    kernels.bin_pairs_local(pc, res, A)
    kernels.bin_pairs_local_banded(pc, res, B)
    assert torch.equal(A.buf, B.buf)
    # uint8 chromosome columns, fed in two chunks (the PCIe-overlapped path)
    Cb = DenseBatch(sizes, cuda_device)
    bb = kernels.BandedBinning(Cb, res)
    t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(cuda_device)
    u1 = np.where(c1 < 0, 255, c1).astype(np.uint8); u2 = np.where(c2 < 0, 255, c2).astype(np.uint8)
    h = 1_100_000 // 16 * 16
    for sl in (slice(0, h), slice(h, None)):
        bb.accumulate(t(u1[sl], np.uint8), t(p1[sl], np.int32), t(u2[sl], np.uint8), t(p2[sl], np.int32))
    bb.finish()
    assert torch.equal(A.buf, Cb.buf)


@pytest.mark.parametrize("n,chunk", [(0, 64), (5, 16), (100_003, 4096), (100_003, 1 << 24)])
def test_stage_from_host_chunks_equals_whole_upload(mb, cuda_device, n, chunk):
    """`LocalStage.run_from_host` (chunked H2D on a copy stream, uint8 chromosome columns binned as
    they land) gives the same tiles, records and weights as upload-then-run, and as the oracle."""
    from hichap_master_b200.pipeline import HostPairs, LocalStage
    genome = {c: l for c, l in SMALL_GENOME.items() if c != "M"}
    order = list(genome)
    res = 40000
    c1, p1, c2, p2 = synth.genome_pairs(genome, order, max(n, 1), 77, trans_frac=0.1)
    c1, p1, c2, p2 = c1[:n].copy(), p1[:n], c2[:n].copy(), p2[:n]
    if n > 10:
        c1[::13] = -1
    sizes = [genome[c] // res + 1 for c in order]
    host = HostPairs(c1, p1, c2, p2)
    st = LocalStage(sizes, max(n, 16), cuda_device)
    o1 = st.run(st.upload(host), res, records=True)
    tiles1 = [st.batch.to_numpy(i).copy() for i in range(len(sizes))]
    w1 = o1["bias"].cpu().numpy().copy()
    rec1 = [r.copy() for r in o1["records"]]
    o2 = st.run_from_host(host, res, records=True, chunk_pairs=chunk)
    keep = (c1 >= 0) & (c2 >= 0)
    exp = ho.bin_local_dense(c1[keep], p1[keep], c2[keep], p2[keep], sizes, res)
    for i in range(len(sizes)):
        assert np.array_equal(st.batch.to_numpy(i), tiles1[i]) and np.array_equal(tiles1[i], exp[i])
        assert np.array_equal(o2["records"][i], rec1[i])
    assert np.array_equal(o2["bias"].cpu().numpy(), w1, equal_nan=True)


@pytest.mark.parametrize("n,seed", [(5, 0), (1000, 1), (70_001, 2), (300_000, 3)])
def test_mad_filter_grid_wide_equals_single_cta_and_numpy(mb, cuda_device, monkeypatch, n, seed):
    """hc_ice_filter_bins: the grid-wide radix select (default) against the single-CTA kernel (HC_ICE_MAD_SINGLE=1) and
    against NumPy's medians -- marginals with ties, zeros (excluded bins) and a heavy tail; the bias masks must be equal."""
    import ctypes as C
    import torch
    from hichap_master_b200 import kernels
    from hichap_master_b200._abi import check, lib
    from hichap_master_b200.device import ptr, stream_ptr
    rng = np.random.default_rng(seed)
    marg = np.exp(rng.normal(0, 0.4, n)) * 1000
    marg[rng.random(n) < 0.1] = 0.0                         # uncovered bins
    marg[rng.random(n) < 0.05] *= 1e-3                      # low outliers (what MAD-max removes)
    marg[::7] = np.round(marg[::7])                         # ties
    nnz = np.full(n, 100.0)
    chrom_off = np.array([0, n // 3, n], np.int64)
    params = kernels.ice_params(mad_max=5, min_nnz=10)
    out = {}
    for mode in ("0", "1"):
        monkeypatch.setenv("HC_ICE_MAD_SINGLE", mode)
        t = lambda a: torch.from_numpy(a.copy()).to(cuda_device)
        d_nnz, d_marg, d_off = t(nnz), t(marg), t(chrom_off)
        bias = torch.empty(n, dtype=torch.float64, device=cuda_device)
        work = torch.empty(2 * n, dtype=torch.float64, device=cuda_device)
        check(lib().hc_ice_filter_bins(ptr(d_nnz), ptr(d_marg), n, ptr(d_off), 2, C.byref(params), ptr(bias), ptr(work),
                                       stream_ptr()), "hc_ice_filter_bins")
        out[mode] = bias.cpu().numpy()
    assert np.array_equal(out["0"], out["1"])
    # cooler's rule in NumPy
    m = marg.copy()
    for lo, hi in zip(chrom_off[:-1], chrom_off[1:]):
        c = m[lo:hi]
        m[lo:hi] = c / np.median(c[c > 0])
    lg = np.log(m[m > 0])
    med = np.median(lg)
    mad = np.median(np.abs(lg - med))
    cutoff = np.exp(med - 5 * mad)
    exp = np.ones(n)
    exp[m < cutoff] = 0.0
    assert np.array_equal(out["0"], exp)
