"""Allelic mode on CSR matrices: local resolutions whose dense working set (traditional + haplotype tiles + float64
corrected matrices) exceeds the dense budget are binned by the sort path and corrected by hc_twostep_csr_batch.
The sparse path is forced with HC_DENSE_BUDGET_GB=0 (genome-wide resolutions stay dense by contract) and checked
against the reference's golden outputs, the dense path and the NumPy oracle."""
import os

import numpy as np
import pytest
import scipy.sparse as sp

from conftest import CHROMS, load_golden, unflatten
from hichap_master_b200 import synth
from oracle import hichap_oracle as ho
from test_gpu_drivers import write_allelic_beds

RTOL = 1e-6
STORES = ("S_Traditional_Multi.npz", "S_UnImputated_Haplotype_Multi.npz", "S_Imputated_Haplotype_Multi.npz")


def test_allelic_dense_working_set_decides_per_resolution():
    """host logic: the dense working set of hg19 chr1-22,X (T + Un + Imp tiles + float64 M and P) against the default
    budget of a 180 GB card (a third): 40 kb and 20 kb stay dense, 10 kb and 5 kb go sparse"""
    from hichap_master_b200.construction import _allelic_dense_bytes
    genome = {c: l for c, l in synth.HG19.items() if c not in ("Y", "M")}
    need = {res: _allelic_dense_bytes([l // res + 1 for l in genome.values()]) / 1e9 for res in (40000, 20000, 10000, 5000)}
    assert 10 < need[40000] < 11.5 and 40 < need[20000] < 45 and 165 < need[10000] < 175 and 670 < need[5000] < 690
    budget = 180e9 / 3 / 1e9
    assert [res for res, gb in need.items() if gb > budget] == [10000, 5000]


def _gaps_equal(a, b):
    return np.array_equal(np.asarray(a, np.int64), np.asarray(b, np.int64))


def _records_close(got, exp, what):
    assert np.array_equal(got["bin1"], exp["bin1"]) and np.array_equal(got["bin2"], exp["bin2"]), what
    np.testing.assert_allclose(got["IF"], exp["IF"], rtol=RTOL, err_msg=what)


def _stores_match(dense_path, sparse_path, what):
    """integer records bit-exact, float records and weights within RTOL (same NaN mask)"""
    a, b = np.load(dense_path, allow_pickle=True), np.load(sparse_path, allow_pickle=True)
    keys = sorted(k for k in a.files if "|" in k)
    assert keys == sorted(k for k in b.files if "|" in k), what
    for k in keys:
        if k.startswith("weight_attrs"):
            continue
        if k.startswith("weight|"):
            wa, wb = a[k], b[k]
            assert np.array_equal(np.isnan(wa), np.isnan(wb)), (what, k)
            ok = ~np.isnan(wa)
            assert np.max(np.abs(wa[ok] - wb[ok]) / np.abs(wa[ok])) < RTOL, (what, k)
        elif k.startswith("bins|") or not what.endswith("_Imputated_Haplotype_Multi.npz"):
            assert a[k].dtype == b[k].dtype and all(np.array_equal(a[k][f], b[k][f]) for f in a[k].dtype.names), (what, k)
        else:
            _records_close(b[k], a[k], (what, k))


def _gap_npz_equal(pa, pb):
    a, b = np.load(pa, allow_pickle=True), np.load(pb, allow_pickle=True)
    assert a.files == b.files
    for r in a.files:
        ga, gb = a[r].item(), b[r].item()
        assert set(ga) == set(gb)
        for k in ga:
            assert _gaps_equal(ga[k], gb[k]) and np.asarray(ga[k]).dtype == np.asarray(gb[k]).dtype, (r, k)


@pytest.mark.gpu
def test_haplotype_building_sparse_golden(cuda_device, tmp_path, small_genome_file, monkeypatch):
    from hichap_master_b200 import matrixBuilding as mb
    g = load_golden("allelic_small.npz")
    beds = write_allelic_beds(str(tmp_path / "beds"), g)
    dense, sparse = str(tmp_path / "dense"), str(tmp_path / "sparse")
    os.makedirs(dense), os.makedirs(sparse)
    mb.HaplotypeMatrixBuilding(dense, beds, small_genome_file, [500000], [80000], 10000000, 2, 0.9, CHROMS)
    monkeypatch.setenv("HC_DENSE_BUDGET_GB", "0")
    _, ds = mb.HaplotypeMatrixBuilding(sparse, beds, small_genome_file, [500000], [80000], 10000000, 2, 0.9, CHROMS)
    # the local matrices are scipy CSR, equal to the reference's dense matrices
    for key in ("Tradition_Local", "UnImputated_Local", "Imputated_Local"):
        ref = unflatten(g, key)["80000"]
        assert set(ds[key][80000]) == set(ref)
        for c in ref:
            m = ds[key][80000][c]
            assert isinstance(m, sp.csr_matrix) and np.array_equal(m.toarray(), ref[c]), (key, c)
    # the genome-wide resolution stays dense
    assert isinstance(ds["Imputated_Whole"][500000]["Matrix"], np.ndarray)
    un = np.load(os.path.join(sparse, STORES[1]), allow_pickle=True)
    for c, m in unflatten(g, "UnImputated_Local")["80000"].items():
        exp = ho.dense_to_triu_records(m)
        assert all(np.array_equal(un["80000|" + c][f], exp[f]) for f in ("bin1", "bin2", "IF")), c
    imp = np.load(os.path.join(sparse, STORES[2]), allow_pickle=True)
    for c, rec in unflatten(g, "Balanced_Local")["80000"].items():
        _records_close(imp["80000|" + c], rec, c)
    gap = np.load(os.path.join(sparse, "S_Imputated_Gap.npz"), allow_pickle=True)["80000"].item()
    ref = unflatten(g, "Gap")["80000"]
    assert set(gap) == set(ref) and all(_gaps_equal(gap[k], ref[k]) for k in ref)
    # everything else equals the dense run: records, traditional weights, the 500 kb outputs, the gap NPZ
    for f in STORES:
        _stores_match(os.path.join(dense, f), os.path.join(sparse, f), f)
    _gap_npz_equal(os.path.join(dense, "S_Imputated_Gap.npz"), os.path.join(sparse, "S_Imputated_Gap.npz"))


@pytest.mark.gpu
def test_twostep_correction_sparse_golden(cuda_device):
    from hichap_master_b200 import matrixBuilding as mb
    g = load_golden("twostep_cases.npz")
    for tag in ("nogap", "gappy"):
        nm, npm, gm, gp = mb.TwoStepCorrection(*(sp.csr_matrix(g[tag + "|" + k]) for k in ("TM", "MM", "PM")))
        assert _gaps_equal(gm, g[tag + "|Gap_M"]) and _gaps_equal(gp, g[tag + "|Gap_P"]), tag
        for got, exp in ((nm, g[tag + "|Nor_MM"]), (npm, g[tag + "|Nor_PM"])):
            assert sp.isspmatrix_csr(got) and (got != got.T).nnz == 0, tag
            np.testing.assert_allclose(got.toarray(), exp, rtol=RTOL, atol=0, err_msg=tag)


def _random_case(rng, n, kind):
    """(TM, MM, PM) dense int64 with an asymmetric imputed part"""
    base = rng.poisson(3.0 / (1 + np.abs(np.subtract.outer(np.arange(n), np.arange(n)))) * 8)
    TM = np.triu(base) + np.triu(base, 1).T
    hap = []
    for p in (0.12, 0.1):
        both = rng.binomial(np.triu(TM), p)
        X = both + np.triu(both, 1).T
        one = rng.binomial(TM, p / 2) * (rng.random((n, n)) < 0.5)       # one-sided: (i, j) without (j, i)
        hap.append(X + one)
    MM, PM = hap
    if kind == "gapfree":
        MM, PM = MM + 1, PM + 1
    elif kind == "gappy" and n > 4:
        gap = np.arange(1, n, 7)
        for X in (MM, PM):
            d = X[gap, gap] + 1
            X[gap, :] = 0
            X[:, gap] = 0
            X[gap, gap] = d                                        # diagonal-only rows
            X[gap[1::2], gap[:-1:2][:len(gap[1::2])]] = 2          # and one (i, j) between two gap rows: the max rule
    return TM, MM, PM


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 63, 64, 65, 300, 2000])
def test_twostep_sparse_against_oracle(cuda_device, n):
    from hichap_master_b200 import matrixBuilding as mb
    rng = np.random.default_rng(n)
    for kind in ("gapfree", "gappy", "plain"):
        TM, MM, PM = _random_case(rng, n, kind)
        try:
            exp = ho.two_step_correction(TM, MM, PM)
        except IndexError:                    # no covered row in a matrix: the reference has no percentile
            continue
        got = mb.TwoStepCorrection(sp.csr_matrix(TM), sp.csr_matrix(MM), sp.csr_matrix(PM))
        assert _gaps_equal(got[2], exp[2]) and _gaps_equal(got[3], exp[3]), (n, kind)
        for a, b in ((got[0], exp[0]), (got[1], exp[1])):
            np.testing.assert_allclose(a.toarray(), b, rtol=RTOL, atol=0, err_msg="%d %s" % (n, kind))


@pytest.mark.gpu
def test_twostep_sparse_empty_paternal_matrix(cuda_device):
    """a chromosome whose P matrix has no contact (the paternal X of a male sample): gaps equal the dense batch path;
    the sparse path emits no record for that matrix (the dense path writes an all-NaN matrix, the reference raises)"""
    from hichap_master_b200 import matrixBuilding as mb
    rng = np.random.default_rng(7)
    tra, hap = {}, {}
    for c, n in (("1", 300), ("X", 200)):
        TM, MM, PM = _random_case(rng, n, "plain")
        tra[c], hap["M" + c], hap["P" + c] = TM, MM, PM if c == "1" else np.zeros_like(PM)
    nor_d, gap_d = mb.IntraChromMatrixCorrection(tra, hap)
    nor_s, gap_s = mb.IntraChromMatrixCorrection({c: sp.csr_matrix(m) for c, m in tra.items()},
                                                 {c: sp.csr_matrix(m) for c, m in hap.items()})
    assert set(gap_s) == set(gap_d) and all(_gaps_equal(gap_s[k], gap_d[k]) for k in gap_d)
    assert nor_s["PX"].nnz == 0 and np.isnan(nor_d["PX"]).all()
    for k in ("M1", "P1", "MX"):
        np.testing.assert_allclose(nor_s[k].toarray(), nor_d[k], rtol=RTOL, atol=0, err_msg=k)


@pytest.mark.gpu
def test_haplotype_construction_sparse_equals_dense(cuda_device, tmp_path, small_genome_file, monkeypatch):
    from hichap_master_b200 import matrixBuilding as mb
    g = load_golden("allelic_small.npz")
    rng = np.random.default_rng(5)
    reps = []
    for i in range(2):                         # two different replicates: the first one, and a subsample of it
        keep = rng.random(g["c1"].size) < (1.0 if i == 0 else 0.6)
        sub = {k: (g[k][keep] if k in ("c1", "p1", "c2", "p2", "cls", "mark") else g[k]) for k in g.files}
        reps.append(write_allelic_beds(str(tmp_path / ("rep%d" % i)), sub))
    runs = {}
    for mode in ("dense", "sparse"):
        if mode == "sparse":
            monkeypatch.setenv("HC_DENSE_BUDGET_GB", "0")
        runs[mode] = str(tmp_path / mode)
        os.makedirs(runs[mode])
        mb.HaplotypeMatrixConstruction(runs[mode], reps, small_genome_file, [500000], [80000], chroms=CHROMS)
    for prefix in ("S_", "Merged_"):
        for f in STORES:
            f = f.replace("S_", prefix)
            _stores_match(os.path.join(runs["dense"], "Cooler", f), os.path.join(runs["sparse"], "Cooler", f), f)
        gf = prefix + "Imputated_Gap.npz"
        _gap_npz_equal(os.path.join(runs["dense"], "Cooler", gf), os.path.join(runs["sparse"], "Cooler", gf))


@pytest.mark.gpu
def test_directed_entry_count_overflow(cuda_device, tmp_path, small_genome_file, monkeypatch):
    """a cell count beyond the entry count field never wraps: same stores as without the narrow field, or
    CountFieldOverflow"""
    from hichap_master_b200 import kernels, matrixBuilding as mb
    g = load_golden("allelic_small.npz")
    beds = write_allelic_beds(str(tmp_path / "beds"), g)
    monkeypatch.setenv("HC_DENSE_BUDGET_GB", "0")
    ref = str(tmp_path / "ref"); os.makedirs(ref)
    mb.HaplotypeMatrixBuilding(ref, beds, small_genome_file, [500000], [80000], chroms=CHROMS)
    monkeypatch.setenv("HC_ENTRY_CNT_BITS", "2")
    out = str(tmp_path / "narrow"); os.makedirs(out)
    try:
        mb.HaplotypeMatrixBuilding(out, beds, small_genome_file, [500000], [80000], chroms=CHROMS)
    except kernels.CountFieldOverflow:
        return
    for f in STORES:
        _stores_match(os.path.join(ref, f), os.path.join(out, f), f)


# ---- full size: C3-like synthetic pairs (the generator and seeds of bench.py's C3 section) ----------------------------
def _c3_pairs(genome, order, n, dev):
    """(rest, M_M, P_P) PairColumns: 86 % bi-allelic (+ M_P / P_M), 6 % M_M, 6 % P_P; Both / R1 / R2 = 30 / 35 / 35 %"""
    import torch
    from hichap_master_b200.device import PairColumns
    c1, p1, c2, p2 = synth.genome_pairs_torch(genome, order, n, 3, dev, trans_frac=0.0)
    gen = torch.Generator(device=dev); gen.manual_seed(33)
    cls = torch.rand(n, generator=gen, device=dev)
    mark = torch.multinomial(torch.tensor([0.30, 0.35, 0.35], device=dev), n, replacement=True, generator=gen).to(torch.uint8)
    out = []
    for sel in ((cls < 0.86) | (cls >= 0.98), (cls >= 0.86) & (cls < 0.92), (cls >= 0.92) & (cls < 0.98)):
        out.append(PairColumns(c1[sel], p1[sel], c2[sel], p2[sel], mark[sel], device=dev))
    return out


def _sparse_run(genome, cols, res, dev):
    from hichap_master_b200 import kernels
    from hichap_master_b200.construction import HaplotypeData, _bin_haplotype_sparse
    data = HaplotypeData()
    _bin_haplotype_sparse(data, cols, genome, res, dev)
    T, H = data.tra_local[res], data.imp_local[res]
    return kernels.twostep_csr_batch(T.csr, T.off, H.csr, H.off), data


@pytest.mark.gpu
def test_fullsize_chr1_40kb_sparse_equals_dense_batch(cuda_device):
    from hichap_master_b200 import _abi, kernels
    from hichap_master_b200.construction import _sub_batch
    from hichap_master_b200.device import DenseBatch
    from hichap_master_b200.matrixBuilding import IntraMatrixToSparseDict
    genome, res = {"1": synth.HG19["1"]}, 40000
    rest, mm, pp = _c3_pairs(genome, ["1"], 8_000_000, cuda_device)
    (recs, gaps), _ = _sparse_run(genome, {"Bi_Allelic": rest, "M_M": mm, "P_P": pp}, res, cuda_device)
    n = genome["1"] // res + 1
    assert n == 6232
    T, H = DenseBatch([n], cuda_device), DenseBatch([n, n], cuda_device)
    for p in (rest, mm, pp):
        kernels.bin_pairs_local(p, res, T)
    for k, p in enumerate((mm, pp)):
        kernels.bin_pairs_local(p, res, _sub_batch(H, k, 1), _abi.HC_BIN_SYM_BOTH)
        kernels.bin_pairs_local(p, res, _sub_batch(H, k, 1), _abi.HC_BIN_ONESIDED)
    mats, dgaps = kernels.twostep_batch(T, H)
    for k in range(2):
        assert _gaps_equal(gaps[k], dgaps[k]), k
        _records_close(recs[k], IntraMatrixToSparseDict({"x": mats[k]})["x"], k)


@pytest.mark.gpu
def test_fullsize_chr21_10kb_sparse_equals_oracle(cuda_device):
    genome, res = {"21": synth.HG19["21"]}, 10000
    rest, mm, pp = _c3_pairs(genome, ["21"], 2_000_000, cuda_device)
    (recs, gaps), data = _sparse_run(genome, {"Bi_Allelic": rest, "M_M": mm, "P_P": pp}, res, cuda_device)
    T = data.tra_local[res].matrices()["21"].toarray()
    H = data.imp_local[res].matrices()
    assert T.shape == (4813, 4813)
    exp = ho.two_step_correction(T, H["M21"].toarray(), H["P21"].toarray())
    for k in range(2):
        assert _gaps_equal(gaps[k], exp[2 + k]), k
        _records_close(recs[k], ho.dense_to_triu_records(exp[k]), k)


@pytest.mark.gpu
def test_allelic_driver_completes_at_5kb(cuda_device, tmp_path, monkeypatch):
    """hg19 chr1-22,X at 5 kb: the dense allelic working set would be ~680 GB, so completing shows no n^2 allocation"""
    import torch
    from hichap_master_b200 import matrixBuilding as mb
    genome = {c: l for c, l in synth.HG19.items() if c not in ("Y", "M")}
    order = [str(i) for i in range(1, 23)] + ["X"]
    gfile = synth.write_genome_size(str(tmp_path / "genomeSize"), genome)
    cls_of = {"Bi_Allelic": 0, "M_M": 1, "P_P": 2}
    parts = _c3_pairs(genome, order, 3_000_000, cuda_device)
    beds = str(tmp_path / "beds"); os.makedirs(beds)
    for tag, p in zip(("Bi_Allelic", "M_M", "P_P"), parts):
        cols = [t.cpu().numpy() for t in (p.c1, p.p1, p.c2, p.p2, p.mark)]
        with open(os.path.join(beds, "S_Valid_%s.bed" % tag), "w") as fh:
            fh.writelines(synth.allelic_lines(order, *cols[:4], cols[4] if cls_of[tag] else None))
    bi = [t[:10].cpu().numpy() for t in (parts[0].c1, parts[0].p1, parts[0].c2, parts[0].p2)]
    for tag in ("M_P", "P_M"):
        with open(os.path.join(beds, "S_Valid_%s.bed" % tag), "w") as fh:
            fh.writelines(synth.allelic_lines(order, *bi))
    out = str(tmp_path / "out"); os.makedirs(out)
    monkeypatch.delenv("HC_DENSE_BUDGET_GB", raising=False)
    torch.cuda.reset_peak_memory_stats(cuda_device)
    _, ds = mb.HaplotypeMatrixBuilding(out, beds, gfile, [], [5000], chroms=CHROMS)
    assert torch.cuda.max_memory_allocated(cuda_device) < 40e9
    assert isinstance(ds["Imputated_Local"][5000]["M1"], sp.csr_matrix)
    st = np.load(os.path.join(out, STORES[2]), allow_pickle=True)
    assert st["5000|M1"].size > 0 and np.isfinite(st["5000|M1"]["IF"]).all()
    gap = np.load(os.path.join(out, "S_Imputated_Gap.npz"), allow_pickle=True)["5000"].item()
    assert set(gap) == {h + c for h in "MP" for c in order}
