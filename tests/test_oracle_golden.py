"""CPU tests: the oracle restatements (oracle/hichap_oracle.py, oracle/cooler_ice.py) against
the committed golden vectors that were produced by the UNMODIFIED reference run through
oracle/ref_shim.py (oracle/make_golden.py).  Integer work is compared bit-exactly; floating
point at 1e-12 (the reference's own NumPy arithmetic re-expressed, only summation order differs)."""
import numpy as np

from conftest import CHROMS, SORTED_SMALL, load_golden, unflatten
from hichap_master_b200 import synth
from oracle import cooler_ice
from oracle import hichap_oracle as ho


def assert_records_equal(a, b):
    assert a.dtype == b.dtype == ho.S_DTYPE
    assert a.shape == b.shape
    for f in ("bin1", "bin2", "IF"):
        assert np.array_equal(a[f], b[f]), f


def test_traditional_binning_matches_reference_golden(small_genome_file):
    g = load_golden("traditional_small.npz")
    names = [str(x) for x in g["names"]]
    lines = list(synth.valid23_lines(names, g["c1"], g["p1"], g["c2"], g["p2"]))
    whole, local = ho.traditional_matrix_building(lines, small_genome_file, [500000], [40000], CHROMS)
    gw, gl = unflatten(g, "whole")["500000"], unflatten(g, "local")["40000"]
    assert set(whole[500000]) == set(gw) and set(local[40000]) == set(gl)
    assert set(gl) == set(SORTED_SMALL)
    for k in gw:
        assert_records_equal(whole[500000][k], gw[k])
    for k in gl:
        assert_records_equal(local[40000][k], gl[k])
    # count conservation: every kept cis pair lands once in the upper triangle
    genome = ho.load_genome(small_genome_file, CHROMS)
    c1, p1, c2, p2, _ = ho.parse_pairs(lines, genome, CHROMS, "valid23")
    assert sum(int(gl[c]["IF"].sum()) for c in gl) == int((c1 == c2).sum())


def _allelic_columns(g, genome):
    names = [str(x) for x in g["names"]]
    order = ho.sort_chromosomes(genome)
    remap = np.array([order.index(n) if n in order else -1 for n in names])
    c1, c2 = remap[g["c1"]], remap[g["c2"]]
    keep = (c1 >= 0) & (c2 >= 0)
    return order, c1, g["p1"], c2, g["p2"], g["cls"], g["mark"], keep


def test_allelic_binning_restatement_matches_reference_golden(small_genome_file):
    g = load_golden("allelic_small.npz")
    genome = ho.load_genome(small_genome_file, CHROMS)
    order, c1, p1, c2, p2, cls, mark, keep = _allelic_columns(g, genome)
    res = 80000
    nb = [genome[c] // res + 1 for c in order]
    # traditional = all five classes
    tl = ho.bin_local_dense(c1[keep], p1[keep], c2[keep], p2[keep], nb, res)
    gt = unflatten(g, "Tradition_Local")[str(res)]
    for i, c in enumerate(order):
        assert np.array_equal(tl[i], gt[c])
    # un-imputed: 'Both' rows of M_M (class 1) / P_P (class 2); imputed adds R1/R2 one-sided
    for tag, k in (("M", 1), ("P", 2)):
        sel = keep & (cls == k)
        both = sel & (mark == 0)
        un = ho.bin_local_dense(c1[both], p1[both], c2[both], p2[both], nb, res)
        gu = unflatten(g, "UnImputated_Local")[str(res)]
        for i, c in enumerate(order):
            assert np.array_equal(un[i], gu[tag + c])
        imp = ho.bin_local_onesided(c1[sel], p1[sel], c2[sel], p2[sel], mark[sel], nb, res, [m.copy() for m in un])
        gi = unflatten(g, "Imputated_Local")[str(res)]
        for i, c in enumerate(order):
            assert np.array_equal(imp[i], gi[tag + c])
            assert not np.array_equal(gi[tag + c], gi[tag + c].T) or gi[tag + c].sum() == 0  # asymmetric
    # whole-genome haplotype matrix (un-imputed): M_M/P_P Both + M_P + P_M
    wres = 500000
    hb, htot = ho.chro_bins_haplotypes(genome, wres)
    sm = np.array([hb["M" + c][0] for c in order]); sp = np.array([hb["P" + c][0] for c in order])
    H = np.zeros((htot, htot), np.int64)
    for k, (s1, s2, need_both) in {1: (sm, sm, True), 2: (sp, sp, True), 3: (sm, sp, False), 4: (sp, sm, False)}.items():
        sel = keep & (cls == k) & ((mark == 0) | (not need_both))
        ho.bin_whole_dense(c1[sel], p1[sel], c2[sel], p2[sel], s1, s2, htot, wres, out=H)
    gw = unflatten(g, "UnImputated_Whole")[str(wres)]
    assert np.array_equal(H, gw["Matrix"])
    for c in order:
        assert tuple(gw["Bins"]["M" + c]) == hb["M" + c] and tuple(gw["Bins"]["P" + c]) == hb["P" + c]


def test_two_step_correction_matches_reference_golden():
    g = load_golden("twostep_cases.npz")
    for tag in ("nogap", "gappy"):
        nm, npm, gm, gp = ho.two_step_correction(g[tag + "|TM"], g[tag + "|MM"], g[tag + "|PM"])
        assert np.array_equal(gm, g[tag + "|Gap_M"]) and np.array_equal(gp, g[tag + "|Gap_P"])
        np.testing.assert_allclose(nm, g[tag + "|Nor_MM"], rtol=1e-12, atol=0)
        np.testing.assert_allclose(npm, g[tag + "|Nor_PM"], rtol=1e-12, atol=0)
        np.testing.assert_allclose(nm, nm.T, rtol=1e-12)          # corrected matrices are symmetric
        np.testing.assert_allclose(nm.mean(), g[tag + "|MM"].mean(), rtol=1e-12)  # rescaled to raw mean


def test_intra_chrom_correction_and_gaps_match_reference_golden():
    g = load_golden("allelic_small.npz")
    res = "80000"
    tra = unflatten(g, "Tradition_Local")[res]
    hap = unflatten(g, "Imputated_Local")[res]
    nor, gaps = ho.intra_chrom_matrix_correction(tra, hap)
    gn, gg = unflatten(g, "Nor_Local")[res], unflatten(g, "Gap")[res]
    for k in gn:
        np.testing.assert_allclose(nor[k], gn[k], rtol=1e-12, atol=0)
        assert np.array_equal(gaps[k], gg[k])
    # what the reference hands to the cool writer: triu records of the corrected matrices
    gb = unflatten(g, "Balanced_Local")[res]
    for k in gb:
        rec = ho.dense_to_triu_records(nor[k])
        assert np.array_equal(rec["bin1"], gb[k]["bin1"]) and np.array_equal(rec["bin2"], gb[k]["bin2"])
        np.testing.assert_allclose(rec["IF"], gb[k]["IF"], rtol=1e-12)


def test_genome_wide_correction_matches_reference_golden():
    g = load_golden("allelic_small.npz")
    tw = unflatten(g, "Tradition_Whole")["500000"]
    iw = unflatten(g, "Imputated_Whole")["500000"]
    bins = {k: tuple(int(x) for x in v) for k, v in tw["Bins"].items()}
    hbins = {k: tuple(int(x) for x in v) for k, v in iw["Bins"].items()}
    out = ho.genome_wide_matrix_correction(bins, hbins, tw["Matrix"], iw["Matrix"])
    np.testing.assert_allclose(out, g["GenomeWide|500000"], rtol=1e-12, atol=0)


def test_bin_tables():
    genome = {c: l for c, l in synth.HG19.items() if ho.chrom_passes(c, CHROMS)}
    assert ho.sort_chromosomes(genome)[:3] == ["1", "2", "3"] and ho.sort_chromosomes(genome)[-1] == "X"
    for res, total in ((40000, 75918), (10000, 303641), (5000, 607271)):   # SURVEY.md section 8
        table, n = ho.chro_bins(genome, res)
        assert n == total
        ht, hn = ho.chro_bins_haplotypes(genome, res)
        assert hn == 2 * total and ht["P1"][0] == total
    t, _ = ho.chro_bins(genome, 40000)
    assert t["1"] == (0, 6231) and t["21"][1] - t["21"][0] + 1 == 1204


# ---- ICE restatement (parity unpinned: no reference implementation exists to pin it) --------
def test_ice_restatement_regression_and_properties():
    g = load_golden("ice_restated.npz")
    off = g["chrom_offsets"]
    n = int(off[-1])
    w, st = cooler_ice.balance(g["bin1"], g["bin2"], g["count"], n, off, cis_only=True, ignore_diags=1)
    assert np.array_equal(np.isnan(w), np.isnan(g["weight_cis"]))
    np.testing.assert_allclose(w, g["weight_cis"], rtol=1e-12, equal_nan=True)
    assert list(st["iters"]) == list(g["iters_cis"])
    # balanced marginals of every converged chromosome are 1 +- sqrt(tol)-ish after rescaling
    b1, b2 = g["bin1"], g["bin2"]
    data = g["count"].astype(float)
    data[np.abs(b1 - b2) < 1] = 0
    wz = np.nan_to_num(w)
    marg = cooler_ice.marginalize(b1, b2, wz[b1] * wz[b2] * data, n)
    for c, (lo, hi) in enumerate(zip(off[:-1], off[1:])):
        if st["converged_per_chrom"][c]:
            m = marg[lo:hi][~np.isnan(w[lo:hi])]
            assert abs(m.mean() - 1.0) < 1e-2 and m.std() < 1e-2
    w2, st2 = cooler_ice.balance(g["gw_bin1"], g["gw_bin2"], g["gw_count"], n, off, cis_only=False, ignore_diags=1)
    np.testing.assert_allclose(w2, g["weight_gw"], rtol=1e-12, equal_nan=True)
    assert st2["iters"] == int(g["iters_gw"]) and st2["converged"]


def test_ice_edge_cases():
    # all-zero matrix -> every bin filtered, weights NaN, no exception
    w, st = cooler_ice.balance(np.array([0, 1]), np.array([1, 2]), np.array([0, 0]), 4, [0, 4])
    assert np.isnan(w).all()
    # empty pixel table
    w, st = cooler_ice.balance(np.zeros(0, int), np.zeros(0, int), np.zeros(0, int), 3, [0, 3])
    assert np.isnan(w).all()
    # dense helper equals the pixel path
    rng = np.random.default_rng(5)
    M = rng.poisson(4.0, size=(40, 40)); M = M + M.T
    w1, _ = cooler_ice.balance_dense(M, mad_max=0, min_nnz=0)
    x, y = np.nonzero(np.triu(M))
    w2, _ = cooler_ice.balance(x, y, M[x, y], 40, [0, 40], mad_max=0, min_nnz=0)
    assert np.array_equal(w1, w2)


def _imputation_case(g, k, genome):
    """Inputs of the oracle's imputation for case k of imputation_small.npz."""
    order, c1, p1, c2, p2, cls, mark, keep = _allelic_columns(g, genome)
    region, imin, ratio = g["case%d|params" % k]
    whole_res = [int(r) for r in g["case%d|whole_res" % k]]
    files = {}
    for tag, kcls in (("M_M", 1), ("P_P", 2)):
        sel = cls == kcls                          # file order; filtered chromosomes stay as -1
        files[tag] = (c1[sel], p1[sel], c2[sel], p2[sel], mark[sel])
    starts = {}
    for res in whole_res:
        hb, _ = ho.chro_bins_haplotypes(genome, res)
        starts[res] = (np.array([hb["M" + c][0] for c in order]), np.array([hb["P" + c][0] for c in order]))
    return order, files, starts, whole_res, int(region), int(imin), float(ratio)


def test_inter_chromosomal_imputation_matches_reference_golden(small_genome_file):
    """Bug-for-bug restatement of matrixBuilding.py:1302-1378 / :1416-1492 against matrices the
    reference itself produced (several resolutions / region / min / ratio settings)."""
    g = load_golden("imputation_small.npz")
    genome = ho.load_genome(small_genome_file, CHROMS)
    fired = 0
    for k in range(int(g["ncases"])):
        order, files, starts, whole_res, region, imin, ratio = _imputation_case(g, k, genome)
        un = {res: g["case%d|un|%d" % (k, res)].astype(np.int64) for res in whole_res}
        imp = {res: un[res].copy() for res in whole_res}
        for res in whole_res:
            for tag, own in (("M_M", 0), ("P_P", 1)):
                ho.bin_whole_onesided(*files[tag], starts[res][own], res, imp[res])
        cis_only = {res: imp[res].copy() for res in whole_res}
        ho.impute_inter_chromosomal(un, imp, whole_res, starts, files, region, imin, ratio)
        for res in whole_res:
            assert np.array_equal(imp[res], g["case%d|imp|%d" % (k, res)]), (k, res)
            fired += int((imp[res] - cis_only[res]).sum())
    assert fired > 1000          # the fixtures do exercise the neighbourhood vote


def test_imputation_error_behaviour_of_the_oracle(tmp_path):
    """The oracle half of test_oracle_vs_reference's error test, which needs no reference: NameError when the P_P
    loop needs `M_M_sub` and the M_M loop never set it, IndexError when the stale window belongs to a coarser
    resolution (the reference's own behaviour on the same inputs, checked live where its source is present)."""
    import pytest
    from test_oracle_vs_reference import _live_imputation
    (tmp_path / "a").mkdir()
    (tmp_path / "b").mkdir()
    _, oracle = _live_imputation(tmp_path / "a", 204, [500000], (1500000, 2, 0.7), drop_mm_onesided=True)
    with pytest.raises(NameError):
        oracle({"UnImputated_Whole": {500000: {"Matrix": np.zeros((82, 82), np.int64)}}})
    _, oracle = _live_imputation(tmp_path / "b", 205, [250000, 500000], (1500000, 2, 0.7))
    with pytest.raises(IndexError):
        oracle({"UnImputated_Whole": {250000: {"Matrix": np.zeros((160, 160), np.int64)},
                                      500000: {"Matrix": np.zeros((82, 82), np.int64)}}})


def test_building_blocks_golden():
    """oracle restatements of the reference's helper functions vs outputs of the reference itself
    (Coverage_M :904, Gap_defined :915, Gap_definedLowRes :742, Trans2symmetry :945, Correct_VC :780)."""
    g = load_golden("building_blocks.npz")
    for tag in ("nogap", "gappy"):
        M = g[tag + "|M"]
        assert np.array_equal(ho.coverage(M), g[tag + "|Coverage"])
        assert np.array_equal(np.asarray(ho.gap_defined(M), np.int64), np.asarray(g[tag + "|Gap"], np.int64))
        assert np.array_equal(np.asarray(ho.gap_defined_lowres(M), np.int64), np.asarray(g[tag + "|GapLowRes"], np.int64))
        np.testing.assert_allclose(ho.trans2symmetry(g[tag + "|S"], g[tag + "|Gap"]), g[tag + "|Sym"], rtol=1e-14)
        np.testing.assert_allclose(ho.trans2symmetry(g[tag + "|S"], np.array([])), g[tag + "|SymLowRes"], rtol=1e-14)
        np.testing.assert_allclose(ho.correct_vc(g[tag + "|Sym"], 2.0 / 3), g[tag + "|VC"], rtol=1e-13)
    np.testing.assert_allclose(ho.trans2symmetry(g["forced|S"], g["forced|Gap"]), g["forced|Sym"], rtol=1e-14)
    np.testing.assert_allclose(ho.correct_vc(g["rect|X"], 0.5), g["rect|VC"], rtol=1e-13)


def test_consumers_golden():
    """oracle restatements of StructureFind's first consumers of the stage outputs vs the reference's own methods
    (Distance_Decay :201-272, the O/E loop of Get_PCA :318-326, Get_DI :804-840)."""
    g = load_golden("consumers.npz")
    np.testing.assert_array_equal(ho.balanced_matrix(g["M"], g["weight"]), g["cM"])
    db, G, NG = ho.distance_decay(g["cM"], None)
    np.testing.assert_allclose(db, g["dd_auto"], rtol=1e-13)
    assert np.array_equal(G, g["dd_auto_G"]) and np.array_equal(NG, g["dd_auto_NG"])
    db, G, NG = ho.distance_decay(g["cM"], g["dd_given_G"])
    np.testing.assert_allclose(db, g["dd_given"], rtol=1e-13)
    assert np.array_equal(NG, g["dd_given_NG"])
    np.testing.assert_allclose(ho.observed_expected(g["cM"], g["dd_auto"]), g["OE"], rtol=1e-13)
    for t in ("ttest", "chitest"):
        np.testing.assert_allclose(ho.get_di(g["cM"], g["gap"], g["window"], t), g["DI_" + t], rtol=1e-12, equal_nan=True)
