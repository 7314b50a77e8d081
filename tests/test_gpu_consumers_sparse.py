"""The downstream consumers (hichap_master_b200/structureFind.py) on scipy.sparse matrices: the CSR kernels of
csrc/hc_consumers.cu against the reference's golden outputs, the dense path (bit for bit where the arithmetic is the
same), and the oracle."""
import numpy as np
import pytest
import scipy.sparse as sp

from conftest import SMALL_GENOME, load_golden
from oracle import hichap_oracle as ho

RTOL = 1e-9        # distance sums: the same terms as the dense kernel and NumPy, added in another (fixed) order


@pytest.fixture(scope="module")
def sf(cuda_device):
    from hichap_master_b200 import structureFind
    return structureFind


def _hic(rng, n, nnz_per_row, asym=False):
    """Hi-C-shaped counts: contact probability ~ 1/distance, a bias per bin, symmetric unless ``asym``; a gap block
    (rows and columns 100-139 empty) and an all-zero row / column 7"""
    m = n * nnz_per_row
    i = rng.integers(0, n, m)
    d = np.minimum(np.exp(rng.uniform(0, np.log(n), m)).astype(np.int64) - 1, n - 1)
    j = i + np.where(rng.random(m) < 0.5, -d, d)
    ok = (j >= 0) & (j < n)
    i, j = i[ok], j[ok]
    bias = np.exp(rng.normal(0, 0.4, n))
    v = rng.poisson(2.0 * bias[i] * bias[j]) + 1
    M = sp.csr_matrix((v, (i, j)), shape=(n, n))                 # duplicates summed
    if not asym:
        M = sp.triu(M) + sp.triu(M, 1).T
    keep = np.ones(n)
    keep[100:140] = 0
    keep[7] = 0
    D = sp.diags(keep)
    return sp.csr_matrix(D @ M @ D).astype(np.int64)


def _weights(M):
    s = np.asarray(M.sum(axis=1)).ravel().astype(float)
    w = 1.0 / np.sqrt(np.maximum(s, 1.0))
    w[s < np.percentile(s, 3)] = np.nan                        # filtered bins: whole rows and columns of NaN weight
    return w


def _csr_equal(a, b):
    a, b = sp.csr_matrix(a), sp.csr_matrix(b)
    return (a.shape == b.shape and np.array_equal(a.indptr, b.indptr) and np.array_equal(a.indices, b.indices)
            and np.array_equal(a.data, b.data))


def _snapshot(M):
    return M.format, M.dtype, M.shape, [np.array(x, copy=True) for x in (getattr(M, a) for a in ("data", "indices", "indptr", "row", "col")
                                                                         if hasattr(M, a))]


def _same_snapshot(a, b):
    return a[:3] == b[:3] and len(a[3]) == len(b[3]) and all(np.array_equal(x, y) for x, y in zip(a[3], b[3]))


@pytest.mark.gpu
def test_consumers_sparse_golden(sf):
    g = load_golden("consumers.npz")
    cM = sf.balanced_matrix(sp.csr_matrix(g["M"].astype(np.int64)), g["weight"])
    assert isinstance(cM, sp.csr_matrix) and cM.dtype == np.float64
    np.testing.assert_allclose(cM.toarray(), g["cM"], rtol=1e-15)
    assert np.array_equal(cM.toarray() != 0, g["cM"] != 0)
    S = sp.csr_matrix(g["cM"])
    db, G, NG = sf.Distance_Decay(S, None)
    np.testing.assert_allclose(db, g["dd_auto"], rtol=RTOL)
    assert np.array_equal(G, g["dd_auto_G"]) and np.array_equal(NG, g["dd_auto_NG"])
    db2, G2, NG2 = sf.Distance_Decay(S, g["dd_given_G"])
    np.testing.assert_allclose(db2, g["dd_given"], rtol=RTOL)
    assert np.array_equal(NG2, g["dd_given_NG"])
    OE = sf.Observed_Expected(S, g["dd_auto"].copy())
    assert isinstance(OE, sp.csr_matrix)
    np.testing.assert_allclose(OE.toarray(), g["OE"], rtol=RTOL)
    for t in ("ttest", "chitest"):
        np.testing.assert_allclose(sf.Get_DI(S, g["gap"], g["window"], t), g["DI_" + t], rtol=RTOL, atol=1e-12, equal_nan=True)


@pytest.fixture(scope="module")
def big(sf):
    """about 12 000 bins and a few million stored entries, with its dense counterpart"""
    rng = np.random.default_rng(2024)
    n = 12_000
    M = _hic(rng, n, 400)
    w = _weights(M)
    window = rng.integers(1, 60, n)
    return M, w, window


@pytest.mark.gpu
def test_sparse_equals_dense_bit_for_bit(sf, big):
    M, w, window = big
    n = M.shape[0]
    assert 1_000_000 < M.nnz < 5_000_000
    cM = sf.balanced_matrix(M, w)
    dense_cM = sf.balanced_matrix(M.toarray(), w)
    assert np.array_equal(cM.toarray(), dense_cM)
    assert cM.nnz == np.count_nonzero(dense_cM)
    del dense_cM
    D = cM.toarray()
    for given in (None, np.concatenate([[7], np.arange(100, 140)])):
        db, G, NG = sf.Distance_Decay(cM, given)
        db_again, _, _ = sf.Distance_Decay(cM, given)
        assert np.array_equal(db, db_again)                        # fixed summation order
        ddb, dG, dNG = sf.Distance_Decay(D, given)
        rb, rG, rNG = ho.distance_decay(D, given)
        assert np.array_equal(G, dG) and np.array_equal(NG, dNG) and np.array_equal(G, rG) and np.array_equal(NG, rNG)
        assert 100 in G and 7 in G and (given is None or NG.size == n - 41)   # auto rule: nearly every column at this density
        np.testing.assert_allclose(db, ddb, rtol=RTOL)
        np.testing.assert_allclose(db, rb, rtol=RTOL)
    decline = ddb.copy()
    OE = sf.Observed_Expected(cM, decline.copy())
    assert np.array_equal(OE.indptr, cM.indptr) and np.array_equal(OE.indices, cM.indices)    # the pattern of M
    assert np.array_equal(OE.toarray(), sf.Observed_Expected(D, decline.copy()))
    for t in ("ttest", "chitest"):
        assert np.array_equal(sf.Get_DI(cM, G, window, t), sf.Get_DI(D, G, window, t), equal_nan=True), t


@pytest.mark.gpu
def test_asymmetric_matrix_against_oracle(sf):
    """a general matrix (the allelic imputed matrices are): DI reads column j, the distance sums drop gap COLUMNS"""
    rng = np.random.default_rng(5)
    n = 1500
    M = _hic(rng, n, 150, asym=True).astype(np.float64) * 0.37
    assert (M != M.T).nnz > 0
    D = M.toarray()
    db, G, NG = sf.Distance_Decay(M)
    rb, rG, rNG = ho.distance_decay(D)
    np.testing.assert_allclose(db, rb, rtol=RTOL)
    assert np.array_equal(G, rG) and np.array_equal(NG, rNG)
    given = np.array([3, 50, 51, 52, 700, 1499])
    db2, _, NG2 = sf.Distance_Decay(M, given)
    rb2, _, rNG2 = ho.distance_decay(D, given)
    np.testing.assert_allclose(db2, rb2, rtol=RTOL)
    assert np.array_equal(NG2, rNG2)
    window = rng.integers(2, 40, n)
    for t in ("ttest", "chitest"):
        got = sf.Get_DI(M, G, window, t)
        np.testing.assert_allclose(got, ho.get_di(D, G, window, t), rtol=1e-8, atol=1e-12)
        assert np.array_equal(got, sf.Get_DI(D, G, window, t), equal_nan=True)
    np.testing.assert_allclose(sf.Observed_Expected(M, rb.copy()).toarray(), ho.observed_expected(D, rb), rtol=RTOL)


def _messy(M, rng, integer):
    """the same matrix as a CSR with unsorted indices, duplicate cells and explicit zeros"""
    C = sp.coo_matrix(M)
    r, c, v = C.row, C.col, C.data
    split = rng.random(v.size) < 0.3
    if integer:
        a = v[split] // 2
    else:
        a = v[split] * 0.5                                       # exact halves: the duplicates sum back exactly
    v = v.copy()
    v[split] -= a
    r = np.concatenate([r, r[split], rng.integers(0, M.shape[0], 500)])
    c = np.concatenate([c, c[split], rng.integers(0, M.shape[0], 500)])
    v = np.concatenate([v, a, np.zeros(500, v.dtype)])
    p = rng.permutation(v.size)
    r, c, v = r[p], c[p], v[p]
    o = np.argsort(r, kind="stable")
    indptr = np.concatenate([[0], np.cumsum(np.bincount(r, minlength=M.shape[0]))])
    X = sp.csr_matrix((v[o], c[o], indptr), shape=M.shape)
    assert not X.has_sorted_indices
    return X, sp.coo_array((v, (r, c)), shape=M.shape)


@pytest.mark.gpu
def test_input_forms_and_no_mutation(sf):
    rng = np.random.default_rng(9)
    n = 900
    M = _hic(rng, n, 80)
    w = _weights(M)
    cM = sf.balanced_matrix(M, w)
    db, G, _ = sf.Distance_Decay(cM)
    window = rng.integers(1, 30, n)
    ref = {"oe": sf.Observed_Expected(cM, db.copy()), "di_t": sf.Get_DI(cM, G, window, "ttest"),
           "di_c": sf.Get_DI(cM, G, window, "chitest")}
    Mx, Mcoo = _messy(M, rng, True)
    for form in (M.tocoo(), M.tocsc(), sp.csr_array(M), Mx, Mcoo):
        snap = _snapshot(form)
        assert _csr_equal(sf.balanced_matrix(form, w), cM), type(form)
        assert _same_snapshot(snap, _snapshot(form)), type(form)
    Fx, Fcoo = _messy(cM, rng, False)
    for form in (cM.tocoo(), cM.tocsc(), sp.csr_array(cM), Fx, Fcoo):
        snap = _snapshot(form)
        got_db, got_G, _ = sf.Distance_Decay(form)
        assert np.array_equal(got_db, db) and np.array_equal(got_G, G), type(form)
        assert _csr_equal(sf.Observed_Expected(form, db.copy()), ref["oe"]), type(form)
        assert np.array_equal(sf.Get_DI(form, G, window, "ttest"), ref["di_t"], equal_nan=True), type(form)
        assert np.array_equal(sf.Get_DI(form, G, window, "chitest"), ref["di_c"], equal_nan=True), type(form)
        assert _same_snapshot(snap, _snapshot(form)), type(form)
    assert np.array_equal(sf.Get_DI(cM, G, window, "other"), np.zeros(n))


def test_non_square_input_raises():
    from hichap_master_b200 import structureFind as sf
    R = sp.csr_matrix(np.ones((3, 4)))
    for call in (lambda: sf.balanced_matrix(R.astype(np.int64), np.ones(3)), lambda: sf.Distance_Decay(R),
                 lambda: sf.Observed_Expected(R, np.ones(4)), lambda: sf.Get_DI(R, [], np.ones(4, int), "ttest")):
        with pytest.raises(ValueError):
            call()


@pytest.mark.gpu
def test_edges(sf):
    # one bin
    one = sp.csr_matrix(np.array([[5]]))
    assert np.array_equal(sf.balanced_matrix(one, [0.5]).toarray(), sf.balanced_matrix(np.array([[5]]), [0.5]))
    db, G, NG = sf.Distance_Decay(one.astype(float))
    ddb, dG, dNG = sf.Distance_Decay(np.array([[5.0]]))
    assert np.array_equal(db, ddb) and np.array_equal(G, dG) and np.array_equal(NG, dNG)
    for t in ("ttest", "chitest"):
        assert np.array_equal(sf.Get_DI(one.astype(float), [], [0], t), sf.Get_DI(np.array([[5.0]]), [], [0], t))
    # windows reaching either end, w == 1 (the t-test's 0/0 NaN), w == 0, gap bins
    rng = np.random.default_rng(3)
    n = 400
    M = _hic(rng, n, 50).astype(np.float64)
    D = M.toarray()
    window = rng.integers(0, 60, n)
    window[[0, 1, 2, 60, 61, 200, 397, 398, 399]] = [1, 1, 3, 60, 1, 1, 2, 1, 1]
    for t in ("ttest", "chitest"):
        got = sf.Get_DI(M, [5, 200], window, t)
        assert np.array_equal(got, sf.Get_DI(D, [5, 200], window, t), equal_nan=True), t
        np.testing.assert_allclose(got, ho.get_di(D, [5, 200], window, t), rtol=1e-8, atol=1e-12)
    assert np.isnan(sf.Get_DI(M, [], window, "ttest")[61])
    # whole rows / columns of NaN weight: their entries vanish from the sparse result
    C = _hic(rng, n, 50)
    w = _weights(C)
    w[10:20] = np.nan
    cM = sf.balanced_matrix(C, w)
    assert cM.nnz == np.count_nonzero(sf.balanced_matrix(C.toarray(), w))
    assert cM[10:20].nnz == 0 and cM[:, 10:20].nnz == 0
    # an all-zero matrix
    Z = sp.csr_matrix((50, 50), dtype=np.int64)
    assert sf.balanced_matrix(Z, np.ones(50)).nnz == 0
    db, G, NG = sf.Distance_Decay(Z.astype(float))
    ddb, dG, dNG = sf.Distance_Decay(np.zeros((50, 50)))
    assert np.array_equal(db, ddb) and np.array_equal(G, dG) and np.array_equal(NG, dNG)
    win = np.full(50, 3); win[25] = 1
    for t in ("ttest", "chitest"):
        assert np.array_equal(sf.Get_DI(Z.astype(float), [], win, t), sf.Get_DI(np.zeros((50, 50)), [], win, t), equal_nan=True)
    with pytest.raises(ValueError) as dense_err:
        sf.Observed_Expected(np.zeros((50, 50)), ddb.copy())
    with pytest.raises(ValueError) as sparse_err:
        sf.Observed_Expected(Z.astype(float), db.copy())
    assert str(sparse_err.value) == str(dense_err.value)


@pytest.mark.gpu
def test_cis_csr_pipeline_5kb(sf, cuda_device):
    """a CisCsr chromosome at 5 kb from the sort path, ICE weights of the CSR balancer, through all four consumers,
    against the dense consumers on the same chromosome densified"""
    from hichap_master_b200 import matrixBuilding as mb, synth
    from hichap_master_b200.device import PairColumns
    genome = {c: SMALL_GENOME[c] for c in ("1", "2")}
    order = mb.Sort_Chromosomes(genome)
    c1, p1, c2, p2 = synth.genome_pairs(genome, order, 1_500_000, 41, trans_frac=0.0)
    res = 5000
    bins, csr = mb.bin_traditional_sparse(PairColumns(c1, p1, c2, p2), genome, res, cis_only=True)
    w, _ = mb.ice_balance_sparse(csr, bins, cis_only=True)
    cis = mb.CisCsr(csr, bins, order)
    M = cis.matrices()["1"]
    lo, hi = bins["1"][0], bins["1"][1] + 1
    wc = w[lo:hi]
    D = M.toarray()
    cM = sf.balanced_matrix(M, wc)
    dcM = sf.balanced_matrix(D, wc)
    assert np.array_equal(cM.toarray(), dcM)
    db, G, NG = sf.Distance_Decay(cM)
    ddb, dG, dNG = sf.Distance_Decay(dcM)
    assert np.array_equal(G, dG) and np.array_equal(NG, dNG)
    np.testing.assert_allclose(db, ddb, rtol=RTOL)
    assert np.array_equal(sf.Observed_Expected(cM, ddb.copy()).toarray(), sf.Observed_Expected(dcM, ddb.copy()))
    window = np.full(M.shape[0], 2_000_000 // res)
    for t in ("ttest", "chitest"):
        assert np.array_equal(sf.Get_DI(cM, G, window, t), sf.Get_DI(dcM, G, window, t), equal_nan=True), t


@pytest.mark.gpu
def test_allelic_correction_output_pipeline(sf):
    """the symmetric sparse output of IntraChromMatrixCorrection on sparse inputs into Distance_Decay / Get_DI"""
    from hichap_master_b200 import matrixBuilding as mb
    from test_gpu_allelic_sparse import _random_case
    rng = np.random.default_rng(11)
    tra, hap = {}, {}
    for c, n in (("1", 700), ("2", 450)):
        TM, MM, PM = _random_case(rng, n, "gappy")
        tra[c], hap["M" + c], hap["P" + c] = sp.csr_matrix(TM), sp.csr_matrix(MM), sp.csr_matrix(PM)
    nor, gaps = mb.IntraChromMatrixCorrection(tra, hap)
    for k, S in nor.items():
        assert sp.issparse(S)
        D = S.toarray()
        db, G, NG = sf.Distance_Decay(S)
        ddb, dG, dNG = sf.Distance_Decay(D)
        assert np.array_equal(G, dG) and np.array_equal(NG, dNG), k
        np.testing.assert_allclose(db, ddb, rtol=RTOL, err_msg=k)
        db_g, _, _ = sf.Distance_Decay(S, gaps[k])
        np.testing.assert_allclose(db_g, sf.Distance_Decay(D, gaps[k])[0], rtol=RTOL, err_msg=k)
        window = rng.integers(1, 25, S.shape[0])
        for t in ("ttest", "chitest"):
            assert np.array_equal(sf.Get_DI(S, gaps[k], window, t), sf.Get_DI(D, gaps[k], window, t), equal_nan=True), (k, t)
