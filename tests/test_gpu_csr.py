"""GPU parity tests of the sort path: hand-written radix sort, reduce-by-key into the symmetric
CSR, the upper-triangular records and ICE on the CSR, against NumPy / the oracle."""
import numpy as np
import pytest

from conftest import CHROMS, SMALL_GENOME, load_golden
from hichap_master_b200 import synth
from oracle import cooler_ice
from oracle import hichap_oracle as ho

pytestmark = pytest.mark.gpu
RTOL = 1e-6


@pytest.fixture(scope="module")
def K(cuda_device):
    from hichap_master_b200 import kernels
    return kernels


@pytest.mark.parametrize("n,bits", [(0, 40), (1, 40), (5, 16), (4095, 40), (4096, 40), (4097, 34), (100_000, 40),
                                    (3_000_001, 40), (1_000_000, 64), (50_000, 8)])
def test_radix_sort_matches_numpy(K, cuda_device, n, bits):
    import torch
    rng = np.random.default_rng(n + bits)
    hi = (1 << bits) - 1 if bits < 64 else (1 << 63) - 1
    keys = rng.integers(0, hi, size=n, dtype=np.int64, endpoint=True)
    if n > 10:
        keys[::7] = keys[3]                       # duplicates
    t = torch.from_numpy(keys.copy()).to(cuda_device)
    out, _ = K.sort_keys_u64(t, bits if bits < 64 else 63)
    assert np.array_equal(out.cpu().numpy(), np.sort(keys))


def test_radix_sort_padding_keys_sort_last(K, cuda_device):
    import torch
    rng = np.random.default_rng(1)
    keys = rng.integers(0, 1 << 34, size=20_000, dtype=np.int64)
    keys[rng.random(keys.size) < 0.3] = -1        # ~0 as uint64
    out, _ = K.sort_keys_u64(torch.from_numpy(keys.copy()).to(cuda_device), 34)
    exp = np.sort(keys.view(np.uint64)).view(np.int64)
    assert np.array_equal(out.cpu().numpy(), exp)


def small_case(seed, n_pairs, trans):
    genome = {c: l for c, l in SMALL_GENOME.items() if ho.chrom_passes(c, CHROMS)}
    order = ho.sort_chromosomes(genome)
    c1, p1, c2, p2 = synth.genome_pairs(genome, order, n_pairs, seed, trans_frac=trans)
    return genome, order, c1, p1, c2, p2


@pytest.mark.parametrize("keys_per_pair", ["1", "2"])
@pytest.mark.parametrize("res,cis_only,npairs", [(40000, False, 60_000), (40000, True, 60_000), (500000, False, 5_000),
                                                 (10000, False, 7), (40000, False, 0)])
def test_pairs_to_csr_matches_oracle(K, cuda_device, res, cis_only, npairs, keys_per_pair):
    """keys_per_pair=1: the default (one upper-triangle entry per pair, lower list by a row-bits re-sort);
    2: the first version (both orientations sorted), the fallback on count-field overflow."""
    import torch
    from hichap_master_b200 import matrixBuilding as mb
    from hichap_master_b200.device import PairColumns
    genome, order, c1, p1, c2, p2 = small_case(5, max(npairs, 1), 0.2)
    c1, p1, c2, p2 = c1[:npairs], p1[:npairs], c2[:npairs], p2[:npairs]
    bins, csr = mb.bin_traditional_sparse(PairColumns(c1, p1, c2, p2), genome, res, cis_only=cis_only)
    table, total = ho.chro_bins(genome, res)
    assert bins == table and csr.nbins == total
    start = np.array([table[c][0] for c in order], np.int64)
    if keys_per_pair == "2":
        chrom_bins = torch.tensor([genome[c] // res + 1 for c in order], dtype=torch.int32, device=cuda_device)
        csr = K._pairs_to_csr_two_keys(PairColumns(c1, p1, c2, p2, device=cuda_device), res,
                                       torch.from_numpy(start).to(cuda_device), chrom_bins, total, cis_only)
        assert csr.nbins == total
    keep = (c1 == c2) if cis_only else np.ones(c1.size, bool)
    M = ho.bin_whole_dense(c1[keep], p1[keep], c2[keep], p2[keep], start, start, total, res)
    # full symmetric CSR
    rp = csr.row_ptr.cpu().numpy(); col = csr.col.cpu().numpy(); cnt = csr.cnt.cpu().numpy()
    x, y = np.nonzero(M)
    assert rp[-1] == x.size == col.size
    assert np.array_equal(np.repeat(np.arange(total), np.diff(rp)), x)
    assert np.array_equal(col, y) and np.array_equal(cnt, M[x, y])
    # the reference's per-block dictionary
    got = mb.WholeCsrToSparseDict(bins, csr)
    exp = ho.whole_matrix_to_sparse_dict(table, M)
    assert set(got) == set(exp)
    for k in exp:
        for f in ("bin1", "bin2", "IF"):
            assert np.array_equal(got[k][f], exp[k][f]), (k, f)


def csr_from_pixels(K, dev, b1, b2, cnt, n):
    """symmetric CSR tensors from upper-triangular pixels (host construction, test helper)"""
    import torch
    off = b1 != b2
    r = np.concatenate([b1, b2[off]]); c = np.concatenate([b2, b1[off]]); v = np.concatenate([cnt, cnt[off]])
    o = np.lexsort((c, r))
    r, c, v = r[o], c[o], v[o]
    rp = np.zeros(n + 1, np.int64)
    np.add.at(rp, r + 1, 1)
    rp = np.cumsum(rp)
    t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(dev)
    return K.SymCsr(t(rp, np.int64), t(c, np.int32), t(v, np.int32), n)


def check_weights(w, ref, what):
    assert np.array_equal(np.isnan(w), np.isnan(ref)), what + ": NaN mask differs"
    ok = ~np.isnan(ref)
    err = np.max(np.abs(w[ok] - ref[ok]) / np.abs(ref[ok])) if ok.any() else 0.0
    print("%s: max rel err %.3e over %d bins" % (what, err, int(ok.sum())))
    assert err < RTOL, what


@pytest.mark.parametrize("blocked", ["1", "0"])
def test_ice_csr_restated_golden(K, cuda_device, monkeypatch, blocked):
    """blocked=1: the default column-blocked encoding (hc_ice_csrb.cu); blocked=0: the row-major gather kernel."""
    monkeypatch.setenv("HC_CSR_BLOCKED", blocked)
    g = load_golden("ice_restated.npz")
    off = g["chrom_offsets"]
    n = int(off[-1])
    csr = csr_from_pixels(K, cuda_device, g["gw_bin1"], g["gw_bin2"], g["gw_count"], n)
    bias, st = K.ice_balance_csr(csr, np.array([0, n]), chrom_off=off)
    check_weights(bias.cpu().numpy(), g["weight_gw"], "csr genome-wide")
    assert st["iters"] == int(g["iters_gw"]) and st["converged"]
    csr = csr_from_pixels(K, cuda_device, g["bin1"], g["bin2"], g["count"], n)
    bias, st = K.ice_balance_csr(csr, off, chrom_off=off)
    check_weights(bias.cpu().numpy(), g["weight_cis"], "csr cis-only")
    assert st["iters"] == [int(i) for i in g["iters_cis"]]
    np.testing.assert_allclose(st["scale"], g["scale_cis"], rtol=RTOL)


@pytest.mark.parametrize("kw", [dict(), dict(ignore_diags=0), dict(ignore_diags=3), dict(mad_max=0, min_nnz=0),
                                dict(max_iters=4)])
def test_ice_csr_end_to_end_vs_oracle(K, cuda_device, kw):
    """pairs -> sort path -> CSR -> ICE, against the pixel-based oracle."""
    from hichap_master_b200 import matrixBuilding as mb
    from hichap_master_b200.device import PairColumns
    genome, order, c1, p1, c2, p2 = small_case(9, 300_000, 0.25)
    res = 40000
    bins, csr = mb.bin_traditional_sparse(PairColumns(c1, p1, c2, p2), genome, res)
    w, st = mb.ice_balance_sparse(csr, bins, cis_only=False, **kw)
    table, total = ho.chro_bins(genome, res)
    start = np.array([table[c][0] for c in order], np.int64)
    b1 = p1.astype(np.int64) // res + start[c1]; b2 = p2.astype(np.int64) // res + start[c2]
    lo, hi = np.minimum(b1, b2), np.maximum(b1, b2)
    key, cnt = np.unique(lo * total + hi, return_counts=True)
    off = mb.chrom_offsets_from_bins(bins)
    ref, rst = cooler_ice.balance(key // total, key % total, cnt, total, off, cis_only=False, **kw)
    check_weights(w, ref, "e2e %r" % (kw,))
    assert st["iters"] == rst["iters"] and st["converged"] == rst["converged"]


def test_power_of_two_bins_last_diagonal_cell_survives_padding(K, cuda_device):
    """nbins == 2^col_bits (256 bins): the key of cell (255, 255) is all ones in the low 2*col_bits bits and would tie
    with the padding key of dropped pairs; the sort must look at one more bit (kernels.key_sort_bits)."""
    import torch
    from hichap_master_b200 import kernels
    from hichap_master_b200.device import PairColumns
    res, nb = 1000, 256
    assert kernels.key_sort_bits(nb) == 17 and kernels.key_sort_bits(255) == 16 and kernels.key_sort_bits(257) == 18
    # dropped pairs (filtered chromosome -1) come FIRST in the input: a stable sort on 16 bits would leave their
    # padding keys in front of the (255, 255) key
    c1 = np.array([-1, -1, -1, 0, 0, 0, 0], np.int32)
    p1 = np.array([5, 5, 5, 255_500, 255_100, 1_000, 254_000], np.int32)
    p2 = np.array([5, 5, 5, 255_900, 255_200, 2_000, 255_999], np.int32)
    start = torch.zeros(1, dtype=torch.int64, device=cuda_device)
    chrom_bins = torch.tensor([nb], dtype=torch.int32, device=cuda_device)
    csr = kernels.pairs_to_csr(PairColumns(c1, p1, c1, p2, device=cuda_device), res, start, chrom_bins, nb, False)
    b1, b2, v = (t.cpu().numpy() for t in kernels.csr_upper_records(csr))
    got = {(int(a), int(b)): int(c) for a, b, c in zip(b1, b2, v)}
    assert got == {(1, 2): 1, (254, 255): 1, (255, 255): 2}


def _banded_pixels(n, seed, band, far_per_row, big=None):
    """upper-triangular pixels of an n-bin matrix: a dense band (long segments in the diagonal column block), random
    far pixels (short segments in every other block), a masked stretch of rows, optionally one huge count"""
    rng = np.random.default_rng(seed)
    bias = np.exp(rng.normal(0, 0.3, n))
    b1, b2, cnt = [], [], []
    for k in range(0, band):
        i = np.arange(n - k)
        v = rng.poisson(60.0 / (k + 1) * bias[i] * bias[i + k])
        keep = v > 0
        b1.append(i[keep]); b2.append(i[keep] + k); cnt.append(v[keep])
    m = n * far_per_row
    i = rng.integers(0, n, m); j = rng.integers(0, n, m)
    lo, hi = np.minimum(i, j), np.maximum(i, j)
    ok = hi - lo >= band
    key = np.unique(lo[ok].astype(np.int64) * n + hi[ok])
    b1.append(key // n); b2.append(key % n); cnt.append(rng.integers(1, 4, key.size))
    b1, b2, cnt = (np.concatenate(x) for x in (b1, b2, cnt))
    dead = (b1 >= 3000) & (b1 < 3040) | (b2 >= 3000) & (b2 < 3040)
    b1, b2, cnt = b1[~dead], b2[~dead], cnt[~dead].astype(np.int64)
    if big is not None:
        cnt[np.argmax((b1 == 100) & (b2 == 101))] = big
    o = np.lexsort((b2, b1))
    return b1[o], b2[o], cnt[o]


@pytest.mark.parametrize("n,band,far,cis,kw", [
    (20_000, 12, 6, False, dict()),                 # 3 column blocks: long diagonal-block segments, short far ones
    (20_000, 300, 2, False, dict(ignore_diags=0, max_iters=40)),  # segments of several hundred entries (whole-warp groups); diagonal counted twice
    (9_000, 4, 2, False, dict(ignore_diags=2, min_nnz=1, mad_max=0, max_iters=50)),     # very short segments (2-lane groups)
    (26_000, 12, 4, True, dict(max_iters=60)),      # cis-only: 4 problems, chromosome borders inside column blocks
])
def test_ice_csr_column_blocked_vs_oracle(K, cuda_device, n, band, far, cis, kw):
    b1, b2, cnt = _banded_pixels(n, 3 + band, band, far)
    off = np.array([0, n // 3, n // 2, n - 700, n], np.int64) if cis else np.array([0, n // 2, n], np.int64)
    if cis:         # cis-only keys: drop the pixels between different chromosomes
        ch = np.searchsorted(off[1:], np.arange(n), side="right")
        keep = ch[b1] == ch[b2]
        b1, b2, cnt = b1[keep], b2[keep], cnt[keep]
    csr = csr_from_pixels(K, cuda_device, b1, b2, cnt, n)
    bias, st = K.ice_balance_csr(csr, off if cis else np.array([0, n]), chrom_off=off, **kw)
    assert "column-blocked" in st["encoding"]
    ref, rst = cooler_ice.balance(b1, b2, cnt, n, off, cis_only=cis, **kw)
    check_weights(bias.cpu().numpy(), ref, "blocked n=%d band=%d" % (n, band))
    assert st["iters"] == rst["iters"]
    if cis:
        assert st["converged_per_chrom"] == rst["converged_per_chrom"]
        np.testing.assert_allclose(st["scale"], rst["scale"], rtol=RTOL)


def test_ice_csr_count_beyond_19_bits_uses_the_row_major_kernel(K, cuda_device):
    n = 9_000
    b1, b2, cnt = _banded_pixels(n, 8, 6, 2, big=700_000)
    csr = csr_from_pixels(K, cuda_device, b1, b2, cnt, n)
    bias, st = K.ice_balance_csr(csr, np.array([0, n]))
    assert "row-major" in st["encoding"]
    ref, rst = cooler_ice.balance(b1, b2, cnt, n, np.array([0, n]), cis_only=False)
    check_weights(bias.cpu().numpy(), ref, "count overflow fallback")
    assert st["iters"] == rst["iters"]


def _random_pairs_one_chrom(nb, res, npairs, seed, hot=0.0):
    rng = np.random.default_rng(seed)
    p1 = rng.integers(0, nb * res, npairs).astype(np.int32)
    p2 = np.clip(p1 + rng.integers(-30 * res, 30 * res, npairs), 0, nb * res - 1).astype(np.int32)
    if hot:                                                 # a heavy cell
        k = int(hot * npairs)
        p1[:k] = 5 * res + 1; p2[:k] = 9 * res + 3
    return np.zeros(npairs, np.int32), p1, p2


@pytest.mark.parametrize("nb", [1024, 777, 1])
def test_entry_path_equals_two_key_path(K, cuda_device, nb):
    """Same symmetric CSR from both versions of the sort path, incl. a power-of-two bin count (padding-bit case)
    and dropped pairs (padding keys in the middle of the list)."""
    import torch
    from hichap_master_b200.device import PairColumns
    res = 1000
    c1, p1, p2 = _random_pairs_one_chrom(nb, res, 300_000, nb)
    c1[::11] = -1                                           # filtered chromosome -> padding entries
    p1[7::13] = nb * res - 1; p2[7::13] = nb * res - 1      # the last diagonal cell (all-ones key when nb is 2^k)
    start = torch.zeros(1, dtype=torch.int64, device=cuda_device)
    chrom_bins = torch.tensor([nb], dtype=torch.int32, device=cuda_device)
    out = {}
    for mode, build in (("1", K.pairs_to_csr), ("2", K._pairs_to_csr_two_keys)):
        csr = build(PairColumns(c1, p1, c1, p2, device=cuda_device), res, start, chrom_bins, nb, False)
        out[mode] = [t.cpu().numpy() for t in (csr.row_ptr, csr.col, csr.cnt)]
    for a, b in zip(out["1"], out["2"]):
        assert np.array_equal(a, b)
    keep = c1 >= 0
    M = np.zeros((nb, nb), np.int64)
    np.add.at(M, (p1[keep] // res, p2[keep] // res), 1)
    M = M + M.T - np.diag(np.diag(M))
    x, y = np.nonzero(M)
    assert np.array_equal(out["1"][1], y) and np.array_equal(out["1"][2], M[x, y])
    assert np.array_equal(np.repeat(np.arange(nb), np.diff(out["1"][0])), x)


def test_entry_count_field_overflow_falls_back(K, cuda_device, monkeypatch):
    """A cell with more pairs than the count field holds: the entry path reports it and the two-key path (run lengths
    as int32 counts, no field limit) produces the matrix."""
    import torch
    from hichap_master_b200.device import PairColumns
    monkeypatch.setenv("HC_ENTRY_CNT_BITS", "6")            # test hook: 63 pairs per cell at most
    nb, res = 300, 1000
    c1, p1, p2 = _random_pairs_one_chrom(nb, res, 40_000, 3, hot=0.05)
    start = torch.zeros(1, dtype=torch.int64, device=cuda_device)
    chrom_bins = torch.tensor([nb], dtype=torch.int32, device=cuda_device)
    pairs = PairColumns(c1, p1, c1, p2, device=cuda_device)
    with pytest.raises(K.CountFieldOverflow):
        K.pairs_to_entry_lists(pairs, res, start, chrom_bins, nb, False)
    csr = K.pairs_to_csr(pairs, res, start, chrom_bins, nb, False)
    M = np.zeros((nb, nb), np.int64)
    np.add.at(M, (p1 // res, p2 // res), 1)
    M = M + M.T - np.diag(np.diag(M))
    x, y = np.nonzero(M)
    assert M.max() > 63
    assert np.array_equal(csr.col.cpu().numpy(), y) and np.array_equal(csr.cnt.cpu().numpy(), M[x, y])


def test_reduce_entries_adds_counts(K, cuda_device):
    """unit=False (merging lists from several ranks): counts of equal cells are added."""
    import torch
    nb = 5000
    cb, vb = K.key_col_bits(nb), K.entry_cnt_bits(nb)
    rng = np.random.default_rng(9)
    cells = rng.integers(0, nb * 40, 200_000)
    r, c = cells // 40, np.minimum(cells // 40 + cells % 40, nb - 1)
    v = rng.integers(1, 1000, cells.size)
    ent = (((r << cb) | c) << vb) | v
    t = torch.from_numpy(ent.astype(np.int64)).to(cuda_device)
    sent, free = K.sort_entries(t, nb, vb, 2)
    nv = torch.tensor([ent.size], dtype=torch.int64, device=cuda_device)
    got = K.reduce_entries(sent, nv, nb, unit=False).cpu().numpy()
    key = (r << cb) | c
    uk, inv = np.unique(key, return_inverse=True)
    tot = np.bincount(inv, weights=v).astype(np.int64)
    assert np.array_equal(got >> vb, uk) and np.array_equal(got & ((1 << vb) - 1), tot)


def test_fused_emit_equals_unfused_building_blocks(K, cuda_device):
    """hc_entries_emit (reduce + transpose in one pass) against hc_entries_reduce followed by hc_entries_transpose, on a list
    with runs that cross warp chunks and tiles (one cell holds 20 000 pairs) and padding entries."""
    import ctypes as C
    import torch
    from hichap_master_b200._abi import check, lib
    from hichap_master_b200.device import ptr, stream_ptr
    nb = 3000
    cb, vb = K.key_col_bits(nb), K.entry_cnt_bits(nb)
    rng = np.random.default_rng(11)
    r = rng.integers(0, nb, 150_000); c = np.minimum(r + rng.integers(0, 50, r.size), nb - 1)
    r[:20_000] = 7; c[:20_000] = 9                      # a long run
    r[20_000:21_000] = 100; c[20_000:21_000] = 100      # a diagonal cell
    ent = (((r << cb) | c) << vb) | 1
    ent = np.concatenate([ent, np.full(5_000, -1, np.int64)])       # padding keys (dropped pairs)
    rng.shuffle(ent)
    t = torch.from_numpy(ent.astype(np.int64)).to(cuda_device)
    sent, free = K.sort_entries(t, nb, vb, 2)
    nv = torch.tensor([r.size], dtype=torch.int64, device=cuda_device)
    up, lo, n_lo = K.reduce_entries(sent, nv, nb, unit=True, want_lower=True)
    # unfused
    n = int(sent.numel())
    work = torch.empty(int(lib().hc_csr_work_bytes(n)), dtype=torch.uint8, device=cuda_device)
    nu = C.c_int64(0)
    check(lib().hc_entries_count(ptr(sent), n, ptr(nv), vb, ptr(work), C.byref(nu), stream_ptr()), "count")
    nu = int(nu.value)
    assert nu == up.numel()
    out2 = torch.empty(nu, dtype=torch.int64, device=cuda_device)
    upos = torch.empty(nu, dtype=torch.int64, device=cuda_device)
    d_ovf = torch.zeros(1, dtype=torch.int32, device=cuda_device); h_ovf = C.c_int32(0)
    check(lib().hc_entries_reduce(ptr(sent), n, ptr(nv), ptr(work), nu, vb, 1, ptr(upos), ptr(out2), ptr(d_ovf), C.byref(h_ovf),
                                  stream_ptr()), "reduce")
    lo2 = torch.empty(nu, dtype=torch.int64, device=cuda_device)
    n_lo2 = torch.zeros(1, dtype=torch.int64, device=cuda_device)
    check(lib().hc_entries_transpose(ptr(out2), nu, cb, vb, ptr(lo2), ptr(n_lo2), stream_ptr()), "transpose")
    assert torch.equal(up, out2) and torch.equal(lo, lo2) and int(n_lo.item()) == int(n_lo2.item())
    key = (r << cb) | c
    uk, cnts = np.unique(key, return_counts=True)
    got = up.cpu().numpy()
    assert np.array_equal(got >> vb, uk) and np.array_equal(got & ((1 << vb) - 1), cnts)


@pytest.mark.parametrize("n,pad,longrun", [(1, 0, 0), (31, 3, 0), (32, 0, 0), (33, 1, 40), (511, 0, 600), (512, 7, 0), (513, 0, 0),
                                           (4095, 0, 0), (4096, 5, 5000), (4097, 0, 0), (8191, 2, 9000), (8193, 0, 0),
                                           (100_003, 11, 30_000)])
def test_entry_reduce_sizes_around_chunk_and_tile_edges(K, cuda_device, n, pad, longrun):
    """ent_count / ent_emit at list lengths around the 32-entry, 512-entry (warp chunk) and 4096-entry (tile) edges, with padding
    entries behind n_valid and one run longer than a tile; both count modes; the swapped list checked too."""
    import torch
    nb = 70_000
    cb, vb = K.key_col_bits(nb), K.entry_cnt_bits(nb)
    rng = np.random.default_rng(n + pad)
    r = rng.integers(0, nb, n); c = np.minimum(r + rng.integers(0, 3, n), nb - 1)
    if longrun:
        m = min(longrun, n)
        r[:m] = 123; c[:m] = 456
    for unit in (True, False):
        v = np.ones(n, np.int64) if unit else rng.integers(1, 50, n)
        ent = np.concatenate([(((r << cb) | c) << vb) | v, np.full(pad, -1, np.int64)]).astype(np.int64)
        t = torch.from_numpy(ent[rng.permutation(ent.size)].copy()).to(cuda_device)
        sent, _ = K.sort_entries(t, nb, vb, 2)
        nv = torch.tensor([n], dtype=torch.int64, device=cuda_device)
        up, lo, n_lo = K.reduce_entries(sent, nv, nb, unit=unit, want_lower=True)
        key = (r << cb) | c
        uk, inv = np.unique(key, return_inverse=True)
        tot = np.bincount(inv, weights=v).astype(np.int64)
        got = up.cpu().numpy()
        assert np.array_equal(got >> vb, uk) and np.array_equal(got & ((1 << vb) - 1), tot), (n, unit)
        ur, uc = uk >> cb, uk & ((1 << cb) - 1)
        exp_lo = np.where(ur != uc, (((uc << cb) | ur) << vb) | tot, -1)
        assert np.array_equal(lo.cpu().numpy(), exp_lo) and int(n_lo.item()) == int((ur != uc).sum())
