"""B200 drop-ins for the first consumers of the matrix stage's outputs in ``HiCHap/StructureFind.py`` (SURVEY.md
section 8f row 4): how ``CallPeaks`` ingests the ICE weights and the gap NPZ, the distance-decay curve and the
observed/expected matrix of the compartment analysis, and the directionality index of the TAD caller.  Same names,
argument order and return values as the reference methods (``self`` dropped); the arithmetic runs in the kernels of
``csrc/hc_consumers.cu`` behind the C ABI.  Citations are ``file:line`` in the reference tree.

Every matrix argument may also be a ``scipy.sparse`` matrix (any format): the sparse outputs of the matrix stage at
10 kb and 5 kb (``CisCsr.matrices()``, the allelic corrections).  Those run on a canonical CSR on the device (the
CSR kernels of the same file) and never build the n x n matrix; ``balanced_matrix`` and ``Observed_Expected`` then
return a float64 ``scipy.sparse.csr_matrix``.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _abi
from .device import DenseBatch, require_cuda
from .kernels import GenCsr, ptr, stream_ptr
from .matrixBuilding import _device_csr


def _f64(M):
    if isinstance(M, torch.Tensor):
        return M.to(device=require_cuda(), dtype=torch.float64).contiguous()
    return torch.from_numpy(np.ascontiguousarray(np.asarray(M), dtype=np.float64)).to(require_cuda())


def _sparse(M, dtype, transpose=False):
    """scipy.sparse ``M`` -> canonical device CSR (``transpose``: the CSR of M.T, i.e. the column-compressed M), or
    None for any other input"""
    import scipy.sparse as sp
    if not sp.issparse(M):
        return None
    if M.ndim != 2 or M.shape[0] != M.shape[1]:
        raise ValueError("a square matrix is expected, got shape %s" % (M.shape,))
    return _device_csr(M.T if transpose else M, GenCsr, dtype)


def _like(c, values):
    """float64 scipy CSR with the pattern of the canonical CSR ``c`` and the device ``values`` of its entries"""
    import scipy.sparse as sp
    h = c.host
    return sp.csr_matrix((values.cpu().numpy(), h.indices, h.indptr), shape=h.shape)


def _flags(n, idx, dev):
    f = np.zeros(n, dtype=np.uint8)
    idx = np.asarray(idx, dtype=np.int64).reshape(-1)
    f[idx[(idx >= 0) & (idx < n)]] = 1
    return torch.from_numpy(f).to(dev)


# ---- CallPeaks: weights and gaps --------------------------------------------------------------------------------
def balanced_matrix(M, weight):
    """``np.nan_to_num(cooler.matrix(balance=True).fetch(chrom))`` (StructureFind.py:2005-2007): count * w_i * w_j with
    the filtered (NaN-weight) bins zeroed.  ``M``: integer matrix, ``scipy.sparse`` matrix of counts or ``(DenseBatch,
    index)``; ``weight``: the chromosome's slice of the ICE weight vector.  A sparse ``M`` gives a float64
    ``scipy.sparse.csr_matrix`` whose non-zeros are those of the dense result (the entries of filtered bins are
    dropped)."""
    c = _sparse(M, np.int32)
    if c is not None:
        w = _f64(weight).reshape(-1)
        if w.numel() != c.nbins:
            raise ValueError("weight has %d entries for a %d-bin matrix" % (w.numel(), c.nbins))
        out = torch.empty(c.nnz, dtype=torch.float64, device=w.device)
        _abi.check(_abi.lib().hc_balance_apply_csr_i32(ptr(c.row_ptr), ptr(c.col), ptr(c.cnt), c.nbins, ptr(w), ptr(out),
                                                       stream_ptr()), "hc_balance_apply_csr_i32")
        r = _like(c, out)
        r.eliminate_zeros()
        return r
    b, i = M if isinstance(M, tuple) else (DenseBatch.from_numpy([np.asarray(M)]), 0)
    n = b.sizes[i]
    w = _f64(weight).reshape(-1)
    assert w.numel() == n
    out = torch.empty((n, n), dtype=torch.float64, device=b.device)
    _abi.check(_abi.lib().hc_balance_apply_i32(b.mat_ptr(i), b.lds[i], n, ptr(w), ptr(out), out.stride(0), stream_ptr()),
               "hc_balance_apply_i32")
    return out.cpu().numpy()


def peak_biases(weight):
    """StructureFind.py:2008-2011: ``biases = 1 / weight`` wherever the weight is non-zero or NaN (a NaN weight stays
    NaN; ``bias_handle`` below turns it into 1), 0 elsewhere.  O(n) host arithmetic."""
    tmp = np.asarray(weight, dtype=np.float64)
    mask = np.logical_not(tmp == 0) | np.isnan(tmp)
    biases = np.zeros_like(tmp)
    with np.errstate(divide="ignore", invalid="ignore"):
        biases[mask] = 1 / tmp[mask]
    return biases


def bias_handle(bias):
    """StructureFind.py:1948-1952."""
    bias = np.array(bias, dtype=np.float64).reshape(np.shape(bias)[0],)
    bias[np.isnan(bias)] = 1.0
    return bias


def load_gap(gap_file, res, chroms):
    """StructureFind.py:1988-1992: the per-chromosome gap rows of ``{prefix}Imputated_Gap.npz`` (written by
    ``HaplotypeMatrixBuilding``) at one resolution."""
    Gap = np.load(gap_file, allow_pickle=True)
    Gap = Gap[str(res)][()]
    return {chro: Gap[chro] for chro in chroms}


# ---- compartment analysis -----------------------------------------------------------------------------------------
def Distance_Decay(M, G_array=None):
    """StructureFind.py:201-272 -> (distance_bin, G_array, NG_array).  Mean contact per genomic distance over the
    non-zero entries whose COLUMN is not a gap; without ``G_array`` the gaps are the columns with at most 5 % non-zero
    entries.  The per-distance sums run on the device; the O(n) normalisation by the number of contributing bins is the
    reference's own arithmetic on prefix counts.  A ``scipy.sparse`` ``M`` runs on its stored entries."""
    c = _sparse(M, np.float64)
    t = _f64(M) if c is None else None
    size = t.shape[0] if c is None else c.nbins
    dev = t.device if c is None else c.device
    bin_arange = np.arange(size)
    if G_array is None:
        nz = torch.empty(size, dtype=torch.int32, device=dev)
        if c is None:
            _abi.check(_abi.lib().hc_colnnz_f64(ptr(t), t.stride(0), size, ptr(nz), stream_ptr()), "hc_colnnz_f64")
        else:
            _abi.check(_abi.lib().hc_colnnz_csr(ptr(c.col), c.nnz, size, ptr(nz), stream_ptr()), "hc_colnnz_csr")
        gap_mask = (nz.cpu().numpy() / float(size)) <= 0.05
        G_array, NG_array = bin_arange[gap_mask], bin_arange[~gap_mask]
    else:
        G_array = np.asarray(G_array)
        keep = np.ones(size, dtype=bool)
        g = G_array.astype(np.int64)
        keep[g[(g >= 0) & (g < size)]] = False
        NG_array = bin_arange[keep]
    gf = _flags(size, G_array, dev)
    dsum = torch.empty(size, dtype=torch.float64, device=dev)
    if c is None:
        _abi.check(_abi.lib().hc_distance_sums_f64(ptr(t), t.stride(0), size, ptr(gf), ptr(dsum), stream_ptr()),
                   "hc_distance_sums_f64")
    else:
        work = torch.empty(int(_abi.lib().hc_distance_sums_csr_work_bytes(c.nnz)), dtype=torch.uint8, device=dev)
        _abi.check(_abi.lib().hc_distance_sums_csr_f64(ptr(c.row_ptr), ptr(c.col), ptr(c.cnt), c.nnz, size, ptr(gf),
                                                       ptr(dsum), ptr(work), stream_ptr()), "hc_distance_sums_csr_f64")
    distance_bin = dsum.cpu().numpy()
    # gaps among the first / last bins of each diagonal (:253-268), via prefix counts instead of per-distance scans
    g = np.asarray(G_array, dtype=np.int64)
    g = g[(g >= 0) & (g <= size - 1)]
    cnt = np.bincount(g, minlength=size)                       # a gap listed twice counts twice, as in the reference
    pre = np.concatenate([[0], np.cumsum(cnt)])
    i = np.arange(size)
    start = pre[size - i]                                      # gaps in [0, size-1-i]
    end = pre[size] - pre[i]                                   # gaps in [i, size-1]
    bin_num = np.where(i == 0, float(size) - end, (size - i) * 2.0 - (start + end))
    ok = bin_num > 0
    distance_bin[ok] = distance_bin[ok] / bin_num[ok]
    return distance_bin, G_array, NG_array


def Observed_Expected(M, distance_bin):
    """The O/E matrix ``Get_PCA`` builds from the decay curve (StructureFind.py:318-326, SA = False): zeros of the curve
    are first replaced by its smallest non-zero value (in place, like the reference), then every non-zero entry is
    divided by the expected value at its distance.  A ``scipy.sparse`` ``M`` gives a float64
    ``scipy.sparse.csr_matrix`` with the pattern of ``M``."""
    decline = distance_bin
    decline[decline == 0] = decline[np.nonzero(decline)].min()
    c = _sparse(M, np.float64)
    if c is not None:
        d = torch.from_numpy(np.ascontiguousarray(decline, dtype=np.float64)).to(c.device)
        if d.numel() < c.nbins:
            raise ValueError("distance_bin has %d entries for a %d-bin matrix" % (d.numel(), c.nbins))
        out = torch.empty(c.nnz, dtype=torch.float64, device=c.device)
        _abi.check(_abi.lib().hc_observed_expected_csr_f64(ptr(c.row_ptr), ptr(c.col), ptr(c.cnt), c.nbins, ptr(d),
                                                           ptr(out), stream_ptr()), "hc_observed_expected_csr_f64")
        return _like(c, out)
    t = _f64(M)
    n = t.shape[0]
    d = torch.from_numpy(np.ascontiguousarray(decline, dtype=np.float64)).to(t.device)
    out = torch.empty_like(t)
    _abi.check(_abi.lib().hc_observed_expected_f64(ptr(t), t.stride(0), n, ptr(d), ptr(out), out.stride(0), stream_ptr()),
               "hc_observed_expected_f64")
    return out.cpu().numpy()


# ---- TAD caller ---------------------------------------------------------------------------------------------------------
def Get_DI(M, Gap, window_bin, test_type="ttest"):
    """StructureFind.py:804-840: directionality index per bin from the ``window_bin[j]`` entries above and below the
    diagonal in column j; 0 for gap bins and for bins closer than the window to either end.  A ``scipy.sparse`` ``M``
    is read column by column from its column-compressed form."""
    if test_type not in ("ttest", "chitest"):
        return np.zeros(np.shape(M)[0])                         # the reference appends bias = 0 for any other test type
    c = _sparse(M, np.float64, transpose=True)
    if c is not None:
        n = c.nbins
        gf = _flags(n, Gap, c.device)
        wb = torch.from_numpy(np.ascontiguousarray(np.asarray(window_bin)[:n], dtype=np.int32)).to(c.device)
        if wb.numel() != n:
            raise ValueError("window_bin has %d entries for a %d-bin matrix" % (wb.numel(), n))
        di = torch.empty(n, dtype=torch.float64, device=c.device)
        _abi.check(_abi.lib().hc_directionality_index_csc_f64(ptr(c.row_ptr), ptr(c.col), ptr(c.cnt), n, ptr(gf), ptr(wb),
                                                              int(test_type == "chitest"), ptr(di), stream_ptr()),
                   "hc_directionality_index_csc_f64")
        return di.cpu().numpy()
    t = _f64(M)
    n = t.shape[0]
    gf = _flags(n, Gap, t.device)
    wb = torch.from_numpy(np.ascontiguousarray(np.asarray(window_bin)[:n], dtype=np.int32)).to(t.device)
    di = torch.empty(n, dtype=torch.float64, device=t.device)
    _abi.check(_abi.lib().hc_directionality_index_f64(ptr(t), t.stride(0), n, ptr(gf), ptr(wb), int(test_type == "chitest"),
                                                      ptr(di), stream_ptr()), "hc_directionality_index_f64")
    return di.cpu().numpy()
