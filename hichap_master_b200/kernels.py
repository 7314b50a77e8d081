"""Thin Python wrappers over the C ABI (one function per kernel family).  Everything here
takes / returns device-resident objects from ``device.py``; the reference-named, NumPy-in /
NumPy-out functions live in ``matrixBuilding.py`` and are built from these.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np
import torch

from . import _abi
from ._abi import IceParams, IceResult, IceRunInfo, check, lib
from .device import DenseBatch, PairColumns, ptr, stream_ptr

S_DTYPE = np.dtype([("bin1", "<i8"), ("bin2", "<i8"), ("IF", "<f8")])  # matrixBuilding.py:460-461


# --------------------------------------------------------------------------------------
# (a) binning
# --------------------------------------------------------------------------------------
def _oob_counter(dev):
    return torch.zeros(1, dtype=torch.int64, device=dev)


def _raise_oob(oob, what):
    n = int(oob.item())
    if n:
        # the reference indexes a NumPy matrix with the bin and raises IndexError
        raise IndexError("%d pair(s) fall outside the %s matrix (position beyond the chromosome "
                         "length in the genomeSize file)" % (n, what))


def bin_pairs_local(pairs: PairColumns, res: int, batch: DenseBatch, mode=_abi.HC_BIN_SYM_ALL,
                    check_bounds=True, oob=None):
    """Accumulate cis pairs into the per-chromosome matrices of ``batch`` (matrix i <->
    chromosome index i).  matrixBuilding.py:595-603 and the allelic variants.  ``oob``: device
    int64[1] counter of out-of-range pairs to add to (the caller checks it later)."""
    oob = _oob_counter(batch.device) if oob is None else oob
    check(lib().hc_bin_pairs_local(ptr(pairs.c1), ptr(pairs.p1), ptr(pairs.c2), ptr(pairs.p2),
                                   ptr(pairs.mark), pairs.n, int(res), int(mode), ptr(batch.buf),
                                   ptr(batch.mat_off), ptr(batch.mat_n), ptr(batch.mat_ld),
                                   len(batch), ptr(oob), stream_ptr()), "hc_bin_pairs_local")
    if check_bounds:
        _raise_oob(oob, "intra-chromosomal")


def bin_pairs_local_banded(pairs: PairColumns, res: int, batch: DenseBatch, mode=_abi.HC_BIN_SYM_ALL,
                           check_bounds=True, work=None, band_width=128, oob=None):
    """``bin_pairs_local`` for the symmetric modes on matrices that are symmetric on entry
    (freshly zeroed tiles): upper-triangle-only updates with an L2-resident near-diagonal band
    accumulator, band merge, mirror.  Falls back to the direct kernel outside its limits.
    Returns the work buffer (reusable)."""
    if len(batch) > 256 or mode == _abi.HC_BIN_ONESIDED or batch.nbins == 0:
        bin_pairs_local(pairs, res, batch, mode, check_bounds, oob=oob)
        return work
    oob = _oob_counter(batch.device) if oob is None else oob
    nbytes = int(lib().hc_bin_band_work_bytes(batch.nbins, band_width))
    if work is None or work.numel() < nbytes:
        work = torch.empty(nbytes, dtype=torch.uint8, device=batch.device)
    check(lib().hc_bin_pairs_local_banded(ptr(pairs.c1), ptr(pairs.p1), ptr(pairs.c2), ptr(pairs.p2),
                                          ptr(pairs.mark), pairs.n, int(res), int(mode), ptr(batch.buf),
                                          ptr(batch.mat_off), ptr(batch.mat_n), ptr(batch.mat_ld),
                                          ptr(batch.bin_off), len(batch), batch.h_mat_n, band_width, ptr(oob),
                                          ptr(work), stream_ptr()), "hc_bin_pairs_local_banded")
    if check_bounds:
        _raise_oob(oob, "intra-chromosomal")
    return work


class BandedBinning:
    """begin -> accumulate(chunk) x N -> finish: banded binning fed chunk by chunk (e.g. while later
    chunks are still in flight over PCIe).  Chromosome columns may be int32 or uint8 (255 = filtered)."""

    def __init__(self, batch: DenseBatch, res: int, mode=_abi.HC_BIN_SYM_ALL, work=None, band_width=128, oob=None):
        if len(batch) > 256 or mode == _abi.HC_BIN_ONESIDED:
            raise ValueError("banded binning: symmetric modes, at most 256 matrices")
        self.batch, self.res, self.mode = batch, int(res), int(mode)
        self.bw = int(band_width)
        self.oob = _oob_counter(batch.device) if oob is None else oob
        nbytes = int(lib().hc_bin_band_work_bytes(batch.nbins, self.bw))
        if work is None or work.numel() < nbytes:
            work = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=batch.device)
        self.work = work
        check(lib().hc_bin_band_begin(ptr(work), batch.nbins, self.bw, stream_ptr()), "hc_bin_band_begin")

    def accumulate(self, c1, p1, c2, p2, mark=None):
        b = self.batch
        u8 = c1.dtype == torch.uint8
        assert c2.dtype == c1.dtype and p1.dtype == torch.int32 and p2.dtype == torch.int32
        check(lib().hc_bin_band_accumulate(ptr(c1), ptr(p1), ptr(c2), ptr(p2), ptr(mark), int(p1.numel()), int(u8),
                                           self.res, self.mode, ptr(b.buf), ptr(b.mat_off), ptr(b.mat_n), ptr(b.mat_ld),
                                           ptr(b.bin_off), len(b), self.bw, ptr(self.oob), ptr(self.work), stream_ptr()),
              "hc_bin_band_accumulate")

    def finish(self, check_bounds=True):
        b = self.batch
        check(lib().hc_bin_band_finish(ptr(b.buf), ptr(b.mat_off), ptr(b.mat_n), ptr(b.mat_ld), ptr(b.bin_off), len(b),
                                       b.h_mat_n, self.bw, ptr(self.work), stream_ptr()), "hc_bin_band_finish")
        if check_bounds:
            _raise_oob(self.oob, "intra-chromosomal")
        return self.work


def impute_inter(pairs: PairColumns, res: int, start_m, start_p, own_is_p: bool, un: DenseBatch, imp: DenseBatch,
                 half_width: int, nb_i, nb_j, imin: int, ratio: float, stale_state=0, stale_sum=0,
                 last_qualifying=None, stale_needed=None):
    """Inter-chromosomal imputation of the one-sided lines of an M_M / P_P bed on the genome-wide
    haplotype matrix (``hc_impute_inter``; matrixBuilding.py:1302-1378, :1416-1492)."""
    assert len(un) == 1 and len(imp) == 1 and un.sizes[0] == imp.sizes[0] and un.lds[0] == imp.lds[0]
    check(lib().hc_impute_inter(ptr(pairs.c1), ptr(pairs.p1), ptr(pairs.c2), ptr(pairs.p2), ptr(pairs.mark), pairs.n,
                                int(res), ptr(start_m), ptr(start_p), int(start_m.numel()), int(bool(own_is_p)),
                                ptr(un.buf), ptr(imp.buf), un.sizes[0], un.lds[0], int(half_width), ptr(nb_i), ptr(nb_j),
                                int(nb_i.numel()), int(imin), float(ratio), int(stale_state), int(stale_sum),
                                ptr(last_qualifying), ptr(stale_needed), stream_ptr()), "hc_impute_inter")


def bin_pairs_whole(pairs: PairColumns, res: int, start1, start2, whole: DenseBatch,
                    mode=_abi.HC_BIN_SYM_ALL, check_bounds=True):
    """Accumulate pairs into the single genome-wide matrix ``whole`` (a 1-matrix batch) with
    per-side chromosome start tables (device int64).  matrixBuilding.py:582-592."""
    assert len(whole) == 1
    oob = _oob_counter(whole.device)
    check(lib().hc_bin_pairs_whole(ptr(pairs.c1), ptr(pairs.p1), ptr(pairs.c2), ptr(pairs.p2),
                                   ptr(pairs.mark), pairs.n, int(res), int(mode), ptr(start1),
                                   ptr(start2), int(start1.numel()), ptr(whole.buf), whole.sizes[0],
                                   whole.lds[0], ptr(oob), stream_ptr()), "hc_bin_pairs_whole")
    if check_bounds:
        _raise_oob(oob, "genome-wide")


def dense_nonzero_records(base_ptr: int, ld: int, nrows: int, ncols: int, triu: bool, is_f64: bool,
                          device) -> np.ndarray:
    """np.triu/np.nonzero marshalling (matrixBuilding.py:489-503, :515-521) on the device;
    returns the reference's structured array (bin1, bin2, IF) in row-major order."""
    row_ptr = torch.empty(nrows + 1, dtype=torch.int64, device=device)
    check(lib().hc_dense_nonzero_count(C.c_void_p(base_ptr), ld, nrows, ncols, int(triu), int(is_f64),
                                       ptr(row_ptr), stream_ptr()), "hc_dense_nonzero_count")
    nnz = int(row_ptr[-1].item())
    rec = np.zeros(nnz, dtype=S_DTYPE)
    if nnz == 0:
        return rec
    b1 = torch.empty(nnz, dtype=torch.int32, device=device)
    b2 = torch.empty(nnz, dtype=torch.int32, device=device)
    val = torch.empty(nnz, dtype=torch.float64 if is_f64 else torch.int32, device=device)
    check(lib().hc_dense_nonzero_extract(C.c_void_p(base_ptr), ld, nrows, ncols, int(triu), int(is_f64),
                                         ptr(row_ptr), ptr(b1), ptr(b2), ptr(val), stream_ptr()),
          "hc_dense_nonzero_extract")
    rec["bin1"], rec["bin2"], rec["IF"] = b1.cpu().numpy(), b2.cpu().numpy(), val.cpu().numpy()
    return rec


class PinnedPool:
    """Grow-only pinned host buffer + device staging buffer reused across calls (pinned
    allocation is far too slow to repeat per call)."""

    def __init__(self):
        self.host = None
        self.dev = None

    def get(self, nbytes: int, device):
        if self.host is None or self.host.numel() < nbytes:
            cap = int(nbytes * 1.25) + 4096
            self.host = torch.empty(cap, dtype=torch.uint8).pin_memory()
            self.dev = torch.empty(cap, dtype=torch.uint8, device=device)
        return self.host, self.dev


_RECORD_POOL = PinnedPool()


def dense_batch_triu_records(batch: DenseBatch, pool: PinnedPool = None, sync=True):
    """Upper-triangular records of EVERY matrix of the batch in the reference's structured
    layout (matrixBuilding.py:508-524), produced on the device and copied to the host once.
    Returns (list of S_DTYPE arrays, one per matrix, that are views of one pinned buffer --
    valid until the next call with the same pool --, bytes copied)."""
    pool = _RECORD_POOL if pool is None else pool
    dev, n = batch.device, batch.nbins
    row_ptr = torch.empty(n + 1, dtype=torch.int64, device=dev)
    check(lib().hc_dense_batch_triu_count(ptr(batch.buf), ptr(batch.mat_off), ptr(batch.mat_n), ptr(batch.mat_ld),
                                          ptr(batch.bin_off), len(batch), n, ptr(row_ptr), stream_ptr()),
          "hc_dense_batch_triu_count")
    bounds = row_ptr[batch.bin_off].cpu().numpy()          # one small D2H: record range per matrix
    total = int(bounds[-1])
    host, dbuf = pool.get(24 * max(total, 1), dev)
    if total:
        check(lib().hc_dense_batch_triu_records(ptr(batch.buf), ptr(batch.mat_off), ptr(batch.mat_n),
                                                ptr(batch.mat_ld), ptr(batch.bin_off), len(batch), n, ptr(row_ptr),
                                                ptr(dbuf), stream_ptr()), "hc_dense_batch_triu_records")
        host[:24 * total].copy_(dbuf[:24 * total], non_blocking=True)
        if sync:                                  # sync=False: the caller synchronises the stream it issued this on
            torch.cuda.current_stream().synchronize()
    rec = host[:24 * total].numpy().view(S_DTYPE)
    return [rec[int(bounds[i]):int(bounds[i + 1])] for i in range(len(batch))], 24 * total


# --------------------------------------------------------------------------------------
# (b) ICE
# --------------------------------------------------------------------------------------
def ice_params(ignore_diags=1, mad_max=5, min_nnz=10, min_count=0, tol=1e-5, max_iters=200,
               rescale_marginals=True, poll_every=8) -> IceParams:
    return IceParams(float(tol), float(mad_max), int(min_nnz), int(min_count), int(ignore_diags),
                     int(max_iters), int(bool(rescale_marginals)), int(poll_every))


def ice_dense_filters(batch: DenseBatch, params: IceParams, chrom_off=None):
    """Pre-iteration bin filters of ``cooler balance`` -> initial bias (device float64)."""
    dev, n = batch.device, batch.nbins
    nnz_marg = torch.empty(n, dtype=torch.float64, device=dev)
    marg = torch.empty(n, dtype=torch.float64, device=dev)
    check(lib().hc_ice_dense_marginals(ptr(batch.buf), ptr(batch.mat_off), ptr(batch.mat_n),
                                       ptr(batch.mat_ld), ptr(batch.bin_off), len(batch),
                                       params.ignore_diags, ptr(nnz_marg), ptr(marg), stream_ptr()),
          "hc_ice_dense_marginals")
    if chrom_off is None:
        chrom_off = batch.bin_off
    bias = torch.empty(n, dtype=torch.float64, device=dev)
    work = torch.empty(2 * max(n, 1), dtype=torch.float64, device=dev)
    check(lib().hc_ice_filter_bins(ptr(nnz_marg), ptr(marg), n, ptr(chrom_off), int(chrom_off.numel()) - 1,
                                   C.byref(params), ptr(bias), ptr(work), stream_ptr()),
          "hc_ice_filter_bins")
    return bias


def ice_dense_iterate(batch: DenseBatch, bias, params: IceParams):
    """Run every problem of the batch to convergence on the device; ``bias`` is updated in
    place to the final weights.  Returns (results ndarray of IceResult fields, IceRunInfo)."""
    dev, n = batch.device, batch.nbins
    res = torch.zeros(len(batch) * C.sizeof(IceResult), dtype=torch.uint8, device=dev)
    info = IceRunInfo(0, 0.0)
    check(lib().hc_ice_dense_balance(ptr(batch.buf), ptr(batch.mat_off), ptr(batch.mat_n),
                                     ptr(batch.mat_ld), ptr(batch.bin_off), len(batch), batch.h_mat_n,
                                     C.byref(params), ptr(bias), ptr(res), C.byref(info),
                                     stream_ptr()), "hc_ice_dense_balance")
    rdt = np.dtype([("scale", "<f8"), ("var", "<f8"), ("iters", "<i4"), ("converged", "<i4")])
    return res.cpu().numpy().view(rdt), info


def ice_balance_dense(batch: DenseBatch, chrom_off=None, **kw):
    """``cooler balance --ignore-diags K --cis-only`` for a batch of intra-chromosomal
    matrices (one independent problem per matrix), or genome-wide balancing for a 1-matrix
    batch with ``chrom_off`` giving the chromosome boundaries used by the MAD-max filter.
    Returns (weights float64 ndarray over the concatenated bins, stats dict)."""
    params = ice_params(**kw)
    bias = ice_dense_filters(batch, params, chrom_off)
    results, info = ice_dense_iterate(batch, bias, params)
    w = bias.cpu().numpy()
    cis = len(batch) > 1 or chrom_off is None
    stats = dict(tol=params.tol, min_nnz=params.min_nnz, min_count=params.min_count,
                 mad_max=params.mad_max, cis_only=cis, ignore_diags=params.ignore_diags,
                 divisive_weights=False, launches=int(info.launches), loop_ms=float(info.loop_ms))
    if len(batch) == 1 and chrom_off is not None:
        stats.update(scale=float(results["scale"][0]), var=float(results["var"][0]),
                     converged=bool(results["converged"][0]), iters=int(results["iters"][0]))
    else:
        stats.update(scale=results["scale"].copy(), var=float(results["var"][-1]),
                     converged=bool(results["var"][-1] < params.tol),
                     iters=[int(i) for i in results["iters"]],
                     converged_per_chrom=[bool(c) for c in results["converged"]])
    return w, stats


# --------------------------------------------------------------------------------------
# (c) two-step allelic correction
# --------------------------------------------------------------------------------------
def rowstats(base_ptr: int, ld: int, nrows: int, ncols: int, device, want_nnz=True):
    rs = torch.empty(nrows, dtype=torch.int64, device=device)
    nz = torch.empty(nrows, dtype=torch.int32, device=device) if want_nnz else None
    check(lib().hc_rowstats_i32(C.c_void_p(base_ptr), ld, nrows, ncols, ptr(rs), ptr(nz), stream_ptr()),
          "hc_rowstats_i32")
    return rs, nz


def twostep_alpha(rs_t, rs_m, rs_p, nnz_a, nnz_b, n, ncols, gap_mode, device):
    alpha = torch.empty(n, dtype=torch.float64, device=device)
    gf_a = torch.empty(n, dtype=torch.uint8, device=device)
    gi_a = torch.empty(n, dtype=torch.int32, device=device)
    gf_b = torch.empty(n, dtype=torch.uint8, device=device) if nnz_b is not None else None
    gi_b = torch.empty(n, dtype=torch.int32, device=device) if nnz_b is not None else None
    ngap = torch.zeros(2, dtype=torch.int32, device=device)
    work = torch.empty(2 * n, dtype=torch.float64, device=device)
    check(lib().hc_twostep_alpha(ptr(rs_t), ptr(rs_m), ptr(rs_p), ptr(nnz_a), ptr(nnz_b), n, ncols,
                                 gap_mode, ptr(alpha), ptr(gf_a), ptr(gf_b), ptr(gi_a), ptr(gi_b),
                                 ptr(ngap), ptr(work), stream_ptr()), "hc_twostep_alpha")
    return alpha, (gf_a, gi_a), (gf_b, gi_b), ngap


def twostep_correct(x_ptr: int, ld: int, n: int, alpha, gapflag, has_gap: bool, rowsum_x, device,
                    out=None):
    """X/alpha -> Trans2symmetry -> Correct_VC(2/3) -> rescale, fused; returns an (n, n)
    float64 device tensor."""
    if out is None:
        out = torch.empty((n, n), dtype=torch.float64, device=device)
    work = torch.empty(int(lib().hc_twostep_work_bytes(n)), dtype=torch.uint8, device=device)
    check(lib().hc_twostep_correct(C.c_void_p(x_ptr), ld, n, ptr(alpha), ptr(gapflag), int(has_gap),
                                   ptr(rowsum_x), ptr(out), out.stride(0), ptr(work), stream_ptr()),
          "hc_twostep_correct")
    return out


# --------------------------------------------------------------------------------------
# (a') sort path: pairs -> keys -> radix sort -> reduce-by-key -> symmetric CSR
# --------------------------------------------------------------------------------------
def sort_keys_u64(keys, nbits: int, tmp=None):
    """Ascending radix sort of a uint64 device tensor (viewed as int64 by torch) on its low
    ``nbits`` bits.  Returns the sorted tensor (one of ``keys`` / ``tmp``)."""
    n = int(keys.numel())
    if tmp is None:
        tmp = torch.empty_like(keys)
    work = torch.empty(int(lib().hc_sort_work_bytes(n)), dtype=torch.uint8, device=keys.device)
    in_tmp = C.c_int32(0)
    check(lib().hc_sort_keys_u64(ptr(keys), ptr(tmp), n, 0, int(nbits), ptr(work), C.byref(in_tmp), stream_ptr()),
          "hc_sort_keys_u64")
    return (tmp, keys) if in_tmp.value else (keys, tmp)


class SymCsr:
    """Symmetric CSR of one contact matrix over ``nbins`` concatenated bins (both triangles
    stored); ``row0`` / ``nloc`` describe the row block held locally (all rows on one GPU)."""

    def __init__(self, row_ptr, col, cnt, nbins, row0=0):
        self.row_ptr, self.col, self.cnt = row_ptr, col, cnt
        self.nbins, self.row0 = int(nbins), int(row0)
        self.nloc = int(row_ptr.numel()) - 1
        self.nnz = int(col.numel())
        self.device = col.device


def keys_to_csr(sorted_keys, n_valid, col_bits: int, nrows: int, scratch=None, row0: int = 0):
    """Reduce-by-key over sorted keys -> (row_ptr int64[nrows+1], col int32, cnt int32)."""
    dev, nkeys = sorted_keys.device, int(sorted_keys.numel())
    work = torch.empty(int(lib().hc_csr_work_bytes(nkeys)), dtype=torch.uint8, device=dev)
    nnz = C.c_int64(0)
    check(lib().hc_csr_count(ptr(sorted_keys), nkeys, ptr(n_valid), ptr(work), C.byref(nnz), stream_ptr()),
          "hc_csr_count")
    nnz = int(nnz.value)
    row_ptr = torch.empty(nrows + 1, dtype=torch.int64, device=dev)
    col = torch.empty(nnz, dtype=torch.int32, device=dev)
    cnt = torch.empty(nnz, dtype=torch.int32, device=dev)
    ukey = scratch if (scratch is not None and scratch.numel() >= nnz) else torch.empty(max(nnz, 1), dtype=torch.int64, device=dev)
    upos = torch.empty(max(nnz, 1), dtype=torch.int64, device=dev)
    check(lib().hc_csr_emit(ptr(sorted_keys), nkeys, ptr(n_valid), ptr(work), nnz, int(col_bits), int(row0), int(nrows),
                            ptr(ukey), ptr(upos), ptr(row_ptr), ptr(col), ptr(cnt), stream_ptr()), "hc_csr_emit")
    return row_ptr, col, cnt


def key_col_bits(nbins: int) -> int:
    return max(1, int(nbins - 1).bit_length())


def key_sort_bits(nbins: int) -> int:
    """Bits the radix sort must look at so that the padding key ~0 sorts strictly after every real
    key: 2*col_bits, plus one when nbins is a power of two -- the key of the last diagonal cell
    (nbins-1, nbins-1) is then all ones in the low 2*col_bits bits and would tie with the padding."""
    cb = key_col_bits(nbins)
    return 2 * cb + (1 if int(nbins) == (1 << cb) else 0)


def pairs_to_sorted_keys(pairs: PairColumns, res: int, start, chrom_bins, nbins: int, cis_only: bool,
                         check_bounds=True):
    """pairs -> (row << col_bits | col) keys, both orientations, radix-sorted; padding keys
    (dropped pairs) sort last.  Returns (sorted_keys, free_buffer, n_valid device scalar)."""
    dev = pairs.device
    col_bits = key_col_bits(nbins)
    keys = torch.empty(2 * max(pairs.n, 1), dtype=torch.int64, device=dev)
    n_valid = torch.zeros(1, dtype=torch.int64, device=dev)
    oob = torch.zeros(1, dtype=torch.int64, device=dev)
    check(lib().hc_pairs_to_keys(ptr(pairs.c1), ptr(pairs.p1), ptr(pairs.c2), ptr(pairs.p2), pairs.n, int(res),
                                 ptr(start), ptr(chrom_bins), int(start.numel()), int(bool(cis_only)), col_bits,
                                 ptr(keys), ptr(n_valid), ptr(oob), stream_ptr()), "hc_pairs_to_keys")
    if check_bounds:
        _raise_oob(oob, "genome-wide")
    keys = keys[:2 * pairs.n]
    skeys, free = sort_keys_u64(keys, key_sort_bits(nbins)) if pairs.n else (keys, None)
    return skeys, free, n_valid


def entry_cnt_bits(nbins: int) -> int:
    """Width of the count field of a 64-bit entry (row | col | count): what two column fields and the
    padding bit leave, at most 31 (counts are int32 in the CSR)."""
    room = min(31, 63 - 2 * key_col_bits(nbins))
    return min(room, int(os.environ.get("HC_ENTRY_CNT_BITS", room)))       # the variable is a test hook


def sort_entries(ent, nbins: int, begin_bit: int, nfields: int, tmp=None):
    """Stable radix sort of entries on ``nfields`` bin fields starting at ``begin_bit`` (plus the bit above them
    when nbins is a power of two, so that the padding key ~0 sorts strictly last)."""
    cb = key_col_bits(nbins)
    end_bit = begin_bit + nfields * cb + (1 if int(nbins) == (1 << cb) else 0)
    n = int(ent.numel())
    if n <= 1:
        return ent, tmp
    if tmp is None:
        tmp = torch.empty_like(ent)
    work = torch.empty(int(lib().hc_sort_work_bytes(n)), dtype=torch.uint8, device=ent.device)
    in_tmp = C.c_int32(0)
    check(lib().hc_sort_keys_u64(ptr(ent), ptr(tmp), n, int(begin_bit), int(end_bit), ptr(work), C.byref(in_tmp),
                                 stream_ptr()), "hc_sort_keys_u64")
    return (tmp, ent) if in_tmp.value else (ent, tmp)


class CountFieldOverflow(OverflowError):
    """A cell count does not fit the count field of the 64-bit entries."""


def reduce_entries(sorted_ent, n_valid, nbins: int, unit: bool, lower_into=None, want_lower=False):
    """Reduce-by-cell over sorted entries.  Returns the reduced entries [nuniq] (a fresh tensor) -- and, with
    ``want_lower``, also (lo [nuniq], n_lo device scalar): the same cells with row and col swapped (padding key for the
    diagonal ones), written by the same pass into ``lower_into`` when that tensor is large enough."""
    dev, n = sorted_ent.device, int(sorted_ent.numel())
    cb, cnt_bits = key_col_bits(nbins), entry_cnt_bits(nbins)
    work = torch.empty(int(lib().hc_csr_work_bytes(n)), dtype=torch.uint8, device=dev)
    nuniq = C.c_int64(0)
    check(lib().hc_entries_count(ptr(sorted_ent), n, ptr(n_valid), cnt_bits, ptr(work), C.byref(nuniq), stream_ptr()),
          "hc_entries_count")
    nuniq = int(nuniq.value)
    out = torch.empty(nuniq, dtype=torch.int64, device=dev)
    lo = n_lo = None
    if want_lower:
        lo = lower_into[:nuniq] if (lower_into is not None and lower_into.numel() >= nuniq) else \
            torch.empty(nuniq, dtype=torch.int64, device=dev)
        n_lo = torch.zeros(1, dtype=torch.int64, device=dev)
    d_ovf = torch.zeros(1, dtype=torch.int32, device=dev)
    h_ovf = C.c_int32(0)
    check(lib().hc_entries_emit(ptr(sorted_ent), n, ptr(n_valid), ptr(work), nuniq, cb, cnt_bits, int(bool(unit)), ptr(out),
                                ptr(lo), ptr(n_lo), ptr(d_ovf), C.byref(h_ovf), stream_ptr()), "hc_entries_emit")
    if h_ovf.value:
        raise CountFieldOverflow("a cell holds more than 2^%d - 1 pairs" % cnt_bits)
    return (out, lo, n_lo) if want_lower else out


def pairs_to_entry_lists(pairs: PairColumns, res: int, start, chrom_bins, nbins: int, cis_only: bool,
                         check_bounds=True):
    """pairs -> one entry per pair (its upper-triangle cell) -> sorted -> reduced; the lower-triangle list (swapped
    cells) comes out of the same reduction pass and is re-sorted on its row bits.  Returns (up [nuniq] ordered by
    (row, col), lo_sorted [nuniq] ordered by (row, col) with the padding keys of the diagonal cells behind the first
    n_lo entries, n_lo device scalar)."""
    dev = pairs.device
    cb, cnt_bits = key_col_bits(nbins), entry_cnt_bits(nbins)
    ent = torch.empty(max(pairs.n, 1), dtype=torch.int64, device=dev)
    n_valid = torch.zeros(1, dtype=torch.int64, device=dev)
    oob = torch.zeros(1, dtype=torch.int64, device=dev)
    check(lib().hc_pairs_to_entries(ptr(pairs.c1), ptr(pairs.p1), ptr(pairs.c2), ptr(pairs.p2), pairs.n, int(res),
                                    ptr(start), ptr(chrom_bins), int(start.numel()), int(bool(cis_only)), cb, cnt_bits,
                                    ptr(ent), ptr(n_valid), ptr(oob), stream_ptr()), "hc_pairs_to_entries")
    if check_bounds:
        _raise_oob(oob, "genome-wide")
    ent = ent[:pairs.n]
    sent, free = sort_entries(ent, nbins, cnt_bits, 2)
    # the lower list goes into the free half of the ping-pong pair; the sorted pair entries are dead after the reduction
    # and serve as the ping-pong partner of the lower list's sort
    up, lo, n_lo = reduce_entries(sent, n_valid, nbins, unit=True, lower_into=free, want_lower=True)
    nuniq = int(up.numel())
    slo, _ = sort_entries(lo, nbins, cnt_bits + cb, 1, tmp=sent[:nuniq] if sent.numel() >= nuniq else None)
    return up, slo, n_lo


def entries_to_csr(up, lo, n_lo, nbins: int, nrows: int, row0: int = 0, total=None):
    """Symmetric CSR tensors (row_ptr, col, cnt) from the upper list and (optionally) the sorted lower list."""
    dev = up.device
    cb, cnt_bits = key_col_bits(nbins), entry_cnt_bits(nbins)
    n_up = int(up.numel())
    if total is None:
        total = n_up + (int(n_lo.item()) if lo is not None else 0)
    row_ptr = torch.empty(nrows + 1, dtype=torch.int64, device=dev)
    col = torch.empty(total, dtype=torch.int32, device=dev)
    cnt = torch.empty(total, dtype=torch.int32, device=dev)
    work = torch.empty(int(lib().hc_entries_csr_work_bytes(nrows)), dtype=torch.uint8, device=dev)
    check(lib().hc_entries_to_csr(ptr(up), n_up, ptr(lo) if lo is not None else None, ptr(n_lo) if lo is not None else None,
                                  cb, cnt_bits, int(row0), int(nrows), ptr(work), ptr(row_ptr), ptr(col), ptr(cnt),
                                  stream_ptr()), "hc_entries_to_csr")
    return row_ptr, col, cnt


def _pairs_to_csr_two_keys(pairs: PairColumns, res: int, start, chrom_bins, nbins: int, cis_only: bool,
                           check_bounds=True) -> SymCsr:
    """The first version of the sort path: two keys per off-diagonal pair, five digit passes over all of them.
    Kept as the fallback for counts that overflow the entry count field."""
    skeys, free, n_valid = pairs_to_sorted_keys(pairs, res, start, chrom_bins, nbins, cis_only, check_bounds)
    row_ptr, col, cnt = keys_to_csr(skeys, n_valid, key_col_bits(nbins), nbins, scratch=free)
    return SymCsr(row_ptr, col, cnt, nbins)


def pairs_to_csr(pairs: PairColumns, res: int, start, chrom_bins, nbins: int, cis_only: bool,
                 check_bounds=True) -> SymCsr:
    """Binning through the sort path (north_star kernel (a)): every pair becomes ONE 64-bit entry of its
    upper-triangle cell; the entries are radix-sorted and reduced by cell; the lower triangle is the swapped list
    re-sorted on its row bits only; the symmetric CSR is the row-wise concatenation of the two lists."""
    if pairs.n == 0:
        return _pairs_to_csr_two_keys(pairs, res, start, chrom_bins, nbins, cis_only, check_bounds)
    try:
        up, slo, n_lo = pairs_to_entry_lists(pairs, res, start, chrom_bins, nbins, cis_only, check_bounds)
    except CountFieldOverflow:
        return _pairs_to_csr_two_keys(pairs, res, start, chrom_bins, nbins, cis_only, check_bounds)
    row_ptr, col, cnt = entries_to_csr(up, slo, n_lo, nbins, nbins)
    return SymCsr(row_ptr, col, cnt, nbins)


class GenCsr(SymCsr):
    """General (asymmetric) CSR over ``nbins`` concatenated bins, rows column-sorted, nothing mirrored.  ``t``: its
    transpose without the diagonal (a GenCsr), when it was built."""
    t = None


def pairs_to_directed_csr(parts, res: int, chrom_bins, nbins: int, onesided: bool, transpose: bool) -> GenCsr:
    """Haplotype matrices of allelic mode through the sort path.  ``parts``: [(PairColumns of an M_M / P_P bed,
    device start table of its chromosomes in the concatenated haplotype bins)].  Both pairs count symmetrically; with
    ``onesided`` the R1 / R2 pairs are added at (b1, b2) / (b2, b1) -- the cells of ``bin_pairs_local`` with
    HC_BIN_SYM_BOTH then HC_BIN_ONESIDED.  Directed entries -> radix sort -> reduce-by-cell -> CSR; with ``transpose``
    the swapped list of the same reduction, re-sorted on its row bits, becomes ``.t``.  A cell count that does not fit
    the entry count field raises ``CountFieldOverflow``."""
    dev = chrom_bins.device
    cb, cnt_bits = key_col_bits(nbins), entry_cnt_bits(nbins)
    total = sum(p.n for p, _ in parts)
    ent = torch.empty(2 * max(total, 1), dtype=torch.int64, device=dev)
    n_valid = torch.zeros(1, dtype=torch.int64, device=dev)
    oob = torch.zeros(1, dtype=torch.int64, device=dev)
    done = 0
    for pairs, start in parts:
        check(lib().hc_pairs_to_directed_entries(ptr(pairs.c1), ptr(pairs.p1), ptr(pairs.c2), ptr(pairs.p2), ptr(pairs.mark),
                                                 pairs.n, int(res), ptr(start), ptr(chrom_bins), int(start.numel()),
                                                 int(bool(onesided)), cb, cnt_bits, C.c_void_p(ent.data_ptr() + 16 * done),
                                                 ptr(n_valid), ptr(oob), stream_ptr()), "hc_pairs_to_directed_entries")
        done += pairs.n
    _raise_oob(oob, "intra-chromosomal")
    sent, free = sort_entries(ent[:2 * total], nbins, cnt_bits, 2)
    red = reduce_entries(sent, n_valid, nbins, unit=True, lower_into=free, want_lower=transpose)
    up = red[0] if transpose else red
    X = GenCsr(*entries_to_csr(up, None, None, nbins, nbins), nbins)
    if transpose:
        _, lo, n_lo = red
        nuniq = int(up.numel())
        slo, _ = sort_entries(lo, nbins, cnt_bits + cb, 1, tmp=sent[:nuniq] if sent.numel() >= nuniq else None)
        X.t = GenCsr(*entries_to_csr(slo[:int(n_lo.item())], None, None, nbins, nbins), nbins)
    return X


def twostep_csr_batch(T: SymCsr, t_bin_off, X: GenCsr, h_bin_off):
    """``twostep_batch`` on CSR matrices (``hc_twostep_csr_batch``): ``T`` the symmetric CSR of the nchrom traditional
    matrices over their concatenated bins (host offsets ``t_bin_off``), ``X`` the imputed haplotype matrices (all
    maternal, then all paternal; host offsets ``h_bin_off``) with its transpose in ``X.t``.  Returns (list of 2*nchrom
    S_DTYPE arrays: the upper-triangle records of every corrected matrix in chromosome-local bins, row-major -- what
    ``IntraMatrixToSparseDict`` takes from the dense corrected matrix --, list of 2*nchrom host gap-index arrays)."""
    nchrom = len(t_bin_off) - 1
    dev = T.device
    t_off = torch.from_numpy(np.ascontiguousarray(t_bin_off, dtype=np.int64)).to(dev)
    h_off = torch.from_numpy(np.ascontiguousarray(h_bin_off, dtype=np.int64)).to(dev)
    alpha = torch.empty(max(T.nbins, 1), dtype=torch.float64, device=dev)
    gapflag = torch.empty(max(X.nbins, 1), dtype=torch.uint8, device=dev)
    gapidx = torch.empty(max(X.nbins, 1), dtype=torch.int32, device=dev)
    ngap = torch.zeros(2 * nchrom, dtype=torch.int32, device=dev)
    rec_ptr = torch.empty(X.nbins + 1, dtype=torch.int64, device=dev)
    recs = torch.empty(24 * max(X.nnz + X.t.nnz, 1), dtype=torch.uint8, device=dev)   # the union has at most this many cells
    work = torch.empty(int(lib().hc_twostep_csr_batch_work_bytes(T.nbins, X.nbins, nchrom)), dtype=torch.uint8, device=dev)
    nrec = C.c_int64(0)
    check(lib().hc_twostep_csr_batch(ptr(T.row_ptr), ptr(T.cnt), ptr(X.row_ptr), ptr(X.col), ptr(X.cnt), ptr(X.t.row_ptr),
                                     ptr(X.t.col), ptr(X.t.cnt), ptr(t_off), ptr(h_off), nchrom, T.nbins, X.nbins, ptr(alpha),
                                     ptr(gapflag), ptr(gapidx), ptr(ngap), ptr(rec_ptr), ptr(recs), C.byref(nrec), ptr(work),
                                     stream_ptr()), "hc_twostep_csr_batch")
    bounds = rec_ptr[h_off].cpu().numpy()
    rec = recs[:24 * int(nrec.value)].cpu().numpy().view(S_DTYPE)
    ng, gi = ngap.cpu().numpy(), gapidx.cpu().numpy()
    recs_out, gaps = [], []
    for k in range(2 * nchrom):
        recs_out.append(rec[int(bounds[k]):int(bounds[k + 1])])
        c, hap = k % nchrom, k // nchrom
        cnt = int(ng[2 * c + hap])
        lo = int(h_bin_off[k])
        gaps.append(gi[lo:lo + cnt].astype(np.int64) if cnt else np.array([]))
    return recs_out, gaps


def csr_upper_records(csr: SymCsr):
    """Upper-triangular (bin1, bin2, count) int32 device tensors of the local rows, row-major
    (global bin indices)."""
    dev = csr.device
    out_ptr = torch.empty(csr.nloc + 1, dtype=torch.int64, device=dev)
    check(lib().hc_csr_upper_count(ptr(csr.row_ptr), ptr(csr.col), csr.row0, csr.nloc, ptr(out_ptr), stream_ptr()),
          "hc_csr_upper_count")
    n = int(out_ptr[-1].item())
    b1 = torch.empty(n, dtype=torch.int32, device=dev)
    b2 = torch.empty(n, dtype=torch.int32, device=dev)
    v = torch.empty(n, dtype=torch.int32, device=dev)
    if n:
        check(lib().hc_csr_upper_emit(ptr(csr.row_ptr), ptr(csr.col), ptr(csr.cnt), csr.row0, csr.nloc, ptr(out_ptr),
                                      ptr(b1), ptr(b2), ptr(v), stream_ptr()), "hc_csr_upper_emit")
    return b1, b2, v


def ice_balance_csr(csr: SymCsr, prob_off, chrom_off=None, comm=None, allreduce=None, **kw):
    """ICE on the symmetric CSR.  ``prob_off``: host int64 array of problem boundaries over the
    bins ([0, nbins] = genome-wide; per-chromosome offsets on cis-only keys = --cis-only).
    ``chrom_off``: chromosome boundaries for the MAD-max filter (defaults to prob_off).
    Row-block sharding: ``comm`` = handle from nccl_comm_init (in-loop allreduce) and
    ``allreduce`` = callable used for the two filter vectors (torch.distributed.all_reduce)."""
    params = ice_params(**kw)
    dev, n = csr.device, csr.nbins
    prob_off = np.ascontiguousarray(prob_off, dtype=np.int64)
    chrom_off = prob_off if chrom_off is None else np.ascontiguousarray(chrom_off, dtype=np.int64)
    d_prob = torch.from_numpy(prob_off).to(dev)
    d_chrom = torch.from_numpy(chrom_off).to(dev)
    nnz_marg = torch.zeros(n, dtype=torch.float64, device=dev)
    marg = torch.zeros(n, dtype=torch.float64, device=dev)
    check(lib().hc_ice_csr_marginals(ptr(csr.row_ptr), ptr(csr.col), ptr(csr.cnt), csr.row0, csr.nloc,
                                     params.ignore_diags, ptr(nnz_marg), ptr(marg), stream_ptr()),
          "hc_ice_csr_marginals")
    if allreduce is not None:
        allreduce(nnz_marg)
        allreduce(marg)
    bias = torch.empty(n, dtype=torch.float64, device=dev)
    fwork = torch.empty(2 * max(n, 1), dtype=torch.float64, device=dev)
    check(lib().hc_ice_filter_bins(ptr(nnz_marg), ptr(marg), n, ptr(d_chrom), len(chrom_off) - 1,
                                   C.byref(params), ptr(bias), ptr(fwork), stream_ptr()), "hc_ice_filter_bins")
    nprob = len(prob_off) - 1
    work = torch.empty(int(lib().hc_ice_csr_work_bytes(n, nprob)), dtype=torch.uint8, device=dev)
    res = torch.zeros(nprob * C.sizeof(IceResult), dtype=torch.uint8, device=dev)
    info = IceRunInfo(0, 0.0)
    h_off = (C.c_int64 * len(prob_off))(*[int(x) for x in prob_off])
    # the library re-encodes the CSR into stream-ordered scratch of its own (~4.3 B per stored entry + ~100 B per row and
    # column block): hand torch's cached-but-unused blocks back to the driver first when the device could not serve that
    need = int(4.3 * csr.nnz) + 16 * csr.nloc * ((n + 8191) // 8192) + (64 << 20)
    free_dev, pool_free = torch.cuda.mem_get_info(dev)[0], int(lib().hc_mempool_free_bytes())
    if os.environ.get("HC_DEBUG_MEM") == "1":
        import sys
        sys.stderr.write("[ice_balance_csr] need %.2f GB, device free %.2f GB, pool free %.2f GB, torch reserved %.2f GB\n"
                         % (need / 1e9, free_dev / 1e9, pool_free / 1e9, torch.cuda.memory_reserved(dev) / 1e9))
    if free_dev + pool_free < need:
        torch.cuda.empty_cache()
    check(lib().hc_ice_csr_balance(ptr(csr.row_ptr), ptr(csr.col), ptr(csr.cnt), csr.row0, csr.nloc, ptr(d_prob),
                                   nprob, h_off, C.byref(params), ptr(bias), ptr(work), ptr(res), C.byref(info),
                                   C.c_void_p(comm or 0), stream_ptr()), "hc_ice_csr_balance")
    rdt = np.dtype([("scale", "<f8"), ("var", "<f8"), ("iters", "<i4"), ("converged", "<i4")])
    results = res.cpu().numpy().view(rdt)
    stats = dict(tol=params.tol, min_nnz=params.min_nnz, min_count=params.min_count, mad_max=params.mad_max,
                 cis_only=nprob > 1, ignore_diags=params.ignore_diags, divisive_weights=False,
                 launches=int(info.launches), loop_ms=float(info.loop_ms), pack_ms=float(info.pack_ms),
                 stream_full_ms=float(info.stream_full_ms), stream_full_launches=int(info.stream_full_launches))
    if int(info.packed) == 2:       # column-blocked encoding (hc_ice_csrb.cu): 4-byte entries, padded segments
        stats.update(encoding="column-blocked symmetric CSR: 4 B per stored entry (13-bit column in an 8192-bin block + 19-bit "
                              "weighted count), bias block staged in shared memory by cp.async.bulk",
                     stored_entries=int(info.overflow_cells),
                     bytes_per_entry=4.0 * int(info.overflow_cells) / max(csr.nnz, 1))
    else:
        stats.update(encoding="row-major symmetric CSR: int32 column + int32 count per stored entry, bias gathered from L2",
                     stored_entries=int(csr.nnz), bytes_per_entry=8.0)
    if nprob == 1:
        stats.update(scale=float(results["scale"][0]), var=float(results["var"][0]),
                     converged=bool(results["converged"][0]), iters=int(results["iters"][0]))
    else:
        stats.update(scale=results["scale"].copy(), var=float(results["var"][-1]),
                     converged=bool(results["var"][-1] < params.tol), iters=[int(i) for i in results["iters"]],
                     converged_per_chrom=[bool(c) for c in results["converged"]])
    return bias, stats


# ---- NCCL communicator for the row-block sharded ICE -------------------------------------
def nccl_unique_id() -> bytes:
    buf = (C.c_char * 128)()
    check(lib().hc_nccl_unique_id(buf), "hc_nccl_unique_id")
    return bytes(buf)


def nccl_comm_init(uid: bytes, nranks: int, rank: int) -> int:
    comm = C.c_void_p(0)
    buf = (C.c_char * 128).from_buffer_copy(uid)
    check(lib().hc_nccl_comm_init(buf, nranks, rank, C.byref(comm)), "hc_nccl_comm_init")
    return int(comm.value)


def nccl_allreduce_f64(comm: int, t):
    """In-place sum-allreduce of a float64 device tensor on the library's communicator (current stream)."""
    check(lib().hc_nccl_allreduce_sum_f64(C.c_void_p(comm), ptr(t), int(t.numel()), stream_ptr()), "hc_nccl_allreduce_sum_f64")


def nccl_comm_destroy(comm: int):
    check(lib().hc_nccl_comm_destroy(C.c_void_p(comm)), "hc_nccl_comm_destroy")


def twostep_batch(T: DenseBatch, H: DenseBatch):
    """IntraChromMatrixCorrection (matrixBuilding.py:1026-1041) for all chromosomes in one library
    call: ``T`` holds the nchrom traditional matrices, ``H`` the 2*nchrom haplotype matrices (all
    maternal, then all paternal).  Returns (list of 2*nchrom (n, n) float64 device tensors in H's
    order, list of 2*nchrom host gap-index arrays)."""
    nchrom = len(T)
    assert len(H) == 2 * nchrom and H.sizes[:nchrom] == T.sizes and H.sizes[nchrom:] == T.sizes
    dev = T.device
    sizes = T.sizes
    out_off = np.concatenate([[0], np.cumsum([n * n for n in H.sizes])]).astype(np.int64)
    out = torch.empty(int(out_off[-1]), dtype=torch.float64, device=dev)
    alpha = torch.empty(max(T.nbins, 1), dtype=torch.float64, device=dev)
    gapflag = torch.empty(max(H.nbins, 1), dtype=torch.uint8, device=dev)
    gapidx = torch.empty(max(H.nbins, 1), dtype=torch.int32, device=dev)
    ngap = torch.zeros(2 * nchrom, dtype=torch.int32, device=dev)
    work = torch.empty(int(lib().hc_twostep_batch_work_bytes(T.nbins, H.nbins, max(sizes) if sizes else 0)),
                       dtype=torch.uint8, device=dev)
    i32 = lambda xs: (C.c_int32 * len(xs))(*[int(x) for x in xs])
    i64 = lambda xs: (C.c_int64 * len(xs))(*[int(x) for x in xs])
    check(lib().hc_twostep_batch(ptr(T.buf), ptr(T.mat_off), ptr(T.mat_n), ptr(T.mat_ld), ptr(T.bin_off),
                                 ptr(H.buf), ptr(H.mat_off), ptr(H.mat_n), ptr(H.mat_ld), ptr(H.bin_off), nchrom,
                                 i32(sizes), i64(H.offsets), i32(H.lds), i64(T.h_bin_off), i64(H.h_bin_off), ptr(out),
                                 i64(out_off), ptr(alpha), ptr(gapflag), ptr(gapidx), ptr(ngap), ptr(work), stream_ptr()),
          "hc_twostep_batch")
    ng = ngap.cpu().numpy()                       # the only host round trip of the whole batch
    gi = gapidx.cpu().numpy()
    mats, gaps = [], []
    for k in range(2 * nchrom):
        n = H.sizes[k]
        mats.append(out[int(out_off[k]):int(out_off[k + 1])].view(n, n))
        c, hap = k % nchrom, k // nchrom
        cnt = int(ng[2 * c + hap])
        lo = int(H.h_bin_off[k])
        gaps.append(gi[lo:lo + cnt].astype(np.int64) if cnt else np.array([]))
    return mats, gaps
