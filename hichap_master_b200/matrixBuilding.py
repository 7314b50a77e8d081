"""B200 drop-in for the numeric functions of ``HiCHap/matrixBuilding.py`` (the ``matrix`` stage).

Same callables, argument order and return layouts as the reference; the arithmetic runs in
hand-written sm_100a kernels behind the C ABI (``include/hichap_b200.h``).  Citations are
``file:line`` in the reference tree.

Besides the reference's NumPy-in / NumPy-out signatures, every heavy function accepts the
device-resident objects of ``device.py`` so a pipeline can keep matrices in HBM between the
binning, ICE and correction kernels (``bin_traditional`` -> ``ice_balance_dense`` ->
``two_step_device``).
"""
from __future__ import annotations

import logging

import numpy as np
import torch

from . import _abi, kernels
from .device import DenseBatch, PairColumns, as_int32_counts, require_cuda
from .pairs import chrom_passes, read_pairs

log = logging.getLogger(__name__)

S_dtype = kernels.S_DTYPE


# ======================================================================================
# genome / bin tables (host; matrixBuilding.py:349-454)
# ======================================================================================
def Load_Genome(genomeSize, chroms):
    """matrixBuilding.py:349-366 -- ``{chrom: length}`` for chromosomes passing the filter.
    ``lstrip('chr')`` strips the character set {c,h,r}, exactly as the reference does."""
    genome = {}
    with open(genomeSize, "r") as fh:
        for line in fh:
            parts = line.strip().split()
            c = parts[0].lstrip("chr")
            if chrom_passes(c, chroms):
                genome[c] = int(parts[1])
    return genome


def Load_HaplotypeGenome(genomeSize, chroms):
    """matrixBuilding.py:369-386."""
    genome = {}
    for c, l in Load_Genome(genomeSize, chroms).items():
        genome["M" + c] = l
        genome["P" + c] = l
    return genome


def Sort_Chromosomes(chro_lst):
    """matrixBuilding.py:388-406 -- numeric labels ascending, then the others sorted."""
    num, other = [], []
    for name in chro_lst:
        name = name.lstrip("chr")
        try:
            num.append(int(name))
        except ValueError:
            other.append(name)
    return [str(v) for v in sorted(num)] + sorted(other)


def _bins_from_genome(genome, Resolution, order):
    table, nxt = {}, 0
    for key, c in order:
        span = genome[c] // Resolution
        table[key] = (nxt, nxt + span)      # inclusive end, matrixBuilding.py:420-422
        nxt += span + 1
    return table, nxt


def Get_Chro_Bins(genomeSize, Resolution, chroms):
    """matrixBuilding.py:409-426 -- ({chrom: (start, end_inclusive)}, total bins)."""
    genome = Load_Genome(genomeSize, chroms)
    return _bins_from_genome(genome, Resolution, [(c, c) for c in Sort_Chromosomes(genome)])


def Get_Chro_Bins_Haplotypes(genomeSize, Resolution, chroms):
    """matrixBuilding.py:429-454 -- maternal chromosomes first, then paternal."""
    genome = Load_Genome(genomeSize, chroms)
    order = Sort_Chromosomes(genome)
    return _bins_from_genome(genome, Resolution,
                             [("M" + c, c) for c in order] + [("P" + c, c) for c in order])


# ======================================================================================
# (a) binning
# ======================================================================================
def _start_table(bins, keys, device):
    return torch.tensor([bins[k][0] for k in keys], dtype=torch.int64, device=device)


def _to_pair_columns(bed_IO, order, chroms, layout, device):
    if isinstance(bed_IO, PairColumns):
        return bed_IO
    c1, p1, c2, p2, mark = read_pairs(bed_IO, order, chroms, layout)
    return PairColumns(c1, p1, c2, p2, mark, device)


def dense_budget_bytes(device=None) -> int:
    """Largest dense int32 tile set the binning may allocate before it switches to the sort path (symmetric
    CSR).  The reference always allocates ``np.zeros((Sum, Sum))`` (matrixBuilding.py:559), which at 10 kb
    genome-wide is 369 GB.  ``HC_DENSE_BUDGET_GB`` overrides; default: a third of the device memory."""
    import os
    env = os.environ.get("HC_DENSE_BUDGET_GB")
    if env is not None:
        return int(float(env) * 1e9)
    dev = require_cuda(device)
    return int(torch.cuda.get_device_properties(dev).total_memory // 3)


def _dense_bytes(sizes) -> int:
    return int(sum(4 * n * max(128, (n + 127) // 128 * 128) for n in sizes))


def _check_fits(nbytes, dev, what):
    free, _ = torch.cuda.mem_get_info(dev)
    if nbytes > free:
        raise MemoryError("the dense %s matrices need %.1f GB of device memory (%.1f GB free); this entry point returns "
                          "dense matrices like the reference -- use the sparse path (bin_traditional_sparse / "
                          "TraditionalMatrixBuilding) for this resolution" % (what, nbytes / 1e9, free / 1e9))


class CisCsr:
    """All intra-chromosomal matrices of one resolution as ONE CSR over the concatenated bins (keys built cis-only):
    the sparse counterpart of the per-chromosome ``DenseBatch``.  Symmetric for the traditional and un-imputed
    matrices; the imputed haplotype matrices are a general ``kernels.GenCsr``.  ``order`` names the matrices in bin
    order (chromosomes, or M chromosomes then P chromosomes)."""

    def __init__(self, csr, bins, order):
        self.csr, self.bins, self.order = csr, bins, list(order)
        self.off = np.array([bins[c][0] for c in self.order] + [bins[self.order[-1]][1] + 1], dtype=np.int64)

    def matrices(self):
        """{chrom: scipy.sparse.csr_matrix (int64 counts)}: the per-chromosome blocks of the CSR"""
        import scipy.sparse as sp
        c = self.csr
        full = sp.csr_matrix((c.cnt.cpu().numpy().astype(np.int64), c.col.cpu().numpy(), c.row_ptr.cpu().numpy()),
                             shape=(c.nbins, c.nbins))
        return {name: full[a:b, a:b] for name, a, b in zip(self.order, self.off[:-1], self.off[1:])}

    def records(self):
        """{chrom: upper-triangular S_dtype records in chromosome-local coordinates} (matrixBuilding.py:508-524)"""
        b1, b2, v = (t.cpu().numpy() for t in kernels.csr_upper_records(self.csr))
        cut = np.searchsorted(b1, self.off)
        out = {}
        for i, c in enumerate(self.order):
            lo, hi = int(cut[i]), int(cut[i + 1])
            rec = np.zeros(hi - lo, dtype=S_dtype)
            rec["bin1"], rec["bin2"], rec["IF"] = b1[lo:hi].astype(np.int64) - self.off[i], b2[lo:hi].astype(np.int64) - self.off[i], v[lo:hi]
            out[c] = rec
        return out


def bin_traditional(pairs: PairColumns, genome: dict, wholeRes, localRes, device=None, budget=None):
    """Device-resident binning: returns ({res: (bins, DenseBatch[1] | SymCsr)}, {res: DenseBatch[nchrom] | CisCsr})
    with chromosomes in ``Sort_Chromosomes`` order.  matrixBuilding.py:553-603.  Matrices whose dense int32 tiles
    exceed ``budget`` bytes (``dense_budget_bytes``) go through the sort path (radix sort + reduce-by-key into a
    symmetric CSR) instead of the dense accumulation."""
    dev = require_cuda(device)
    order = Sort_Chromosomes(genome)
    budget = dense_budget_bytes(dev) if budget is None else int(budget)
    whole, local = {}, {}
    for res in wholeRes:
        bins, total = _bins_from_genome(genome, res, [(c, c) for c in order])
        start = _start_table(bins, order, dev)
        if _dense_bytes([total]) > budget:
            chrom_bins = torch.tensor([genome[c] // res + 1 for c in order], dtype=torch.int32, device=dev)
            whole[res] = (bins, kernels.pairs_to_csr(pairs, res, start, chrom_bins, total, False))
            continue
        _check_fits(_dense_bytes([total]), dev, "genome-wide %d bp" % res)
        W = DenseBatch([total], dev)
        kernels.bin_pairs_whole(pairs, res, start, start, W)
        whole[res] = (bins, W)
    for res in localRes:
        sizes = [genome[c] // res + 1 for c in order]                # matrixBuilding.py:564
        if _dense_bytes(sizes) > budget:
            bins, csr = bin_traditional_sparse(pairs, genome, res, cis_only=True, device=dev)
            local[res] = CisCsr(csr, bins, order)
            continue
        _check_fits(_dense_bytes(sizes), dev, "intra-chromosomal %d bp" % res)
        L = DenseBatch(sizes, dev)
        kernels.bin_pairs_local_banded(pairs, res, L)            # freshly zeroed tiles: symmetric on entry
        local[res] = L
    return whole, local


def WholeMatrixToSparseDict(Bins, Matrix):
    """matrixBuilding.py:457-506.  ``Matrix`` may be a NumPy array (uploaded) or a 1-matrix
    ``DenseBatch`` already in HBM.  Intra blocks: upper triangle; inter blocks ``c1_c2`` (c1
    before c2 in sorted order): all non-zeros, block-local coordinates."""
    if isinstance(Matrix, kernels.SymCsr):
        return WholeCsrToSparseDict(Bins, Matrix)
    W = Matrix if isinstance(Matrix, DenseBatch) else DenseBatch.from_numpy([np.asarray(Matrix)])
    ld, base = W.lds[0], W.buf.data_ptr()
    chroms = Sort_Chromosomes(Bins.keys())
    out = {}
    for i, ca in enumerate(chroms):
        a0, a1 = Bins[ca][0], Bins[ca][1] + 1
        out[ca] = kernels.dense_nonzero_records(base + 4 * (a0 * ld + a0), ld, a1 - a0, a1 - a0, True,
                                                False, W.device)
        for cb in chroms[i + 1:]:
            b0, b1 = Bins[cb][0], Bins[cb][1] + 1
            out[ca + "_" + cb] = kernels.dense_nonzero_records(base + 4 * (a0 * ld + b0), ld, a1 - a0,
                                                               b1 - b0, False, False, W.device)
    return out


def IntraMatrixToSparseDict(Dict):
    """matrixBuilding.py:508-524.  Values may be int or float NumPy matrices, or
    ``(DenseBatch, index)`` / float64 device tensors produced by this package."""
    out = {}
    for chro, M in Dict.items():
        if isinstance(M, torch.Tensor):              # float64 (n, n) device tensor
            n = M.shape[0]
            out[chro] = kernels.dense_nonzero_records(M.data_ptr(), M.stride(0), n, n, True, True, M.device)
        elif isinstance(M, tuple):                   # (DenseBatch, i)
            b, i = M
            out[chro] = kernels.dense_nonzero_records(b.buf.data_ptr() + 4 * b.offsets[i], b.lds[i],
                                                      b.sizes[i], b.sizes[i], True, False, b.device)
        else:
            M = np.asarray(M)
            if np.issubdtype(M.dtype, np.floating):
                t = torch.from_numpy(np.ascontiguousarray(M, dtype=np.float64)).to(require_cuda())
                out[chro] = kernels.dense_nonzero_records(t.data_ptr(), t.stride(0), M.shape[0], M.shape[1],
                                                          True, True, t.device)
            else:
                b = DenseBatch.from_numpy([M])
                out[chro] = kernels.dense_nonzero_records(b.buf.data_ptr(), b.lds[0], b.sizes[0], b.sizes[0],
                                                          True, False, b.device)
    return out


def TraditionalMatrixBuilding(bed_IO, genomeSize, wholeRes, localRes, chroms):
    """matrixBuilding.py:528-613.  ``bed_IO``: stream of 23-column valid-pair lines (or a
    ``PairColumns`` already in HBM).  Returns (Whole_Lib, Local_Lib) of structured arrays."""
    genome = Load_Genome(genomeSize, chroms)
    order = Sort_Chromosomes(genome)
    dev = require_cuda()
    pairs = _to_pair_columns(bed_IO, order, chroms, "valid23", dev)
    whole, local = bin_traditional(pairs, genome, wholeRes, localRes, dev)
    Whole_Lib = {res: WholeMatrixToSparseDict(bins, W) for res, (bins, W) in whole.items()}
    Local_Lib = {}
    for res, L in local.items():
        if isinstance(L, CisCsr):
            Local_Lib[res] = L.records()
            continue
        recs, _ = kernels.dense_batch_triu_records(L)
        Local_Lib[res] = {c: recs[i].copy() for i, c in enumerate(order)}   # own the memory (pool is reused)
    return Whole_Lib, Local_Lib


def TraditionalMatrixInAllelic(bed_IO, genomeSize, wholeRes, localRes, chroms):
    """matrixBuilding.py:793-854 -- same accumulation on the 4/5-column allelic beds; returns
    the RAW dense matrices: ({res: {'Bins', 'Matrix'}}, {res: {chrom: ndarray int64}})."""
    genome = Load_Genome(genomeSize, chroms)
    order = Sort_Chromosomes(genome)
    dev = require_cuda()
    pairs = _to_pair_columns(bed_IO, order, chroms, "allelic", dev)
    whole, local = bin_traditional(pairs, genome, wholeRes, localRes, dev, budget=1 << 62)   # dense by contract
    Whole_Lib = {res: {"Bins": bins, "Matrix": W.to_numpy(0)} for res, (bins, W) in whole.items()}
    Local_Lib = {res: {c: L.to_numpy(i) for i, c in enumerate(order)} for res, L in local.items()}
    return Whole_Lib, Local_Lib


def bin_haplotype_local(pairs: PairColumns, genome: dict, res: int, onesided: bool, out: DenseBatch = None,
                        device=None):
    """Per-chromosome haplotype matrices from an M_M or P_P bed: 'Both' pairs symmetric
    (matrixBuilding.py:1153-1161), or -- ``onesided`` -- the R1/R2 pairs added asymmetrically
    on top of ``out`` (:1295-1301, :1409-1415)."""
    dev = require_cuda(device)
    order = Sort_Chromosomes(genome)
    L = out if out is not None else DenseBatch([genome[c] // res + 1 for c in order], dev)
    kernels.bin_pairs_local(pairs, res, L, _abi.HC_BIN_ONESIDED if onesided else _abi.HC_BIN_SYM_BOTH)
    return L


def GetNeighborhoodIndex(L):
    """matrixBuilding.py:721-732: window indices (i, j) of a (2L+1)x(2L+1) window closer than
    sqrt(L) to (L+1, L+1) -- the reference's centre, one off the window centre."""
    i, j = np.mgrid[0:2 * L + 1, 0:2 * L + 1]
    near = np.sqrt(((i - (L + 1)) ** 2 + (j - (L + 1)) ** 2).astype(np.float64)) < np.sqrt(np.float64(L))
    return [int(x) for x in i[near]], [int(x) for x in j[near]]


def impute_inter_chromosomal(un: dict, imp: dict, mm: PairColumns, pp: PairColumns, starts: dict, wholeRes,
                             Imputation_region, Imputation_min, Imputation_ratio):
    """Inter-chromosomal branches of the imputation loops (matrixBuilding.py:1302-1378 for the M_M
    file, :1416-1492 for P_P) on the genome-wide haplotype matrices, bug for bug.

    un / imp: {res: one-matrix DenseBatch} (un-imputed, read only / imputed, credited);
    starts: {res: (start_M, start_P)} device int64 tables; mm / pp: the bed columns in FILE order.

    The P_P R1 branch of the reference votes with the window object `M_M_sub` left behind by the M_M
    loop (:1448).  That window belongs to the last M_M line -- and, within it, the last resolution
    of `wholeRes` -- that reached the window cut; it is located on the device (atomic max of the line
    index), fetched, and its disc sum per resolution handed to the P_P pass.  Where the reference
    would raise (no such line: NameError; stale window of a coarser resolution too small for this
    resolution's indices: IndexError) the same exception is raised here if a P_P R1 line gets that far.
    """
    dev = mm.device
    wholeRes = list(wholeRes)
    half = {res: int(Imputation_region) // res for res in wholeRes}
    nb = {}
    for res in wholeRes:
        ii, jj = GetNeighborhoodIndex(half[res])
        nb[res] = (torch.tensor(ii, dtype=torch.int32, device=dev), torch.tensor(jj, dtype=torch.int32, device=dev), ii, jj)
    last = torch.full((len(wholeRes),), -1, dtype=torch.int64, device=dev)
    for k, res in enumerate(wholeRes):
        kernels.impute_inter(mm, res, starts[res][0], starts[res][1], False, un[res], imp[res], half[res], nb[res][0],
                             nb[res][1], Imputation_min, Imputation_ratio, last_qualifying=last[k:k + 1])
    if pp.n == 0:
        return
    # ---- the stale `M_M_sub` window -------------------------------------------------------------
    h_last = last.cpu().numpy()
    line = int(h_last.max()) if len(h_last) else -1
    stale = None
    if line >= 0:
        k = max(i for i in range(len(wholeRes)) if h_last[i] == line)
        res = wholeRes[k]
        ca, pa, cb, pb, mk = (int(t[line].item()) for t in (mm.c1, mm.p1, mm.c2, mm.p2, mm.mark))
        sm, sp = starts[res][0].cpu().numpy(), starts[res][1].cpu().numpy()
        b1, b2, s = pa // res, pb // res, half[res]
        if mk == 1:
            r0, c0 = b1 + int(sm[ca]), b2 + int(sm[cb])          # Matrix[bin1 +- s, M_bin2 +- s]   (:1327)
        else:
            r0, c0 = b1 + int(sm[cb]), b2 + int(sm[ca])          # Matrix[M_bin1 +- s, bin2 +- s]   (:1363)
        n, ld = un[res].sizes[0], un[res].lds[0]
        U = un[res].buf[un[res].offsets[0]:un[res].offsets[0] + n * ld].view(n, ld)
        stale = U[r0 - s:r0 + s + 1, c0 - s:c0 + s + 1].cpu().numpy().astype(np.int64)
    needed = torch.zeros(len(wholeRes), dtype=torch.int32, device=dev)
    states = []
    for k, res in enumerate(wholeRes):
        ii, jj = nb[res][2], nb[res][3]
        if stale is None:
            state, ksum = 1, 0
        elif ii and (max(ii) >= stale.shape[0] or max(jj) >= stale.shape[1]):
            state, ksum = 2, 0
        else:
            state, ksum = 0, int(stale[ii, jj].sum())
        states.append(state)
        kernels.impute_inter(pp, res, starts[res][0], starts[res][1], True, un[res], imp[res], half[res], nb[res][0],
                             nb[res][1], Imputation_min, Imputation_ratio, stale_state=state, stale_sum=ksum,
                             stale_needed=needed[k:k + 1])
    h_needed = needed.cpu().numpy()
    for k, res in enumerate(wholeRes):
        if h_needed[k] and states[k] == 1:
            raise NameError("name 'M_M_sub' is not defined")          # what the reference dies with at :1448
        if h_needed[k] and states[k] == 2:
            raise IndexError("stale M_M_sub window of another resolution is too small for resolution %d (:1448)" % res)


# ======================================================================================
# (c) two-step allelic correction
# ======================================================================================
def _f64_device(X):
    """float64 device copy (row-major) of a host matrix or device tensor."""
    if isinstance(X, torch.Tensor):
        return X.to(device=require_cuda(), dtype=torch.float64).contiguous()
    return torch.from_numpy(np.ascontiguousarray(np.asarray(X), dtype=np.float64)).to(require_cuda())


def _row_nnz(Matrix):
    """Per-row non-zero counts on the device: (int32 device tensor, nrows, ncols)."""
    dev = require_cuda()
    if isinstance(Matrix, torch.Tensor) or np.issubdtype(np.asarray(Matrix).dtype, np.floating):
        t = _f64_device(Matrix)
        nr, nc = t.shape
        nz = torch.empty(nr, dtype=torch.int32, device=dev)
        _abi.check(_abi.lib().hc_rownnz_f64(kernels.ptr(t), t.stride(0), nr, nc, kernels.ptr(nz), kernels.stream_ptr()),
                   "hc_rownnz_f64")
        return nz, nr, nc
    M = np.asarray(Matrix)
    if M.shape[0] != M.shape[1]:
        return _row_nnz(M.astype(np.float64))
    b = DenseBatch.from_numpy([M])
    _, nz = kernels.rowstats(b.buf.data_ptr(), b.lds[0], b.sizes[0], b.sizes[0], dev)
    return nz, b.sizes[0], b.sizes[0]


def _gap_rows(Matrix, gap_mode):
    nz, nr, nc = _row_nnz(Matrix)
    dev = nz.device
    cov = torch.empty(nr, dtype=torch.float64, device=dev)
    gf = torch.empty(nr, dtype=torch.uint8, device=dev)
    gi = torch.empty(nr, dtype=torch.int32, device=dev)
    ng = torch.zeros(1, dtype=torch.int32, device=dev)
    _abi.check(_abi.lib().hc_gap_rows(kernels.ptr(nz), nr, nc, gap_mode, kernels.ptr(cov), kernels.ptr(gf), kernels.ptr(gi),
                                      kernels.ptr(ng), kernels.stream_ptr()), "hc_gap_rows")
    return cov, gf, gi, int(ng.item())


def Coverage_M(Matrix):
    """matrixBuilding.py:904-912 -- fraction of non-zero entries per row."""
    return _gap_rows(Matrix, _abi.HC_GAP_FIXED)[0].cpu().numpy()


def Gap_defined(Matrix):
    """matrixBuilding.py:915-929 -- rows whose coverage is below min(25th percentile of the non-zero
    coverages, 0.2).  A matrix without a covered row has no percentile: the reference raises IndexError
    there (np.percentile of an empty array), and so does this."""
    cov, _, gi, n = _gap_rows(Matrix, _abi.HC_GAP_PERCENTILE)
    if not bool((cov != 0).any().item()):
        raise IndexError("index -1 is out of bounds for axis 0 with size 0")     # what np.percentile([]) raises
    return _gap_array(gi, n)


def Gap_definedLowRes(Matrix):
    """matrixBuilding.py:742-753 -- fixed 0.1 coverage threshold."""
    _, _, gi, n = _gap_rows(Matrix, _abi.HC_GAP_FIXED)
    return _gap_array(gi, n)


def Non_Gap_Defined(N, gap):
    """matrixBuilding.py:932-943 -- the rows of range(N) that are not gaps (host: O(N) index bookkeeping)."""
    keep = np.ones(int(N), dtype=bool)
    g = np.asarray(gap, dtype=np.int64)
    keep[g[(g >= 0) & (g < N)]] = False
    return np.nonzero(keep)[0] if keep.any() else np.array([])


Non_Gap_DefinedLowRes = Non_Gap_Defined          # matrixBuilding.py:756-767: same body


def Trans2symmetry(Matrix, gap):
    """matrixBuilding.py:945-979 -- no gap rows: S_ij + S_ji off the diagonal; otherwise max for pairs of
    gap rows and the mean for every other pair; the diagonal is kept."""
    S = _f64_device(Matrix)
    n = S.shape[0]
    assert S.shape[1] == n
    gap = np.asarray(gap)
    gf = None
    if gap.size:
        flags = np.zeros(n, dtype=np.uint8)
        flags[gap.astype(np.int64)] = 1
        gf = torch.from_numpy(flags).to(S.device)
    out = torch.empty_like(S)
    _abi.check(_abi.lib().hc_trans2symmetry_f64(kernels.ptr(S), S.stride(0), n, kernels.ptr(gf), kernels.ptr(out),
                                                out.stride(0), kernels.stream_ptr()), "hc_trans2symmetry_f64")
    return out.cpu().numpy()


def Trans2symmetryLowRes(Matrix):
    """matrixBuilding.py:770-776."""
    return Trans2symmetry(Matrix, np.array([]))


def Correct_VC(X, alpha):
    """matrixBuilding.py:780-790 -- one-shot vanilla-coverage style scaling
    x / (colsum**alpha [None, :] * rowsum**alpha [:, None]), zero sums replaced by 1."""
    x = _f64_device(X)
    nr, nc = x.shape
    out = torch.empty_like(x)
    work = torch.empty(int(_abi.lib().hc_correct_vc_work_bytes(nr, nc)), dtype=torch.uint8, device=x.device)
    _abi.check(_abi.lib().hc_correct_vc_f64(kernels.ptr(x), x.stride(0), nr, nc, float(alpha), kernels.ptr(out), out.stride(0),
                                            kernels.ptr(work), kernels.stream_ptr()), "hc_correct_vc_f64")
    return out.cpu().numpy()


def _gap_array(idx_t, count):
    # the reference returns np.array(python list): int64, or float64 when empty
    return idx_t[:count].cpu().numpy().astype(np.int64) if count else np.array([])


def two_step_device(T: DenseBatch, ti: int, M: DenseBatch, mi: int, P: DenseBatch, pi: int):
    """TwoStepCorrection on matrices already in HBM; returns device float64 tensors and the
    host gap arrays."""
    n, dev = T.sizes[ti], T.device
    assert M.sizes[mi] == n and P.sizes[pi] == n
    if M is P and pi == mi + 1 and n > 0:
        # M and P next to each other in one batch: the batched driver (one launch per pass over both matrices, the gap
        # decision read on the device -- no host round trip in the middle)
        from .construction import _sub_batch
        mats, gaps = kernels.twostep_batch(_sub_batch(T, ti, 1), _sub_batch(M, mi, 2))
        return mats[0], mats[1], gaps[0], gaps[1]
    tp, mp, pp = (b.buf.data_ptr() + 4 * b.offsets[i] for b, i in ((T, ti), (M, mi), (P, pi)))
    rs_t, _ = kernels.rowstats(tp, T.lds[ti], n, n, dev, want_nnz=False)
    rs_m, nz_m = kernels.rowstats(mp, M.lds[mi], n, n, dev)
    rs_p, nz_p = kernels.rowstats(pp, P.lds[pi], n, n, dev)
    alpha, (gf_m, gi_m), (gf_p, gi_p), ngap = kernels.twostep_alpha(
        rs_t, rs_m, rs_p, nz_m, nz_p, n, n, _abi.HC_GAP_PERCENTILE, dev)
    ng = ngap.cpu().numpy()
    nor_m = kernels.twostep_correct(mp, M.lds[mi], n, alpha, gf_m, ng[0] > 0, rs_m, dev)
    nor_p = kernels.twostep_correct(pp, P.lds[pi], n, alpha, gf_p, ng[1] > 0, rs_p, dev)
    return nor_m, nor_p, _gap_array(gi_m, int(ng[0])), _gap_array(gi_p, int(ng[1]))


def _is_sparse(*mats):
    import scipy.sparse as sp
    return any(sp.issparse(m) for m in mats)


def _device_csr(m, cls, dtype=np.int32):
    """host matrix (scipy.sparse or dense) -> device CSR: duplicates summed, explicit zeros dropped (coverage counts the
    stored entries), columns sorted.  ``dtype`` int32: integer counts (``as_int32_counts``); float64: values as they
    are.  The input is not modified; the canonical host copy is kept as ``.host``."""
    import scipy.sparse as sp
    m = sp.csr_matrix(m, copy=True)
    m.sum_duplicates()
    m.eliminate_zeros()
    m.sort_indices()
    dev = require_cuda()
    up = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(dev)
    vals = as_int32_counts(m.data) if dtype == np.int32 else m.data
    X = cls(up(m.indptr, np.int64), up(m.indices, np.int32), up(vals, dtype), m.shape[0])
    X.host = m
    return X


def _twostep_sparse(tra, hap):
    """TwoStepCorrection of nchrom chromosomes on the CSR path: ``tra`` nchrom square count matrices, ``hap`` their
    2*nchrom haplotype matrices (all M, then all P).  Returns (2*nchrom symmetric float64 scipy CSR matrices, both
    triangles stored, and 2*nchrom gap arrays)."""
    import scipy.sparse as sp
    sizes = [m.shape[0] for m in tra]
    if any(m.shape != (n, n) for m, n in zip(list(tra) + list(hap), sizes * 3)) or len(hap) != 2 * len(tra):
        raise ValueError("square traditional and haplotype matrices of matching sides expected")
    t_off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    h_off = np.concatenate([[0], np.cumsum(sizes + sizes)]).astype(np.int64)
    H = sp.block_diag(hap, format="csr")
    X = _device_csr(H, kernels.GenCsr)
    X.t = _device_csr(H.T, kernels.GenCsr)
    recs, gaps = kernels.twostep_csr_batch(_device_csr(sp.block_diag(tra, format="csr"), kernels.SymCsr), t_off, X, h_off)
    mats = []
    for r, n in zip(recs, sizes + sizes):
        b1, b2, v = r["bin1"], r["bin2"], r["IF"]
        off = b1 != b2
        mats.append(sp.csr_matrix((np.concatenate([v, v[off]]), (np.concatenate([b1, b2[off]]), np.concatenate([b2, b1[off]]))),
                                  shape=(n, n)))
    return mats, gaps


def TwoStepCorrection(TM, MM, PM):
    """matrixBuilding.py:984-1023 -> (Nor_MM, Nor_PM, Gap_M, Gap_P).  With ``scipy.sparse`` inputs the correction runs
    on the non-zeros (``hc_twostep_csr_batch``) and Nor_MM / Nor_PM are symmetric ``scipy.sparse`` CSR matrices."""
    if _is_sparse(TM, MM, PM):
        mats, gaps = _twostep_sparse([TM], [MM, PM])
        return mats[0], mats[1], gaps[0], gaps[1]
    b = DenseBatch.from_numpy([np.asarray(TM), np.asarray(MM), np.asarray(PM)])
    nor_m, nor_p, gap_m, gap_p = two_step_device(b, 0, b, 1, b, 2)
    return nor_m.cpu().numpy(), nor_p.cpu().numpy(), gap_m, gap_p


def IntraChromMatrixCorrection(Tra_Lib, Hap_Lib):
    """matrixBuilding.py:1026-1041 -> (Nor_Lib, Gap_Lib) keyed 'M'+chrom / 'P'+chrom.  All
    chromosomes are corrected by one batched library call (``kernels.twostep_batch``; with ``scipy.sparse``
    inputs ``kernels.twostep_csr_batch``, and the corrected matrices are symmetric ``scipy.sparse`` CSR)."""
    chros = list(Tra_Lib.keys())
    if _is_sparse(*Tra_Lib.values(), *Hap_Lib.values()):
        mats, gaps = _twostep_sparse([Tra_Lib[c] for c in chros], [Hap_Lib["M" + c] for c in chros] + [Hap_Lib["P" + c] for c in chros])
        keys = ["M" + c for c in chros] + ["P" + c for c in chros]
        return dict(zip(keys, mats)), dict(zip(keys, gaps))
    T = DenseBatch.from_numpy([np.asarray(Tra_Lib[c]) for c in chros])
    H = DenseBatch.from_numpy([np.asarray(Hap_Lib["M" + c]) for c in chros] +
                              [np.asarray(Hap_Lib["P" + c]) for c in chros])
    mats, gaps = kernels.twostep_batch(T, H)
    Nor_Lib, Gap_Lib = {}, {}
    for i, c in enumerate(chros):
        Nor_Lib["M" + c], Nor_Lib["P" + c] = mats[i].cpu().numpy(), mats[len(chros) + i].cpu().numpy()
        Gap_Lib["M" + c], Gap_Lib["P" + c] = gaps[i], gaps[len(chros) + i]
    return Nor_Lib, Gap_Lib


def GenomeWideMatrixCorrection(Bins_Pos, Hap_Bins_Pos, T_M, H_M):
    """matrixBuilding.py:857-901 -- low-resolution genome-wide haplotype matrix: per-chromosome
    alpha from the intra blocks (gaps by the fixed 0.1 coverage rule on the traditional block),
    concatenated in sorted chromosome order and repeated for the P half; H/alpha ->
    sum-symmetrise -> Correct_VC(2/3) -> rescale to the raw mean."""
    dev = require_cuda()
    Tb = T_M if isinstance(T_M, DenseBatch) else DenseBatch.from_numpy([np.asarray(T_M)])
    Hb = H_M if isinstance(H_M, DenseBatch) else DenseBatch.from_numpy([np.asarray(H_M)])
    n_h = Hb.sizes[0]
    alphas = {}
    for chro, (lo, hi) in Bins_Pos.items():
        n = hi - lo + 1
        ml, pl = Hap_Bins_Pos["M" + chro][0], Hap_Bins_Pos["P" + chro][0]
        tptr = Tb.buf.data_ptr() + 4 * (lo * Tb.lds[0] + lo)
        mptr = Hb.buf.data_ptr() + 4 * (ml * Hb.lds[0] + ml)
        pptr = Hb.buf.data_ptr() + 4 * (pl * Hb.lds[0] + pl)
        rs_t, nz_t = kernels.rowstats(tptr, Tb.lds[0], n, n, dev)
        rs_m, _ = kernels.rowstats(mptr, Hb.lds[0], n, n, dev, want_nnz=False)
        rs_p, _ = kernels.rowstats(pptr, Hb.lds[0], n, n, dev, want_nnz=False)
        alpha, _, _, _ = kernels.twostep_alpha(rs_t, rs_m, rs_p, nz_t, None, n, n, _abi.HC_GAP_FIXED, dev)
        alphas[chro] = alpha
    alpha = torch.cat([alphas[c] for c in Sort_Chromosomes(alphas.keys())])
    alpha = torch.cat([alpha, alpha])                      # matrixBuilding.py:892
    rs_h, _ = kernels.rowstats(Hb.buf.data_ptr(), Hb.lds[0], n_h, n_h, dev, want_nnz=False)
    out = kernels.twostep_correct(Hb.buf.data_ptr(), Hb.lds[0], n_h, alpha, None, False, rs_h, dev)
    return out.cpu().numpy()


# ======================================================================================
# (b) ICE  (`cooler balance`, call sites matrixBuilding.py:708, :713, :1537, :1542)
# ======================================================================================
def ice_balance_dense(mats, chrom_offsets=None, ignore_diags=1, mad_max=5, min_nnz=10, min_count=0,
                      tol=1e-5, max_iters=200, rescale_marginals=True):
    """Balance dense symmetric matrices.

    ``mats``: list of square integer matrices / a ``DenseBatch`` -> ``--cis-only`` semantics
    (each matrix is one chromosome with its own loop, scale and early exit; weights are
    returned concatenated).  With ``chrom_offsets`` (nchrom+1 bin offsets) and ONE matrix ->
    genome-wide balancing of that matrix (`cooler balance` without --cis-only)."""
    batch = mats if isinstance(mats, DenseBatch) else DenseBatch.from_numpy([np.asarray(m) for m in mats])
    off = None
    if chrom_offsets is not None:
        assert len(batch) == 1, "genome-wide balancing takes exactly one matrix"
        off = torch.tensor(np.asarray(chrom_offsets, dtype=np.int64), device=batch.device)
    return kernels.ice_balance_dense(batch, off, ignore_diags=ignore_diags, mad_max=mad_max,
                                     min_nnz=min_nnz, min_count=min_count, tol=tol, max_iters=max_iters,
                                     rescale_marginals=rescale_marginals)


# ======================================================================================
# sort path (genome-wide matrices that do not fit dense tiles): pairs -> symmetric CSR
# ======================================================================================
def bin_traditional_sparse(pairs: PairColumns, genome: dict, res: int, cis_only=False, device=None):
    """Genome-wide binning through radix sort + reduce-by-key (north_star kernel (a)).
    Same bins as ``Get_Chro_Bins`` (matrixBuilding.py:409-426).  Returns (Bins, SymCsr)."""
    dev = require_cuda(device)
    order = Sort_Chromosomes(genome)
    bins, total = _bins_from_genome(genome, res, [(c, c) for c in order])
    start = _start_table(bins, order, dev)
    chrom_bins = torch.tensor([genome[c] // res + 1 for c in order], dtype=torch.int32, device=dev)
    return bins, kernels.pairs_to_csr(pairs, res, start, chrom_bins, total, cis_only)


def chrom_offsets_from_bins(Bins):
    """nchrom+1 bin offsets in ``Sort_Chromosomes`` order (the cool file's indexes/chrom_offset)."""
    order = Sort_Chromosomes(Bins.keys())
    return np.array([Bins[c][0] for c in order] + [Bins[order[-1]][1] + 1], dtype=np.int64)


def WholeCsrToSparseDict(Bins, csr):
    """``WholeMatrixToSparseDict`` (matrixBuilding.py:457-506) for a genome-wide symmetric CSR:
    intra blocks keyed 'c' (upper triangle), inter blocks 'c1_c2' (c1 before c2), block-local
    coordinates, row-major order inside each block."""
    b1, b2, v = (t.cpu().numpy() for t in kernels.csr_upper_records(csr))
    b1 = b1.astype(np.int64)
    order = Sort_Chromosomes(Bins.keys())
    off = chrom_offsets_from_bins(Bins)
    ca = np.searchsorted(off, b1, side="right") - 1
    cb = np.searchsorted(off, b2, side="right") - 1
    out = {}
    # upper-triangular pixels have chrom(bin1) <= chrom(bin2); group by (ca, cb) preserving order
    grp = ca * len(order) + cb
    idx = np.argsort(grp, kind="stable")
    bounds = np.searchsorted(grp[idx], np.arange(len(order) * len(order) + 1))
    for i, c1 in enumerate(order):
        for j in range(i, len(order)):
            c2 = order[j]
            sel = idx[bounds[i * len(order) + j]:bounds[i * len(order) + j + 1]]
            rec = np.zeros(sel.size, dtype=S_dtype)
            rec["bin1"], rec["bin2"], rec["IF"] = b1[sel] - off[i], b2[sel].astype(np.int64) - off[j], v[sel]
            out[c1 if i == j else c1 + "_" + c2] = rec
    return out


def ice_balance_sparse(csr, Bins, cis_only=False, ignore_diags=1, mad_max=5, min_nnz=10, min_count=0,
                       tol=1e-5, max_iters=200, rescale_marginals=True, comm=None, allreduce=None):
    """`cooler balance --ignore-diags K [--cis-only]` on the symmetric CSR.  With ``cis_only``
    the CSR must have been built from cis pairs only (``bin_traditional_sparse(cis_only=True)``):
    every chromosome then iterates on its own."""
    off = chrom_offsets_from_bins(Bins)
    prob = off if cis_only else np.array([0, off[-1]], dtype=np.int64)
    bias, stats = kernels.ice_balance_csr(csr, prob, chrom_off=off, comm=comm, allreduce=allreduce,
                                          ignore_diags=ignore_diags, mad_max=mad_max, min_nnz=min_nnz,
                                          min_count=min_count, tol=tol, max_iters=max_iters,
                                          rescale_marginals=rescale_marginals)
    return bias.cpu().numpy(), stats


# drivers (replicate loop, merge, stores): same names as the reference, defined in construction.py (which imports this
# module): resolved on first use so that either module can be imported first
_DRIVERS = ("Check_Bed", "HaplotypeMatrixBuilding", "HaplotypeMatrixConstruction", "Merge_beds", "TraditionalMatrixConstruction")


def __getattr__(name):
    if name in _DRIVERS:
        from . import construction
        return getattr(construction, name)
    raise AttributeError("module %r has no attribute %r" % (__name__, name))
