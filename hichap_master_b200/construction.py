"""Drivers of the matrix stage with the reference's signatures:
``TraditionalMatrixConstruction`` (matrixBuilding.py:617-717) and ``HaplotypeMatrixBuilding`` /
``HaplotypeMatrixConstruction`` (matrixBuilding.py:1044-1860).

Host orchestration re-expressed around the device kernels: replicate loop, bed concatenation
(the reference pipes ``cat``; here the files are chained in Python), replicate merge (dense
``+=`` as at :1700-1719, on the device), ICE (the reference shells out to ``cooler balance``),
two-step correction, gap NPZ.  The reference stores everything in multi-resolution ``.cool``
files through the un-vendored ``cooler`` package (needs ``h5py``; neither is available here), so
matrices and weights are written as ``.npz`` stores with the same content: per resolution the
(bin1, bin2, IF) records of every chromosome / chromosome pair exactly as ``NPZ2Cooler`` receives
them, plus the ``weight`` vector and balancing stats that ``cooler balance`` would put in
``bins/weight``.  ``{prefix}Imputated_Gap.npz`` is written with the reference's key structure
(consumed at StructureFind.py:1988-1992).

Deviations (documented in DESIGN.md): allelic mode accepts a single replicate (the reference
raises TypeError there, matrixBuilding.py:1676-1683).  Inter-chromosomal imputation
(:1302-1378, :1416-1492) is performed bug for bug (``matrixBuilding.impute_inter_chromosomal``).
"""
from __future__ import annotations

import itertools
import logging
import os

import numpy as np
import torch

from . import _abi, kernels
from .device import DenseBatch, PairColumns, require_cuda
from .matrixBuilding import (CisCsr, GenomeWideMatrixCorrection, IntraMatrixToSparseDict, Load_Genome, Sort_Chromosomes,
                             WholeMatrixToSparseDict, _bins_from_genome, _dense_bytes, _start_table, bin_traditional,
                             bin_traditional_sparse, chrom_offsets_from_bins, dense_budget_bytes, ice_balance_sparse,
                             impute_inter_chromosomal)
from .pairs import read_pair_files

log = logging.getLogger(__name__)


def _say(msg):
    print(msg)
    log.log(21, msg)


def Merge_beds(bed_lst):
    """matrixBuilding.py:307-313 returned a ``cat`` command line; here: one chained line stream."""
    return itertools.chain.from_iterable(open(f, "r") for f in bed_lst)


def Check_Bed(bed_lst):
    """matrixBuilding.py:316-346."""
    for tag in ("Bi_Allelic", "M_M", "P_P", "M_P", "P_M"):
        if not any((tag + ".bed") in f for f in bed_lst):
            return False, tag
    return True, ""


class MatrixStore:
    """``.npz`` stand-in for the multi-resolution cool file written by ``NPZ2Cooler``
    (matrixBuilding.py:100-303): ``add(res, lib)`` takes the same ``{key: records}`` dictionaries."""

    def __init__(self, path):
        self.path = path
        self.data = {}

    def add(self, res, lib, bins=None):
        for key, rec in lib.items():
            self.data["%d|%s" % (res, key)] = rec
        if bins is not None:
            self.data["bins|%d" % res] = np.array([(k, v[0], v[1]) for k, v in bins.items()],
                                                  dtype=[("chrom", "U16"), ("start", "<i8"), ("end", "<i8")])

    def set_weight(self, res, weight, stats, names=None):
        """``names``: chromosomes (in order) the weight vector covers when this rank balanced only its own
        chromosomes; the pieces of all ranks are gathered and rank 0 stores the full vector."""
        dist, rank, world = _dist()
        if names is not None and world > 1:
            pieces = [None] * world
            dist.all_gather_object(pieces, (list(names), np.asarray(weight), stats))
            if rank != 0:
                return
            self.data["weight_chroms|%d" % res] = np.array([c for nm, _, _ in pieces for c in nm])
            weight = np.concatenate([w for _, w, _ in pieces])
            stats = dict(stats, iters=[i for _, _, st in pieces for i in st["iters"]],
                         scale=np.concatenate([np.atleast_1d(st["scale"]) for _, _, st in pieces]))
        elif world > 1 and rank != 0:
            return
        self.data["weight|%d" % res] = weight
        self.data["weight_attrs|%d" % res] = np.array(repr({k: (v.tolist() if isinstance(v, np.ndarray) else v)
                                                            for k, v in stats.items()}))

    def save(self):
        _, rank, world = _dist()
        path = self.path if rank == 0 else self.path[:-4] + ".part%d.npz" % rank
        if rank == 0 and world > 1:
            self.data["parts"] = np.array(world)
        np.savez(path, **self.data)
        return path

    @staticmethod
    def load(path):
        """{key: array} of a store, the per-rank parts concatenated in rank order (row blocks / chromosomes are
        assigned to ranks in ascending order of rows, so record order is preserved)."""
        main = dict(np.load(path, allow_pickle=True))
        for r in range(1, int(main.get("parts", 1))):
            part = np.load(path[:-4] + ".part%d.npz" % r, allow_pickle=True)
            for k in part.files:
                if k in main and main[k].dtype.names and part[k].dtype.names:
                    main[k] = np.concatenate([main[k], part[k]])
                elif k not in main:
                    main[k] = part[k]
        return main


def _add_into(dst: DenseBatch, src: DenseBatch):
    """replicate merge, matrixBuilding.py:1703-1719 (dense +=), on the device"""
    _abi.check(_abi.lib().hc_add_i32(C_ptr(dst.buf), C_ptr(src.buf), dst.buf.numel(), kernels.stream_ptr()),
               "hc_add_i32")


def C_ptr(t):
    return kernels.ptr(t)


def _balance(store, whole, local, wholeRes, localRes):
    """ICE of one store: genome-wide for the whole resolutions, --cis-only for the local ones
    (matrixBuilding.py:706-714)."""
    for res in wholeRes:
        bins, W = whole[res]
        if isinstance(W, kernels.SymCsr):              # sort path (dense tiles would not fit) / row-block shard
            w, st = ice_balance_sparse(W, bins, cis_only=False, ignore_diags=1, comm=getattr(W, "comm", None),
                                       allreduce=getattr(W, "allreduce", None))
        else:
            off = torch.from_numpy(chrom_offsets_from_bins(bins)).to(W.device)
            w, st = kernels.ice_balance_dense(W, off, ignore_diags=1)
        store.set_weight(res, w, st)
    for res in localRes:
        L = local[res]
        if isinstance(L, CisCsr):
            w, st = ice_balance_sparse(L.csr, L.bins, cis_only=True, ignore_diags=1)
            names = L.order
        else:
            w, st = kernels.ice_balance_dense(L, None, ignore_diags=1)
            names = getattr(L, "chrom_names", None)
        store.set_weight(res, w, st, names=names if _dist()[2] > 1 else None)


def _store_traditional(path, genome, whole, local):
    order = Sort_Chromosomes(genome)
    store = MatrixStore(path)
    for res, (bins, W) in whole.items():
        store.add(res, WholeMatrixToSparseDict(bins, W), bins)
    for res, L in local.items():
        if isinstance(L, CisCsr):
            store.add(res, L.records())
            continue
        recs, _ = kernels.dense_batch_triu_records(L)
        store.add(res, {c: recs[i].copy() for i, c in enumerate(getattr(L, "chrom_names", order))})
    return store


def _dist():
    """(torch.distributed, rank, world) when the process runs under torchrun with an initialised group."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        return dist, dist.get_rank(), dist.get_world_size()
    return None, 0, 1


_COMM = {}


def _library_comm(dev):
    """one NCCL communicator of the library per process (in-loop allreduce of the row-block sharded ICE)"""
    from . import distributed as hd
    if "comm" not in _COMM:
        _COMM["comm"] = hd.nccl_comm_from_process_group(dev)
    return _COMM["comm"]


def _bin_replicate(cols, genome, wholeRes, localRes, dev):
    """Binning of one replicate's host columns.  One process: ``bin_traditional`` (dense tiles, or the sort path when
    they would not fit).  Under torchrun (SURVEY.md section 8e): genome-wide matrices become row-block sharded CSRs
    (each rank sorts a slice of the pairs, keys are exchanged), intra-chromosomal matrices are LPT-sharded by
    chromosome -- every rank bins and balances only its own chromosomes, no collective on that path."""
    dist, rank, world = _dist()
    c1, p1, c2, p2 = cols
    if world == 1:
        return bin_traditional(PairColumns(c1, p1, c2, p2, device=dev), genome, wholeRes, localRes, dev)
    from . import distributed as hd, shard
    from .matrixBuilding import _check_fits, _dense_bytes, bin_traditional_sparse, dense_budget_bytes
    order = Sort_Chromosomes(genome)
    whole, local = {}, {}
    if wholeRes:
        sl = slice(rank, None, world)
        pr = PairColumns(c1[sl], p1[sl], c2[sl], p2[sl], device=dev)
        comm = _library_comm(dev)
        for res in wholeRes:
            bins, total = _bins_from_genome(genome, res, [(c, c) for c in order])
            start = _start_table(bins, order, dev)
            chrom_bins = torch.tensor([genome[c] // res + 1 for c in order], dtype=torch.int32, device=dev)
            csr, _ = hd.build_row_block_csr(pr, res, start, chrom_bins, total)
            csr.comm, csr.allreduce = comm, (lambda t: dist.all_reduce(t))
            whole[res] = (bins, csr)
    for res in localRes:
        sizes = [genome[c] // res + 1 for c in order]
        mine = shard.chromosome_shards(sizes, world)[rank]
        remap = np.full(len(order) + 1, -1, np.int32)
        remap[mine] = np.arange(len(mine), dtype=np.int32)
        lc = np.where(c1 == c2, remap[np.where(c1 >= 0, c1, len(order))], -1).astype(np.int32)
        sel = lc >= 0
        pr = PairColumns(lc[sel], p1[sel], lc[sel], p2[sel], device=dev)
        names = [order[i] for i in mine]
        my_sizes = [sizes[i] for i in mine]
        if _dense_bytes(my_sizes) > dense_budget_bytes(dev):
            bins, csr = bin_traditional_sparse(pr, {c: genome[c] for c in names}, res, cis_only=True, device=dev)
            local[res] = CisCsr(csr, bins, names)
        else:
            _check_fits(_dense_bytes(my_sizes), dev, "intra-chromosomal %d bp" % res)
            L = DenseBatch(my_sizes, dev)
            L.chrom_names = names
            kernels.bin_pairs_local_banded(pr, res, L)
            local[res] = L
    return whole, local


def _is_sparse(whole, local):
    return any(isinstance(W, kernels.SymCsr) for _, W in whole.values()) or any(isinstance(L, CisCsr) for L in local.values())


def TraditionalMatrixConstruction(OutPath, RepPath, genomeSize, wholeRes, localRes, chroms=["#", "X"],
                                  balance=True):
    """matrixBuilding.py:617-717.  Writes ``Cooler/{prefix}Multi.npz`` per replicate and
    ``Cooler/Merged_Multi.npz``; returns the list of written files.  Under torchrun every rank writes the
    records it owns (``*.partK.npz`` for rank K > 0; ``MatrixStore.load`` reassembles them) and rank 0 the weights."""
    _say("Building Replicate Matrix respectively")
    dev = require_cuda()
    CoolerPath = os.path.join(OutPath, "Cooler")
    os.makedirs(CoolerPath, exist_ok=True)
    genome = Load_Genome(genomeSize, chroms)
    order = Sort_Chromosomes(genome)
    written, merged, all_cols = [], None, []
    for rep_p in RepPath:
        files = [i for i in os.listdir(rep_p) if "_Valid.bed" in i]
        prefix = files[0].split("Valid")[0]
        files = [os.path.join(rep_p, f) for f in files]
        c1, p1, c2, p2, _ = read_pair_files(files, order, chroms, "valid23")   # `cat files` + per-line parse
        whole, local = _bin_replicate((c1, p1, c2, p2), genome, wholeRes, localRes, dev)
        store = _store_traditional(os.path.join(CoolerPath, prefix + "Multi.npz"), genome, whole, local)
        if balance:
            _balance(store, whole, local, wholeRes, localRes)
        written.append(store.save())
        _say("    %s finished" % store.path)
        all_cols.append((c1, p1, c2, p2))
        if merged is None:
            merged = (whole, local)
        elif not _is_sparse(whole, local):          # cooler.merge_coolers (:692) sums the pixels
            for res in wholeRes:
                _add_into(merged[0][res][1], whole[res][1])
            for res in localRes:
                _add_into(merged[1][res], local[res])
    _say("Merging the replicates ...")
    if len(RepPath) > 1 and _is_sparse(*merged):    # sparse matrices: the merged pixels are those of the concatenated pairs
        del whole, local
        merged = _bin_replicate(tuple(np.concatenate([c[k] for c in all_cols]) for k in range(4)), genome, wholeRes, localRes, dev)
    store = _store_traditional(os.path.join(CoolerPath, "Merged_Multi.npz"), genome, merged[0], merged[1])
    if balance:
        _say("    Balancing start ...")
        _balance(store, merged[0], merged[1], wholeRes, localRes)
    written.append(store.save())
    _say("All Done!")
    return written


# ======================================================================================
# allelic mode
# ======================================================================================
class HaplotypeData:
    """Device-resident counterpart of the reference's ``DataSets`` dictionary (:1059-1500).  A local resolution in
    ``sparse_res`` holds ``CisCsr`` matrices (T: the cis CSR of the traditional matrices; un / imp: CSRs over the
    concatenated haplotype bins, the imputed one general with its transpose); ``cols`` then keeps the pair columns
    they were binned from, so that merged replicates can be re-binned."""

    def __init__(self):
        self.tra_whole, self.tra_local = {}, {}
        self.un_whole, self.un_local = {}, {}
        self.imp_whole, self.imp_local = {}, {}
        self.hap_bins = {}
        self.sparse_res, self.cols = [], None

    def add(self, other):
        """dense replicate merge (+=); the sparse resolutions are re-binned from all replicates' pairs by the caller"""
        for a, b in ((self.tra_whole, other.tra_whole), (self.un_whole, other.un_whole), (self.imp_whole, other.imp_whole)):
            for res in a:
                _add_into(a[res][1], b[res][1])
        for a, b in ((self.tra_local, other.tra_local), (self.un_local, other.un_local), (self.imp_local, other.imp_local)):
            for res in a:
                if res not in self.sparse_res:
                    _add_into(a[res], b[res])

    def to_datasets(self, order):
        """the reference's DataSets layout with NumPy matrices (for parity checks / callers)"""
        hap_order = ["M" + c for c in order] + ["P" + c for c in order]
        out = {}
        for name, whole, local, keys in (("Tradition", self.tra_whole, self.tra_local, order),
                                         ("UnImputated", self.un_whole, self.un_local, hap_order),
                                         ("Imputated", self.imp_whole, self.imp_local, hap_order)):
            out[name + "_Whole"] = {res: {"Bins": b, "Matrix": W.to_numpy(0)} for res, (b, W) in whole.items()}
            out[name + "_Local"] = {res: L.matrices() if isinstance(L, CisCsr) else {k: L.to_numpy(i) for i, k in enumerate(keys)}
                                    for res, L in local.items()}
        return out


def _haplotype_counts(bed_files, genome, wholeRes, localRes, chroms, dev, imputation=(10000000, 2, 0.9)):
    """Binning part of HaplotypeMatrixBuilding (matrixBuilding.py:1079-1500) for one replicate."""
    order = Sort_Chromosomes(genome)
    nchrom = len(order)
    data = HaplotypeData()
    cols = {}
    for tag in ("Bi_Allelic", "M_M", "P_P", "M_P", "P_M"):
        fs = [f for f in bed_files if (tag + ".bed") in f]
        c1, p1, c2, p2, mark = read_pair_files(fs, order, chroms, "allelic")
        cols[tag] = PairColumns(c1, p1, c2, p2, mark, dev)
    sizes = lambda res: [genome[c] // res + 1 for c in order]
    budget = dense_budget_bytes(dev)
    data.sparse_res = [res for res in localRes if _allelic_dense_bytes(sizes(res)) > budget]
    dense_res = [res for res in localRes if res not in data.sparse_res]
    # traditional matrices: all five classes together (:1081-1094)
    allp = _all_pairs(cols, dev)
    data.tra_whole, data.tra_local = bin_traditional(allp, genome, wholeRes, dense_res, dev, budget=1 << 62)   # the correction reads dense tiles
    del allp
    if data.sparse_res:
        data.cols = cols
        for res in data.sparse_res:
            _bin_haplotype_sparse(data, cols, genome, res, dev)
    for res in dense_res:
        # haplotype local matrices live in one batch: M chromosomes then P chromosomes
        un = DenseBatch(sizes(res) + sizes(res), dev)
        for hap, tag in ((0, "M_M"), (1, "P_P")):
            view = _sub_batch(un, hap * nchrom, nchrom)
            kernels.bin_pairs_local(cols[tag], res, view, _abi.HC_BIN_SYM_BOTH)          # :1153-1161
        imp = DenseBatch(un.sizes, dev)
        imp.buf.copy_(un.buf)                                                             # deepcopy :1255-1256
        for hap, tag in ((0, "M_M"), (1, "P_P")):
            view = _sub_batch(imp, hap * nchrom, nchrom)
            kernels.bin_pairs_local(cols[tag], res, view, _abi.HC_BIN_ONESIDED)           # :1295-1301
        data.un_local[res], data.imp_local[res] = un, imp
    starts, un_w, imp_w = {}, {}, {}
    for res in wholeRes:
        hb, htot = _bins_from_genome(genome, res, [("M" + c, c) for c in order] + [("P" + c, c) for c in order])
        sm = _start_table(hb, ["M" + c for c in order], dev)
        sp = _start_table(hb, ["P" + c for c in order], dev)
        un = DenseBatch([htot], dev)
        kernels.bin_pairs_whole(cols["M_M"], res, sm, sm, un, _abi.HC_BIN_SYM_BOTH)       # :1144-1151
        kernels.bin_pairs_whole(cols["P_P"], res, sp, sp, un, _abi.HC_BIN_SYM_BOTH)       # :1182-1189
        kernels.bin_pairs_whole(cols["M_P"], res, sm, sp, un, _abi.HC_BIN_SYM_ALL)        # :1217-1221
        kernels.bin_pairs_whole(cols["P_M"], res, sp, sm, un, _abi.HC_BIN_SYM_ALL)        # :1239-1243
        imp = DenseBatch([htot], dev)
        imp.buf.copy_(un.buf)
        kernels.bin_pairs_whole(cols["M_M"], res, sm, sm, imp, _abi.HC_BIN_ONESIDED)      # :1285-1293 (cis)
        kernels.bin_pairs_whole(cols["P_P"], res, sp, sp, imp, _abi.HC_BIN_ONESIDED)      # :1399-1407 (cis)
        data.un_whole[res], data.imp_whole[res] = (hb, un), (hb, imp)
        data.hap_bins[res] = hb
        starts[res], un_w[res], imp_w[res] = (sm, sp), un, imp
    # inter-chromosomal one-sided contacts: neighbourhood vote on the un-imputed matrix (:1302-1378, :1416-1492)
    impute_inter_chromosomal(un_w, imp_w, cols["M_M"], cols["P_P"], starts, wholeRes, *imputation)
    return data


def _allelic_dense_bytes(sizes) -> int:
    """Dense working set of one local resolution in allelic mode: the traditional tiles, the un-imputed and imputed
    maternal and paternal tiles, and the float64 corrected maternal and paternal matrices."""
    return 5 * _dense_bytes(sizes) + 16 * sum(n * n for n in sizes)


def _all_pairs(cols, dev):
    """the five allelic classes as one set of pairs (the traditional matrix, matrixBuilding.py:1081-1094)"""
    return PairColumns(*(torch.cat([getattr(cols[t], a) for t in cols]) for a in ("c1", "p1", "c2", "p2")), device=dev)


def _bin_haplotype_sparse(data: HaplotypeData, cols, genome, res, dev):
    """One local resolution through the sort path, for a dense working set beyond ``dense_budget_bytes``: T as the
    cis CSR of the traditional binning, the un-imputed (Both pairs, symmetric) and imputed (Both pairs plus the
    one-sided ones, asymmetric, with its transpose) haplotype matrices as CSRs over the concatenated haplotype bins in
    the order of the dense batch: all M chromosomes, then all P chromosomes."""
    order = Sort_Chromosomes(genome)
    bins, csr = bin_traditional_sparse(_all_pairs(cols, dev), genome, res, cis_only=True, device=dev)
    data.tra_local[res] = CisCsr(csr, bins, order)
    hap_order = ["M" + c for c in order] + ["P" + c for c in order]
    hb, htot = _bins_from_genome(genome, res, [(h, h[1:]) for h in hap_order])
    chrom_bins = torch.tensor([genome[c] // res + 1 for c in order], dtype=torch.int32, device=dev)
    parts = [(cols["M_M"], _start_table(hb, hap_order[:len(order)], dev)),
             (cols["P_P"], _start_table(hb, hap_order[len(order):], dev))]
    data.un_local[res] = CisCsr(kernels.pairs_to_directed_csr(parts, res, chrom_bins, htot, False, False), hb, hap_order)
    data.imp_local[res] = CisCsr(kernels.pairs_to_directed_csr(parts, res, chrom_bins, htot, True, True), hb, hap_order)


def _sub_batch(batch: DenseBatch, first: int, count: int) -> DenseBatch:
    """A view of ``count`` consecutive matrices of a batch (shares the buffer)."""
    sub = DenseBatch.__new__(DenseBatch)
    sub.sizes = batch.sizes[first:first + count]
    sub.lds = batch.lds[first:first + count]
    sub.offsets = batch.offsets[first:first + count]
    sub.buf = batch.buf
    sub.numel = batch.numel
    sub.device = batch.device
    sub.mat_off = batch.mat_off[first:first + count]
    sub.mat_n = batch.mat_n[first:first + count]
    sub.mat_ld = batch.mat_ld[first:first + count]
    bo = np.concatenate([[0], np.cumsum(sub.sizes)]).astype(np.int64)
    sub.h_bin_off = bo
    sub.bin_off = torch.from_numpy(bo).to(batch.device)
    import ctypes as C
    sub.h_mat_n = (C.c_int32 * len(sub.sizes))(*sub.sizes)
    sub.nbins = int(bo[-1])
    return sub


def _haplotype_outputs(OutPath, prefix, genome, data: HaplotypeData, wholeRes, localRes):
    """Correction + stores of HaplotypeMatrixBuilding (matrixBuilding.py:1502-1638).  ``nor_local[res]`` holds float64
    device matrices for a dense resolution and the upper-triangle records for a sparse one."""
    order = Sort_Chromosomes(genome)
    nchrom = len(order)
    hap_order = ["M" + c for c in order] + ["P" + c for c in order]
    _say("    Traditional Matrix starting ...")
    tra = _store_traditional(os.path.join(OutPath, prefix + "Traditional_Multi.npz"), genome, data.tra_whole,
                             data.tra_local)
    _say("    ICE Balance for Traditional Matrix ...")
    _balance(tra, data.tra_whole, data.tra_local, wholeRes, localRes)
    tra.save()
    with open(os.path.join(OutPath, "Hap_genomeSize"), "w") as out:                      # :1551-1564
        for c in genome:
            out.write("M%s\t%d\n" % (c, genome[c]))
            out.write("P%s\t%d\n" % (c, genome[c]))
    _say("    UnImputated Matrix start ...")
    un = MatrixStore(os.path.join(OutPath, prefix + "UnImputated_Haplotype_Multi.npz"))
    for res in wholeRes:
        hb, W = data.un_whole[res]
        un.add(res, WholeMatrixToSparseDict(hb, W), hb)
    for res in localRes:
        L = data.un_local[res]
        if isinstance(L, CisCsr):
            un.add(res, L.records())
            continue
        recs, _ = kernels.dense_batch_triu_records(L)
        un.add(res, {k: recs[i].copy() for i, k in enumerate(hap_order)})
    un.save()
    _say("    Two-Step balancing for Imputated Matrix ...")
    imp = MatrixStore(os.path.join(OutPath, prefix + "Imputated_Haplotype_Multi.npz"))
    nor_whole, nor_local, gap_local = {}, {}, {}
    for res in wholeRes:
        bins, T = data.tra_whole[res]
        hb, H = data.imp_whole[res]
        nor_whole[res] = GenomeWideMatrixCorrection(bins, hb, T, H)                       # :1601-1605
        imp.add(res, WholeMatrixToSparseDict_float(hb, nor_whole[res]), hb)
    for res in localRes:
        T, H = data.tra_local[res], data.imp_local[res]
        if isinstance(H, CisCsr):                   # sparse: the corrected matrices come out as their upper-triangle records
            recs, gl = kernels.twostep_csr_batch(T.csr, T.off, H.csr, H.off)
            nor_local[res] = dict(zip(hap_order, recs))
            gap_local[str(res)] = dict(zip(hap_order, gl))
            imp.add(res, nor_local[res])
            continue
        mats, gl = kernels.twostep_batch(T, H)                                            # :1031-1039, one call
        nor = {("M" if k < nchrom else "P") + order[k % nchrom]: mats[k] for k in range(2 * nchrom)}
        gaps = {("M" if k < nchrom else "P") + order[k % nchrom]: gl[k] for k in range(2 * nchrom)}
        nor_local[res], gap_local[str(res)] = nor, gaps
        imp.add(res, IntraMatrixToSparseDict(nor))
    np.savez(os.path.join(OutPath, prefix + "Imputated_Gap.npz"), **gap_local)            # :1616-1617
    imp.save()
    _say("    Done !!")
    return nor_whole, nor_local, gap_local


def WholeMatrixToSparseDict_float(Bins, Matrix):
    """``WholeMatrixToSparseDict`` (matrixBuilding.py:457-506) for a float64 genome-wide matrix
    (the corrected haplotype matrix handed to the cool writer at :1605)."""
    dev = require_cuda()
    t = Matrix if isinstance(Matrix, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(Matrix, dtype=np.float64)).to(dev)
    ld, base = t.stride(0), t.data_ptr()
    chroms = Sort_Chromosomes(Bins.keys())
    out = {}
    for i, ca in enumerate(chroms):
        a0, a1 = Bins[ca][0], Bins[ca][1] + 1
        out[ca] = kernels.dense_nonzero_records(base + 8 * (a0 * ld + a0), ld, a1 - a0, a1 - a0, True, True, t.device)
        for cb in chroms[i + 1:]:
            b0, b1 = Bins[cb][0], Bins[cb][1] + 1
            out[ca + "_" + cb] = kernels.dense_nonzero_records(base + 8 * (a0 * ld + b0), ld, a1 - a0, b1 - b0, False,
                                                               True, t.device)
    return out


def HaplotypeMatrixBuilding(OutPath, BedPath, genomeSize, wholeRes, localRes, Imputation_region=10000000,
                            Imputation_min=2, Imputation_ratio=0.9, chroms=["#", "X"], _return_device=False):
    """matrixBuilding.py:1044-1638 for one replicate.  Returns (prefix, DataSets) like the
    reference (NumPy matrices), inter-chromosomal imputation included (bug for bug, see
    ``matrixBuilding.impute_inter_chromosomal``)."""
    dev = require_cuda()
    files = sorted(i for i in os.listdir(BedPath)
                   if any((t + ".bed") in i for t in ("Bi_Allelic", "M_M", "M_P", "P_P", "P_M")))
    if not files:
        raise Exception("Missing file Bi_Allelic.bed in %s" % BedPath)
    prefix = files[0].split("Valid")[0]
    _say("Matrix Construction for %s " % prefix)
    if len(files) != 5:
        ok, tag = Check_Bed(files)
        if not ok:
            raise Exception("Missing file %s.bed in %s" % (tag, BedPath))            # :1075
    files = [os.path.join(BedPath, f) for f in files]
    genome = Load_Genome(genomeSize, chroms)
    data = _haplotype_counts(files, genome, wholeRes, localRes, chroms, dev,
                             (Imputation_region, Imputation_min, Imputation_ratio))
    _haplotype_outputs(OutPath, prefix, genome, data, wholeRes, localRes)
    if _return_device:
        return prefix, data
    return prefix, data.to_datasets(Sort_Chromosomes(genome))


def HaplotypeMatrixConstruction(OutPath, RepPath, genomeSize, wholeRes, localRes, Imputation_region=10000000,
                                Imputation_min=2, Imputation_ratio=0.9, chroms=["#", "X"]):
    """matrixBuilding.py:1641-1860: per-replicate stores, then the replicate-merged stores
    (dense += of every matrix, :1700-1719) under the ``Merged_`` prefix."""
    _say("Building Replicate Matrix respectively !!!")
    CoolerPath = os.path.join(OutPath, "Cooler")
    os.makedirs(CoolerPath, exist_ok=True)
    genome = Load_Genome(genomeSize, chroms)
    total, rep_cols = None, []
    for rep_p in RepPath:
        _, data = HaplotypeMatrixBuilding(CoolerPath, rep_p, genomeSize, wholeRes, localRes, Imputation_region,
                                          Imputation_min, Imputation_ratio, chroms, _return_device=True)
        rep_cols.append(data.cols)
        if total is None:
            total = data
        else:
            total.add(data)
    if len(RepPath) == 1:
        _say("    No replicates to merge.")
        _say("All Done !!!")
        return
    _say("Merging the Replicates...")
    if total.sparse_res:            # sparse matrices: the merged counts are those of all replicates' pairs binned at once
        dev = require_cuda()
        cols = {t: PairColumns(*(torch.cat([getattr(c[t], a) for c in rep_cols]) for a in ("c1", "p1", "c2", "p2", "mark")),
                               device=dev) for t in rep_cols[0]}
        del rep_cols
        for res in total.sparse_res:
            _bin_haplotype_sparse(total, cols, genome, res, dev)
    _haplotype_outputs(CoolerPath, "Merged_", genome, total, wholeRes, localRes)
    _say("All Done !!!")
