"""Multi-GPU plumbing (one process per GPU, torch.distributed over NCCL for setup and data
exchange; the per-iteration allreduce inside the ICE loop is issued by the library itself on
the compute stream -- see hc_ice_csr_balance).

Genome-wide matrices are row-block sharded (SURVEY.md section 8e): every rank bins the pairs it
was handed into sorted keys, the ranks agree on row boundaries with ~equal numbers of stored
entries, exchange keys so that each rank owns the complete rows of its block, and reduce them
into a local symmetric CSR.  ICE then needs exactly one allreduce of the marginal vector per
iteration.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.distributed as dist

from . import kernels
from .device import PairColumns


def nccl_comm_from_process_group(device) -> int:
    """A NCCL communicator for the library's in-loop allreduce, bootstrapped through the
    existing torch.distributed process group (rank 0's unique id is broadcast)."""
    rank, world = dist.get_rank(), dist.get_world_size()
    uid = torch.zeros(128, dtype=torch.uint8)
    if rank == 0:
        uid = torch.frombuffer(bytearray(kernels.nccl_unique_id()), dtype=torch.uint8).clone()
    backend = dist.get_backend()
    buf = uid.to(device) if backend == "nccl" else uid
    dist.broadcast(buf, src=0)
    return kernels.nccl_comm_init(bytes(buf.cpu().numpy().tobytes()), world, rank)


def row_cuts_from_counts(row_counts: np.ndarray, world: int):
    """Row boundaries (world+1) giving every rank ~the same number of stored entries."""
    from .shard import row_block_splits
    row_ptr = np.concatenate([[0], np.cumsum(row_counts, dtype=np.int64)])
    return row_block_splits(row_ptr, world)


def exchange_plan(sorted_rows_hist_local: np.ndarray, cuts):
    """Number of local keys destined to each rank, given the local per-row key counts."""
    c = np.concatenate([[0], np.cumsum(sorted_rows_hist_local, dtype=np.int64)])
    return [int(c[cuts[r + 1]] - c[cuts[r]]) for r in range(len(cuts) - 1)]


def exchange_entry_lists(up, lo, nbins: int):
    """Collective.  ``up`` / ``lo``: this rank's reduced upper and lower entry lists (int64, each ordered by row).
    The ranks agree on row boundaries with ~equal numbers of cells and every entry is sent to the owner of its row.
    Returns (inbox = [upper runs of every rank | lower runs of every rank], cuts).  Works on any backend (the host
    logic is covered by a gloo test)."""
    world = dist.get_world_size()
    dev = up.device
    cb, cnt_bits = kernels.key_col_bits(nbins), kernels.entry_cnt_bits(nbins)
    # rows are the top field of an entry: the first entry of every row is a binary search away.  This bookkeeping,
    # used to agree on the row boundaries, is the only torch math on the path.
    edges = torch.arange(nbins + 1, dtype=torch.int64, device=dev) << (cb + cnt_bits)
    pos_up, pos_lo = torch.searchsorted(up, edges), torch.searchsorted(lo, edges)
    hist_up, hist_lo = pos_up[1:] - pos_up[:-1], pos_lo[1:] - pos_lo[:-1]
    # cut on the cells per row (what the owner will store, give or take cells held by several ranks)
    total = hist_up + hist_lo
    dist.all_reduce(total)
    cuts = row_cuts_from_counts(total.cpu().numpy(), world)
    send_up, send_lo = exchange_plan(hist_up.cpu().numpy(), cuts), exchange_plan(hist_lo.cpu().numpy(), cuts)
    send_t = torch.tensor([send_up, send_lo], dtype=torch.int64, device=dev).t().contiguous()      # [dest][up, lo]
    recv_t = torch.empty(world, 2, dtype=torch.int64, device=dev)
    dist.all_to_all_single(recv_t, send_t)
    recv = recv_t.cpu().numpy()
    recv_up, recv_lo = [int(x) for x in recv[:, 0]], [int(x) for x in recv[:, 1]]
    n_in_up, n_in = sum(recv_up), sum(recv_up) + sum(recv_lo)
    inbox = torch.empty(n_in, dtype=torch.int64, device=dev)
    dist.all_to_all_single(inbox[:n_in_up], up.contiguous(), output_split_sizes=recv_up, input_split_sizes=send_up)
    dist.all_to_all_single(inbox[n_in_up:], lo.contiguous(), output_split_sizes=recv_lo, input_split_sizes=send_lo)
    return inbox, cuts


def _build_row_block_csr_two_keys(pairs: PairColumns, res: int, start, chrom_bins, nbins: int, cis_only=False):
    """First version (two keys per pair, keys exchanged unreduced); the fallback on count-field overflow."""
    rank, world = dist.get_rank(), dist.get_world_size()
    dev = pairs.device
    col_bits = kernels.key_col_bits(nbins)
    skeys, _, n_valid = kernels.pairs_to_sorted_keys(pairs, res, start, chrom_bins, nbins, cis_only)
    m = int(n_valid.item())
    skeys = skeys[:m]
    edges = torch.arange(nbins + 1, dtype=torch.int64, device=dev) << col_bits
    pos = torch.searchsorted(skeys, edges)                       # first key with row >= r
    hist = pos[1:] - pos[:-1]
    if m > 1:
        first = torch.ones(m, dtype=torch.int32, device=dev)
        first[1:] = (skeys[1:] != skeys[:-1]).to(torch.int32)
        cd = torch.zeros(m + 1, dtype=torch.int64, device=dev)
        torch.cumsum(first, 0, out=cd[1:])
        del first
        total = cd[pos[1:]] - cd[pos[:-1]]
        del cd
    else:
        total = hist.clone()
    dist.all_reduce(total)
    cuts = row_cuts_from_counts(total.cpu().numpy(), world)
    send = exchange_plan(hist.cpu().numpy(), cuts)
    send_t = torch.tensor(send, dtype=torch.int64, device=dev)
    recv_t = torch.empty(world, dtype=torch.int64, device=dev)
    dist.all_to_all_single(recv_t, send_t)
    recv = [int(x) for x in recv_t.cpu().numpy()]
    inbox = torch.empty(sum(recv), dtype=torch.int64, device=dev)
    dist.all_to_all_single(inbox, skeys.contiguous(), output_split_sizes=recv, input_split_sizes=send)
    merged, free = kernels.sort_keys_u64(inbox, kernels.key_sort_bits(nbins)) if inbox.numel() > 1 else (inbox, None)
    nv = torch.tensor([merged.numel()], dtype=torch.int64, device=dev)
    row0, row1 = cuts[rank], cuts[rank + 1]
    row_ptr, col, cnt = kernels.keys_to_csr(merged, nv, col_bits, row1 - row0, scratch=free, row0=row0)
    return kernels.SymCsr(row_ptr, col, cnt, nbins, row0=row0), cuts


def build_row_block_csr(pairs: PairColumns, res: int, start, chrom_bins, nbins: int, cis_only=False):
    """Collective: returns (SymCsr of this rank's row block, cuts).

    Every rank reduces ITS pairs to unique upper-triangle cells with counts (one 64-bit entry per cell), derives the
    lower-triangle list (same cells, row and col swapped, re-sorted on the row bits), and sends each list's rows to
    their owner; the owner sorts what it received once more and adds the counts of equal cells -- the cells travel
    reduced, and a row's lower and upper parts interleave into CSR order by that one sort."""
    import os
    import time
    rank, world = dist.get_rank(), dist.get_world_size()
    dev = pairs.device
    timing = os.environ.get("HC_DIST_TIMING") == "1"      # per-phase wall times of this rank on stderr (synchronises)
    marks = []

    def mark(what):
        if timing:
            torch.cuda.synchronize(dev)
            marks.append((what, time.perf_counter()))
    mark("start")
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    lists = None
    try:
        lists = kernels.pairs_to_entry_lists(pairs, res, start, chrom_bins, nbins, cis_only)
    except kernels.CountFieldOverflow:
        flag += 1
    dist.all_reduce(flag)                      # all ranks take the same path
    if int(flag.item()):
        del lists
        return _build_row_block_csr_two_keys(pairs, res, start, chrom_bins, nbins, cis_only)
    up, slo, n_lo = lists
    mark("local lists (entries, sort, reduce, lower sort)")
    cb, cnt_bits = kernels.key_col_bits(nbins), kernels.entry_cnt_bits(nbins)
    lo = slo[:int(n_lo.item())]
    inbox, cuts = exchange_entry_lists(up, lo, nbins)
    mark("cuts + exchange")
    del up, lo, slo, lists
    merged, mfree = kernels.sort_entries(inbox, nbins, cnt_bits, 2)
    mark("merge sort of the inbox (%d entries)" % int(inbox.numel()))
    nv = torch.tensor([inbox.numel()], dtype=torch.int64, device=dev)
    try:
        cells = kernels.reduce_entries(merged, nv, nbins, unit=False)
        ok = 0
    except kernels.CountFieldOverflow:
        ok = 1
    flag = torch.tensor([ok], dtype=torch.int32, device=dev)
    dist.all_reduce(flag)
    if int(flag.item()):
        return _build_row_block_csr_two_keys(pairs, res, start, chrom_bins, nbins, cis_only)
    mark("add-counts reduce")
    row0, row1 = cuts[rank], cuts[rank + 1]
    row_ptr, col, cnt = kernels.entries_to_csr(cells, None, None, nbins, row1 - row0, row0=row0, total=int(cells.numel()))
    mark("CSR")
    if timing:
        import sys
        sys.stderr.write("[build_row_block_csr rank %d] " % rank + "; ".join(
            "%s %.2f ms" % (marks[i][0], 1e3 * (marks[i][1] - marks[i - 1][1])) for i in range(1, len(marks))) + "\n")
    return kernels.SymCsr(row_ptr, col, cnt, nbins, row0=row0), cuts
