"""Allelic mode on the CSR path, measured: C3 mix (hg19 chr1-22,X; 86 % bi-allelic, 6 % M_M, 6 % P_P; Both / R1 / R2 =
30 / 35 / 35 %; the generator and seeds of bench.py's C3 section).

  40 kb: dense and sparse on the same inputs in the same process, alternated; both times and the agreement of their
         outputs (gaps exact, corrected records within 1e-6).
  10 kb and 5 kb: sparse only (the dense working set would be 171 GB / 682 GB).

Per configuration one JSON line: binning, ICE of the traditional matrices and two-step times (CUDA events around work
that ends in a device synchronise; the last of `--reps` passes, the first warms up), nnz, peak device memory of the
torch allocator, and the algorithmic bytes of the two-step passes with their share of the HBM peak (7.7 TB/s):

  4 nnz(T) + 28 nnz(X) + 24 nnz(XT) + 24 records + 64 n_H bytes
  (row sums read T's and X's counts; the ROWSUM, TOTAL and EMIT passes each read X and XT (int32 column + int32 count);
  EMIT writes 24-byte records; per haplotype row a few int64 / float64 vectors)

Usage: python profiles/c3_sparse_run.py [--pairs 100000000] [--reps 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_PEAK = 7.7e12


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines() or ["?, ?"])[0].split(", ")
    return {"gpu": name, "power_limit": power}


def c3_pairs(genome, order, n, dev):
    from hichap_master_b200 import synth
    from hichap_master_b200.device import PairColumns
    c1, p1, c2, p2 = synth.genome_pairs_torch(genome, order, n, 3, dev, trans_frac=0.0)
    g = torch.Generator(device=dev); g.manual_seed(33)
    cls = torch.rand(n, generator=g, device=dev)
    mark = torch.multinomial(torch.tensor([0.30, 0.35, 0.35], device=dev), n, replacement=True, generator=g).to(torch.uint8)
    cols = {}
    for tag, sel in (("Bi_Allelic", (cls < 0.86) | (cls >= 0.98)), ("M_M", (cls >= 0.86) & (cls < 0.92)),
                     ("P_P", (cls >= 0.92) & (cls < 0.98))):
        cols[tag] = PairColumns(c1[sel], p1[sel], c2[sel], p2[sel], mark[sel], device=dev)
    return cols


def ev(fn):
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(); out = fn(); b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b), out


def run_sparse(genome, cols, res, dev):
    from hichap_master_b200 import kernels
    from hichap_master_b200.construction import HaplotypeData, _bin_haplotype_sparse
    from hichap_master_b200.matrixBuilding import ice_balance_sparse
    data = HaplotypeData()
    t = {}
    t["binning_ms"], _ = ev(lambda: _bin_haplotype_sparse(data, cols, genome, res, dev))
    T, H = data.tra_local[res], data.imp_local[res]
    t["ice_traditional_ms"], _ = ev(lambda: ice_balance_sparse(T.csr, T.bins, cis_only=True, ignore_diags=1))
    t["two_step_ms"], (recs, gaps) = ev(lambda: kernels.twostep_csr_batch(T.csr, T.off, H.csr, H.off))
    nnz = {"T": T.csr.nnz, "X": H.csr.nnz, "XT": H.csr.t.nnz, "UnImputated": data.un_local[res].csr.nnz,
           "records": int(sum(r.size for r in recs))}
    return t, nnz, recs, gaps, H.csr.nbins


def run_dense(genome, order, cols, res, dev):
    from hichap_master_b200 import _abi, kernels
    from hichap_master_b200.construction import _all_pairs, _sub_batch
    from hichap_master_b200.device import DenseBatch
    nchrom = len(order)
    sizes = [genome[c] // res + 1 for c in order]
    allp = _all_pairs(cols, dev)
    T, H = DenseBatch(sizes, dev), DenseBatch(sizes + sizes, dev)

    def bin_all():
        kernels.bin_pairs_local_banded(allp, res, T)
        for k, tag in enumerate(("M_M", "P_P")):
            v = _sub_batch(H, k * nchrom, nchrom)
            kernels.bin_pairs_local(cols[tag], res, v, _abi.HC_BIN_SYM_BOTH)
            kernels.bin_pairs_local(cols[tag], res, v, _abi.HC_BIN_ONESIDED)
    t = {}
    t["binning_ms"], _ = ev(bin_all)
    t["ice_traditional_ms"], _ = ev(lambda: kernels.ice_balance_dense(T, None, ignore_diags=1))
    t["two_step_ms"], (mats, gaps) = ev(lambda: kernels.twostep_batch(T, H))
    recs = [kernels.dense_nonzero_records(m.data_ptr(), m.stride(0), m.shape[0], m.shape[0], True, True, dev) for m in mats]
    return t, recs, gaps


def agree(recs_a, gaps_a, recs_b, gaps_b):
    gaps_ok = all(np.array_equal(np.asarray(a, np.int64), np.asarray(b, np.int64)) for a, b in zip(gaps_a, gaps_b))
    bins_ok = all(np.array_equal(a["bin1"], b["bin1"]) and np.array_equal(a["bin2"], b["bin2"]) for a, b in zip(recs_a, recs_b))
    rel = max((float(np.max(np.abs(a["IF"] - b["IF"]) / np.abs(b["IF"]))) if a.size else 0.0)
              for a, b in zip(recs_a, recs_b)) if bins_ok else None
    return {"gaps_equal": gaps_ok, "records_bins_equal": bins_ok, "max_rel_diff_IF": rel, "agree": bool(gaps_ok and bins_ok and rel < 1e-6)}


def two_step_bytes(nnz, n_h):
    return 4 * nnz["T"] + 28 * nnz["X"] + 24 * nnz["XT"] + 24 * nnz["records"] + 64 * n_h


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=100_000_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from hichap_master_b200 import synth
    from hichap_master_b200.construction import _allelic_dense_bytes
    from hichap_master_b200.device import require_cuda
    dev = require_cuda()
    info = gpu_info()
    genome = {c: l for c, l in synth.HG19.items() if c not in ("Y", "M")}
    order = [str(i) for i in range(1, 23)] + ["X"]
    cols = c3_pairs(genome, order, args.pairs, dev)
    lines = []
    for res in (40000, 10000, 5000):
        row = dict(info, workload="C3 allelic, %d pairs, local %d bp" % (args.pairs, res), res=res,
                   dense_working_set_gb=_allelic_dense_bytes([genome[c] // res + 1 for c in order]) / 1e9)
        hist = {"sparse": [], "dense": []}
        for _ in range(args.reps):
            if res == 40000:
                torch.cuda.empty_cache(); torch.cuda.reset_peak_memory_stats(dev)
                td, rd, gd = run_dense(genome, order, cols, res, dev)
                hist["dense"].append(td)
                row["dense_peak_mem_gb"] = torch.cuda.max_memory_allocated(dev) / 1e9
            torch.cuda.empty_cache(); torch.cuda.reset_peak_memory_stats(dev)
            ts, nnz, rs, gs, n_h = run_sparse(genome, cols, res, dev)
            hist["sparse"].append(ts)
            row["sparse_peak_mem_gb"] = torch.cuda.max_memory_allocated(dev) / 1e9
        row["sparse"] = hist["sparse"][-1]
        row["sparse_all_reps"] = hist["sparse"]
        row["nnz"] = nnz
        b = two_step_bytes(nnz, n_h)
        row["two_step_roofline"] = {"algorithmic_bytes": b, "achieved_GBps": b / (row["sparse"]["two_step_ms"] * 1e6),
                                    "share_of_hbm_peak": b / (row["sparse"]["two_step_ms"] * 1e-3) / HBM_PEAK}
        if res == 40000:
            row["dense"] = hist["dense"][-1]
            row["dense_all_reps"] = hist["dense"]
            row["outputs"] = agree(rs, gs, rd, gd)
            del rd, gd
        del rs, gs
        line = json.dumps(row)
        print(line, flush=True)
        lines.append(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
