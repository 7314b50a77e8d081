"""The downstream consumers on sparse matrices, measured: hg19 chr1 at C2 density (its share of bench.py's 400 M cis
pairs, ~32.8 M pairs from `synth.cis_pairs`), binned at 10 kb and 5 kb by the sort path
(`bin_traditional_sparse(cis_only=True)`), ICE weights from `ice_balance_sparse`, then the four consumers in the order
CallPeaks / Get_PCA / Get_DI use them: balanced matrix -> distance decay -> O/E -> DI (t-test and chi-square).

Per resolution one JSON line:
  - per CSR kernel: CUDA-event time per launch over --launches launches after a warm-up, on device-resident inputs;
    algorithmic bytes (below), achieved GB/s and share of the 7.7 TB/s HBM peak;
  - per public call (structureFind): wall time including the host canonicalisation and the transfers;
  - nnz, bins, and at 10 kb (--dense, default on) the dense path on `toarray()` with its wall times and whether the
    outputs agree (balanced matrix, O/E and DI bit for bit, distance decay within 1e-9).

Algorithmic bytes (n bins, nnz stored entries, P = radix passes of the distance sort, B = entries in the DI windows):
  balance apply      16 nnz + 16 n   (col + count in, value out; row_ptr and weight per row)
  colnnz              4 nnz +  4 n
  distance sums      key build 12 nnz + 9 n; sort 8 nnz (histogram) + 16 nnz per pass; segmented sum 16 nnz + 8 n
  O/E                20 nnz + 16 n   (col + value in, value out; row_ptr and expected value per row)
  DI                 12 B + 21 n     (row + value of every entry in a window; col_ptr, window, gap flag, result)
The weight / decline gathers and the DI window reads hit L2 (n doubles); they are counted once per row.

Usage: python profiles/consumers_sparse_run.py [--pairs N] [--launches 20] [--window-bp 2000000] [--no-dense] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_PEAK = 7.7e12
HG19_CIS_PAIRS = 400_000_000          # bench.py's C2 workload: cis pairs over chr1-22,X in proportion to length


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines() or ["?, ?"])[0].split(", ")
    return {"gpu": name, "power_limit": power}


def chr1_c2_pairs():
    from hichap_master_b200 import synth
    lens = np.array([synth.HG19[c] for c in [str(i) for i in range(1, 23)] + ["X"]], dtype=np.float64)
    return int(np.floor(HG19_CIS_PAIRS * lens[0] / lens.sum()))


def sort_passes(nnz, n):
    idx_bits = max(int(nnz) - 1, 0).bit_length()
    return (int(n).bit_length() + 7) // 8 if nnz > 1 else 0, idx_bits


def kernel_bytes(nnz, n, window_entries):
    passes, _ = sort_passes(nnz, n)
    return {"balance_apply": 16 * nnz + 16 * n, "colnnz": 4 * nnz + 4 * n,
            "distance_sums": (12 * nnz + 9 * n) + (8 * nnz + 16 * nnz * passes) + (16 * nnz + 8 * n),
            "observed_expected": 20 * nnz + 16 * n, "di_ttest": 12 * window_entries + 21 * n,
            "di_chitest": 12 * window_entries + 21 * n}


def window_entries(C, gap, window):
    """stored entries (i, j), |i - j| <= window[j], of the columns Get_DI evaluates"""
    n = C.shape[0]
    cols = np.repeat(np.arange(n), np.diff(C.indptr))
    w = window[cols]
    ok = (np.abs(C.indices - cols) <= w) & ~gap[cols] & (cols >= w) & (cols <= n - w - 1) & (w >= 1)
    return int(ok.sum())


def time_launches(fn, launches):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(launches):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / launches


def wall(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3, out


def kernels_on_device(M_i32, w, cM, decline, gap_idx, window, launches):
    """CUDA-event time per launch of each CSR kernel on device-resident canonical inputs"""
    from hichap_master_b200 import _abi
    from hichap_master_b200.device import ptr, stream_ptr
    from hichap_master_b200.kernels import GenCsr
    from hichap_master_b200.matrixBuilding import _device_csr
    lib, chk = _abi.lib(), _abi.check
    ci = _device_csr(M_i32, GenCsr)
    cf = _device_csr(cM, GenCsr, np.float64)
    cc = _device_csr(cM.T, GenCsr, np.float64)
    dev, n = cf.device, cf.nbins
    w = torch.from_numpy(np.ascontiguousarray(w, dtype=np.float64)).to(dev)
    out_i = torch.empty(max(ci.nnz, 1), dtype=torch.float64, device=dev)
    out_f = torch.empty(max(cf.nnz, 1), dtype=torch.float64, device=dev)
    nz = torch.empty(n, dtype=torch.int32, device=dev)
    gf = np.zeros(n, np.uint8); gf[gap_idx] = 1
    gf = torch.from_numpy(gf).to(dev)
    dsum = torch.empty(n, dtype=torch.float64, device=dev)
    work = torch.empty(int(lib.hc_distance_sums_csr_work_bytes(cf.nnz)), dtype=torch.uint8, device=dev)
    d = torch.from_numpy(np.ascontiguousarray(decline, dtype=np.float64)).to(dev)
    wb = torch.from_numpy(np.ascontiguousarray(window, dtype=np.int32)).to(dev)
    di = torch.empty(n, dtype=torch.float64, device=dev)
    s = stream_ptr()
    calls = {
        "balance_apply": lambda: chk(lib.hc_balance_apply_csr_i32(ptr(ci.row_ptr), ptr(ci.col), ptr(ci.cnt), n, ptr(w),
                                                                  ptr(out_i), s), "balance"),
        "colnnz": lambda: chk(lib.hc_colnnz_csr(ptr(cf.col), cf.nnz, n, ptr(nz), s), "colnnz"),
        "distance_sums": lambda: chk(lib.hc_distance_sums_csr_f64(ptr(cf.row_ptr), ptr(cf.col), ptr(cf.cnt), cf.nnz, n, ptr(gf),
                                                                  ptr(dsum), ptr(work), s), "dsum"),
        "observed_expected": lambda: chk(lib.hc_observed_expected_csr_f64(ptr(cf.row_ptr), ptr(cf.col), ptr(cf.cnt), n, ptr(d),
                                                                          ptr(out_f), s), "oe"),
        "di_ttest": lambda: chk(lib.hc_directionality_index_csc_f64(ptr(cc.row_ptr), ptr(cc.col), ptr(cc.cnt), n, ptr(gf), ptr(wb),
                                                                    0, ptr(di), s), "di"),
        "di_chitest": lambda: chk(lib.hc_directionality_index_csc_f64(ptr(cc.row_ptr), ptr(cc.col), ptr(cc.cnt), n, ptr(gf),
                                                                      ptr(wb), 1, ptr(di), s), "di"),
    }
    ms = {k: time_launches(f, launches) for k, f in calls.items()}
    # the distance sums twice more: bit-identical from one call to the next
    r = []
    for _ in range(2):
        calls["distance_sums"]()
        r.append(dsum.cpu().numpy().copy())
    return ms, bool(np.array_equal(r[0], r[1])), ci.nnz, cf.nnz


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=None, help="chr1 cis pairs (default: its share of C2's 400 M)")
    ap.add_argument("--launches", type=int, default=20)
    ap.add_argument("--window-bp", type=int, default=2_000_000, help="DI window in bp (window_bin = window-bp // res for every bin)")
    ap.add_argument("--no-dense", action="store_true", help="skip the dense comparison at 10 kb")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.launches < 20:
        ap.error("--launches must be at least 20")
    pairs = args.pairs if args.pairs is not None else chr1_c2_pairs()

    from hichap_master_b200 import matrixBuilding as mb, structureFind as sf, synth
    from hichap_master_b200.device import PairColumns, require_cuda
    dev = require_cuda()
    info = gpu_info()
    L = synth.HG19["1"]
    p1, p2 = synth.cis_pairs("1", L, pairs, seed=1)
    z = np.zeros(p1.size, np.int32)
    P = PairColumns(z, p1, z, p2, device=dev)
    wbins, wcsr = mb.bin_traditional_sparse(PairColumns(z[:100000], p1[:100000], z[:100000], p2[:100000], device=dev),
                                            {"1": L}, 100000, cis_only=True, device=dev)
    warm = mb.CisCsr(wcsr, wbins, ["1"]).matrices()["1"]
    wc = sf.balanced_matrix(warm, np.ones(warm.shape[0]))       # first launches and library set-up, untimed
    sf.Get_DI(wc, [], np.full(warm.shape[0], 3), "ttest")
    sf.Observed_Expected(wc, sf.Distance_Decay(wc)[0])
    lines = []
    for res in (10000, 5000):
        bins, csr = mb.bin_traditional_sparse(P, {"1": L}, res, cis_only=True, device=dev)
        w, _ = mb.ice_balance_sparse(csr, bins, cis_only=True)
        M = mb.CisCsr(csr, bins, ["1"]).matrices()["1"]
        n = M.shape[0]
        window = np.full(n, args.window_bp // res, dtype=np.int32)
        row = dict(info, workload="hg19 chr1, %d synthetic cis pairs (C2 density), %d bp, sparse consumers" % (pairs, res),
                   res=res, bins=n, pairs=pairs, window_bins=int(window[0]))
        t = {}
        t["balanced_matrix_ms"], cM = wall(lambda: sf.balanced_matrix(M, w))
        t["distance_decay_ms"], (db, G, NG) = wall(lambda: sf.Distance_Decay(cM))
        t["observed_expected_ms"], OE = wall(lambda: sf.Observed_Expected(cM, db.copy()))
        t["di_ttest_ms"], di_t = wall(lambda: sf.Get_DI(cM, G, window, "ttest"))
        t["di_chitest_ms"], di_c = wall(lambda: sf.Get_DI(cM, G, window, "chitest"))
        row["public_call_wall_ms"] = t
        row["gap_columns"] = int(G.size)
        decline = db.copy()
        decline[decline == 0] = decline[np.nonzero(decline)].min()
        gap = np.zeros(n, bool); gap[G] = True
        ms, dsum_repeatable, ci_nnz, nnz = kernels_on_device(M, w, cM, decline, G, window, args.launches)
        row["nnz"] = {"counts": ci_nnz, "balanced": nnz}
        passes, idx_bits = sort_passes(nnz, n)
        row["distance_sort"] = {"passes": passes, "key_bits": idx_bits + int(n).bit_length()}
        be = window_entries(cM.tocsc(), gap, window)
        nbytes = kernel_bytes(nnz, n, be)
        nbytes["balance_apply"] = 16 * ci_nnz + 16 * n
        row["kernels"] = {k: {"ms_per_launch": v, "launches": args.launches, "algorithmic_bytes": nbytes[k],
                              "GBps": nbytes[k] / (v * 1e6), "share_of_hbm_peak": nbytes[k] / (v * 1e-3) / HBM_PEAK}
                          for k, v in ms.items()}
        row["distance_sums_bit_identical_across_calls"] = dsum_repeatable
        if res == 10000 and not args.no_dense:
            row["dense"] = dense_check(sf, M, w, window, cM, db, G, NG, OE, di_t, di_c)
        line = json.dumps(row)
        print(line, flush=True)
        lines.append(line)
        del cM, OE, M, csr
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


def same_at_pattern(D, S):
    """the dense matrix D has exactly the non-zeros of the canonical CSR S, with the same values"""
    r = np.repeat(np.arange(S.shape[0]), np.diff(S.indptr))
    return bool(np.count_nonzero(D) == S.nnz and np.array_equal(D[r, S.indices], S.data))


def dense_check(sf, M, w, window, cM, db, G, NG, OE, di_t, di_c):
    """the dense consumers on the densified chromosome: wall times and agreement with the sparse outputs"""
    D = M.toarray()
    t = {}
    t["balanced_matrix_ms"], dcM = wall(lambda: sf.balanced_matrix(D, w))
    del D
    ok_b = same_at_pattern(dcM, cM)
    t["distance_decay_ms"], (ddb, dG, dNG) = wall(lambda: sf.Distance_Decay(dcM))
    ok_d = bool(np.array_equal(G, dG) and np.array_equal(NG, dNG) and np.allclose(db, ddb, rtol=1e-9, atol=0))
    rel = float(np.max(np.abs(db - ddb) / np.where(ddb != 0, np.abs(ddb), 1.0)))
    t["observed_expected_ms"], dOE = wall(lambda: sf.Observed_Expected(dcM, db.copy()))
    ok_o = same_at_pattern(dOE, OE)
    del dOE
    t["di_ttest_ms"], ddt = wall(lambda: sf.Get_DI(dcM, G, window, "ttest"))
    t["di_chitest_ms"], ddc = wall(lambda: sf.Get_DI(dcM, G, window, "chitest"))
    ok_i = bool(np.array_equal(di_t, ddt, equal_nan=True) and np.array_equal(di_c, ddc, equal_nan=True))
    return {"public_call_wall_ms": t, "balanced_equal": ok_b, "distance_decay_close": ok_d, "distance_decay_max_rel": rel,
            "observed_expected_equal": ok_o, "di_equal": ok_i, "agree": ok_b and ok_d and ok_o and ok_i}


if __name__ == "__main__":
    main()
