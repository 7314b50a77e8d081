#!/usr/bin/env python
"""bench.py -- the matrix-stage hot path.

Headline (BASELINE.json configs[1], "C2"): hg19 chr1-22,X intra-chromosomal matrices at 40 kb from
synthetic cis valid pairs, binned on the GPU and ICE-balanced (`cooler balance --ignore-diags 1
--cis-only` semantics) to convergence.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--pairs P] [--impl ours|reference] [--dump-outputs DIR]

One "step" = zero the dense tiles, bin all pairs, run the bin filters and iterate every chromosome to
convergence.  `value` = device-resident step time (ms, lower is better); `e2e` = the same through the
host-facing call: pinned host columns -> HBM, the step, the upper-triangular records and the weight
vector back to the host.  N > 1: chromosomes are LPT-sharded over ranks (no collective on the data
path); time = max over ranks.

The same JSON line also carries
  parity_check      the GPU matrices / weights of two chromosomes of THIS run against the CPU oracle on the
                    same pairs (counts bit-exact, NaN mask and iteration count equal, weights <= 1e-6);
  cpu_baseline      (N = 1) that oracle computation, timed on one host core;
  roofline          the dominant kernel (fused ICE iteration) + roofline_secondary (binning, two-step);
  c4                BASELINE.json configs[3]: hg19 genome-wide 10 kb (303 641 bins, 1 G pairs), sort path ->
                    row-block sharded symmetric CSR -> ICE with one NCCL allreduce per iteration, at the
                    same N, with its own roofline (SURVEY's 8Z + 24n bytes per iteration) and, at every N,
                    a sharded-vs-oracle parity check run in-process.

`--impl reference` times the reference's CPU path (the oracle port: the Python-2 reference cannot be
installed) on the FULL C2 workload over all host cores -- nothing is extrapolated.

`--dump-outputs DIR` writes what the last timed step returned as .npy files (see `dump_outputs`).  The
inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

RES = 40000
METRIC = "matrix_stage_time_to_ice_convergence"
UNIT = "ms"
RTOL = 1e-6        # north_star: bias vectors within 1e-6 relative


def c2_genome():
    from hichap_master_b200 import synth
    g = {c: l for c, l in synth.HG19.items() if c not in ("Y", "M")}
    order = [str(i) for i in range(1, 23)] + ["X"]
    return g, order


def pair_shares(genome, order, total):
    lens = np.array([genome[c] for c in order], dtype=np.float64)
    share = np.floor(total * lens / lens.sum()).astype(np.int64)
    share[0] += total - share.sum()
    return share


def workload_name(pairs):
    return ("C2: hg19 chr1-22,X intra-chromosomal 40 kb matrices, %d synthetic cis valid pairs, "
            "binning + cis-only ICE (ignore_diags=1, cooler defaults) to convergence" % pairs)


def workload_config(pairs):
    """Keys shared by both arms (the driver compares them)."""
    genome, order = c2_genome()
    return {"workload": workload_name(pairs), "pairs": int(pairs),
            "bins": int(sum(genome[c] // RES + 1 for c in order)), "resolution": RES, "chromosomes": len(order)}


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


# ------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.tmp = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=self.tmp, stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.tmp.flush()
        rows = [r.strip().split(", ") for r in open(self.tmp.name) if r.strip()]
        os.unlink(self.tmp.name)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for nm, v in zip(names, r[5:9]):
                if v.strip().lower() == "active":
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        busy = [s for s in sm if s > 0.5 * max(sm)] or sm
        return {"sm_mhz": float(np.median(busy)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------
# CPU oracle on one chromosome (the only place bench.py executes oracle/): used as the checker of
# `parity_check`, as `cpu_baseline`, and by the reference arm
# ------------------------------------------------------------------------------------------
def _cpu_one_chrom(job, keep=False):
    """oracle port on one chromosome: bin (NumPy restatement of matrixBuilding.py:595-603), upper-triangular
    records (:515-521), cis-only ICE restatement (cooler balance)"""
    from oracle import cooler_ice, hichap_oracle as ho
    c, length, p1, p2 = job
    if isinstance(p1, str):
        p1, p2 = np.load(p1, mmap_mode="r"), np.load(p2, mmap_mode="r")
        p1, p2 = np.asarray(p1), np.asarray(p2)
    n = length // RES + 1
    z = np.zeros(p1.size, np.int32)
    t0 = time.perf_counter()
    M = ho.bin_local_dense(z, p1, z, p2, [n], RES)[0]
    rec = ho.dense_to_triu_records(M)
    t1 = time.perf_counter()
    w, st = cooler_ice.balance(rec["bin1"], rec["bin2"], rec["IF"].astype(np.int32), n, [0, n], cis_only=True)
    t2 = time.perf_counter()
    out = dict(chrom=c, bin_s=t1 - t0, ice_s=t2 - t1, iters=int(st["iters"][0]), nnz=int(rec.size), pairs=int(p1.size))
    if keep:
        out.update(M=M, w=w)
    return out


def parity_and_cpu_baseline(sample, stage, out, sizes, pairs_total, world):
    """sample: [(local index, chrom name, length, p1 host, p2 host)].  Runs the oracle on exactly the pairs the
    GPU binned for these chromosomes and compares; its time is the single-core CPU baseline."""
    off = stage.batch.h_bin_off
    w_gpu = out["bias"].cpu().numpy()
    iters_gpu = out["results"]["iters"]
    checks, per, t_all = [], [], time.perf_counter()
    for li, c, length, a, b in sample:
        r = _cpu_one_chrom((c, length, a, b), keep=True)
        Mg = stage.batch.to_numpy(li)
        wg, wr = w_gpu[off[li]:off[li + 1]], r["w"]
        good = ~np.isnan(wr)
        err = float(np.max(np.abs(wg[good] - wr[good]) / np.abs(wr[good]))) if good.any() else 0.0
        checks.append({"chrom": c, "bins": int(sizes[li]), "pairs": r["pairs"], "counts_equal": bool(np.array_equal(Mg, r["M"])),
                       "nan_mask_equal": bool(np.array_equal(np.isnan(wg), np.isnan(wr))),
                       "iters_gpu": int(iters_gpu[li]), "iters_oracle": r["iters"], "max_rel_err": err})
        per.append({k: r[k] for k in ("chrom", "bin_s", "ice_s", "iters", "nnz", "pairs")})
    wall = time.perf_counter() - t_all
    ok = all(ch["counts_equal"] and ch["nan_mask_equal"] and ch["iters_gpu"] == ch["iters_oracle"] and ch["max_rel_err"] < RTOL
             for ch in checks)
    parity = {"ok": bool(ok), "tolerance": RTOL, "against": "oracle/ (NumPy restatement) on the same pairs", "chromosomes": checks}
    cpu = None
    if world == 1:
        # scale to the full workload: binning by pairs, ICE by nnz x iterations (both known for every chromosome
        # from the GPU run: upper-triangle nnz from the tiles, iteration counts from the results)
        import torch
        bin_s = sum(p["bin_s"] for p in per); ice_s = sum(p["ice_s"] for p in per)
        s_pairs = sum(p["pairs"] for p in per); s_work = sum(p["nnz"] * p["iters"] for p in per)
        nnz_all = []
        for i, n in enumerate(sizes):
            v = stage.batch.view(i)[:, :n]
            nnz_all.append(int((torch.count_nonzero(v).item() + torch.count_nonzero(torch.diagonal(v)).item()) // 2))
        work_all = float(sum(z * int(it) for z, it in zip(nnz_all, iters_gpu)))
        est = bin_s * pairs_total / max(s_pairs, 1) + ice_s * work_all / max(s_work, 1)
        cpu = {"value": est * 1e3, "unit": UNIT, "cores": 1, "kind": "port",
               "sample": ("oracle port (NumPy restatement of matrixBuilding.py:595-603, :515-521 + cooler balance --cis-only) on "
                          "chromosomes %s of THIS run's pairs (%d of %d pairs), %.1f s measured on one core; value = binning time "
                          "x pair ratio (%.1f) + ICE time x (nnz x iterations) ratio (%.1f), both ratios measured on the GPU "
                          "matrices -- a model, not a measurement; `bench.py --impl reference` measures the full workload on all cores"
                          % ("+".join(p["chrom"] for p in per), s_pairs, pairs_total, wall, pairs_total / max(s_pairs, 1),
                             work_all / max(s_work, 1))),
               "measured_s": wall, "per_chrom": per, "host_cores": os.cpu_count()}
    return parity, cpu


DUMP_CELLS = 1 << 21    # matrix cells sampled by --dump-outputs: the int32 tiles of C2 are ~1.2 GB, the sample ~32 MB


def dump_outputs(d, stage, out, rank, world):
    """Write the result of one `LocalStage.run` step as .npy files in `d`, every value finite:
      ice_weights      float64, one weight per bin of every chromosome; 0 = filtered bin (NaN in the weights
                       the step returns; the weight of a kept bin is positive)
      ice_scale, ice_var, ice_iters, ice_converged   float64, one value per chromosome; the scale is 0 where
                       every bin of the chromosome is filtered (NaN in the step's results; the library sets the
                       variance of such a chromosome to 0, so a non-finite variance is a fault and is written as is)
      cells_sampled    float32 (k, 3): chromosome index, row, column of the sampled matrix cells
      counts_sampled   float32 (k,): the binned contact counts of those cells
    The cells are drawn uniformly over all matrix cells with a fixed seed, so the same arguments give the same
    cells.  With several ranks every rank writes the chromosomes it holds, with a `_rank<r>` suffix, and samples
    DUMP_CELLS / ranks cells, so that the dump stays near 33 MB in all."""
    import torch
    os.makedirs(d, exist_ok=True)
    b = stage.batch
    n = np.array(b.sizes, np.int64)
    start = np.concatenate([[0], np.cumsum(n * n)])
    flat = np.unique(np.random.default_rng(20240601).integers(0, start[-1], size=min(DUMP_CELLS // world, int(start[-1]))))
    ci = np.searchsorted(start, flat, side="right") - 1
    row, col = np.divmod(flat - start[ci], n[ci])
    at = np.array(b.offsets, np.int64)[ci] + row * np.array(b.lds, np.int64)[ci] + col
    res = out["results"]
    filtered_as_zero = lambda a: np.where(np.isnan(a), 0.0, a).astype(np.float64)
    arrays = {"ice_weights": filtered_as_zero(out["bias"].cpu().numpy()),
              "ice_scale": filtered_as_zero(res["scale"]), "ice_var": res["var"].astype(np.float64),
              "ice_iters": res["iters"].astype(np.float64), "ice_converged": res["converged"].astype(np.float64),
              "cells_sampled": np.stack([ci, row, col], axis=1).astype(np.float32),
              "counts_sampled": b.buf[torch.from_numpy(at).to(b.device)].cpu().numpy().astype(np.float32)}
    suffix = "_rank%d" % rank if world > 1 else ""
    for name, a in arrays.items():
        np.save(os.path.join(d, name + suffix + ".npy"), a)


# ------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from hichap_master_b200 import _abi, kernels, shard, synth
    from hichap_master_b200.device import PairColumns
    from hichap_master_b200.pipeline import HostPairs, LocalStage

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus or world == 1, "launch with torchrun --nproc-per-node == --gpus"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    peaks = load_peaks()
    peak = float(peaks.get("hbm_gbs", 6650.0))

    genome, order = c2_genome()
    sizes_all = [genome[c] // RES + 1 for c in order]
    shares = pair_shares(genome, order, args.pairs)
    mine = shard.chromosome_shards(sizes_all, world)[rank]
    sizes = [sizes_all[i] for i in mine]

    # ---- synthetic inputs, generated on the device, one seeded stream per chromosome ---------
    # chromosomes the oracle re-computes from this run's pairs (rank 0): the two smallest -- and, on one GPU, the largest as
    # well (chr1: ~15 s on one core), so that the single-core baseline is extrapolated from a cache-unfriendly chromosome
    # too and the in-run parity check covers a full-size matrix
    by_size = sorted(range(len(mine)), key=lambda li: sizes[li])
    sample_li = (by_size[:2] + ([by_size[-1]] if world == 1 and len(by_size) > 2 and not args.no_cpu_baseline else [])) if rank == 0 else []
    sample = []
    cs, p1s, p2s = [], [], []
    for li, gi in enumerate(mine):
        c = order[gi]
        _, a, _, b = synth.genome_pairs_torch({c: genome[c]}, [c], int(shares[gi]), 2000 + gi, dev)
        if li in sample_li:
            sample.append((li, c, genome[c], a.cpu().numpy(), b.cpu().numpy()))
        cs.append(torch.full((a.numel(),), li, dtype=torch.int32, device=dev)); p1s.append(a); p2s.append(b)
    c1 = torch.cat(cs); p1 = torch.cat(p1s); p2 = torch.cat(p2s)
    del cs, p1s, p2s
    g = torch.Generator(device=dev); g.manual_seed(99 + rank)
    perm = torch.randperm(c1.numel(), generator=g, device=dev)
    c1, p1, p2 = c1[perm].contiguous(), p1[perm].contiguous(), p2[perm].contiguous()
    del perm
    n_local = int(c1.numel())
    pairs = PairColumns(c1, p1, c1, p2, device=dev)
    stage = LocalStage(sizes, n_local, dev)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """device time of `steps` calls, max over ranks (ms per step) + last result"""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = None
        for _ in range(steps):
            out = fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1) / steps], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        barrier()
        return float(ms.item()), out

    os.environ.setdefault("HC_ICE_TIME_KERNEL", "1")    # per-launch events around the ICE stream kernel (roofline)
    step = lambda: stage.run(pairs, RES, records=False, weights_to_host=False)
    for _ in range(args.warmup):
        step()
    launches0 = _abi.launch_count()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_step, out = timed(step, args.steps)
    launches = (_abi.launch_count() - launches0) // args.steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, stage, out, rank, world)
    # roofline of the dominant kernel (the fused ICE iteration), from the same timed steps
    iters = out["results"]["iters"].astype(np.int64)
    info = out["info"]
    mode = int(info.packed)            # 3: symmetric blocks, persistent dataflow kernel; 1: full-matrix uint8; 0: int32 tiles
    packed = mode != 0
    # algorithmic bytes of the stream kernel: the matrix once per iteration -- SURVEY 8(d) counts 4 B per cell (int32
    # tiles); the packed encoding streams 1 B per cell + 8 B per overflow cell (col, extra count); the symmetric
    # encoding (default) streams only the 256 x 256 uint8 blocks on or above the diagonal
    cell_iters = float(sum(int(it) * n * n for it, n in zip(iters, sizes)))
    mean_iters = cell_iters / max(float(sum(n * n for n in sizes)), 1.0)
    nblk = [(n + 255) // 256 for n in sizes]
    sym_bytes = [65536.0 * nb * (nb + 1) // 2 for nb in nblk]
    if mode == 3:
        ice_bytes = float(sum(int(it) * b for it, b in zip(iters, sym_bytes))) + 8.0 * float(info.overflow_cells) * mean_iters
        ice_kernel = "sym_ice_kernel"
    elif mode == 1:
        ice_bytes = 1.0 * cell_iters + 8.0 * float(info.overflow_cells) * mean_iters
        ice_kernel = "ice_q8_mma_kernel"
    else:
        ice_bytes = 4.0 * cell_iters
        ice_kernel = "ice_dense_stream_kernel"
    loop_ms = float(info.loop_ms)
    n_iter_launches = int(max(iters)) if len(iters) else 0

    if args.skip_e2e:
        if rank == 0:
            sampler.stop()
            print(json.dumps({"tuning_only": True, "ms_per_step": ms_step, "ice_loop_ms": loop_ms,
                              "ice_GBps": ice_bytes / (loop_ms * 1e6), "ice_launches": n_iter_launches, "ice_kernel": ice_kernel,
                              "stream_full_ms": float(info.stream_full_ms), "stream_full_launches": int(info.stream_full_launches),
                              "pack_ms": float(info.pack_ms), "overflow_cells": int(info.overflow_cells), "iters_max": int(max(iters)),
                              "variant": os.environ.get("HC_ICE_VARIANT"), "item_kb": os.environ.get("HC_ICE_ITEM_KB")}))
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- parity of this very run against the oracle (+ the single-core CPU baseline at N = 1) ----
    parity, cpu = (None, None)
    if rank == 0 and not args.no_cpu_baseline:
        parity, cpu = parity_and_cpu_baseline(sample, stage, out, sizes, args.pairs, world)

    # ---- end to end through the host-facing call ---------------------------------------------
    host = HostPairs(c1.cpu(), p1.cpu(), c1.cpu(), p2.cpu())
    if os.environ.get("HC_E2E_CHUNKED", "1") == "1":     # chunked H2D overlapped with binning (default)
        e2e_step = lambda: stage.run_from_host(host, RES, records=True, weights_to_host=True)
    else:                                                   # A/B: whole-column upload, then the step
        e2e_step = lambda: stage.run(stage.upload(host), RES, records=True, weights_to_host=True)
    for _ in range(max(1, min(args.warmup, 2))):
        o2 = e2e_step()
    e2e_steps = max(1, min(args.steps, 3))
    ms_e2e, o2 = timed(e2e_step, e2e_steps)
    clocks = sampler.stop() if rank == 0 else None
    h2d = torch.tensor([float(host.nbytes)], dtype=torch.float64, device=dev)
    d2h = torch.tensor([float(o2["d2h_bytes"])], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(h2d); dist.all_reduce(d2h)
    del host

    # ---- per-kernel breakdown (rank 0, outside the timed regions) ----------------------------
    def ev_time(fn, reps=3):
        fn(); torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record(); torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    breakdown, secondary = None, []
    if rank == 0:
        t_zero = ev_time(lambda: stage.batch.buf.zero_())
        t_bin = ev_time(lambda: (stage.batch.buf.zero_(), kernels.bin_pairs_local_banded(
            pairs, RES, stage.batch, check_bounds=False, work=stage.bin_work))) - t_zero
        params = kernels.ice_params()
        t_filt = ev_time(lambda: kernels.ice_dense_filters(stage.batch, params))
        sq = float(sum(n * n for n in sizes))
        breakdown = {
            "zero_tiles_ms": t_zero, "binning_ms": t_bin, "ice_filters_ms": t_filt, "ice_pack_ms": float(info.pack_ms),
            "ice_loop_ms": loop_ms, "binning_Gpairs_per_s": n_local / (t_bin * 1e6),
            "ice_iters": [int(i) for i in iters], "ice_iter_launches": n_iter_launches,
        }
        bin_bytes = 16.0 * n_local + 8.0 * sq
        secondary.append({"kernel": "banded binning (bin_pairs_band + band_merge + mirror_upper)", "bound": "hbm / L2 atomics",
                          "algorithmic_bytes": bin_bytes, "formula": "16*P + 8*N^2 (SURVEY 8d dense-tile path)", "ms": t_bin,
                          "achieved": bin_bytes / (t_bin * 1e6), "peak": peak, "unit": "GB/s", "frac": bin_bytes / (t_bin * 1e6) / peak})
        secondary.append({"kernel": "ICE filters (marginals + min_nnz + MAD-max)", "bound": "hbm", "algorithmic_bytes": 4.0 * sq,
                          "formula": "4*N^2", "ms": t_filt, "achieved": 4.0 * sq / (t_filt * 1e6), "peak": peak, "unit": "GB/s",
                          "frac": 4.0 * sq / (t_filt * 1e6) / peak})
    del pairs, c1, p1, p2
    stage_batch_numel = stage.batch.numel
    del stage, out, o2
    torch.cuda.empty_cache()

    c1 = c3 = None
    if rank == 0 and not args.skip_secondary:
        secondary.append(twostep_roofline(dev, peak, ev_time))
        if world == 1:          # the other single-GPU configs of BASELINE.json, at their stated sizes
            c1 = c1_section(dev)
            c3 = c3_section(100_000_000, dev, peak)
            r = c3["two_step_roofline"]
            secondary.append({"kernel": "two-step correction, C3: 23 chromosomes, M and P, one batched call (every pass one launch over "
                                        "the tile pairs of all 46 matrices)", "bound": "hbm", "algorithmic_bytes": r["algorithmic_bytes"],
                              "formula": r["formula"], "ms": c3["two_step_ms"], "achieved": r["achieved"], "peak": peak, "unit": "GB/s",
                              "frac": r["frac"]})
    c4 = None
    if not args.skip_c4:
        c4 = run_c4_section(args, world, rank, dev, peak)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    traffic = None          # dram__bytes_read.sum + dram__bytes_write.sum of one full launch, from the committed ncu capture
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        traffic = float(tj["traffic_bytes_per_launch"]) if world == 1 and str(tj.get("kernel", "")).startswith(ice_kernel) else None
        traffic_note = tj.get("note", "")
    except Exception:
        traffic, traffic_note = None, ""
    loop_achieved = ice_bytes / (loop_ms * 1e6) if loop_ms > 0 else 0.0
    # the stream kernel on its own: the first launch of every graph replay is bracketed by CUDA events inside the graph
    # (HC_ICE_TIME_KERNEL=1) and those with all chromosomes still active are averaged; falls back to the loop-level figure
    sq = float(sum(n * n for n in sizes))
    if mode == 3:       # ONE launch runs every iteration of every chromosome: the launch's bytes are the loop's bytes
        full_bytes, survey_bytes = ice_bytes, 4.0 * cell_iters
    else:
        full_bytes = (1.0 if packed else 4.0) * sq + (8.0 * float(info.overflow_cells) if packed else 0.0)
        survey_bytes = 4.0 * sq      # SURVEY.md 8(d): dense-tile ICE iteration = 4*N^2
    kernel_ms = float(info.stream_full_ms) if int(info.stream_full_launches) > 0 else 0.0
    achieved = full_bytes / (kernel_ms * 1e6) if kernel_ms > 0 else loop_achieved
    launch_ms = kernel_ms if kernel_ms > 0 else loop_ms / max(n_iter_launches, 1)
    cfg = workload_config(args.pairs)
    cfg.update({"parallelism": "chromosomes LPT-sharded by N^2 over %d GPU(s), no collective" % world,
                "host_format": "pinned columns: chromosome uint8 + mid-point int32 per mate (10 B/pair)",
                "l2": "inputs larger than L2 (%.1f GB pair columns, %.2f GB int32 tiles on rank 0)" % (16e-9 * n_local, 4e-9 * stage_batch_numel)})
    line = {
        "metric": METRIC, "value": ms_step, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": False, "scaling": "strong",
        "vs_baseline": None,
        "dtype": "int32 counts (ICE streams them as u8 + overflow list, s32 tensor-core plane sums) / f64 weights" if packed else "int32 counts / f64 weights",
        "ice_mode": {3: "symmetric blocks, persistent dataflow kernel", 1: "full-matrix uint8, one launch pair per iteration", 0: "int32 tiles"}.get(mode),
        "data": "synthetic", "config": cfg,
        "throughput_Mpairs_per_s": args.pairs / (ms_step * 1e3),
        "e2e": {"value": ms_e2e, "unit": UNIT, "h2d_bytes_per_step": int(h2d.item()),
                "d2h_bytes_per_step": int(d2h.item()), "steps": e2e_steps,
                "Mpairs_per_s": args.pairs / (ms_e2e * 1e3)},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "kernel": ice_kernel, "achieved": achieved, "peak": peak,
                     "unit": "GB/s", "frac": achieved / peak, "frac_of_nominal_8TBps": achieved / 8000.0,
                     "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured copy)" if peaks else "fallback 6650",
                     "algorithmic_bytes_per_launch": full_bytes if kernel_ms > 0 else ice_bytes / max(n_iter_launches, 1),
                     "bytes_definition": ("symmetric packed encoding: the 256 x 256 uint8 blocks on or above the diagonal, once per iteration of "
                                          "each chromosome, + 8 B per overflow cell -- the bytes this kernel must stream; one launch = the whole loop"
                                          if mode == 3 else
                                          "packed encoding: 1 B per cell + 8 B per overflow cell -- the bytes this kernel must stream"
                                          if packed else "int32 tiles: 4 B per cell (SURVEY 8d)"),
                     "survey_4N2": {"algorithmic_bytes_per_launch": survey_bytes, "effective": survey_bytes / (launch_ms * 1e6) if launch_ms > 0 else 0.0,
                                    "frac": survey_bytes / (launch_ms * 1e6) / peak if launch_ms > 0 else 0.0,
                                    "note": "the same launch against SURVEY.md 8(d)'s 4*N^2 (int32 tiles): above 1 because the "
                                            "packed encoding moves a quarter of those bytes, exactly"},
                     "launches": int(info.stream_full_launches) if kernel_ms > 0 else n_iter_launches,
                     "avg_launch_ms": launch_ms,
                     "timing": ("CUDA events around the single persistent launch that runs all iterations of all chromosomes "
                                "(block streaming, partial-sum reduction, bias update and convergence test inside it)") if mode == 3 else
                               ("CUDA events around the first stream-kernel launch of every graph replay of the last timed step in "
                                "which every chromosome was still active (event-record nodes inside the replayed graph)") if kernel_ms > 0
                               else "CUDA events around the whole iteration loop (stream + update kernels, launch gaps, polls)",
                     "loop": {"achieved": loop_achieved, "frac": loop_achieved / peak, "ms": loop_ms, "launches": n_iter_launches,
                              "note": "algorithmic bytes of all iterations / time of the whole loop incl. update kernels and gaps"},
                     "encoding": ("upper-triangular 256 x 256 uint8 blocks + overflow list, built once per call in %.3f ms (%d overflow cells)"
                                  % (float(info.pack_ms), int(info.overflow_cells))) if mode == 3 else
                                 ("uint8 cells + overflow list, built once per call in %.3f ms (%d overflow cells)"
                                  % (float(info.pack_ms), int(info.overflow_cells))) if packed else "int32 tiles",
                     "traffic": traffic, "traffic_note": traffic_note},
        "roofline_secondary": secondary,
        "breakdown": breakdown, "clocks": clocks,
    }
    if parity is not None:
        line["parity_check"] = parity
    if cpu is not None:
        line["cpu_baseline"] = cpu
    if c1 is not None:
        line["c1"] = c1
    if c3 is not None:
        line["c3"] = c3
    if c4 is not None:
        line["c4"] = c4
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    bad = ((parity is not None and not parity["ok"]) or (c4 is not None and c4.get("parity_check") and not c4["parity_check"]["ok"])
           or (c1 is not None and not c1["parity_check"]["ok"]))
    if bad:
        sys.stderr.write("bench.py: PARITY CHECK FAILED (see parity_check in the line above)\n")
        sys.exit(3)


def twostep_roofline(dev, peak, ev_time, n=6232):
    """kernel (c): the two-step allelic correction of one chr1-sized chromosome (M and P), SURVEY 8(d): 52*N^2"""
    import torch
    from hichap_master_b200 import matrixBuilding as mb
    from hichap_master_b200.device import DenseBatch
    g = torch.Generator(device=dev); g.manual_seed(7)
    b = DenseBatch([n, n, n], dev)
    idx = torch.arange(n, device=dev)
    dist = (idx[:, None] - idx[None, :]).abs().clamp_(min=1).to(torch.float32)
    lam = 40.0 / dist
    del dist
    for k, f in enumerate((1.0, 0.06, 0.05)):
        m = torch.poisson(lam * f, generator=g).to(torch.int32)
        m = torch.triu(m) + torch.triu(m, 1).t()
        b.view(k)[:, :n].copy_(m)
    del lam, m
    ms = ev_time(lambda: mb.two_step_device(b, 0, b, 1, b, 2))
    by = 52.0 * n * n
    return {"kernel": "two-step correction of ONE chromosome, M and P, one call (9 launches for ~0.5 ms of streaming: set-up bound; "
                      "the batched C3 entry below is the throughput figure)", "bound": "hbm",
            "algorithmic_bytes": by, "formula": "52*N^2 (SURVEY 8d), N = %d" % n, "ms": ms, "achieved": by / (ms * 1e6),
            "peak": peak, "unit": "GB/s", "frac": by / (ms * 1e6) / peak}


# ------------------------------------------------------------------------------------------
# C4: genome-wide 10 kb, sort path -> row-block sharded CSR -> ICE with one allreduce per iteration
# ------------------------------------------------------------------------------------------
def csr_parity_small(world, rank, dev, comm):
    """The row-block sharded path on a small genome against the oracle (what tests/dist_gpu_check.py checks),
    run in-process so that the driver's own bench run carries the evidence at every N."""
    import torch
    import torch.distributed as dist
    from hichap_master_b200 import distributed as hd, kernels, matrixBuilding as mb, synth
    from hichap_master_b200.device import PairColumns
    from oracle import cooler_ice, hichap_oracle as ho
    small = {"1": 6_010_000, "2": 4_800_000, "10": 3_333_333, "X": 5_000_001}
    order = ho.sort_chromosomes(small)
    res = 20000
    c1, p1, c2, p2 = synth.genome_pairs(small, order, 1_500_000, 17, trans_frac=0.25)
    mine = np.arange(c1.size) % world == rank
    table, total = ho.chro_bins(small, res)
    start = torch.tensor([table[c][0] for c in order], dtype=torch.int64, device=dev)
    chrom_bins = torch.tensor([small[c] // res + 1 for c in order], dtype=torch.int32, device=dev)
    pairs = PairColumns(c1[mine], p1[mine], c2[mine], p2[mine], device=dev)
    if world > 1:
        csr, _ = hd.build_row_block_csr(pairs, res, start, chrom_bins, total)
        w, st = mb.ice_balance_sparse(csr, table, cis_only=False, comm=comm, allreduce=lambda t: dist.all_reduce(t))
    else:
        csr = kernels.pairs_to_csr(pairs, res, start, chrom_bins, total, False)
        w, st = mb.ice_balance_sparse(csr, table, cis_only=False)
    wt = torch.from_numpy(np.nan_to_num(w.copy())).to(dev)
    lo, hi = wt.clone(), wt.clone()
    if world > 1:
        dist.all_reduce(lo, op=dist.ReduceOp.MIN); dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    same = bool(torch.equal(lo, hi))
    if rank != 0:
        return None
    sgl = np.array([table[c][0] for c in order], np.int64)
    b1 = p1.astype(np.int64) // res + sgl[c1]; b2 = p2.astype(np.int64) // res + sgl[c2]
    a, b = np.minimum(b1, b2), np.maximum(b1, b2)
    key, cnt = np.unique(a * total + b, return_counts=True)
    off = mb.chrom_offsets_from_bins(table)
    ref, rst = cooler_ice.balance(key // total, key % total, cnt, total, off, cis_only=False)
    good = ~np.isnan(ref)
    err = float(np.max(np.abs(w[good] - ref[good]) / np.abs(ref[good])))
    nan_same = bool(np.array_equal(np.isnan(w), np.isnan(ref)))
    ok = nan_same and err < RTOL and st["iters"] == rst["iters"] and same
    return {"ok": bool(ok), "tolerance": RTOL, "what": "row-block sharded CSR ICE (%d rank(s), NCCL allreduce per iteration) vs oracle: "
            "4 chromosomes @ 20 kb, 1.5 M pairs, 25 %% trans" % world, "sharded_vs_oracle_max_rel": err, "nan_mask_equal": nan_same,
            "iters_gpu": int(st["iters"]), "iters_oracle": int(rst["iters"]), "iters_equal": bool(st["iters"] == rst["iters"]),
            "identical_across_ranks": same}


def run_c4_section(args, world, rank, dev, peak, config="C4", standalone=False):
    import torch
    import torch.distributed as dist
    from hichap_master_b200 import distributed as hd, kernels, matrixBuilding as mb, synth
    from hichap_master_b200.device import PairColumns

    res = 10000 if config == "C4" else 5000
    npairs = args.c4_pairs if config == "C4" else args.c5_pairs
    genome, order = c2_genome()
    bins, total = mb._bins_from_genome(genome, res, [(c, c) for c in order])
    start = mb._start_table(bins, order, dev)
    chrom_bins = torch.tensor([genome[c] // res + 1 for c in order], dtype=torch.int32, device=dev)
    comm = hd.nccl_comm_from_process_group(dev) if world > 1 else None
    allreduce = (lambda t: dist.all_reduce(t)) if world > 1 else None
    parity = csr_parity_small(world, rank, dev, comm)
    n_local = npairs // world
    c1, p1, c2, p2 = synth.genome_pairs_torch(genome, order, n_local, 4000 + rank, dev, trans_frac=0.25)
    pairs = PairColumns(c1, p1, c2, p2, device=dev)
    del c1, p1, c2, p2
    torch.cuda.synchronize()
    torch.cuda.empty_cache()                   # the generator's temporaries (several times the pair columns)

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def maxr(x):
        t = torch.tensor([float(x)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    os.environ.setdefault("HC_ICE_TIME_KERNEL", "1")
    out, reps = {}, []
    for rep in range(3):                       # rep 0 warms NCCL, allocator and caches; the faster of reps 1 and 2 is reported
        sync_all()
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        e[0].record()
        if world > 1:
            csr, cuts = hd.build_row_block_csr(pairs, res, start, chrom_bins, total)
        else:
            csr, cuts = kernels.pairs_to_csr(pairs, res, start, chrom_bins, total, False), [0, total]
        e[1].record()
        w, st = mb.ice_balance_sparse(csr, bins, cis_only=False, comm=comm, allreduce=allreduce)
        e[2].record()
        torch.cuda.synchronize()
        nnz = torch.tensor([float(csr.nnz)], dtype=torch.float64, device=dev)
        mx = nnz.clone()
        if world > 1:
            dist.all_reduce(nnz); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        out = dict(build_ms=maxr(e[0].elapsed_time(e[1])), ice_ms=maxr(e[1].elapsed_time(e[2])), loop_ms=maxr(st["loop_ms"]),
                   stream_ms=maxr(st.get("stream_full_ms", 0.0)), iters=st["iters"], converged=st["converged"],
                   nnz_stored=float(nnz), nnz_max_rank=float(mx), encoding=st.get("encoding", "symmetric CSR, 8 B per stored entry"),
                   bytes_per_entry=float(st.get("bytes_per_entry", 8.0)), launches=int(st["launches"]),
                   pack_ms=maxr(st.get("pack_ms", 0.0)))
        if rep:
            reps.append(out)
        del csr
    out = min(reps, key=lambda r: r["build_ms"] + r["ice_ms"])
    out["repetitions"] = [{"binning_to_csr_ms": r["build_ms"], "ms_to_convergence": r["ice_ms"], "ice_loop_ms": r["loop_ms"],
                           "ice_encode_ms": r["pack_ms"]} for r in reps]
    # the allreduce on its own (the in-loop one is issued by the library on the compute stream)
    ar_us = None
    if world > 1:
        v = torch.zeros(total, dtype=torch.float64, device=dev)
        for _ in range(5):
            kernels.nccl_allreduce_f64(comm, v)
        sync_all()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(20):
            kernels.nccl_allreduce_f64(comm, v)
        b.record(); torch.cuda.synchronize()
        ar_us = maxr(a.elapsed_time(b) / 20 * 1e3)
    del pairs
    torch.cuda.empty_cache()
    if comm:
        kernels.nccl_comm_destroy(comm)
    if rank != 0:
        return None
    Z = (out["nnz_stored"] + total) / 2
    it = max(int(out["iters"]), 1)
    per_iter = out["loop_ms"] / it
    alg = 8.0 * Z + 24.0 * total                        # SURVEY 8(d): upper-triangular CSR, int32 col + int32 count
    agg = alg / (per_iter * 1e6)
    streamed = out["bytes_per_entry"] * out["nnz_max_rank"]
    k_ms = out["stream_ms"] if out["stream_ms"] > 0 else per_iter
    sec = {
        "workload": "%s: hg19 genome-wide %d kb (%d bins), %d synthetic pairs (75%% cis / 25%% trans), sort path -> row-block "
                    "sharded symmetric CSR over %d GPU(s), ICE with one allreduce of the marginal vector per iteration"
                    % (config, res // 1000, total, npairs, world),
        "n_gpus": world, "pairs": int(npairs), "bins": int(total), "nnz_upper": Z, "nnz_stored_total": out["nnz_stored"],
        "nnz_imbalance": out["nnz_max_rank"] * world / out["nnz_stored"],
        "binning_to_csr_ms": out["build_ms"], "ms_to_convergence": out["ice_ms"], "ice_loop_ms": out["loop_ms"],
        "ice_encode_ms": out["pack_ms"],      # column-blocked re-encoding of the CSR (once per call), part of ms_to_convergence
        "timing": "one warm-up repetition, then two timed ones (CUDA events, max over ranks); the faster one is reported, both are listed",
        "repetitions": out["repetitions"],
        "iters": int(out["iters"]), "converged": bool(out["converged"]), "iter_ms": per_iter, "allreduce_us": ar_us,
        "gpu_launches": out["launches"], "encoding": out["encoding"],
        "roofline": {"bound": "hbm", "kernel": "CSR ICE iteration (stream kernel + update, allreduce included)", "unit": "GB/s",
                     "algorithmic_bytes_per_iteration": alg, "formula": "8*Z + 24*n (SURVEY 8d), aggregate over the GPUs",
                     "achieved": agg / world, "achieved_aggregate": agg, "peak": peak, "frac": agg / world / peak,
                     "stream_kernel": {"ms": k_ms, "streamed_bytes_max_rank": streamed, "achieved": streamed / (k_ms * 1e6),
                                       "frac": streamed / (k_ms * 1e6) / peak,
                                       "note": "bytes the slowest rank's stream kernel reads per launch / its mean launch time"}},
        "sort_path": {"ms": out["build_ms"], "algorithmic_bytes": (40.0 + 16.0 * 5) * npairs + 12.0 * Z,
                      "formula": "(40 + 16*passes)*P + 12*Z, passes = 5 (SURVEY 8d), aggregate",
                      "what": ("one 64-bit entry per pair (upper-triangle cell) -> 5 onesweep passes -> reduce by cell (+ the swapped list) -> "
                               "3 passes over the unique cells on the row bits -> row-wise merge into the symmetric CSR"
                               + ("; reduced cells exchanged between the ranks, one more sort + add-counts reduce" if world > 1 else "")),
                      "achieved": ((40.0 + 16.0 * 5) * npairs + 12.0 * Z) / (out["build_ms"] * 1e6) / world, "peak": peak,
                      "frac": ((40.0 + 16.0 * 5) * npairs + 12.0 * Z) / (out["build_ms"] * 1e6) / world / peak},
        "parity_check": parity,
    }
    return sec


def run_c4_standalone(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    peak = float(load_peaks().get("hbm_gbs", 6650.0))
    sec = run_c4_section(args, world, rank, dev, peak, config=args.config, standalone=True)
    if rank == 0:
        print(json.dumps(sec))
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------
# reference arm: the oracle port on the FULL workload, all host cores
# ------------------------------------------------------------------------------------------
def _gen_chrom(job):
    from hichap_master_b200 import synth
    c, length, n, seed, d = job
    a, b = synth.cis_pairs(c, length, n, seed)
    pa, pb = os.path.join(d, "p1_%s.npy" % c), os.path.join(d, "p2_%s.npy" % c)
    np.save(pa, a); np.save(pb, b)
    return c, length, pa, pb


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle port; the Python-2 reference cannot be installed) on the
    host cores: every chromosome of the C2 workload is binned and balanced, chromosomes spread over a process
    pool (largest first).  Each step is the full workload; when K + W full steps would not fit the time budget the
    step count is reduced (and reported), never the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    import shutil
    genome, order = c2_genome()
    shares = pair_shares(genome, order, args.pairs)
    cores = os.cpu_count() or 1
    nproc = max(1, min(cores, len(order)))
    shm = "/dev/shm" if os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > 10 * args.pairs else None
    d = tempfile.mkdtemp(prefix="hc_ref_", dir=shm)
    budget_s = float(os.environ.get("HC_REF_BUDGET_S", "200"))
    try:
        ctx = mp.get_context("fork")
        big_first = sorted(range(len(order)), key=lambda i: -genome[order[i]])
        with ctx.Pool(nproc) as pool:
            t0 = time.perf_counter()
            jobs = pool.map(_gen_chrom, [(order[i], genome[order[i]], int(shares[i]), 2000 + i, d) for i in big_first], chunksize=1)
            gen_s = time.perf_counter() - t0

            def one_step():
                t = time.perf_counter()
                res = pool.map(_cpu_one_chrom, jobs, chunksize=1)
                return time.perf_counter() - t, res
            t1, res = one_step()
            if t1 * (args.warmup + args.steps) <= budget_s:
                warm, steps, times = args.warmup, args.steps, []
                for _ in range(max(0, warm - 1)):
                    one_step()
                if warm == 0:
                    times.append(t1)
            else:                           # the first full step counts; as many more as the budget allows
                warm, times = 0, [t1]
                steps = max(1, min(args.steps, int(budget_s // t1)))
            while len(times) < steps:
                t, res = one_step()
                times.append(t)
    finally:
        shutil.rmtree(d, ignore_errors=True)
    v = float(np.mean(times)) * 1e3
    crit = max(r["bin_s"] + r["ice_s"] for r in res)
    cb = {"value": v, "unit": UNIT, "cores": nproc, "kind": "port",
          "sample": ("oracle port (NumPy restatement of matrixBuilding.py:595-603, :515-521 + cooler balance --cis-only) on the FULL "
                     "workload: all %d chromosomes, %d pairs, one process per chromosome over %d of %d host cores, largest first; "
                     "every step measured, nothing extrapolated; %s; critical path (largest chromosome, one core) %.1f s; "
                     "pair generation %.1f s untimed"
                     % (len(order), args.pairs, nproc, cores,
                        ("steps as requested" if (steps, warm) == (args.steps, args.warmup) else
                         "%d timed + %d warm-up steps requested, %d + %d run to fit %.0f s" % (args.steps, args.warmup, steps, warm, budget_s)),
                        crit, gen_s)),
          "step_s": times, "host_cores": cores,
          "per_chrom": [{k: r[k] for k in ("chrom", "bin_s", "ice_s", "iters", "nnz", "pairs")} for r in res]}
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
            "steps": steps, "warmup": warm, "steps_requested": args.steps, "warmup_requested": args.warmup,
            "ms_per_step": v, "higher_is_better": False,
            "scaling": "strong", "vs_baseline": None, "dtype": "int64 counts / f64 weights", "data": "synthetic",
            "config": workload_config(args.pairs), "cpu_baseline": cb,
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def c3_section(pairs_n, dev, peak):
    """BASELINE.json configs[2] (C3): allelic maternal/paternal matrices at 40 kb with the two-step (ICE of the
    traditional matrices + SNP-density / coverage) correction.  Single GPU; returns the stage breakdown."""
    import torch
    from hichap_master_b200 import _abi, kernels, synth
    from hichap_master_b200.construction import _sub_batch
    from hichap_master_b200.device import DenseBatch, PairColumns

    genome, order = c2_genome()
    nchrom = len(order)
    c1, p1, c2, p2 = synth.genome_pairs_torch(genome, order, pairs_n, 3, dev, trans_frac=0.0)
    g = torch.Generator(device=dev); g.manual_seed(33)
    cls = torch.rand(pairs_n, generator=g, device=dev)          # Bi 86 %, M_M 6 %, P_P 6 %, M_P 1 %, P_M 1 %
    mark = torch.multinomial(torch.tensor([0.30, 0.35, 0.35], device=dev), pairs_n, replacement=True, generator=g).to(torch.uint8)
    allp = PairColumns(c1, p1, c2, p2, device=dev)
    hap = []
    for lo, hi in ((0.86, 0.92), (0.92, 0.98)):
        sel = (cls >= lo) & (cls < hi)
        hap.append(PairColumns(c1[sel], p1[sel], c2[sel], p2[sel], mark[sel], device=dev))
    del cls, mark
    sizes = [genome[c] // RES + 1 for c in order]
    T = DenseBatch(sizes, dev)
    H = DenseBatch(sizes + sizes, dev)

    def ev(fn):
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); out = fn(); b.record(); torch.cuda.synchronize()
        return a.elapsed_time(b), out

    def bin_all():
        T.buf.zero_(); H.buf.zero_()
        kernels.bin_pairs_local_banded(allp, RES, T, check_bounds=False)
        for k in range(2):
            v = _sub_batch(H, k * nchrom, nchrom)
            kernels.bin_pairs_local(hap[k], RES, v, _abi.HC_BIN_SYM_BOTH, check_bounds=False)
            kernels.bin_pairs_local(hap[k], RES, v, _abi.HC_BIN_ONESIDED, check_bounds=False)

    res_t, outs = {}, None
    for rep in range(3):                         # first pass warms the allocator; report the last
        outs = None                              # release the 4.7 GB of corrected matrices before re-allocating
        res_t["binning_ms"], _ = ev(bin_all)
        res_t["ice_traditional_ms"], (w, st) = ev(lambda: kernels.ice_balance_dense(T, None, ignore_diags=1))
        res_t["two_step_ms"], outs = ev(lambda: kernels.twostep_batch(T, H))
    sq = float(sum(n * n for n in sizes))
    gaps = int(sum(g.size for g in outs[1]))
    del outs, T, H, allp, hap
    torch.cuda.empty_cache()
    return {"workload": "C3: hg19 chr1-22,X allelic matrices at 40 kb, %d synthetic pairs (86%% bi-allelic, 6%% M_M, 6%% P_P; "
                        "Both/R1/R2 = 30/35/35%%), ICE of the traditional matrices + two-step correction of M and P" % pairs_n,
            "n_gpus": 1, **res_t, "total_ms": sum(res_t.values()), "ice_iters_max": int(max(st["iters"])),
            "two_step_roofline": {"formula": "52*N^2 summed over the chromosomes (SURVEY 8d)", "algorithmic_bytes": 52.0 * sq,
                                  "achieved": 52.0 * sq / (res_t["two_step_ms"] * 1e6), "peak": peak,
                                  "frac": 52.0 * sq / (res_t["two_step_ms"] * 1e6) / peak, "unit": "GB/s"},
            "gap_rows_total": gaps}


def c1_section(dev, pairs_n=10_000_000):
    """BASELINE.json configs[0] (C1): chr21 only, 40 kb, 10 M cis pairs: binning + ICE, checked against the oracle."""
    import torch
    from hichap_master_b200 import kernels, synth
    from hichap_master_b200.device import DenseBatch, PairColumns
    from oracle import cooler_ice, hichap_oracle as ho
    L = synth.HG19["21"]
    n = L // RES + 1
    _, a, _, b = synth.genome_pairs_torch({"21": L}, ["21"], pairs_n, 1, dev)
    z = torch.zeros_like(a)
    pairs = PairColumns(z, a, z, b, device=dev)
    batch = DenseBatch([n], dev)

    def step():
        batch.buf.zero_()
        kernels.bin_pairs_local_banded(pairs, RES, batch, check_bounds=False)
        return kernels.ice_balance_dense(batch, None, ignore_diags=1)
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        w, st = step()
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 5
    t0 = time.perf_counter()
    hz = np.zeros(pairs_n, np.int32)
    M = ho.bin_local_dense(hz, a.cpu().numpy(), hz, b.cpu().numpy(), [n], RES)[0]
    ref, rst = cooler_ice.balance_dense(M, cis_only=True)
    cpu_s = time.perf_counter() - t0
    ok = ~np.isnan(ref)
    err = float(np.max(np.abs(w[ok] - ref[ok]) / np.abs(ref[ok])))
    return {"workload": "C1: chr21 (-C 21), 40 kb, 1204 bins, %d synthetic cis pairs, binning + ICE to convergence" % pairs_n,
            "ms_per_step": ms, "iters": int(st["iters"][0]), "cpu_port_one_core_ms": cpu_s * 1e3,
            "parity_check": {"ok": bool(np.array_equal(batch.to_numpy(0), M) and np.array_equal(np.isnan(w), np.isnan(ref))
                                        and st["iters"][0] == rst["iters"][0] and err < RTOL),
                             "counts_equal": bool(np.array_equal(batch.to_numpy(0), M)), "iters_oracle": int(rst["iters"][0]), "max_rel_err": err}}


def run_c3(args):
    import torch
    torch.cuda.set_device(0)
    peak = float(load_peaks().get("hbm_gbs", 6650.0))
    print(json.dumps(c3_section(args.pairs if args.pairs != 400_000_000 else 100_000_000, torch.device("cuda", 0), peak)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5,
                    help="timed steps of the C2 step (`value`), and of --impl reference unless steps + warmup full steps "
                         "exceed HC_REF_BUDGET_S (then `steps` < `steps_requested` in its line); the e2e leg times "
                         "min(steps, 3) steps; the other sections use fixed counts: C1 3 warm-up + 5 timed, C3 the last "
                         "of 3, C4/C5 the faster of 2 after 1 warm-up")
    ap.add_argument("--warmup", type=int, default=3,
                    help="untimed steps before the timed ones; at least 3 for C2 (the line reports the number run)")
    ap.add_argument("--pairs", type=int, default=400_000_000)
    ap.add_argument("--c4-pairs", type=int, default=1_000_000_000)
    ap.add_argument("--c5-pairs", type=int, default=2_000_000_000)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the oracle leg (parity_check + cpu_baseline)")
    ap.add_argument("--skip-e2e", action="store_true", help="kernel tuning runs only: no e2e leg (line is not a bench result)")
    ap.add_argument("--skip-c4", action="store_true", help="leave the genome-wide 10 kb section out of the line")
    ap.add_argument("--skip-secondary", action="store_true")
    ap.add_argument("--config", default="C2", choices=["C2", "C3", "C4", "C5"], help="C2 = the driver's headline workload (its line carries C4 too)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed C2 step computed (weights, ICE results, a seeded sample of the matrices) as .npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.config != "C2"):
        ap.error("--dump-outputs writes the outputs of the C2 workload of --impl ours")
    if args.impl == "reference":
        return run_reference(args)
    if args.config == "C3":
        return run_c3(args)
    if args.config in ("C4", "C5"):
        return run_c4_standalone(args)
    args.warmup = max(args.warmup, 3)
    run_ours(args)


if __name__ == "__main__":
    main()
