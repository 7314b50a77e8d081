#!/usr/bin/env python
"""Where the GPU sits idle during one C2 step (`bench.py`'s timed step: banded binning of 400 M pairs at 40 kb, ICE
filters, packed encoding, iteration loop) on one GPU.  The step runs under torch.profiler with CUDA activities after
three warm-up steps; every kernel, copy and memset on the device is a busy interval, and the gaps between them (over
all streams) longer than --min-gap-us are listed with the operations on either side, followed by their sum.
The profiler does not report the kernels inside the body of a conditional (WHILE) graph node: when the ICE loop runs
as such a graph, its iterations after the first appear as one gap between the first update kernel and
ice_finalize_kernel, and the loop's device time is `ice_loop_ms` (CUDA events) instead.
python profiles/c2_timeline.py [--pairs N] [--min-gap-us 5]  ->  one JSON object on stdout"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=400_000_000)
    ap.add_argument("--min-gap-us", type=float, default=5.0)
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    from bench import RES, c2_genome, pair_shares
    from hichap_master_b200 import synth
    from hichap_master_b200.device import PairColumns
    from hichap_master_b200.pipeline import LocalStage

    os.environ.setdefault("HC_ICE_TIME_KERNEL", "1")     # as bench.py
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    genome, order = c2_genome()
    sizes = [genome[c] // RES + 1 for c in order]
    shares = pair_shares(genome, order, args.pairs)
    cs, p1s, p2s = [], [], []
    for i, c in enumerate(order):          # the same seeded inputs as bench.py on one GPU
        _, a, _, b = synth.genome_pairs_torch({c: genome[c]}, [c], int(shares[i]), 2000 + i, dev)
        cs.append(torch.full((a.numel(),), i, dtype=torch.int32, device=dev)); p1s.append(a); p2s.append(b)
    c1, p1, p2 = torch.cat(cs), torch.cat(p1s), torch.cat(p2s)
    del cs, p1s, p2s
    g = torch.Generator(device=dev); g.manual_seed(99)
    perm = torch.randperm(c1.numel(), generator=g, device=dev)
    c1, p1, p2 = c1[perm].contiguous(), p1[perm].contiguous(), p2[perm].contiguous()
    del perm
    pairs = PairColumns(c1, p1, c1, p2, device=dev)
    stage = LocalStage(sizes, int(c1.numel()), dev)
    step = lambda: stage.run(pairs, RES, records=False, weights_to_host=False)
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = step()
        torch.cuda.synchronize()

    ev = []
    for e in prof.events():
        if e.device_type.name != "CUDA" or e.time_range.elapsed_us() <= 0:
            continue
        ev.append((e.time_range.start, e.time_range.end, e.name))
    ev.sort()
    gaps, busy_end, prev = [], None, None
    for s, t, name in ev:
        if busy_end is not None and s - busy_end > args.min_gap_us:
            gaps.append({"at_us": round(busy_end - ev[0][0], 1), "gap_us": round(s - busy_end, 1),
                         "after": prev[:60], "before": name[:60]})
        if busy_end is None or t > busy_end:
            busy_end, prev = t, name
    info = out["info"]
    print(json.dumps({
        "device": torch.cuda.get_device_name(0), "pairs": args.pairs, "min_gap_us": args.min_gap_us,
        "span_us": round(busy_end - ev[0][0], 1), "device_ops": len(ev), "ice_iters_max": int(out["results"]["iters"].max()),
        "ice_loop_ms": float(info.loop_ms), "idle_gaps": gaps, "n_gaps": len(gaps),
        "idle_sum_us": round(sum(x["gap_us"] for x in gaps), 1)}, indent=1))


if __name__ == "__main__":
    main()
