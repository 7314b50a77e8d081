#!/usr/bin/env python
"""C4 on one GPU: sort path once, then the CSR ICE (filters + column-blocked encoding + iteration graph) twice; prints
the event times.  Under `ncu --metrics gpu__time_duration.sum ... -k regex:'csrb|ice_|mad_|nccl'` it gives the launch
list of the set-up kernels."""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import bench  # noqa: E402
from hichap_master_b200 import kernels, matrixBuilding as mb, synth  # noqa: E402
from hichap_master_b200.device import PairColumns  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--pairs", type=int, default=1_000_000_000)
ap.add_argument("--res", type=int, default=10000)
ap.add_argument("--reps", type=int, default=2)
a = ap.parse_args()
dev = torch.device("cuda:0")
genome, order = bench.c2_genome()
bins, total = mb._bins_from_genome(genome, a.res, [(c, c) for c in order])
start = mb._start_table(bins, order, dev)
chrom_bins = torch.tensor([genome[c] // a.res + 1 for c in order], dtype=torch.int32, device=dev)
c1, p1, c2, p2 = synth.genome_pairs_torch(genome, order, a.pairs, 4000, dev, trans_frac=0.25)
pairs = PairColumns(c1, p1, c2, p2, device=dev)
del c1, p1, c2, p2
csr = kernels.pairs_to_csr(pairs, a.res, start, chrom_bins, total, False)
del pairs
torch.cuda.empty_cache()
out = []
for rep in range(a.reps):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    w, st = mb.ice_balance_sparse(csr, bins, cis_only=False)
    e1.record()
    torch.cuda.synchronize()
    out.append({"ms": e0.elapsed_time(e1), "loop_ms": st["loop_ms"], "pack_ms": st.get("pack_ms"), "iters": st["iters"]})
print(json.dumps(out))
