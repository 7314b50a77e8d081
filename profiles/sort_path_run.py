#!/usr/bin/env python
"""One warm + one measured pass of the sort path (pairs -> symmetric CSR) on the C4 workload, for
   ncu --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum --clock-control none \
       -k regex:'pairs_to|radix|ent_|csr_|rle_' --csv --log-file gpurun_out/X.csv python profiles/sort_path_run.py
and, without ncu, the CUDA-event time of the whole path."""
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
ms = []
for rep in range(a.reps):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    csr = kernels.pairs_to_csr(pairs, a.res, start, chrom_bins, total, False)
    e1.record()
    torch.cuda.synchronize()
    ms.append(e0.elapsed_time(e1))
    nnz = csr.nnz
    del csr
print(json.dumps({"pairs": a.pairs, "bins": total, "nnz_stored": nnz, "ms": ms}))
