"""C4-shaped genome-wide 10 kb CSR (hg19, 25 % trans) + a few ICE iterations, for
`ncu -k regex:csrb_stream`:  python profiles/ncu_csr_ice.py [pairs] [iters]"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from hichap_master_b200 import kernels, matrixBuilding as mb, synth  # noqa: E402
from hichap_master_b200.device import PairColumns  # noqa: E402

P = int(sys.argv[1]) if len(sys.argv) > 1 else 250_000_000
iters = int(sys.argv[2]) if len(sys.argv) > 2 else 4
dev = torch.device("cuda", 0)
genome = {c: l for c, l in synth.HG19.items() if c not in ("Y", "M")}
order = [str(i) for i in range(1, 23)] + ["X"]
c1, p1, c2, p2 = synth.genome_pairs_torch(genome, order, P, 4, dev, trans_frac=0.25)
bins, csr = mb.bin_traditional_sparse(PairColumns(c1, p1, c2, p2, device=dev), genome, 10000)
del c1, p1, c2, p2
w, st = mb.ice_balance_sparse(csr, bins, max_iters=iters)
print("stored entries", csr.nnz, "iters", st["iters"], "loop_ms", st["loop_ms"], st.get("encoding"))
