#!/usr/bin/env python
"""Times the sample-scan kernel (K1, k_scan + k_scan_hits) on a bench workload: the index is built once, then
--reps scans of 2^27 packed k-mers run back to back between two CUDA events.  `--workload l2` keeps every probe line
L2-resident, which gives the kernel's arithmetic floor.  The schemes the round-2 sweeps compared (probe scheme, CTA
size, grid cap, carve-out) are recorded in profiles/round2_sweep_k1_*.txt.
    python profiles/sweep_k1_r2.py [--workload wg] [--reps 10]"""
import argparse
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from malva_b200 import MalvaGpu  # noqa: E402
from malva_b200.kmc import KMER_DTYPE  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--workload", default="wg")
ap.add_argument("--reps", type=int, default=10)
args = ap.parse_args()
wl = bench.WORKLOADS[args.workload]
dev = torch.device("cuda", 0)
gen = torch.Generator(device=dev)
gen.manual_seed(bench.SEED)
alt = bench.rand_kmers(torch, wl["n_alt"], bench.K, gen, dev)
ref = bench.rand_kmers(torch, wl["n_ref"], bench.K, gen, dev)
B = wl["batch"]
g = MalvaGpu(k=bench.K, ref_k=bench.REF_K, bf_bits=wl["bf_bits"])
chunk = 1 << 24
for arr, flag in ((alt, 0), (ref, 1)):
    for o in range(0, arr.shape[0], chunk):
        h = arr[o:o + chunk].cpu().numpy().view(np.uint64).reshape(-1).view(KMER_DTYPE)
        g.add_signatures_packed(h, np.full(len(h), flag, np.uint8))
g.finalize_alt()
g.finalize_context()
batches = [bench.make_sample_batch(torch, B, alt, ref, gen, dev)[:2] for _ in range(2)]
del alt, ref
torch.cuda.synchronize()
for i in range(3):
    g.scan_sample_kmers_ptr(batches[i & 1][0].data_ptr(), batches[i & 1][1].data_ptr(), B, device=True)
g.sync()
g.event_record(0)
for i in range(args.reps):
    g.scan_sample_kmers_ptr(batches[i & 1][0].data_ptr(), batches[i & 1][1].data_ptr(), B, device=True)
g.event_record(1)
ms = g.event_elapsed_ms(0, 1) / args.reps
print(f"workload={args.workload}: {ms:.3f} ms/scan  {B / ms / 1e6:.2f} G k-mers/s  {B * 84 / ms / 1e6:.0f} GB/s algorithmic "
      f"(frac {B * 84 / ms / 1e6 / 6551.4:.3f})", flush=True)
g.close()
