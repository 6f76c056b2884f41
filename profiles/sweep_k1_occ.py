#!/usr/bin/env python
"""K1 sweep on the bench workload: occupancy pre-filter size (MG_OCC_LOG2_BITS, 0 = off) x L2 persistence x deferred hits.
Run on a GPU box:  python profiles/sweep_k1_occ.py [wg|small] > gpurun_out/sweep_k1_occ.txt"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from malva_b200 import MalvaGpu  # noqa: E402
from malva_b200.kmc import KMER_DTYPE  # noqa: E402

wl = bench.WORKLOADS[sys.argv[1] if len(sys.argv) > 1 else "wg"]
dev = torch.device("cuda", 0)
gen = torch.Generator(device=dev)
gen.manual_seed(bench.SEED)
alt = bench.rand_kmers(torch, wl["n_alt"], bench.K, gen, dev)
ref = bench.rand_kmers(torch, wl["n_ref"], bench.K, gen, dev)
B = wl["batch"]
batches = [bench.make_sample_batch(torch, B, alt, ref, gen, dev) for _ in range(2)]
alt_h = alt.cpu().numpy().view(np.uint64).reshape(-1).view(KMER_DTYPE)
ref_h = ref.cpu().numpy().view(np.uint64).reshape(-1).view(KMER_DTYPE)
del alt, ref
p = torch.cuda.get_device_properties(0)
print("L2", p.L2_cache_size, flush=True)

configs = [(29, 1, 1), (29, 1, 0)]
for sig_frac in (1.0, 0.1):
    n_sig = int(len(alt_h) * sig_frac)
    for occ, persist, defer in configs:
        os.environ["MG_SCAN_DEFER_HITS"] = str(defer)
        os.environ["MG_OCC_LOG2_BITS"] = str(occ)
        os.environ["MG_L2_PERSIST"] = str(persist)
        g = MalvaGpu(k=bench.K, ref_k=bench.REF_K, bf_bits=wl["bf_bits"])
        chunk = 1 << 24
        for arr, flag in ((alt_h[:n_sig], 0), (ref_h[:n_sig], 1)):
            for o in range(0, len(arr), chunk):
                g.add_signatures_packed(arr[o:o + chunk], np.full(len(arr[o:o + chunk]), flag, np.uint8))
        g.finalize_alt()
        g.finalize_context()
        for i in range(3):
            g.scan_sample_kmers_ptr(batches[i & 1][0].data_ptr(), batches[i & 1][1].data_ptr(), B, device=True)
        g.sync()
        g.event_record(0)
        n = 10
        for i in range(n):
            g.scan_sample_kmers_ptr(batches[i & 1][0].data_ptr(), batches[i & 1][1].data_ptr(), B, device=True)
        g.event_record(1)
        ms = g.event_elapsed_ms(0, 1) / n
        print(f"signatures={2 * n_sig:.1e} occ_log2={occ} persist={persist} defer_hits={defer}: {ms:.3f} ms/scan  "
              f"{B / ms / 1e6:.2f} G k-mers/s  {B * 84 / ms / 1e6:.0f} GB/s algorithmic", flush=True)
        g.close()
