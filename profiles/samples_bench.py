#!/usr/bin/env python
"""Sample sets on one B200: what genotyping several samples against one index costs and saves.

    python profiles/samples_bench.py [out.json] [Mbp=5] [donors=8]
    python profiles/samples_bench.py devices [out.json] [Mbp=5] [donors=16]

  take          mg_samples_take per sample at the `wg` workload's index (bench.py's build: 2^35-bit filters, 1e8 alt
                + 1e8 ref signature k-mers), after a scan of one bench.py sample batch (2^27 43-mers)
  lookups       k_lookup_packed<K,OUT_SAMPLES> for sets of 1, 8 and 32 samples against one single-sample look-up on the
                same batch
                (bench.py's 2.85e6-variant batch; device time of the look-up phase, mg_genotype_kernel_ms[0])
  whole_program tests/bench_cli_e2e.py's 5 Mbp shape: `malva-geno call` with N donor databases against N single
                calls on the same index; the outputs must be byte-identical

The `devices` part alone (a cohort over several contexts):
  replicate     mg_replicate of the `wg` index (device 0 -> 0, and 0 -> 1 when a second GPU is visible) against the
                sequence that loads an index file onto a context in `call` (mg_create, the imports of the set bits and
                the packed ref keys, both finalizes), from host arrays already read; host clock, best of 3
  cohort        tests/bench_cli_e2e.py's 5 Mbp shape with N donors: `call --out-dir` on one context, with
                --sample-devices over every visible GPU, and with --sample-devices 0,0 (two contexts on one device);
                two runs of each, alternating; every file must be byte-identical across the three

Prints one JSON document (card name and power limit included) and writes it to out.json when given.
"""
import json
import os
import random
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)
import numpy as np  # noqa: E402

import bench  # noqa: E402


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().split("\n")[0] if r.returncode == 0 else "unknown"


def device_part():
    import torch

    from malva_b200.api import PackedSignatureBatch
    from malva_b200.kmc import KMER_DTYPE

    if not torch.cuda.is_available():
        raise SystemExit("samples_bench.py: no CUDA device")
    wl = bench.WORKLOADS["wg"]
    dev = torch.device("cuda", 0)
    gen = torch.Generator(device=dev)
    gen.manual_seed(bench.SEED)
    t0 = time.time()
    g, alt, ref = wg_index(torch, dev, gen)
    stats = g.index_stats()
    rows = stats["bf_ones"] + stats["ref_keys"] - stats["overflow_keys"] + stats["overflow_capacity"]
    B = wl["batch"]
    kk, cc = bench.make_sample_batch(torch, B, alt, ref, gen, dev)[:2]
    vb = bench.make_variant_batch(torch, wl["variants"], alt, ref, gen, dev)
    pb = PackedSignatureBatch(vb["vao"], vb["aso"], vb["sko"], vb["kmers"].cpu().numpy().view(KMER_DTYPE).reshape(-1),
                              vb["freq"], np.zeros(1, np.uint64), b"", np.zeros(0, np.uint32))
    del alt, ref
    torch.cuda.synchronize()
    setup_s = time.time() - t0

    def scan():
        g.scan_sample_kmers_ptr(kk.data_ptr(), cc.data_ptr(), B, device=True)
        g.sync()

    # take: one scan per column, host clock around the synchronous call
    g.samples_begin(32)
    takes = []
    for s in range(32):
        scan()
        t = time.perf_counter()
        g.samples_take(s)
        takes.append((time.perf_counter() - t) * 1e3)
    # look-ups: the live counters hold one more scan for the single-sample path
    scan()
    reps = 5
    single = []
    g.genotype_packed(pb, want_lik=False)     # warm-up
    for _ in range(reps):
        g.genotype_packed(pb, want_lik=False)
        single.append(g.genotype_kernel_ms())
    lookups = {"k_lookup_packed_ms": round(statistics.median(x[0] for x in single), 3),
               "coverage_ms": round(statistics.median(x[1] for x in single), 3),
               "likelihoods_ms": round(statistics.median(x[2] for x in single), 3)}
    ref_res = g.genotype_packed(pb, want_lik=False)
    same = True
    for n in (1, 8, 32):
        if n != 32:
            g.samples_begin(n)
            for s in range(n):
                scan()
                g.samples_take(s)
        g.genotype_samples_packed(pb, want_lik=False)   # warm-up
        ms = []
        for _ in range(reps):
            res = g.genotype_samples_packed(pb, want_lik=False)
            ms.append(g.genotype_kernel_ms())
        same = same and all(np.array_equal(r.gq, ref_res.gq) and np.array_equal(r.cov, ref_res.cov) for r in res)
        lookups[f"samples_G{n}"] = {
            "lookup_ms": round(statistics.median(x[0] for x in ms), 3),
            "coverage_all_samples_ms": round(statistics.median(x[1] for x in ms), 3),
            "likelihoods_all_samples_ms": round(statistics.median(x[2] for x in ms), 3)}
    g.samples_end()
    g.close()
    return {"index": dict(stats, counter_rows=rows, bytes_per_sample=4 * rows), "setup_s": round(setup_s, 1),
            "signature_kmers": int(vb["dims"][3]), "variants": int(vb["dims"][0]),
            "take_ms": {"median": round(statistics.median(takes), 2), "min": round(min(takes), 2),
                        "max": round(max(takes), 2), "n": len(takes)},
            "lookups": lookups,
            "columns_equal_live_genotypes": bool(same)}


def wg_index(torch, dev, gen):
    """bench.py's `wg` index on device 0, and its alt and ref signature k-mers (device tensors)"""
    from malva_b200 import MalvaGpu
    from malva_b200.kmc import KMER_DTYPE

    wl = bench.WORKLOADS["wg"]
    g = MalvaGpu(k=bench.K, ref_k=bench.REF_K, bf_bits=wl["bf_bits"])
    alt = bench.rand_kmers(torch, wl["n_alt"], bench.K, gen, dev)
    ref = bench.rand_kmers(torch, wl["n_ref"], bench.K, gen, dev)
    chunk = 1 << 24
    for arr, flag in ((alt, 0), (ref, 1)):
        for o in range(0, arr.shape[0], chunk):
            h = arr[o:o + chunk].cpu().numpy().view(np.uint64).reshape(-1).view(KMER_DTYPE)
            g.add_signatures_packed(h, np.full(len(h), flag, np.uint8))
    g.finalize_alt()
    g.scan_reference(b"ACGT" * 1000)   # (the context filter does not bear on these timings)
    g.finalize_context()
    return g, alt, ref


def cli_inputs(d, mbp, n_donors):
    """tests/bench_cli_e2e.py's shape in directory d: reference, variants, index, and n_donors donor databases"""
    import bench_cli_e2e as e2e
    import synth
    from malva_b200 import build as mbuild
    from malva_b200 import kmc

    mbuild.build()
    cli = mbuild.CLI
    case = synth.Case("cli_e2e", 20261018 + 42, [("1", int(mbp * 1e6))], mean_gap=41, n_samples=32)
    synth_write = kmc.write_kmc_db
    kmc.write_kmc_db = lambda prefix, uk, uc, k, **kw: e2e.fast_write_kmc(prefix, uk, uc, k)
    try:
        fa, vcf, prefix, _ = synth.build_case(case, d)
        rng = random.Random(case.seed)
        refs = synth.make_reference(rng, case.contigs)
        recs = synth.make_variants(rng, refs, case.mean_gap, case.n_samples, case.haploid, k=case.k)
        dbs = []
        for i in range(n_donors):
            r = random.Random(1000 + i)
            p = os.path.join(d, f"donor{i}")
            synth.sample_kmc_db(r, p, synth.donor_haplotypes(r, refs, recs, False), case.ref_k, case.mean_cov)
            dbs.append(p)
    finally:
        kmc.write_kmc_db = synth_write
    flags = ["-k", "35", "-r", "43", "-b", "1"]
    p = subprocess.run([cli, "index"] + flags + [fa, vcf, prefix], capture_output=True)
    assert p.returncode == 0, p.stderr[-2000:]
    return cli, flags, fa, vcf, dbs


def whole_program(mbp, n_donors):
    import bench_cli_e2e as e2e

    with tempfile.TemporaryDirectory() as d:
        t0 = time.time()
        cli, flags, fa, vcf, dbs = cli_inputs(d, mbp, n_donors)
        gen_s = time.time() - t0
        t = time.time()
        singles = []
        for db in dbs:
            p = subprocess.run([cli, "call"] + flags + [fa, vcf, db], capture_output=True)
            assert p.returncode == 0, p.stderr[-2000:]
            singles.append(p.stdout)
        single_s = time.time() - t
        t = time.time()
        out = os.path.join(d, "out")
        p = subprocess.run([cli, "call"] + flags + [fa, vcf] + dbs + ["--out-dir", out], capture_output=True,
                           text=True)
        multi_s = time.time() - t
        assert p.returncode == 0, p.stderr[-2000:]
        same = all(open(os.path.join(out, os.path.basename(db) + ".vcf"), "rb").read() == s
                   for db, s in zip(dbs, singles))
        n_var = sum(1 for l in open(vcf) if not l.startswith("#"))
        return {"reference_bases": int(mbp * 1e6), "variants": n_var, "donors": n_donors,
                "generate_s": round(gen_s, 1), "single_calls_wall_s": round(single_s, 2),
                "one_call_wall_s": round(multi_s, 2),
                "saving_per_extra_sample_s": round((single_s - multi_s) / max(1, n_donors - 1), 3),
                "outputs_identical": bool(same), "one_call_phases_s": e2e.phases(p.stderr)}


def _export(g, which):
    """set-bit indices of a filter (which 0 / 1) or, which None, the packed ref keys: the arrays of an index file"""
    import ctypes as C

    from malva_b200._lib import check
    from malva_b200.kmc import KMER_DTYPE

    n = C.c_uint64(0)
    if which is None:
        check(g._L.mg_export_ref_keys(g._h, None, 0, C.byref(n)))
        out = np.zeros(max(2 * n.value, 2), np.uint64)
        check(g._L.mg_export_ref_keys(g._h, out.ctypes.data_as(C.POINTER(C.c_uint64)), n.value, C.byref(n)))
        return out[:2 * n.value].view(KMER_DTYPE)
    check(g._L.mg_export_set_bits(g._h, which, None, 0, C.byref(n)))
    out = np.zeros(max(n.value, 1), np.uint64)
    check(g._L.mg_export_set_bits(g._h, which, out.ctypes.data_as(C.POINTER(C.c_uint64)), n.value, C.byref(n)))
    return out[:n.value]


def replicate_part():
    import ctypes as C

    import torch

    from malva_b200 import MalvaGpu
    from malva_b200._lib import check

    if not torch.cuda.is_available():
        raise SystemExit("samples_bench.py: no CUDA device")
    dev = torch.device("cuda", 0)
    gen = torch.Generator(device=dev)
    gen.manual_seed(bench.SEED)
    g, alt, ref = wg_index(torch, dev, gen)
    del alt, ref
    torch.cuda.synchronize()
    bf_idx, ctx_idx, keys = _export(g, 0), _export(g, 1), _export(g, None)
    u64p = C.POINTER(C.c_uint64)

    def load():   # call_main's load sequence (csrc/host/malva_geno.cpp), after the file is read
        h = MalvaGpu(k=g.k, ref_k=g.ref_k, bf_bits=g.bf_bits, device=0)
        check(h._L.mg_import_set_bits(h._h, 0, bf_idx.ctypes.data_as(u64p), len(bf_idx)))
        h.add_signatures_packed(keys, np.ones(len(keys), np.uint8))
        h.finalize_alt()
        check(h._L.mg_import_set_bits(h._h, 1, ctx_idx.ctypes.data_as(u64p), len(ctx_idx)))
        h.finalize_context()
        return h

    def best_of(fn, reps=3):
        ts = []
        for _ in range(reps):
            t = time.perf_counter()
            h = fn()
            ts.append(time.perf_counter() - t)
            same = h.index_stats() == g.index_stats()
            h.close()
            assert same
        return round(min(ts), 3), [round(x, 3) for x in ts]

    res = {"index": g.index_stats(), "bf_bits": g.bf_bits, "load_from_host_arrays_s": best_of(load),
           "replicate_0_to_0_s": best_of(lambda: g.replicate(0))}
    if torch.cuda.device_count() > 1:
        res["replicate_0_to_1_s"] = best_of(lambda: g.replicate(1))
    else:
        res["replicate_0_to_1_s"] = "not measured: one GPU visible"
    g.close()
    return res


def cohort_part(mbp, n_donors):
    import bench_cli_e2e as e2e
    import torch

    n_gpus = torch.cuda.device_count()
    configs = {"one_context": [], "all_gpus": ["--sample-devices", ",".join(str(i) for i in range(n_gpus))],
               "two_contexts_on_gpu0": ["--sample-devices", "0,0"]}
    with tempfile.TemporaryDirectory() as d:
        t0 = time.time()
        cli, flags, fa, vcf, dbs = cli_inputs(d, mbp, n_donors)
        res = {"reference_bases": int(mbp * 1e6), "donors": n_donors, "visible_gpus": n_gpus,
               "generate_s": round(time.time() - t0, 1)}
        walls, outputs, phases = {c: [] for c in configs}, {}, {}
        for rep in range(2):
            for name, extra in configs.items():
                out = os.path.join(d, f"out_{name}_{rep}")
                t = time.time()
                p = subprocess.run([cli, "call"] + flags + extra + [fa, vcf] + dbs + ["--out-dir", out],
                                   capture_output=True, text=True)
                walls[name].append(round(time.time() - t, 2))
                assert p.returncode == 0, p.stderr[-2000:]
                outputs[(name, rep)] = [open(os.path.join(out, os.path.basename(db) + ".vcf"), "rb").read()
                                        for db in dbs]
                phases[name] = e2e.phases(p.stderr)
        first = next(iter(outputs.values()))
        res.update({"wall_s": walls, "last_run_phases_s": phases,
                    "outputs_identical": all(v == first for v in outputs.values())})
    return res


def main():
    args = sys.argv[1:]
    devices = bool(args) and args[0] == "devices"
    if devices:
        args = args[1:]
    out = args[0] if len(args) > 0 else None
    mbp = float(args[1]) if len(args) > 1 else 5.0
    n_donors = int(args[2]) if len(args) > 2 else (16 if devices else 8)
    res = {"gpu": card(), "host_cores": os.cpu_count()}
    if devices:
        res["replicate"] = replicate_part()
        res["cohort"] = cohort_part(mbp, n_donors)
    else:
        res["device"] = device_part()
        res["whole_program"] = whole_program(mbp, n_donors)
    text = json.dumps(res, indent=1)
    print(text)
    if out:
        with open(out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
