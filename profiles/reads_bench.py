"""Genotyping from reads: `malva-geno count` + `call DB` against `call --reads` on the same seeded reads.

    python profiles/reads_bench.py [--mbp 100] [--depth 20] [--out profiles/reads_bench.json] [--keep DIR]

Inputs: a panel and a diploid donor from tests/synth_fast.py (the generator of tests/bench_cli_e2e.py --fast), and
150-base reads of the donor at --depth (over both haplotypes together), either strand, 0.5 % substitutions
(tests/synth_reads.py).  Both ways run from the index that `index` built; their VCFs must be byte-identical, else the
script fails.  Recorded:
  * the phase times of both ways from the CLI's stderr phase lines: counting (`count`) and the sample scan (`call`'s
    "BF weights created": reading the database and K1; for --reads: reading the reads, counting restricted to the
    index, K1), and the wall time of each program;
  * the k-mer table of both: capacity (slots of 32 B), windows examined, ref_k-mers kept (distinct), and the device time
    of the counting kernels per read base.  The full count's table is read from a KmerCounter fed the same reads (the
    CLI's `count` does not print it); the restricted one from `call --reads --trace`;
  * the GPU name and power limit, read with `nvidia-smi --query-gpu` in the same run.
Everything goes to a temporary directory (or --keep DIR); nothing is written to the tree but --out."""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import synth_fast  # noqa: E402
import synth_reads  # noqa: E402
from malva_b200 import KmerCounter  # noqa: E402
from malva_b200 import build as mbuild  # noqa: E402


def phases(stderr: str) -> dict:
    return {m.group(1): float(m.group(2))
            for m in re.finditer(r"\[malva-geno/([^\]]+)\] Execution Time ([0-9.e+-]+)s", stderr)}


def run(cmd, **kw):
    t0 = time.time()
    p = subprocess.run([str(c) for c in cmd], capture_output=True, text=True, **kw)
    if p.returncode != 0:
        sys.stderr.write(p.stderr[-4000:])
        raise SystemExit(f"failed: {' '.join(str(c) for c in cmd[:2])} (exit {p.returncode})")
    return p, time.time() - t0


def full_table(reads: str, ref_k: int, read_len: int) -> dict:
    """an unrestricted KmerCounter over the reads file (fixed-width FASTQ records of synth_reads), 64 MB per add"""
    rec = 2 * read_len + 7
    data = np.memmap(reads, dtype=np.uint8, mode="r").reshape(-1, rec)
    per = (64 << 20) // (read_len + 1)
    c = KmerCounter(ref_k)
    try:
        for a in range(0, len(data), per):
            chunk = np.array(data[a:a + per, 2:3 + read_len])   # '\n' + sequence
            c.add(chunk.tobytes())
        st = c.stats()
    finally:
        c.close()
    return st


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mbp", type=float, default=100.0)
    ap.add_argument("--depth", type=float, default=20.0)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "reads_bench.json"))
    ap.add_argument("--keep", default=None, help="work directory to keep (default: a temporary one)")
    a = ap.parse_args()
    k, ref_k, read_len = 35, 43, 150
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    if not gpu:
        raise SystemExit("no GPU visible (nvidia-smi reports none)")
    mbuild.build()
    cli = mbuild.CLI
    with tempfile.TemporaryDirectory() as tmp:
        d = a.keep or tmp
        os.makedirs(d, exist_ok=True)
        t0 = time.time()
        fa, vcf, donor, n_var = synth_fast.build(d, int(a.mbp * 1e6))
        haps = [ln for ln in open(donor, "rb").read().split(b"\n") if ln and not ln.startswith(b">")]
        haps = [np.frombuffer(h, np.uint8) for h in haps]
        reads = os.path.join(d, "donor.fq")
        bases = synth_reads.write_reads(reads, haps, a.depth / len(haps), 20261022, read_len=read_len)
        t_gen = time.time() - t0
        flags = ["-k", k, "-r", ref_k, "-b", "4"]
        db = os.path.join(d, "donor_db")
        p_count, w_count = run([cli, "count", f"-k{ref_k}", reads, db])
        run([cli, "index"] + flags + [fa, vcf, db])
        p_call, w_call = run([cli, "call"] + flags + [fa, vcf, db])
        p_reads, w_reads = run([cli, "call"] + flags + [fa, vcf, reads, "--reads", "--trace"])
        if p_call.stdout != p_reads.stdout:
            raise SystemExit("call --reads and count + call DB print different VCFs")
        m = re.search(r"\[trace\] reads .*?: (\d+) read bytes, (\d+) windows examined, (\d+) distinct kept \((\d+) seen "
                      r"twice or more\), table capacity (\d+) slots; reading ([0-9.]+) ms \(([0-9.]+) ms waited for\), "
                      r"counting \+ scan ([0-9.]+) ms \(counting kernels ([0-9.]+) ms\)", p_reads.stderr)
        rb, rw, rd, rd2, rcap, t_rd, t_wait, t_cnt, t_kern = m.groups()
        full = full_table(reads, ref_k, read_len)
        mc = re.search(r"(\d+) read bytes, (\d+) k-mer instances, (\d+) distinct, (\d+) written", p_count.stderr)
        pc, pr, pd = phases(p_count.stderr), phases(p_call.stderr), phases(p_reads.stderr)
        res = {
            "gpu": gpu[0], "gpus_visible": len(gpu),
            "inputs": {"generator": "tests/synth_fast.py + tests/synth_reads.py", "mbp": a.mbp, "depth": a.depth,
                       "read_len": read_len, "substitutions": 0.005, "read_bases": bases, "variants": n_var,
                       "generate_s": round(t_gen, 1), "k": k, "ref_k": ref_k, "bf_GB": 4},
            "vcf_identical": True, "vcf_bytes": len(p_call.stdout),
            "count_then_call": {
                "count_s": pc.get("k-mer counting complete"), "count_wall_s": round(w_count, 2),
                "call_scan_s": pr.get("BF weights created"), "call_wall_s": round(w_call, 2),
                "total_wall_s": round(w_count + w_call, 2),
                "db_records": int(mc.group(4)), "db_bytes": os.path.getsize(db + ".kmc_suf") + os.path.getsize(db + ".kmc_pre"),
                "table_capacity_slots": full["capacity"], "windows": full["windows"], "distinct": full["distinct"],
                "count_kernel_ns_per_read_base": full["kernel_us"] * 1e3 / bases,
            },
            "call_reads": {
                "scan_s": pd.get("BF weights created"), "wall_s": round(w_reads, 2),
                "reading_ms": float(t_rd), "waited_for_reads_ms": float(t_wait), "counting_and_scan_ms": float(t_cnt),
                "table_capacity_slots": int(rcap), "windows": int(rw), "distinct_kept": int(rd),
                "kept_seen_twice": int(rd2), "kept_fraction_of_distinct": int(rd) / max(1, full["distinct"]),
                "count_kernel_ns_per_read_base": float(t_kern) * 1e6 / bases, "read_bytes": int(rb),
            },
        }
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
