"""`malva-geno count` when the k-mer table does not fit: one read of the input, a 2-bit copy kept while counting, and
prefix-partitioned passes over that copy.

    python profiles/count_outofcore_bench.py [--mbp 100] [--depth 20] [--out profiles/count_outofcore_bench.json]

Inputs: the donor of profiles/reads_bench.py (tests/synth_fast.py, 150-base reads from tests/synth_reads.py at --depth,
0.5 % substitutions), as plain FASTQ and as gzip FASTQ.  Runs, each `count -k43 --trace`:
  * unlimited: the table grows as device memory allows (one pass, as before);
  * a table cap (MG_COUNT_MAX_SLOTS) of 2^29 slots, and one of 2^27 slots: the table overflows while reading and the
    rest runs as partitioned passes over the copy (about 4 and about 16 ranges for this input);
  * --passes 4.
Every run's .kmc_pre / .kmc_suf must equal the unlimited run's byte for byte (all use the 11-symbol LUT prefix at this
size), else the script fails.  Recorded per run: wall time, the CLI's trace (one read of the input, packed bytes and
runs, where they were kept, passes and splits, reading / counting / pass times, and the device time of the counting
kernels, of the host-to-device copies of the passes and of packing, also per pass), and the GPU name and power
limit read with nvidia-smi in the same run.  Everything goes to a temporary directory; nothing is written to the tree
but --out."""
from __future__ import annotations

import argparse
import gzip
import hashlib
import json
import os
import re
import shutil
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
from malva_b200 import build as mbuild  # noqa: E402

TRACE = re.compile(
    r"\[trace\] count: (\d+) read bytes, one read of the input; ([^;]+); packed copy (\d+) bytes in (\d+) runs "
    r"\((\d+) bytes in host memory, (\d+) bytes in ([^)]+)\); (\d+) passes over the copy, (\d+) splits; reading "
    r"([0-9.]+) ms \(([0-9.]+) ms waited for\), counting \+ packing ([0-9.]+) ms, passes ([0-9.]+) ms; device time: "
    r"counting kernels ([0-9.]+) ms, host-to-device copies ([0-9.]+) ms, packing ([0-9.]+) ms")


def digest(path: str) -> str:
    h = hashlib.sha256()
    with open(path, "rb") as fh:
        while True:
            b = fh.read(1 << 24)
            if not b:
                return h.hexdigest()
            h.update(b)


def count(cli, reads, db, extra=(), env=None):
    e = dict(os.environ)
    e.update(env or {})
    t0 = time.time()
    p = subprocess.run([cli, "count", "-k43", "--trace", *extra, reads, db], capture_output=True, text=True, env=e)
    wall = time.time() - t0
    if p.returncode != 0:
        sys.stderr.write(p.stderr[-4000:])
        raise SystemExit(f"count failed (exit {p.returncode})")
    m = TRACE.search(p.stderr)
    g = m.groups()
    passes = int(g[7])
    r = {"wall_s": round(wall, 2), "read_bytes": int(g[0]), "reads_of_input": 1, "state": g[1],
         "packed_bytes": int(g[2]), "packed_runs": int(g[3]), "packed_in_host_memory_bytes": int(g[4]),
         "packed_spilled_bytes": int(g[5]), "passes_over_copy": passes, "splits": int(g[8]),
         "reading_ms": float(g[9]), "waited_for_reads_ms": float(g[10]), "counting_and_packing_ms": float(g[11]),
         "passes_ms": float(g[12]), "device_counting_kernels_ms": float(g[13]),
         "device_pass_h2d_copies_ms": float(g[14]), "device_packing_ms": float(g[15])}
    if passes:
        r["per_pass_h2d_ms"] = round(float(g[14]) / passes, 2)
        r["per_pass_wall_ms"] = round(float(g[12]) / passes, 1)
    r["summary"] = [ln for ln in p.stderr.splitlines() if ln.startswith("[malva-geno/count]") and "read bytes" in ln][0]
    r["files"] = [digest(db + ".kmc_pre"), digest(db + ".kmc_suf")]
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mbp", type=float, default=100.0)
    ap.add_argument("--depth", type=float, default=20.0)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "count_outofcore_bench.json"))
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    if not gpu:
        raise SystemExit("no GPU visible (nvidia-smi reports none)")
    mbuild.build()
    cli = mbuild.CLI
    with tempfile.TemporaryDirectory() as d:
        t0 = time.time()
        fa, vcf, donor, _ = synth_fast.build(d, int(a.mbp * 1e6))
        haps = [np.frombuffer(h, np.uint8) for h in open(donor, "rb").read().split(b"\n") if h and not h.startswith(b">")]
        fq = os.path.join(d, "donor.fq")
        bases = synth_reads.write_reads(fq, haps, a.depth / len(haps), 20261022, read_len=150)
        gz = fq + ".gz"
        with open(fq, "rb") as src, gzip.open(gz, "wb", compresslevel=1) as dst:
            shutil.copyfileobj(src, dst, 1 << 24)
        t_gen = time.time() - t0
        runs = {}
        for name, reads, extra, env in (
                ("unlimited", fq, (), None),
                ("cap_2^29_slots", fq, (), {"MG_COUNT_MAX_SLOTS": str(1 << 29)}),
                ("cap_2^27_slots", fq, (), {"MG_COUNT_MAX_SLOTS": str(1 << 27)}),
                ("passes_4", fq, ("--passes", "4"), None),
                ("gz_unlimited", gz, (), None),
                ("gz_cap_2^29_slots", gz, (), {"MG_COUNT_MAX_SLOTS": str(1 << 29)})):
            runs[name] = count(cli, reads, os.path.join(d, name), extra, env)
            print(name, json.dumps({x: runs[name][x] for x in ("wall_s", "passes_over_copy", "splits")}), flush=True)
        ref = runs["unlimited"]["files"]
        for name, r in runs.items():
            if r["files"] != ref:
                raise SystemExit(f"{name}: the database differs from the unlimited run's")
        res = {"gpu": gpu[0], "gpus_visible": len(gpu),
               "inputs": {"generator": "tests/synth_fast.py + tests/synth_reads.py", "mbp": a.mbp, "depth": a.depth,
                          "read_len": 150, "substitutions": 0.005, "read_bases": bases,
                          "fastq_bytes": os.path.getsize(fq), "gz_bytes": os.path.getsize(gz),
                          "generate_s": round(t_gen, 1), "k": 43},
               "databases_identical": True, "runs": runs}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
