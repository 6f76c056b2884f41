"""Seeded sequencing reads of a donor for `malva-geno call --reads` (tests/test_gpu_reads.py, profiles/reads_bench.py):
fixed-length reads drawn uniformly from the donor's haplotypes, either strand, with uniform substitutions, written as
FASTQ.  Vectorised with numpy (about 10 s per Gbp of reads).  Test infrastructure only."""
from __future__ import annotations

import gzip

import numpy as np

_COMP = np.zeros(256, np.uint8)
for _a, _b in zip(b"ACGTN", b"TGCAN"):
    _COMP[_a] = _b
_NEXT = {c: np.frombuffer(bytes(x for x in b"ACGT" if x != c), np.uint8) for c in b"ACGT"}


def write_reads(path: str, haps, depth: float, seed: int, read_len: int = 150, sub_rate: float = 0.005,
                batch: int = 1 << 20) -> int:
    """FASTQ of reads covering each haplotype (strings or uint8 arrays) `depth` times; `.gz` paths are gzipped.
    Returns the number of read bases."""
    g = np.random.default_rng(seed)
    seqs = [np.frombuffer(h.encode(), np.uint8) if isinstance(h, str) else np.asarray(h, np.uint8) for h in haps]
    seqs = [s for s in seqs if len(s) >= read_len]
    total = 0
    opener = gzip.open if path.endswith(".gz") else open
    with opener(path, "wb") as fh:
        for s in seqs:
            n = int(len(s) * depth / read_len)
            for a in range(0, n, batch):
                m = min(batch, n - a)
                start = g.integers(0, len(s) - read_len + 1, m)
                r = s[start[:, None] + np.arange(read_len)[None, :]]
                hit = g.random(r.shape) < sub_rate
                if hit.any():
                    pick = g.integers(0, 3, int(hit.sum()))
                    old = r[hit]
                    new = old.copy()
                    for c, alt in _NEXT.items():
                        sel = old == c
                        new[sel] = alt[pick[sel]]
                    r[hit] = new
                rc = g.random(m) < 0.5
                r[rc] = _COMP[r[rc, ::-1]]
                rec = np.empty((m, 2 * read_len + 7), np.uint8)
                rec[:, 0:3] = np.frombuffer(b"@r\n", np.uint8)
                rec[:, 3:3 + read_len] = r
                rec[:, 3 + read_len:6 + read_len] = np.frombuffer(b"\n+\n", np.uint8)
                rec[:, 6 + read_len:6 + 2 * read_len] = ord("I")
                rec[:, -1] = ord("\n")
                fh.write(rec.tobytes())
                total += m * read_len
    return total
