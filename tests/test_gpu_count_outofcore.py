"""Counting read sets larger than the k-mer table with one read of the input (count.cuh: k_pack_*, k_count_packed;
mg_count_set_limit / mg_count_add_keep / mg_count_add_packed; `malva-geno count`): the 2-bit copy against a numpy
restatement, counting from the copy against counting the bytes and oracle/kmc_count.py, the overflow state, and the
CLI's partitioned passes over the copy against an unlimited run."""
import gzip
import os
import random
import subprocess
import threading

import numpy as np
import pytest

import synth_reads
from malva_b200 import KmerCounter, MalvaGpu
from malva_b200 import build as mbuild
from malva_b200._lib import MalvaGpuError
from oracle import kmc_count
from test_gpu_count import random_reads

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "haploid")
_CODE = np.full(256, 255, np.uint8)
for _i, _c in enumerate(b"ACGT"):
    _CODE[_c] = _i


def pack_ref(data: bytes, k: int):
    """the maximal A/C/G/T runs of at least k bytes, 2 bits a base, 4 to a byte, first base high, byte-aligned runs"""
    c = _CODE[np.frombuffer(data, np.uint8)]
    d = np.diff(np.concatenate(([0], (c != 255).astype(np.int8), [0])))
    starts, ends = np.nonzero(d == 1)[0], np.nonzero(d == -1)[0]
    keep = ends - starts >= k
    out = []
    for s, e in zip(starts[keep], ends[keep]):
        r = np.concatenate([c[s:e], np.zeros((-(e - s)) % 4, np.uint8)]).reshape(-1, 4).astype(np.uint32)
        out.append(((r[:, 0] << 6) | (r[:, 1] << 4) | (r[:, 2] << 2) | r[:, 3]).astype(np.uint8))
    return (np.concatenate(out) if out else np.zeros(0, np.uint8)), (ends - starts)[keep].astype(np.uint32)


def edge_calls(rng, k):
    """read byte strings for several add calls: N, lower-case bytes (separators once the host has upper-cased the
    rest), runs of exactly k and k-1, runs far longer than a 1 KiB sub-chunk, a call that is one run"""
    reads = random_reads(rng, 300, read_len=(60, 3000))
    for i in range(0, len(reads), 7):
        r = reads[i]
        if len(r) > 20:
            p = rng.randrange(len(r) - 5)
            reads[i] = r[:p] + r[p:p + 5].lower() + r[p + 5:]
    g = "".join(rng.choice("ACGT") for _ in range(5000))
    reads += [g[:k], g[:k - 1], g[10:10 + k] + "N" + g[20:20 + k - 1], g]
    calls = ["\n".join(reads[i:i + 40]).encode() for i in range(0, len(reads), 40)]
    return calls + [g.encode(), g[:k].encode(), b"", ("N" + g[:2 * k + 3]).encode()]


@pytest.mark.parametrize("k", [1, 21, 31, 43, 63])
def test_pack_equals_the_numpy_restatement(k, monkeypatch):
    monkeypatch.setenv("MG_COUNT_CHUNK", "1024")
    calls = edge_calls(random.Random(300 + k), k)
    c = KmerCounter(k)
    try:
        for b in calls:
            pb, pl = c.add_keep(b)
            eb, el = pack_ref(b, k)
            assert np.array_equal(pl, el) and np.array_equal(pb, eb)
        # the counts of add_keep are those of add
        seqs = [s for b in calls for s in b.decode().split("\n")]
        exp_k, exp_c = kmc_count.count_kmers(["".join(ch if ch in "ACGT" else "N" for ch in s) for s in seqs],
                                             k, 2, 255)
        got_k, got_c = c.finish(2, 255)
        assert np.array_equal(got_k, exp_k) and np.array_equal(got_c, exp_c)
        assert c.stats()["overflowed"] == 0
    finally:
        c.close()


@pytest.mark.parametrize("k", [1, 21, 31, 43, 63])
def test_counting_the_packed_copy_equals_counting_the_bytes(k, monkeypatch):
    """1 KiB sub-chunks: 256-byte staged chunks, so long runs are counted in parts that overlap by k-1 bases"""
    monkeypatch.setenv("MG_COUNT_CHUNK", "1024")
    calls = edge_calls(random.Random(400 + k), k)
    a, b = KmerCounter(k), KmerCounter(k)
    try:
        packs = [a.add_keep(x) for x in calls]
        packed = np.concatenate([p for p, _ in packs])
        lens = np.concatenate([n for _, n in packs])
        bits30 = min(30, 2 * k)
        parts = [(0, 0, 0), (8, 0, 70), (8, 70, 71), (8, 71, 256), (bits30, 0, 1 << (bits30 - 1)),
                 (bits30, 1 << (bits30 - 1), (1 << bits30) - 5), (bits30, (1 << bits30) - 5, 1 << bits30)]
        for pb, lo, hi in parts:
            if pb > 2 * k:
                continue
            a.reset()
            b.reset()
            a.set_partition(pb, lo, hi)
            b.set_partition(pb, lo, hi)
            for x in calls:
                a.add(x)
            b.add_packed(packed, lens)
            assert a.stats()["instances"] == b.stats()["instances"]
            for ci, cs, cx in ((2, 255, 10 ** 9), (1, 3, 10 ** 9), (5, 255, 10 ** 9), (2, 255, 3)):
                ka, na = a.finish(ci, cs, cx)
                kb, nb = b.finish(ci, cs, cx)
                assert np.array_equal(ka, kb) and np.array_equal(na, nb), (pb, lo, hi, ci, cs, cx)
    finally:
        a.close()
        b.close()


def count_split(c, packed, lens, k, depth_seen):
    """the whole prefix space at 30 bits (or 2k), halved on every MG_ERR_NOMEM; results in ascending order"""
    bits = min(30, 2 * k)
    todo = [(0, 1 << bits, 0)]
    keys, counts = [], []
    while todo:
        lo, hi, d = todo.pop(0)
        c.reset()
        c.set_partition(bits, lo, hi)
        try:
            c.add_packed(packed, lens)
            kk, cc = c.finish(2, 255)
        except MalvaGpuError as e:
            assert "error -4" in str(e) and hi - lo >= 2
            mid = (lo + hi) // 2
            todo[:0] = [(lo, mid, d + 1), (mid, hi, d + 1)]
            continue
        depth_seen.append(d)
        keys.append(kk)
        counts.append(cc)
    return np.concatenate(keys), np.concatenate(counts)


def test_overflow_stops_counting_keeps_packing_and_partitions_recover():
    k = 43
    rng = random.Random(77)
    reads = random_reads(rng, 2400, genome_len=60000, read_len=(100, 200))
    calls = ["\n".join(reads[i:i + 50]).encode() for i in range(0, len(reads), 50)]
    exp_k, exp_c = kmc_count.count_kmers(reads, k, 2, 255)
    c = KmerCounter(k)
    try:
        c.set_limit(1 << 16)
        packs, overflow_at, inst = [], None, []
        for i, x in enumerate(calls):
            packs.append(c.add_keep(x))
            st = c.stats()
            inst.append(st["instances"])
            if st["overflowed"] and overflow_at is None:
                overflow_at = i
            eb, el = pack_ref(x, k)
            assert np.array_equal(packs[-1][0], eb) and np.array_equal(packs[-1][1], el)
        assert overflow_at is not None and overflow_at + 3 < len(calls)
        assert len(set(inst[overflow_at:])) == 1 and st["capacity"] <= 1 << 16   # counting stopped at the first
        with pytest.raises(MalvaGpuError, match="error -3"):
            c.finish(2, 255)
        with pytest.raises(MalvaGpuError, match="error -3"):
            c.add(calls[0])
        packed = np.concatenate([p for p, _ in packs])
        lens = np.concatenate([n for _, n in packs])
        depth = []
        got_k, got_c = count_split(c, packed, lens, k, depth)
        assert np.array_equal(got_k, exp_k) and np.array_equal(got_c, exp_c)
        assert max(depth) >= 2                        # a range split more than once
        # without the limit the copy counts in one pass to the same result
        c.set_limit(0)
        c.reset()
        c.set_partition(0, 0, 0)
        c.add_packed(packed, lens)
        got_k, got_c = c.finish(2, 255)
        assert np.array_equal(got_k, exp_k) and np.array_equal(got_c, exp_c)
    finally:
        c.close()


def test_refusals():
    import parity_util as util

    c = KmerCounter(43)
    try:
        with pytest.raises(MalvaGpuError, match="error -1"):
            c.set_limit(1000)
        c.set_limit(1 << 16)
        c.add_keep(b"\n".join(b"ACGT" * 40 + bytes([65 + i % 3]) for i in range(20000)))   # (windows >> the limit)
        assert c.stats()["overflowed"] == 1
        with pytest.raises(MalvaGpuError, match="error -3"):
            c.finish(2, 255)
        with pytest.raises(MalvaGpuError, match="error -3"):
            c.add_packed(np.zeros(11, np.uint8), np.array([43], np.uint32))
        c.reset()
        assert c.stats()["overflowed"] == 0
    finally:
        c.close()
    rng = random.Random(5)
    genome = util.make_genome(rng, 5000)
    nested, _ = util.synth_signatures(rng, genome, 35, 40)
    ks, fl = util.flatten(nested)
    g = MalvaGpu(k=35, ref_k=43, bf_bits=1 << 20)
    c = KmerCounter(43)
    try:
        g.add_signatures(ks, fl)
        g.finalize_alt()
        c.restrict(g)
        with pytest.raises(MalvaGpuError, match="error -3"):
            c.add_keep(genome[:500].encode())
        with pytest.raises(MalvaGpuError, match="error -3"):
            c.add_packed(np.zeros(11, np.uint8), np.array([43], np.uint32))
    finally:
        c.close()
        g.close()


def _run(args, env=None, **kw):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([mbuild.CLI] + [str(a) for a in args], capture_output=True, env=e, **kw)


def _dump(prefix):
    return _run(["kmc-dump", prefix], check=True).stdout


def _lut_len(prefix):
    h = open(str(prefix) + ".kmc_pre", "rb").read()
    return int.from_bytes(h[-8 - 64 + 12:-8 - 64 + 16], "little")


@pytest.fixture(scope="module")
def read_files(tmp_path_factory):
    mbuild.build()
    d = tmp_path_factory.mktemp("ooc")
    g = np.random.default_rng(9)
    genome = "".join("ACGT"[x] for x in g.integers(0, 4, 150000))
    fq = d / "reads.fq"
    synth_reads.write_reads(str(fq), [genome], 8.0, seed=3)
    gz = d / "reads.fq.gz"
    gz.write_bytes(gzip.compress(fq.read_bytes(), 1))
    fa = d / "reads.fa"
    lines = fq.read_text().split("\n")
    with open(fa, "w", newline="") as fh:
        for i in range(1, len(lines), 4):
            s = lines[i]
            fh.write(f">r{i}\r\n")
            for o in range(0, len(s), 61):
                fh.write((s[o:o + 61].lower() if i % 5 == 0 else s[o:o + 61]) + "\r\n")
    return d, {"fq": fq, "gz": gz, "fa": fa}


LIMIT = {"MG_COUNT_MAX_SLOTS": str(1 << 18)}


@pytest.mark.parametrize("kind", ["fq", "gz", "fa"])
def test_cli_partitioned_passes_equal_the_unlimited_run(read_files, kind):
    d, files = read_files
    src = files[kind]
    full, part = d / f"{kind}.full", d / f"{kind}.part"
    r0 = _run(["count", "-k43", src, full])
    assert r0.returncode == 0, r0.stderr.decode()[-2000:]
    tmp = d / f"{kind}.tmp"
    tmp.mkdir()
    r = _run(["count", "-k43", "--trace", src, part, tmp], env=LIMIT)
    assert r.returncode == 0, r.stderr.decode()[-2000:]
    err = r.stderr.decode()
    assert "the table met its limit while reading" in err
    passes = int(err.split(" passes over the copy")[0].rsplit(" ", 1)[1])
    splits = int(err.split(" splits;")[0].rsplit(" ", 1)[1])
    assert passes >= 4 and splits >= 1, err
    assert _dump(full) == _dump(part) and _dump(full).count(b"\n") > 10000
    if _lut_len(full) == _lut_len(part):
        assert open(f"{full}.kmc_suf", "rb").read()[4:] == open(f"{part}.kmc_suf", "rb").read()[4:]
    # the summary line: the read bytes, k-mer instances and distinct k-mers of the single pass
    summary = [[l for l in e.splitlines() if l.startswith("[malva-geno/count]") and "read bytes" in l]
               for e in (r0.stderr.decode(), err)]
    assert len(summary[0]) == 1 and summary[0] == summary[1]
    assert os.listdir(tmp) == []


def test_cli_spills_to_tmp_dir_and_reads_a_fifo(read_files):
    d, files = read_files
    full = d / "spill.full"
    assert _run(["count", "-k43", files["fq"], full]).returncode == 0
    tmp = d / "spill.tmp"
    tmp.mkdir()
    env = dict(LIMIT, MG_COUNT_HOST_BUDGET="1000")
    r = _run(["count", "-k43", "--trace", files["fq"], d / "spill.part", tmp], env=env)
    assert r.returncode == 0, r.stderr.decode()[-2000:]
    assert f"in {tmp}/malva-count-" in r.stderr.decode()
    assert _dump(full) == _dump(d / "spill.part") and os.listdir(tmp) == []
    # a FIFO can be read once only
    fifo = d / "reads.fifo"
    os.mkfifo(fifo)
    data = files["gz"].read_bytes()
    t = threading.Thread(target=lambda: open(fifo, "wb").write(data))
    t.start()
    r = _run(["count", "-k43", fifo, d / "fifo.part", tmp], env=env)
    t.join()
    assert r.returncode == 0, r.stderr.decode()[-2000:]
    assert _dump(full) == _dump(d / "fifo.part") and os.listdir(tmp) == []
    # an output prefix that cannot be written: an error, and no spill file left
    r = _run(["count", "-k43", files["fq"], d / "no" / "such" / "dir" / "db", tmp], env=env)
    assert r.returncode != 0 and os.listdir(tmp) == []


def test_wrapper_with_a_table_limit_prints_the_golden(tmp_path):
    mbuild.build()
    wrapper = os.path.join(os.path.dirname(mbuild.CLI), "MALVA")
    (tmp_path / "haploid.fq").write_bytes(gzip.open(os.path.join(GOLD, "haploid.fq.gz")).read())
    (tmp_path / "haploid.vcf").write_bytes(gzip.open(os.path.join(GOLD, "haploid.vcf.gz")).read())
    os.symlink(os.path.join(GOLD, "haploid.fa"), tmp_path / "haploid.fa")
    cmd = [wrapper, "-1", "-k", "35", "-r", "43", "-b", "1", "-f", "AF", "haploid.fa", "haploid.vcf", "haploid.fq"]
    r = subprocess.run(cmd, capture_output=True, cwd=tmp_path, env=dict(os.environ, MG_COUNT_MAX_SLOTS=str(1 << 16)))
    assert r.returncode == 0, r.stderr.decode()[-2000:]
    assert r.stdout == open(os.path.join(GOLD, "haploid.malva.vcf"), "rb").read()
    assert [p for p in os.listdir(tmp_path) if p.startswith("malva-count-")] == []
