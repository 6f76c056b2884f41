"""Counting restricted to the index (mg_count_restrict, KmerCounter.restrict) and `malva-geno call --reads`.

A ref_k-mer record changes the counters of the sample scan only when its central k-mer sets a bit of bf or is a ref
key of ref_bf, and that depends on the ref_k-mer alone.  So counting only those ref_k-mers and scanning them must leave
exactly the counters of counting everything: at every probe-line key layout (specialised and run-time builds, inline
and wide keys, odd ref_k - k), at filter sizes where keys overflow their line and set bits count outside it, across
the sub-chunk seams of the device, and through the CLI, where `call --reads` must print the bytes of `count` + `call`
on the database."""
import gzip
import os
import random
import re
import subprocess

import numpy as np
import pytest

from malva_b200 import KmerCounter, MalvaGpu, MalvaGpuError, kmc
from malva_b200 import build as mbuild
import parity_util as util
import synth
import synth_reads
import test_gpu_samples as ts

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "haploid")

LAYOUTS = [
    (35, 43),   # the specialised restricted build, inline keys
    (31, 39),   # run-time build
    (36, 43),   # ref_k 43 but k != 35: run-time build; odd ref_k - k
    (47, 55),   # last inline layout
    (48, 56),   # first wide layout: count in key_counts, overflow flag at w3 bit 31
    (60, 63),   # widest counted ref_k (K6 counts k <= 63); odd ref_k - k
]
DENSE, MODULO, SPARSE = 1 << 13, 3 * (1 << 12) + 7, 1 << 22
FILTERS = [pytest.param(DENSE, id="2^13"), pytest.param(MODULO, id="3x2^12+7"), pytest.param(SPARSE, id="2^22")]
NO_CAP = (1 << 32) - 1


def _comp(s: str) -> str:
    return s[::-1].translate(str.maketrans("ACGT", "TGCA"))


def _reads(rng, genome: str, nested, k: int, ref_k: int) -> list:
    """150-base reads of the genome at about 6x (either strand, 0.5 % substitutions, some N's), and sample ref_k-mers
    that carry alt alleles: each seen once, every third one twice"""
    reads = []
    for p in range(0, len(genome) - 150, 25):
        r = list(genome[p:p + 150])
        for i in range(len(r)):
            u = rng.random()
            if u < 0.002:
                r[i] = "N"
            elif u < 0.007:
                r[i] = rng.choice("ACGT")
        r = "".join(r)
        reads.append(_comp(r) if rng.random() < 0.5 else r)
    words, _, _ = util.synth_sample(rng, genome, nested, k, ref_k, 6000)
    return reads + words + words[::3]


def _index(k: int, ref_k: int, bf_bits: int, ks, fl, genome: str) -> MalvaGpu:
    g = MalvaGpu(k=k, ref_k=ref_k, bf_bits=bf_bits)
    g.add_signatures(ks, fl)
    g.finalize_alt()
    g.scan_reference(genome)
    g.finalize_context()
    return g


def _case(k: int, ref_k: int, seed: int):
    rng = random.Random(seed)
    genome = util.make_genome(rng, 30000)
    nested, _ = util.synth_signatures(rng, genome, k, 700)
    ks, fl = util.flatten(nested)
    return rng, genome, nested, ks, fl, _reads(rng, genome, nested, k, ref_k)


def _central(keys: np.ndarray, k: int, ref_k: int) -> list:
    """the k-mer the sample scan takes from each ref_k-mer record: (ref_k - k) // 2 bases of context before it"""
    d = (ref_k - k) // 2
    return [s[d:d + k] for s in kmc.packed_to_strings(keys, ref_k)]


def _line_j(words: np.ndarray, bf_bits: int) -> np.ndarray:
    """number of set bits below each set bit of bf inside its probe line, in rank order"""
    pos = np.flatnonzero(np.unpackbits(words.view(np.uint8), bitorder="little"))
    line = pos[pos < bf_bits] >> 8
    return np.arange(len(line)) - np.searchsorted(line, line, side="left")


@pytest.mark.parametrize("bf_bits", FILTERS)
@pytest.mark.parametrize("k,ref_k", LAYOUTS)
def test_restricted_count_leaves_the_counters_of_the_full_count(k, ref_k, bf_bits):
    """restricted count + scan_counted == full count + scan_counted on a second context of the same index, and the
    restricted table holds exactly the ref_k-mers whose central k-mer is in bf or ref_bf"""
    _, genome, _, ks, fl, reads = _case(k, ref_k, 4000 + 7 * k + bf_bits % 101)
    a, b = _index(k, ref_k, bf_bits, ks, fl, genome), _index(k, ref_k, bf_bits, ks, fl, genome)
    r, u = KmerCounter(ref_k), KmerCounter(ref_k)
    try:
        r.restrict(a)
        r.add(reads)
        u.add(reads)
        # the kept set is the rule, exactly
        rk, rc = r.finish(1, NO_CAP)
        uk, uc = u.finish(1, NO_CAP)
        cen = _central(uk, k, ref_k)
        keep = (a.test_keys(0, cen) | a.test_keys(2, cen)).astype(bool)
        assert np.array_equal(rk, uk[keep]) and np.array_equal(rc, uc[keep])
        assert 100 < len(rk) < len(uk) // 2, (len(rk), len(uk))
        assert (rc == 1).any() and (rc >= 2).any(), "no kept ref_k-mer is dropped by -ci2 next to one that is not"
        sr, su = r.stats(), u.stats()
        assert sr["windows"] == su["instances"] == su["windows"]
        assert sr["instances"] == int(rc.sum()) and sr["distinct"] == len(rk)
        # the counters after the scan
        r.finish(2, 255)
        u.finish(2, 255)
        a.scan_counted(r)
        b.scan_counted(u)
        assert np.array_equal(a.bf_counts(), b.bf_counts()), "bf counters"
        ref_keys = [x for x, f in zip(ks, fl) if f]
        assert np.array_equal(a.get_counts(ref_keys, [1] * len(ref_keys)), b.get_counts(ref_keys, [1] * len(ref_keys)))
        ca, cb = util.counter_arrays(a), util.counter_arrays(b)
        for name, x, y in zip(("bf counters", "line key counts", "overflow counts"), ca, cb):
            assert np.array_equal(x, y), name
        # the edges this filter size is there for
        assert ca[0].any() and ca[1].any()
        if bf_bits in (DENSE, MODULO):
            assert a.index_stats()["overflow_keys"] > 0 and ca[2].any(), "no overflowed key is counted"
        if bf_bits == MODULO:
            j = _line_j(a.bits(0), bf_bits)
            assert (ca[0][j >= 3] > 0).any(), "no counted bit past the three inline counters of its line"
    finally:
        a.close(), b.close(), r.close(), u.close()


@pytest.mark.parametrize("k,ref_k", [(35, 43), (36, 43)])
def test_restricted_count_across_seams_calls_and_partitions(monkeypatch, k, ref_k):
    """device sub-chunks of 1 KiB, one read per call, and three prefix partitions concatenated: the single pass"""
    _, genome, _, ks, fl, reads = _case(k, ref_k, 5100 + k)
    g = _index(k, ref_k, MODULO, ks, fl, genome)
    one = KmerCounter(ref_k)
    try:
        one.restrict(g)
        one.add(reads)
        want_k, want_c = one.finish(1, 255)
        assert len(want_k) > 100
    finally:
        one.close()
    monkeypatch.setenv("MG_COUNT_CHUNK", "1024")
    c = KmerCounter(ref_k)
    try:
        c.restrict(g)
        for rd in reads:
            c.add([rd])
        got_k, got_c = c.finish(1, 255)
        assert np.array_equal(got_k, want_k) and np.array_equal(got_c, want_c)
        parts_k, parts_c = [], []
        for lo, hi in ((0, 70), (70, 71), (71, 256)):
            c.reset()
            c.set_partition(8, lo, hi)
            c.add(reads)
            pk, pc = c.finish(1, 255)
            parts_k.append(pk)
            parts_c.append(pc)
        assert np.array_equal(np.concatenate(parts_k), want_k) and np.array_equal(np.concatenate(parts_c), want_c)
        assert c.stats()["windows"] > c.stats()["instances"]
    finally:
        c.close()
        g.close()


def test_restricted_table_is_smaller(monkeypatch):
    """reads that mostly miss the index, 64 KiB device chunks: the restricted table stays at most 1/8 of the full one"""
    k, ref_k = 35, 43
    _, genome, _, ks, fl, reads = _case(k, ref_k, 5200)
    rnd = np.frombuffer(b"ACGT", np.uint8)[np.random.default_rng(5).integers(0, 4, 1_500_000)].tobytes().decode()
    reads = reads + [rnd[i:i + 150] for i in range(0, len(rnd), 150)]
    g = _index(k, ref_k, SPARSE, ks, fl, genome)
    monkeypatch.setenv("MG_COUNT_CHUNK", str(1 << 16))
    r, u = KmerCounter(ref_k), KmerCounter(ref_k)
    try:
        r.restrict(g)
        r.add(reads)
        u.add(reads)
        sr, su = r.stats(), u.stats()
        assert sr["capacity"] * 8 <= su["capacity"], (sr, su)
        assert sr["windows"] == su["instances"] and sr["instances"] * 8 < su["instances"]
    finally:
        r.close(), u.close(), g.close()


def test_restrict_errors_and_lifting():
    k, ref_k = 35, 43
    _, genome, _, ks, fl, reads = _case(k, ref_k, 5300)
    g = _index(k, ref_k, SPARSE, ks, fl, genome)
    raw = MalvaGpu(k=k, ref_k=ref_k, bf_bits=SPARSE)      # not finalized
    wrong_k = KmerCounter(39)
    c, full = KmerCounter(ref_k), KmerCounter(ref_k)
    try:
        with pytest.raises(MalvaGpuError, match="error -1:"):       # MG_ERR_ARG: the counter's k is not ref_k
            wrong_k.restrict(g)
        raw.add_signatures(ks[:10], fl[:10])
        with pytest.raises(MalvaGpuError, match="error -3:.*mg_finalize_alt"):
            c.restrict(raw)
        c.add(reads[:10])
        with pytest.raises(MalvaGpuError, match="error -3:.*not empty"):
            c.restrict(g)
        c.finish(2, 255)
        with pytest.raises(MalvaGpuError, match="error -3:"):
            c.restrict(g)
        c.reset()
        c.restrict(g)                                              # fresh after a reset
        c.add(reads)
        with pytest.raises(MalvaGpuError, match="error -3:"):
            c.restrict(None)
        c.reset()
        c.restrict(None)                                           # lifted: a full count again
        c.add(reads)
        full.add(reads)
        ck, cc = c.finish(1, 255)
        fk, fc = full.finish(1, 255)
        assert np.array_equal(ck, fk) and np.array_equal(cc, fc)
        assert c.stats()["windows"] == c.stats()["instances"] == full.stats()["instances"]
        if _n_gpus() > 1:
            other = KmerCounter(ref_k, device=1)
            try:
                with pytest.raises(MalvaGpuError, match="error -1:.*different devices"):
                    other.restrict(g)
            finally:
                other.close()
    finally:
        g.close(), raw.close(), wrong_k.close(), c.close(), full.close()


def _n_gpus() -> int:
    from malva_b200 import _lib

    return _lib.load().mg_device_count()


def _run(args, cwd=None):
    mbuild.build()
    return subprocess.run([mbuild.CLI] + [str(a) for a in args], capture_output=True, cwd=cwd)


@pytest.mark.parametrize("verbose,golden", [(False, "haploid.malva.vcf"), (True, "haploid.malva.verbose.vcf")])
def test_cli_call_reads_prints_the_shipped_golden(verbose, golden, tmp_path):
    """README.md:137's example from its reads, plain and gz, in one `call --reads`: the shipped VCF, no database"""
    for f in ("haploid.fa", "haploid.vcf.gz", "haploid.fq.gz"):
        os.symlink(os.path.join(GOLD, f), tmp_path / f)
    (tmp_path / "haploid.fq").write_bytes(gzip.open(os.path.join(GOLD, "haploid.fq.gz")).read())
    flags = ["-1", "-k", "35", "-r", "43", "-b", "1", "-f", "AF"]
    fa, vcf = tmp_path / "haploid.fa", tmp_path / "haploid.vcf.gz"
    r = _run(["index"] + flags + [fa, vcf, os.path.join(GOLD, "haploid")])   # (index opens a database, unused)
    assert r.returncode == 0, r.stderr.decode()[-2000:]
    expected = open(os.path.join(GOLD, golden), "rb").read()
    for reads in ("haploid.fq", "haploid.fq.gz"):
        r = _run(["call"] + flags + (["-v"] if verbose else []) + [fa, vcf, tmp_path / reads, "--reads", "--trace"])
        assert r.returncode == 0, r.stderr.decode()[-2000:]
        assert r.stdout == expected, ts.first_diff(r.stdout, expected)
        for label in (b"KMC output processing", b"BF weights created", b"VCF parsing and genotyping"):
            assert b"[malva-geno/" + label + b"] Execution Time" in r.stderr
        assert re.search(rb"\[trace\] reads .*: \d+ read bytes, \d+ windows examined, \d+ distinct kept", r.stderr)
    assert not [f for f in os.listdir(tmp_path) if ".kmc_" in f], "no database is written"


@pytest.fixture(scope="module")
def read_cohort(tmp_path_factory):
    """haploid_af's panel and index, three read files of donors of it (one gz) and an empty one, and what
    `count` + `call DB` prints for each alone"""
    case = ts._case("haploid_af")
    d = str(tmp_path_factory.mktemp("reads_cohort"))
    fa, vcf, prefix, _ = synth.build_case(case, d)
    rng = random.Random(case.seed)               # (the order of build_case: reference, then variants)
    refs = synth.make_reference(rng, case.contigs)
    recs = synth.make_variants(rng, refs, case.mean_gap, case.n_samples, case.haploid, k=case.k)
    files = []
    for seed, name in ((61, "d61.fq"), (62, "d62.fq.gz"), (63, "d63.fq")):
        haps = synth.donor_haplotypes(random.Random(seed), refs, recs, case.haploid)
        path = os.path.join(d, name)
        synth_reads.write_reads(path, [h for hs in haps.values() for h in hs], 12, seed)
        files.append(path)
    files.append(os.path.join(d, "empty.fq"))
    open(files[-1], "wb").close()
    flags = ts.mk.cli_flags(case, d)
    r = _run(["index"] + flags + [fa, vcf, prefix])
    assert r.returncode == 0, r.stderr.decode()[-2000:]
    single = {}
    for f in files:
        db = f + ".db"
        r = _run(["count", f"-k{case.ref_k}", f, db])
        assert r.returncode == 0, r.stderr.decode()[-2000:]
        r = _run(["call"] + flags + [fa, vcf, db])
        assert r.returncode == 0, r.stderr.decode()[-2000:]
        single[os.path.basename(f)] = r.stdout
    assert len(set(single.values())) == len(single), "the donors are not told apart"
    return {"fa": fa, "vcf": vcf, "flags": flags, "files": files, "single": single, "dir": d}


def _device_sets():
    sets = [None, "0,0"]
    n = _n_gpus()
    if n > 1:
        sets.append(",".join(str(i) for i in range(n)))
    return sets


@pytest.mark.parametrize("devices", _device_sets())
def test_cli_call_reads_cohort_equals_count_then_call(read_cohort, devices, tmp_path):
    c = read_cohort
    out = tmp_path / "out"
    extra = ["--sample-devices", devices] if devices else []
    r = _run(["call"] + c["flags"] + extra + [c["fa"], c["vcf"]] + c["files"] + ["--reads", "--out-dir", out])
    assert r.returncode == 0, r.stderr.decode()[-2000:]
    assert r.stdout == b""
    assert sorted(os.listdir(out)) == sorted(os.path.basename(f) + ".vcf" for f in c["files"])
    for f in c["files"]:
        b = os.path.basename(f)
        got = open(out / (b + ".vcf"), "rb").read()
        assert got == c["single"][b], (b, ts.first_diff(got, c["single"][b]))


def test_cli_call_reads_refusals(read_cohort, tmp_path):
    c = read_cohort
    out = tmp_path / "out"
    r = _run(["call", "--devices", "0,0"] + c["flags"] + [c["fa"], c["vcf"], c["files"][0], "--reads"])
    assert r.returncode == 1 and b"--reads" in r.stderr and b"--devices" in r.stderr, r.stderr
    r = _run(["call"] + c["flags"] + [c["fa"], c["vcf"], c["files"][0], tmp_path / "missing.fq", "--reads",
                                      "--out-dir", out])
    assert r.returncode == 1 and b"cannot open" in r.stderr and b"missing.fq" in r.stderr, r.stderr
    flags64 = [x if x != "43" else "64" for x in c["flags"]]
    assert flags64 != c["flags"]
    r = _run(["call"] + flags64 + [c["fa"], c["vcf"], c["files"][0], "--reads"])
    assert r.returncode == 1 and b"k <= 63" in r.stderr, r.stderr
    assert not os.path.exists(out), "nothing is written after an argument error"
