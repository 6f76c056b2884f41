"""Sample sets: several samples genotyped against one index (include/malva_gpu.h, mg_samples_*), and `malva-geno call`
with several KMC databases.

A sample set keeps one u32 column per sample over the counter rows of the index; mg_samples_take moves the live
counters into a column and zeroes them, the sample-set look-up reads the rows of a batch for every column at once.
Column s must genotype exactly like a fresh context that scanned sample s alone, at every probe-line key layout and at the
filter sizes where counters live in different places (overflowed keys, set bits past the three inline counters of a
line, the partial last line), and a CLI run over N databases must write, per database, the bytes a single-database
run prints."""
import ctypes as C
import gzip
import os
import random
import subprocess
import sys

import numpy as np
import pytest

from malva_b200 import MalvaGpu, MalvaGpuError, SignatureBatch, kmc
from malva_b200.api import IRREGULAR_BIT, PackedSignatureBatch
import parity_util as util

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import make_cli_golden as mk  # noqa: E402
import synth  # noqa: E402
from malva_b200 import build as mbuild  # noqa: E402

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")

LAYOUTS = [(35, 43), (31, 39), (47, 55), (48, 56), (63, 64)]
DENSE, MODULO, SPARSE = 1 << 13, 3 * (1 << 12) + 7, 1 << 22
FILTERS = [pytest.param(DENSE, id="2^13"), pytest.param(MODULO, id="3x2^12+7"), pytest.param(SPARSE, id="2^22")]
FIELDS = ("cov", "n_gts", "status", "best_gt", "gq")


def _find_kmers(L, k: int, bf_bits: int, lo: int, n: int = 1) -> list:
    """n k-mers of k ACGT symbols whose filter index is >= lo (searched in the oracle)"""
    out = C.create_string_buffer((k + 1) * n)
    assert L.mo_find_kmers_at(b"A" * k, k, bf_bits, lo, 0, 1 << 28, out, n) == n
    return [out.raw[j * (k + 1):j * (k + 1) + k].decode() for j in range(n)]


def _window(rng, kmer: str, k: int, ref_k: int) -> str:
    d = (ref_k - k) // 2
    return util.rand_seq(rng, d) + kmer + util.rand_seq(rng, ref_k - k - d)


def _index(oracle_lib, k, ref_k, bf_bits, seed):
    """genome, signatures (irregular k-mers included) and a variant whose ref and alt k-mers sit in the last 7 bits
    of the filter (the partial last probe line of the modulo filter)"""
    rng = random.Random(seed)
    genome = util.make_genome(rng, 30000)
    nested, freqs = util.synth_signatures(rng, genome, k, 700)
    top_ref, top_alt = _find_kmers(oracle_lib, k, bf_bits, bf_bits - 7, n=2)
    nested.append([[[top_ref]], [[top_alt]]])
    freqs.append([0.7, 0.3])
    return rng, genome, nested, freqs, top_ref, top_alt


def _build(k, ref_k, bf_bits, genome, ks, fl):
    g = MalvaGpu(k=k, ref_k=ref_k, bf_bits=bf_bits)
    g.add_signatures(ks, fl)
    g.finalize_alt()
    g.scan_reference(genome)
    g.finalize_context()
    return g


def _samples(rng, genome, nested, k, ref_k, top, n):
    """n samples of the panel; sample 1 with counts past 2^16 per record (bf counters wrap uint16 in get_count)"""
    out = []
    for s in range(n):
        _, packed, counts = util.synth_sample(random.Random(rng.randrange(1 << 30)), genome, nested, k, ref_k,
                                              6000 + 1500 * s, big_counts=s == 1)
        tw = kmc.ints_to_packed([kmc.pack_kmer(_window(rng, t, k, ref_k)) for t in top])
        out.append((np.concatenate([packed, tw]), np.concatenate([counts, np.full(len(top), 300 + s, np.uint32)])))
    return out


def _line_positions(words: np.ndarray, bf_bits: int):
    pos = np.flatnonzero(np.unpackbits(words.view(np.uint8), bitorder="little"))
    pos = pos[pos < bf_bits]
    line = pos >> 8
    return line, np.arange(len(pos)) - np.searchsorted(line, line, side="left")


def _same(a, b, what) -> None:
    for f in FIELDS:
        assert np.array_equal(getattr(a, f), getattr(b, f)), (what, f)
    for v in range(len(a.n_gts)):           # (the slots past n_gts of a variant are not written)
        sl = slice(int(a.lik_off[v]), int(a.lik_off[v]) + int(a.n_gts[v]))
        assert np.array_equal(a.lik[sl].view(np.uint64), b.lik[sl].view(np.uint64)), (what, "lik", v)


@pytest.mark.parametrize("bf_bits", FILTERS)
@pytest.mark.parametrize("k,ref_k", LAYOUTS)
def test_columns_equal_fresh_contexts(oracle_lib, k, ref_k, bf_bits):
    """every column of a set genotypes exactly like a fresh context that scanned that sample alone (cov, n_gts,
    status, GT, GQ and the likelihood bits), diploid and haploid; the inputs reach overflowed keys, set bits past the
    inline counters of their line, the partial last line, and irregular k-mers on both sides"""
    rng, genome, nested, freqs, top_ref, top_alt = _index(oracle_lib, k, ref_k, bf_bits, 9300 + k + bf_bits % 997)
    ks, fl = util.flatten(nested)
    n = 3
    samples = _samples(rng, genome, nested, k, ref_k, [top_ref, top_alt], n)
    batch = SignatureBatch.from_nested(nested, freqs)
    pb = PackedSignatureBatch.from_batch(batch, k)
    assert (pb.kmers["hi"] & np.uint64(IRREGULAR_BIT)).any() and len(pb.irr_kmer) > 5
    g = _build(k, ref_k, bf_bits, genome, ks, fl)
    o = util.OracleRun(oracle_lib, k, ref_k, bf_bits)
    try:
        o.add_signatures(ks, fl)
        o.finalize_alt()
        o.scan_reference(genome)
        o.finalize_context()
        g.samples_begin(n)
        for s, (p, c) in enumerate(samples):
            g.scan_sample_kmers(p, c)
            if s == 1:   # the edges this filter size is there for, on the sample with the big counts
                o.scan_sample_kmers(p, c)
                st = g.index_stats()
                line, j = _line_positions(o.bits(0), bf_bits)
                counts = o.bf_counts()
                if bf_bits in (DENSE, MODULO):
                    assert st["overflow_keys"] > 0
                    assert counts[line == st["probe_lines"] - 1].any(), "the last line's counters are never hit"
                if bf_bits == MODULO:
                    assert (j >= 3).any() and counts[j >= 3].any(), "no counted bit past the inline counters"
                assert (counts.astype(np.int64) > 0).any()
            g.samples_take(s)
        for haploid in (False, True):
            got = g.genotype_samples_packed(pb, 0.001, 10 ** 9, haploid)
            assert len(got) == n
            for s, (p, c) in enumerate(samples):
                f = _build(k, ref_k, bf_bits, genome, ks, fl)
                try:
                    f.scan_sample_kmers(p, c)
                    exp = f.genotype_packed(pb, 0.001, 10 ** 9, haploid)
                finally:
                    f.close()
                _same(got[s], exp, f"sample {s} haploid={haploid}")
                assert (exp.cov > 0).sum() > 100
    finally:
        g.close()
        o.close()


def test_take_resets_and_semantics(oracle_lib):
    """after take every live counter is 0; a sample scanned after a take is not contaminated by the one before; a
    column never taken genotypes as no coverage; a set of one equals genotype_packed on the live counters; misuse
    is refused"""
    k, ref_k, bf_bits = 35, 43, MODULO
    rng, genome, nested, freqs, top_ref, top_alt = _index(oracle_lib, k, ref_k, bf_bits, 4711)
    ks, fl = util.flatten(nested)
    samples = _samples(rng, genome, nested, k, ref_k, [top_ref, top_alt], 2)
    batch = SignatureBatch.from_nested(nested, freqs)
    pb = PackedSignatureBatch.from_batch(batch, k)
    q = ks + [util.rand_seq(rng, k) for _ in range(100)]
    g = _build(k, ref_k, bf_bits, genome, ks, fl)
    try:
        with pytest.raises(MalvaGpuError, match="error -3:"):
            g.genotype_samples_packed(pb, n_samples=1)
        with pytest.raises(MalvaGpuError, match="error -3:"):
            g.samples_take(0)
        with pytest.raises(MalvaGpuError, match="error -1:"):
            g.samples_begin(33)
        with pytest.raises(MalvaGpuError, match="error -1:"):
            g.samples_begin(0)

        # G = 1 on the live counters
        g.scan_sample_kmers(*samples[0])
        live = g.genotype_packed(pb, 0.001, 150, False)
        before = [g.get_counts(q, [f] * len(q)) for f in (0, 1)]
        assert before[0].any() and before[1].any()
        g.samples_begin(1)
        g.samples_take(0)
        for f in (0, 1):
            assert not g.get_counts(q, [f] * len(q)).any(), f"live counters after take (is_ref={f})"
        assert not g.bf_counts().any()
        _same(g.genotype_samples_packed(pb, 0.001, 150, False)[0], live, "G=1")
        with pytest.raises(MalvaGpuError, match="error -1:"):
            g.genotype_samples_packed(pb, n_samples=2)
        with pytest.raises(MalvaGpuError, match="error -1:"):
            g.samples_take(1)
        with pytest.raises(MalvaGpuError, match="error -1:"):
            g.samples_take(-1)

        # a new set: sample 1 scanned after the take of sample 0 is not contaminated; column 2 is never taken
        g.samples_begin(3)
        g.scan_sample_kmers(*samples[0])
        g.samples_take(0)
        g.scan_sample_kmers(*samples[1])
        g.samples_take(1)
        res = g.genotype_samples_packed(pb, 0.001, 150, False)
        for s in (0, 1):
            f = _build(k, ref_k, bf_bits, genome, ks, fl)
            try:
                f.scan_sample_kmers(*samples[s])
                _same(res[s], f.genotype_packed(pb, 0.001, 150, False), f"sample {s}")
            finally:
                f.close()
        nonempty = np.diff(pb.var_allele_off.astype(np.int64)) > 0
        assert (res[2].status[nonempty] == 2).all() and not res[2].cov.any()
        # the live path still works after the set: the same scan genotypes like before
        g.scan_sample_kmers(*samples[0])
        _same(g.genotype_packed(pb, 0.001, 150, False), live, "live after sets")
        g.samples_end()
        with pytest.raises(MalvaGpuError, match="error -3:"):
            g.genotype_samples_packed(pb, n_samples=3)
    finally:
        g.close()


# ------------------------------------------------------------------------------------------------------------------
# CLI: call with several databases
@pytest.fixture(scope="module")
def cli():
    mbuild.build()
    return mbuild.CLI


def _case(name):
    return next(c for c in synth.CASES if c.name == name)


def _donors(case, workdir, seeds, empty=()):
    """the case's inputs, its index, and one KMC database per seed: a donor of the same panel (synth.donor_haplotypes
    with its own random.Random), or an empty database for the seeds in `empty`"""
    fa, vcf, prefix, _ = synth.build_case(case, workdir)
    rng = random.Random(case.seed)               # (the order of build_case: reference, then variants)
    refs = synth.make_reference(rng, case.contigs)
    recs = synth.make_variants(rng, refs, case.mean_gap, case.n_samples, case.haploid, k=case.k)
    dbs = []
    for seed in seeds:
        p = os.path.join(workdir, f"donor{seed}")
        if seed in empty:
            kmc.write_kmc_db(p, np.zeros(0, kmc.KMER_DTYPE), np.zeros(0, np.uint32), case.ref_k)
        else:
            r = random.Random(seed)
            synth.sample_kmc_db(r, p, synth.donor_haplotypes(r, refs, recs, case.haploid), case.ref_k, case.mean_cov)
        dbs.append(p)
    return fa, vcf, prefix, dbs


def _run(cli, args):
    return subprocess.run([cli] + list(args), capture_output=True)


def _index_case(cli, flags, fa, vcf, prefix):
    r = _run(cli, ["index"] + flags + [fa, vcf, prefix])
    assert r.returncode == 0, r.stderr.decode()[-2000:]


def _single(cli, flags, fa, vcf, db):
    r = _run(cli, ["call"] + flags + [fa, vcf, db])
    assert r.returncode == 0, r.stderr.decode()[-2000:]
    return r.stdout


def _multi(cli, flags, fa, vcf, dbs, out_dir):
    r = _run(cli, ["call"] + flags + [fa, vcf] + list(dbs) + ["--out-dir", str(out_dir)])
    assert r.returncode == 0, r.stderr.decode()[-2000:]
    assert r.stdout == b"", "several databases write nothing to stdout"
    return {os.path.basename(d): open(os.path.join(out_dir, os.path.basename(d) + ".vcf"), "rb").read() for d in dbs}


@pytest.mark.parametrize("name,verbose", [("cfg3_chr1_like_snv_indel", True), ("haploid_af", False)])
def test_cli_several_databases_equal_single_runs(cli, name, verbose, tmp_path):
    """three donors of the panel (one of them an empty database) and the case's own database in one call: every file
    equals the stdout of a call with that database alone, and the case's own equals its golden"""
    case = _case(name)
    fa, vcf, prefix, dbs = _donors(case, str(tmp_path), [11, 12, 13], empty=(12,))
    flags = mk.cli_flags(case, str(tmp_path)) + (["-v"] if verbose else [])
    _index_case(cli, mk.cli_flags(case, str(tmp_path)), fa, vcf, prefix)
    got = _multi(cli, flags, fa, vcf, dbs + [prefix], tmp_path / "out")
    assert sorted(os.listdir(tmp_path / "out")) == sorted(os.path.basename(d) + ".vcf" for d in dbs + [prefix])
    for d in dbs + [prefix]:
        want = _single(cli, flags, fa, vcf, d)
        assert got[os.path.basename(d)] == want, (d, first_diff(got[os.path.basename(d)], want))
    if verbose:
        golden = gzip.open(os.path.join(GOLD, "cli", case.name + ".expected.vcf.gz")).read()
        assert got["sample"] == golden, first_diff(got["sample"], golden)
    assert len({v for v in got.values()}) == len(got), "the donors are not told apart"


def test_cli_haploid_example_twice(cli, tmp_path):
    """the shipped haploid example given twice under two prefixes: both files equal its golden"""
    src = os.path.join(GOLD, "haploid")
    for f in ("haploid.fa", "haploid.vcf.gz"):
        os.symlink(os.path.join(src, f), tmp_path / f)
    for d in ("a", "b"):
        os.makedirs(tmp_path / d)
        for ext in ("kmc_pre", "kmc_suf"):
            os.symlink(os.path.join(src, "haploid." + ext), tmp_path / d / ("hap_" + d + "." + ext))
    flags = ["-1", "-k", "35", "-r", "43", "-b", "1", "-f", "AF"]
    fa, vcf = str(tmp_path / "haploid.fa"), str(tmp_path / "haploid.vcf.gz")
    _index_case(cli, flags, fa, vcf, str(tmp_path / "a" / "hap_a"))
    got = _multi(cli, flags, fa, vcf, [str(tmp_path / "a" / "hap_a"), str(tmp_path / "b" / "hap_b")], tmp_path / "out")
    expected = open(os.path.join(src, "haploid.malva.vcf"), "rb").read()
    for v in got.values():
        assert v == expected, first_diff(v, expected)


def test_cli_33_databases_cross_a_group(cli, tmp_path):
    """33 donors: two sample sets and two VCF passes; every file equals its single run"""
    case = _case("haploid_af")
    seeds = list(range(100, 133))
    fa, vcf, prefix, dbs = _donors(case, str(tmp_path), seeds)
    flags = mk.cli_flags(case, str(tmp_path))
    _index_case(cli, flags, fa, vcf, prefix)
    got = _multi(cli, flags + ["-v"], fa, vcf, dbs, tmp_path / "out")
    assert len(got) == 33
    for d in dbs:
        want = _single(cli, flags + ["-v"], fa, vcf, d)
        assert got[os.path.basename(d)] == want, (d, first_diff(got[os.path.basename(d)], want))


def test_cli_several_databases_errors(cli, tmp_path):
    case = _case("haploid_af")
    fa, vcf, prefix, dbs = _donors(case, str(tmp_path), [21])
    flags = mk.cli_flags(case, str(tmp_path))
    _index_case(cli, flags, fa, vcf, prefix)
    out = str(tmp_path / "out")
    r = _run(cli, ["call"] + flags + [fa, vcf, prefix, dbs[0]])
    assert r.returncode == 1 and b"--out-dir" in r.stderr, r.stderr
    os.makedirs(tmp_path / "other")
    for ext in ("kmc_pre", "kmc_suf"):
        os.symlink(dbs[0] + "." + ext, str(tmp_path / "other" / ("donor21." + ext)))
    r = _run(cli, ["call"] + flags + [fa, vcf, dbs[0], str(tmp_path / "other" / "donor21"), "--out-dir", out])
    assert r.returncode == 1 and b"donor21" in r.stderr and b"twice" in r.stderr, r.stderr
    r = _run(cli, ["call"] + flags + [fa, vcf, prefix, dbs[0] + "_nope", "--out-dir", out])
    assert r.returncode == 1 and b"ERROR: cannot open " + (dbs[0] + "_nope").encode() in r.stderr, r.stderr
    assert not os.path.exists(out) or not os.listdir(out), "nothing is written before every database is open"
    r = _run(cli, ["call", "--devices", "0,0"] + flags + [fa, vcf, prefix, dbs[0], "--out-dir", out])
    assert r.returncode == 1 and b"--devices" in r.stderr, r.stderr
    r = _run(cli, ["call"] + flags + [fa, vcf, prefix, "--out-dir", out])
    assert r.returncode == 1 and b"--out-dir" in r.stderr, r.stderr


def first_diff(a: bytes, b: bytes):
    la, lb = a.split(b"\n"), b.split(b"\n")
    for i, (x, y) in enumerate(zip(la, lb)):
        if x != y:
            return f"line {i + 1}:\n  got      {x[:400]!r}\n  expected {y[:400]!r}"
    return f"{len(la)} lines vs {len(lb)} expected"
