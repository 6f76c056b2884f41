"""A cohort over several contexts: index replicas made by device-to-device copies (mg_replicate) and `malva-geno call
... --out-dir DIR --sample-devices A,B,..`, which spreads every round's samples over replicas of one index.

A replica must hold exactly its source's image -- filters, keys, overflow table, rank directory and every live
counter -- at every probe-line key layout and at the filter sizes where counters live in different places, and it must
be independent of its source afterwards.  A CLI run over N databases on several contexts must write, per database, the
bytes a single-database run prints."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from malva_b200 import MalvaGpu, MalvaGpuError, SignatureBatch, kmc
from malva_b200 import _lib
from malva_b200 import build as mbuild
from malva_b200._lib import check
from malva_b200.api import PackedSignatureBatch
import parity_util as util
import test_gpu_samples as ts

pytestmark = pytest.mark.gpu


def _n_gpus() -> int:
    import torch

    return torch.cuda.device_count()


def _export_bits(g, which: int) -> np.ndarray:
    n = C.c_uint64(0)
    check(g._L.mg_export_set_bits(g._h, which, None, 0, C.byref(n)))
    out = np.zeros(max(n.value, 1), np.uint64)
    check(g._L.mg_export_set_bits(g._h, which, out.ctypes.data_as(util.u64p), n.value, C.byref(n)))
    return out[:n.value]


def _export_keys(g) -> list:
    n = C.c_uint64(0)
    check(g._L.mg_export_ref_keys(g._h, None, 0, C.byref(n)))
    out = np.zeros(max(2 * n.value, 2), np.uint64)
    check(g._L.mg_export_ref_keys(g._h, out.ctypes.data_as(util.u64p), n.value, C.byref(n)))
    return sorted(kmc.packed_to_ints(out[:2 * n.value].view(kmc.KMER_DTYPE)))   # (emitted in a racing order)


def _state(g, pb, queries) -> dict:
    """everything a context answers about its index and counters"""
    q, ks, ctx_q = queries
    return {"stats": g.index_stats(), "kmap_size": g.kmap_size(),
            "bits": [_export_bits(g, w) for w in (0, 1)], "keys": _export_keys(g),
            "test_keys": [g.test_keys(0, q), g.test_keys(1, ctx_q), g.test_keys(2, ks)],
            "counters": util.counter_arrays(g),
            "genotypes": [g.genotype_packed(pb, 0.001, 10 ** 9, h) for h in (False, True)]}


def _same_state(a: dict, b: dict, what: str) -> None:
    assert a["stats"] == b["stats"] and a["kmap_size"] == b["kmap_size"], what
    for w in (0, 1):
        assert np.array_equal(a["bits"][w], b["bits"][w]), (what, "bits", w)
    assert a["keys"] == b["keys"], (what, "ref keys")
    for w in range(3):
        assert np.array_equal(a["test_keys"][w], b["test_keys"][w]), (what, "test_keys", w)
    for i in range(3):
        assert np.array_equal(a["counters"][i], b["counters"][i]), (what, "counters", i)
    for h in (0, 1):
        ts._same(a["genotypes"][h], b["genotypes"][h], f"{what} haploid={bool(h)}")


def _replica_parity(oracle_lib, k, ref_k, bf_bits, device):
    rng, genome, nested, freqs, top_ref, top_alt = ts._index(oracle_lib, k, ref_k, bf_bits, 7100 + k + bf_bits % 991)
    ks, fl = util.flatten(nested)
    samples = ts._samples(rng, genome, nested, k, ref_k, [top_ref, top_alt], 3)
    pb = PackedSignatureBatch.from_batch(SignatureBatch.from_nested(nested, freqs), k)
    queries = (ks + [util.rand_seq(rng, k) for _ in range(300)], ks,
               [genome[p:p + ref_k] for p in range(0, len(genome) - ref_k, 37)])
    g = ts._build(k, ref_k, bf_bits, genome, ks, fl)
    made = []

    def replicate(src):
        made.append(src.replicate(device))
        return made[-1]

    try:
        early = replicate(g)                      # before the scan, then fed the same scan
        g.scan_sample_kmers(*samples[0])
        early.scan_sample_kmers(*samples[0])
        r = replicate(g)
        rr = replicate(r)                         # a replica of a replica
        direct = replicate(g)                     # read again after g is destroyed
        want = _state(g, pb, queries)
        assert want["stats"]["irregular_ref_keys"] > 0 and any(c.any() for c in want["counters"])
        if bf_bits != ts.SPARSE:
            assert want["stats"]["overflow_keys"] > 0
        for x, what in ((r, "replica"), (rr, "replica of a replica"), (early, "replica fed the same scan")):
            _same_state(_state(x, pb, queries), want, what)

        # the replica is independent of its source: scanning into it leaves the source's counters alone
        r.scan_sample_kmers(*samples[2])
        after = util.counter_arrays(g)
        assert all(np.array_equal(a, b) for a, b in zip(want["counters"], after)), "a scan into the replica reached the source"
        assert not all(np.array_equal(a, b) for a, b in zip(util.counter_arrays(r), after))

        # a sample set on a replica: the same columns as on the source
        s = replicate(g)
        for x in (g, s):
            x.samples_begin(2)
            x.samples_take(0)                     # samples[0], scanned before the replica was made
            x.scan_sample_kmers(*samples[1])
            x.samples_take(1)
        got, exp = s.genotype_samples_packed(pb, 0.001, 10 ** 9, False), g.genotype_samples_packed(pb, 0.001, 10 ** 9, False)
        for i in range(2):
            ts._same(got[i], exp[i], f"sample set column {i}")
        assert not np.array_equal(exp[0].cov, exp[1].cov)

        # a replica keeps working once its source is gone
        g.close()
        _same_state(_state(direct, pb, queries), want, "replica after the source was destroyed")
    finally:
        g.close()
        for x in made:
            x.close()


@pytest.mark.parametrize("bf_bits", ts.FILTERS)
@pytest.mark.parametrize("k,ref_k", ts.LAYOUTS)
def test_replica_equals_source(oracle_lib, k, ref_k, bf_bits):
    """a replica on the same device answers exactly like its source: index stats, exported bits and keys, filter
    queries, counter images, genotypes with their likelihood bits, and sample-set columns"""
    _replica_parity(oracle_lib, k, ref_k, bf_bits, 0)


def test_replica_on_another_device(oracle_lib):
    if _n_gpus() < 2:
        pytest.skip("one GPU")
    _replica_parity(oracle_lib, 35, 43, ts.MODULO, 1)


def test_replicate_errors():
    L = _lib.load()
    h = C.c_void_p()
    g = MalvaGpu(k=35, ref_k=43, bf_bits=ts.MODULO)
    try:
        assert L.mg_replicate(None, None, 0) == -1
        assert L.mg_replicate(None, g._h, 0) == -1
        assert L.mg_replicate(C.byref(h), None, 0) == -1 and not h.value
        with pytest.raises(MalvaGpuError, match="error -3:"):
            g.replicate(0)
        g.add_signatures(["A" * 35, "C" * 35], [0, 1])
        g.finalize_alt()
        for bad in (-1, L.mg_device_count()):
            with pytest.raises(MalvaGpuError, match="error -2:"):
                g.replicate(bad)
        r = g.replicate(0)
        assert r.index_stats() == g.index_stats() and r.kmap_size() == g.kmap_size() == 1
        r.close()
    finally:
        g.close()


# ------------------------------------------------------------------------------------------------------------------
# CLI: call ... DB1 .. DBn --out-dir DIR --sample-devices A,B,..
def _device_sets():
    n = _n_gpus()
    two = pytest.mark.skipif(n < 2, reason="one GPU")
    return [pytest.param("0,0", id="0,0"), pytest.param("0,0,0", id="0,0,0"),
            pytest.param("0,1", id="0,1", marks=two),
            pytest.param(",".join(str(d) for d in range(max(n, 2))), id="all", marks=two)]


@pytest.fixture(scope="module")
def cli():
    mbuild.build()
    return mbuild.CLI


class Cohort:
    """a case, its index and its donors, with the single-database output of every donor"""

    def __init__(self, cli, name, verbose, workdir, seeds, empty=()):
        self.case = ts._case(name)
        self.fa, self.vcf, self.prefix, donors = ts._donors(self.case, workdir, seeds, empty)
        self.dbs = donors + [self.prefix]
        self.flags = ts.mk.cli_flags(self.case, workdir) + (["-v"] if verbose else [])
        ts._index_case(cli, ts.mk.cli_flags(self.case, workdir), self.fa, self.vcf, self.prefix)
        self.single = {os.path.basename(d): ts._single(cli, self.flags, self.fa, self.vcf, d) for d in self.dbs}


@pytest.fixture(scope="module")
def cohorts(cli, tmp_path_factory):
    """4 databases (one of them empty) of cfg3_chr1_like_snv_indel with -v, and 5 of haploid_af"""
    return {"cfg3_chr1_like_snv_indel": Cohort(cli, "cfg3_chr1_like_snv_indel", True,
                                               str(tmp_path_factory.mktemp("cfg3")), [31, 32, 33], empty=(32,)),
            "haploid_af": Cohort(cli, "haploid_af", False, str(tmp_path_factory.mktemp("hap")), [41, 42, 43, 44],
                                 empty=(42,))}


def _run(cli, args):
    return subprocess.run([cli] + list(args), capture_output=True)


def _spread(cli, flags, fa, vcf, dbs, out_dir, devices):
    """the per-database files of one call on --sample-devices `devices` (None: one context), and the sets per
    context of every round (--trace)"""
    extra = ["--trace"] + (["--sample-devices", devices] if devices else [])
    r = _run(cli, ["call"] + flags + extra + [fa, vcf] + list(dbs) + ["--out-dir", str(out_dir)])
    assert r.returncode == 0, r.stderr.decode()[-2000:]
    assert r.stdout == b"", "several databases write nothing to stdout"
    assert sorted(os.listdir(out_dir)) == sorted(os.path.basename(d) + ".vcf" for d in dbs)
    rounds = [[int(x) for x in m.split()] for m in re.findall(rb"sets per context:([ 0-9]*)\n", r.stderr)]
    return {os.path.basename(d): open(os.path.join(out_dir, os.path.basename(d) + ".vcf"), "rb").read() for d in dbs}, rounds


@pytest.mark.parametrize("devices", _device_sets())
@pytest.mark.parametrize("name", ["cfg3_chr1_like_snv_indel", "haploid_af"])
def test_cli_spread_equals_single_runs(cli, cohorts, name, devices, tmp_path):
    """4 databases, one of them empty, over several contexts: every file equals the single-database call"""
    c = cohorts[name]
    dbs = c.dbs[-4:]
    got, rounds = _spread(cli, c.flags, c.fa, c.vcf, dbs, tmp_path / "out", devices)
    n_ctx = len(devices.split(","))
    per = -(-4 // n_ctx)
    assert rounds == [[min(per, max(0, 4 - per * i)) for i in range(n_ctx)]]
    for d in dbs:
        b = os.path.basename(d)
        assert got[b] == c.single[b], (d, ts.first_diff(got[b], c.single[b]))
    assert len(set(got.values())) == len(got), "the donors are not told apart"


def test_cli_five_over_three_contexts(cli, cohorts, tmp_path):
    """5 databases over 0,0,0 split 2/2/1; every file equals the single-database call"""
    c = cohorts["haploid_af"]
    got, rounds = _spread(cli, c.flags, c.fa, c.vcf, c.dbs, tmp_path / "out", "0,0,0")
    assert len(c.dbs) == 5 and rounds == [[2, 2, 1]]
    for d in c.dbs:
        b = os.path.basename(d)
        assert got[b] == c.single[b], (d, ts.first_diff(got[b], c.single[b]))


def test_cli_65_over_two_contexts(cli, tmp_path):
    """65 databases over 0,0: a round of 32 + 32 and a round in which the second context is idle; every file equals
    the one-context --out-dir run (three rounds of 32, 32 and 1)"""
    case = ts._case("haploid_af")
    fa, vcf, prefix, dbs = ts._donors(case, str(tmp_path), list(range(500, 565)))
    flags = ts.mk.cli_flags(case, str(tmp_path)) + ["-v"]
    ts._index_case(cli, ts.mk.cli_flags(case, str(tmp_path)), fa, vcf, prefix)
    want, rounds = _spread(cli, flags, fa, vcf, dbs, tmp_path / "one", None)
    assert rounds == [[32], [32], [1]]
    got, rounds = _spread(cli, flags, fa, vcf, dbs, tmp_path / "two", "0,0")
    assert rounds == [[32, 32], [1, 0]]
    assert len(got) == 65
    for d in dbs:
        b = os.path.basename(d)
        assert got[b] == want[b], (d, ts.first_diff(got[b], want[b]))


def test_cli_sample_devices_errors(cli, cohorts, tmp_path):
    c = cohorts["haploid_af"]
    out = str(tmp_path / "out")
    r = _run(cli, ["call", "--sample-devices", "0,0"] + c.flags + [c.fa, c.vcf, c.dbs[0]])
    assert r.returncode == 1 and b"--sample-devices" in r.stderr, r.stderr
    r = _run(cli, ["call", "--sample-devices", "0,0", "--devices", "0"] + c.flags + [c.fa, c.vcf] + c.dbs[:2]
             + ["--out-dir", out])
    assert r.returncode == 1 and b"--sample-devices" in r.stderr and b"--devices" in r.stderr, r.stderr
    r = _run(cli, ["call", "--sample-devices", "0,0", "--device", "0"] + c.flags + [c.fa, c.vcf] + c.dbs[:2]
             + ["--out-dir", out])
    assert r.returncode == 1 and b"--sample-devices" in r.stderr and b"--device " in r.stderr, r.stderr
    r = _run(cli, ["call", "--sample-devices", f"0,{_n_gpus()}"] + c.flags + [c.fa, c.vcf] + c.dbs[:2]
             + ["--out-dir", out])
    assert r.returncode == 1 and b"not visible" in r.stderr, r.stderr
    assert not os.path.exists(out) or not os.listdir(out), "nothing is written after an argument error"
