"""Host logic of the malva-geno CLI (malva_b200/csrc/host), checked on CPU against the reference's own
VB::extract_kmers (oracle/_ref hook) and block grouping rules: `malva-geno signatures` prints what the CLI would
send to the device for every var_block.  No GPU involved (the signatures sub-command never touches CUDA)."""
import hashlib
import os
import re
import subprocess

import pytest

import synth
import vcf_blocks
from malva_b200 import build as mbuild
from parity_util import check_digest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "haploid")


@pytest.fixture(scope="module")
def cli():
    mbuild.build()
    assert os.path.exists(mbuild.CLI)
    return mbuild.CLI


def cli_signatures(cli, fa, vcf, flags, index_mode):
    cmd = [cli, "signatures"] + (["--index-blocks"] if index_mode else []) + list(flags) + [fa, vcf]
    out = subprocess.run(cmd, capture_output=True, text=True, check=True).stdout
    blocks, used = {}, None
    for l in out.split("\n"):
        if not l:
            continue
        if l.startswith("#used"):
            used = l.split("\t")[1:]
            continue
        b, contig, pos, vi, allele, kmers = l.split("\t")
        blocks.setdefault(int(b), {}).setdefault((contig, int(pos), int(vi), int(allele)), set()).add(tuple(kmers.split(",")))
    return blocks, used


def expected_signatures(ref_lib, fa, vcf, k, haploid, freq_key, uniform, index_mode, strip_chr=False, sample_cols=None):
    refs, name = {}, None
    for l in open(fa):
        l = l.rstrip("\n")
        if l.startswith(">"):
            name = l[1:].split()[0]
            if strip_chr and name.startswith("chr"):
                name = name[3:]
            refs[name] = []
        else:
            refs[name].append(l.upper())
    refs = {n: "".join(v) for n, v in refs.items()}
    _, recs = vcf_blocks.read_vcf(vcf, freq_key, uniform, sample_cols)
    blocks, used = {}, []
    if recs:
        used.append(recs[0].chrom)
    for b, (contig, blk) in enumerate(vcf_blocks.blocks(recs, k, index_mode=index_mode)):
        if contig not in used or used[-1] != contig:
            used.append(contig)
        nested = vcf_blocks.ref_extract(ref_lib, blk, refs.get(contig, ""), k, haploid)
        for vi, v in enumerate(blk):
            for a, sigs in enumerate(nested[vi]):
                for s in sigs:
                    blocks.setdefault(b, {}).setdefault((contig, v.pos0 + 1, vi, a), set()).add(tuple(s))
    return blocks, used


def signatures_digest(blocks, used):
    h = hashlib.sha256()
    for b in sorted(blocks):
        for key in sorted(blocks[b]):
            h.update(repr((b, key, sorted(blocks[b][key]))).encode())
    h.update(repr(used).encode())
    return h.hexdigest()


def assert_reference_enumeration(ref_lib, key, got, used, *args, **kw):
    """`malva-geno signatures` (got, used) against the reference's VB::extract_kmers on the same files: live through
    oracle/_ref where it is built, else against the digest stored under `key` in tests/golden/signatures.json"""
    if ref_lib is not None:
        exp, exp_used = expected_signatures(ref_lib, *args, **kw)
        assert set(got) == set(exp), f"{key}: different set of blocks with signatures"
        for b in exp:
            assert got[b] == exp[b], f"{key}: block {b} differs"
        assert used == exp_used, key
    n = sum(len(v) for blk in got.values() for v in blk.values())
    check_digest("signatures", key, signatures_digest(got, used), ref_lib is not None, f"({n} signatures, {len(got)} blocks)")


def test_signatures_haploid_example(cli, ref_or_none):
    fa, vcf = os.path.join(GOLD, "haploid.fa"), os.path.join(GOLD, "haploid.vcf.gz")
    for index_mode in (True, False):
        got, used = cli_signatures(cli, fa, vcf, ["-1"], index_mode)
        assert_reference_enumeration(ref_or_none, f"haploid_example/index_mode={index_mode}", got, used,
                                     fa, vcf, 35, True, "AF", False, index_mode)


@pytest.mark.parametrize("case", synth.CASES, ids=[c.name for c in synth.CASES])
def test_signatures_synthetic(cli, ref_or_none, case, tmp_path):
    fa, vcf, _, _ = synth.build_case(case, str(tmp_path))
    uniform = "-u" in case.flags
    if case.sample_subset:
        # the Python twin of the reference reads all samples (the subset is compared with the reference end to end in
        # tests/test_gpu_cli.py); here: the reader's short cuts against its general paths on that case's files
        lst = os.path.join(str(tmp_path), "samples.txt")
        for extra in ([], ["--index-blocks"]):
            a = _signatures_text(cli, fa, vcf, extra + ["-u", "-s", lst], general=False)
            b = _signatures_text(cli, fa, vcf, extra + ["-u", "-s", lst], general=True)
            assert a.returncode == 0 and b.returncode == 0 and a.stdout == b.stdout and a.stdout.count("\n") > 100
        # ... and against VB::extract_kmers fed with the kept columns (header order, whatever the order of the list)
        for index_mode in (True, False):
            got, used = cli_signatures(cli, fa, vcf, ["-u", "-s", lst], index_mode)
            assert_reference_enumeration(ref_or_none, f"synthetic/{case.name}/index_mode={index_mode}", got, used,
                                         fa, vcf, case.k, case.haploid, case.freq_key, True, index_mode,
                                         strip_chr=case.chr_prefix, sample_cols=sorted(case.sample_subset))
        return
    sig_flags = [f for f in case.flags]
    # only the flags the enumeration depends on
    keep, it = [], iter(sig_flags)
    for f in it:
        if f in ("-k", "-f", "-r", "-e", "-c"):
            v = next(it)
            if f in ("-k", "-f"):
                keep += [f, v]
        else:
            keep.append(f)
    for index_mode in (True, False):
        got, used = cli_signatures(cli, fa, vcf, keep, index_mode)
        assert_reference_enumeration(ref_or_none, f"synthetic/{case.name}/index_mode={index_mode}", got, used,
                                     fa, vcf, case.k, case.haploid, case.freq_key, uniform, index_mode,
                                     strip_chr=case.chr_prefix)
        assert sum(len(v) for v in got.values()) > 100


def test_cli_usage_errors(cli):
    r = subprocess.run([cli], capture_output=True, text=True)
    assert r.returncode == 1 and "missing arguments" in r.stderr
    r = subprocess.run([cli, "frobnicate"], capture_output=True, text=True)
    assert r.returncode == 1 and "Could not interpret command" in r.stderr
    r = subprocess.run([cli, "call", "only_one.fa"], capture_output=True, text=True)
    assert r.returncode == 1 and "missing arguments" in r.stderr
    r = subprocess.run([cli, "index", "-h"], capture_output=True, text=True)
    assert r.returncode == 0 and "--bf-size" in r.stdout


@pytest.mark.parametrize("name", ["cfg4_wg_like_multiallelic", "haploid_af"])
def test_cli_goldens_are_what_the_reference_prints(name, tmp_path):
    """tests/golden/cli/*.expected.vcf.gz (used by the GPU end-to-end test) against the reference's own main.cpp
    (oracle/_ref/malva-geno-ref) run now on the regenerated inputs; the other cases are pinned by the manifest."""
    import gzip
    import hashlib
    import json
    import sys

    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import make_cli_golden as mk

    if not os.path.exists(mk.REF_BIN):
        pytest.skip("oracle/_ref/malva-geno-ref not built")
    case = next(c for c in synth.CASES if c.name == name)
    out, hashes, _ = mk.run_reference(case, str(tmp_path))
    manifest = json.load(open(os.path.join(mk.OUT, "manifest.json")))
    assert hashes == manifest[name]["inputs"]
    assert out == gzip.open(os.path.join(mk.OUT, name + ".expected.vcf.gz")).read()
    for n, m in manifest.items():
        blob = gzip.open(os.path.join(mk.OUT, n + ".expected.vcf.gz")).read()
        assert hashlib.sha256(blob).hexdigest() == m["expected_sha256"]


def test_kmc_dump_lists_what_the_python_reader_lists(cli, tmp_path):
    """csrc/host/kmc_db.hpp (the reader `call` uses) against malva_b200.kmc on the haploid database and on random
    databases in both prefix-file layouts"""
    import random

    import numpy as np

    from malva_b200 import kmc

    def dump(prefix):
        out = subprocess.run([cli, "kmc-dump", prefix], capture_output=True, text=True, check=True).stdout
        rows = [l.split("\t") for l in out.split("\n") if l]
        return [r[0] for r in rows], [int(r[1]) for r in rows]

    packed, counts, k = kmc.read_kmc_db(os.path.join(GOLD, "haploid"))
    ks, cs = dump(os.path.join(GOLD, "haploid"))
    assert ks == kmc.packed_to_strings(packed, k) and cs == counts.tolist() and len(ks) == 4503
    rng = random.Random(3)
    for k, version, p, csz in ((43, 0x200, 7, 1), (43, 0, 3, 2), (31, 0x200, 3, 1), (21, 0, 5, 4)):
        vals = sorted({rng.getrandbits(2 * k) for _ in range(3000)})
        cts = np.array([rng.randrange(1, 300 if csz > 1 else 256) for _ in vals], dtype=np.uint32)
        prefix = str(tmp_path / f"db_{k}_{version}_{p}")
        kmc.write_kmc_db(prefix, kmc.ints_to_packed(vals), cts, k, lut_prefix_len=p, version=version, counter_size=csz,
                         min_count=2, max_count=255)
        ks, cs = dump(prefix)
        keep = [(v, int(c)) for v, c in zip(vals, cts) if 2 <= c <= 255]
        assert ks == [kmc.unpack_kmer(v, k) for v, _ in keep] and cs == [c for _, c in keep]
    # several bins (what real KMC2 files look like): sorted within a bin only
    vals = sorted({rng.getrandbits(86) for _ in range(2000)})
    cts = np.array([rng.randrange(2, 200) for _ in vals], dtype=np.uint32)
    prefix = str(tmp_path / "binned")
    kmc.write_kmc_db_binned(prefix, kmc.ints_to_packed(vals), cts, 43, bin_of=lambda v: (v >> 3) % 4, n_bins=4,
                            lut_prefix_len=3)
    listed, lc, _ = kmc.read_kmc_db(prefix)
    ks, cs = dump(prefix)
    assert ks == kmc.packed_to_strings(listed, 43) and cs == lc.tolist() and sorted(kmc.packed_to_ints(listed)) == vals
    r = subprocess.run([cli, "kmc-dump", str(tmp_path / "nope")], capture_output=True, text=True)
    assert r.returncode == 1 and "cannot open" in r.stderr


def test_signatures_fuzz_small_blocks(cli, ref_or_none, tmp_path):
    """many small random VCFs (dense clusters, 20 % multi-allelic, symbolic and long alleles, 1-9 samples, haploid and
    diploid, k from 15 to 35): enumeration == VB::extract_kmers in both grouping modes"""
    import random

    for seed in range(24):
        rng = random.Random(7000 + seed)
        haploid = rng.random() < 0.3
        k = rng.choice([35, 35, 31, 21, 15])
        contigs = [("1", rng.randrange(1500, 6000)), ("2", rng.randrange(800, 3000))]
        refs = synth.make_reference(rng, contigs, n_run_every=1700)
        recs = synth.make_variants(rng, refs, rng.choice([7, 10, 20, 30]), rng.choice([1, 2, 5, 9]), haploid, multi_frac=0.2,
                                   sym_frac=0.03, long_frac=0.02, k=k)
        fa, vcf = str(tmp_path / f"r{seed}.fa"), str(tmp_path / f"v{seed}.vcf")
        synth.write_fasta(fa, refs)
        synth.write_vcf(vcf, refs, recs, len(recs[0].gts) if recs else 1, haploid, 0.05, rng)
        flags = (["-1"] if haploid else []) + ["-k", str(k)]
        for index_mode in (True, False):
            got, used = cli_signatures(cli, fa, vcf, flags, index_mode)
            assert_reference_enumeration(ref_or_none, f"fuzz_small_blocks/seed={seed}/index_mode={index_mode}", got, used,
                                         fa, vcf, k, haploid, "AF", False, index_mode)


def test_index_file_roundtrip(tmp_path):
    """csrc/host/index_file.hpp: sorted set-bit lists (delta-coded) and packed keys survive the zstd-chunked file,
    including sections larger than one chunk and empty sections; a foreign file is refused with a clear message"""
    src = tmp_path / "t.cpp"
    src.write_text(r'''
#include "index_file.hpp"
#include <cstdio>
#include <random>
int main(int argc, char **argv) {
  std::mt19937_64 g(7);
  std::vector<uint64_t> a, b, keys;
  uint64_t x = 0;
  for (int i = 0; i < 9000000; ++i) { x += 1 + g() % 4000; a.push_back(x); }   // 72 MB raw: two chunks
  for (int i = 0; i < 1000; ++i) keys.push_back(g());
  std::vector<uint64_t> a0 = a, b0 = b, k0 = keys;
  { mh::IndexWriter w(argv[1], 35, 43, 1ull << 35); w.write_bits(a); w.write_bits(b); w.write_keys(keys); w.close(); }
  mh::IndexReader r(argv[1]);
  if (r.k != 35 || r.ref_k != 43 || r.bf_bits != (1ull << 35)) return 2;
  if (r.read_bits() != a0) return 3;
  if (r.read_bits() != b0) return 4;
  if (r.read_keys() != k0) return 5;
  try { mh::IndexReader bad(argv[2]); return 6; } catch (const std::exception &e) { if (!strstr(e.what(), "not an index")) return 7; }
  puts("ok");
  return 0;
}
''')
    exe = tmp_path / "t"
    host = os.path.join(os.path.dirname(mbuild.CLI), "csrc", "host")
    zstd = next(p for p in ("/usr/lib/x86_64-linux-gnu/libzstd.so.1", "/lib/x86_64-linux-gnu/libzstd.so.1") if os.path.exists(p))
    stdcxx = next(p for p in ("/usr/lib/x86_64-linux-gnu/libstdc++.so.6", "/lib/x86_64-linux-gnu/libstdc++.so.6") if os.path.exists(p))
    subprocess.run(["g++", "-O1", "-std=c++17", "-I", host, "-o", str(exe), str(src), zstd, "-nostdlib++", stdcxx, "-lm"], check=True)
    other = tmp_path / "other.zst"
    other.write_bytes(b"\x28\xb5\x2f\xfd" + b"\0" * 64)      # (a zstd frame magic: what a CPU-built index starts with)
    r = subprocess.run([str(exe), str(tmp_path / "idx.zst"), str(other)], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.strip() == "ok", (r.returncode, r.stderr)
    assert os.path.getsize(tmp_path / "idx.zst") < 30_000_000   # 72 MB of indices -> deltas -> zstd


def test_fast_decimal_equals_strtod(tmp_path):
    """csrc/host/vcf_io.hpp: the INFO / QUAL float parser takes an exact short cut for plain decimals (<= 19 digits below
    2^53, decimal exponent within +-22: one correctly rounded IEEE operation) and leaves the rest to strtod; htslib
    parses these fields with strtod, so every token must come out bit-identical to strtod's value narrowed to float"""
    src = tmp_path / "t.cpp"
    src.write_text(r'''
#include "vcf_io.hpp"
#include <cstdio>
#include <random>
static int check(const std::string &t, long &fast) {
  double d = 0;
  if (mh::detail::fast_decimal(t.data(), t.data() + t.size(), &d)) {
    ++fast;
    double e = strtod(t.c_str(), nullptr);
    if (memcmp(&d, &e, 8) != 0) { printf("MISMATCH %s: %.17g vs %.17g\n", t.c_str(), d, e); return 1; }
  }
  float f = mh::detail::float_token(t.data(), t.data() + t.size());
  float g = (t.empty() || t == ".") ? mh::detail::missing_float() : (float)strtod(t.c_str(), nullptr);
  if (memcmp(&f, &g, 4) != 0) { printf("TOKEN MISMATCH %s\n", t.c_str()); return 1; }
  return 0;
}
int main() {
  std::mt19937_64 g(11);
  long fast = 0, n = 0; int bad = 0;
  const char *fixed[] = {"0", "-0", "1", "0.5", ".5", "5.", "1e22", "1e-22", "1e23", "1e-23", "9007199254740992", "9007199254740993",
                         "0.000312", "1.5e-05", "3.0E+2", "00012.500", "0.0000000000000000000001", "123456789012345678901",
                         "1.7976931348623157e308", "4.9e-324", "nan", "inf", "-inf", "0x10", "1.5abc", "", ".", "+", "-", "e5", "1e", "1e+",
                         "0.1", "0.2", "0.3", "0.7", "2.2250738585072014e-308", "17.17e1", "1234567890123456789", "9999999999999999999"};
  for (const char *f : fixed) { bad += check(f, fast); ++n; }
  for (int i = 0; i < 2000000; ++i) {
    std::string t;
    if (g() % 8 == 0) t += (g() & 1) ? "-" : "+";
    int ni = (int)(g() % 4), nf = (int)(g() % 21);
    for (int j = 0; j < ni; ++j) t += (char)('0' + g() % 10);
    if (nf || g() % 3 == 0) { t += '.'; for (int j = 0; j < nf; ++j) t += (char)('0' + (g() % 4 ? g() % 10 : 0)); }
    if (g() % 4 == 0) { t += (g() & 1) ? 'e' : 'E'; if (g() % 2) t += (g() & 1) ? '-' : '+'; t += std::to_string(g() % 30); }
    bad += check(t, fast); ++n;
  }
  printf("%ld tokens, %ld through the short cut, %d mismatches\n", n, fast, bad);
  return bad ? 1 : 0;
}
''')
    exe = tmp_path / "t"
    host = os.path.join(os.path.dirname(mbuild.CLI), "csrc", "host")
    stdcxx = next(p for p in ("/usr/lib/x86_64-linux-gnu/libstdc++.so.6", "/lib/x86_64-linux-gnu/libstdc++.so.6") if os.path.exists(p))
    subprocess.run(["g++", "-O2", "-std=c++17", "-I", host, "-o", str(exe), str(src), "-lz", "-nostdlib++", stdcxx, "-lm"], check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-2000:]
    n_fast = int(r.stdout.split(" tokens, ")[1].split(" ")[0])
    assert n_fast > 1_000_000, r.stdout                      # (the short cut is what runs on ordinary AF values)


def test_sample_list_errors_and_subset(cli, tmp_path):
    """-s: an unknown name stops the run with the reference's message and htslib's code (index of the name + 1,
    main.cpp:266-271); a valid list keeps the listed samples in HEADER order whatever the order in the file"""
    case = next(c for c in synth.CASES if c.name == "samples_subset_uniform")
    fa, vcf, _, _ = synth.build_case(case, str(tmp_path))
    bad = tmp_path / "bad.txt"
    bad.write_text("S2\nNOPE\nS1\n")
    r = subprocess.run([cli, "signatures", "-s", str(bad), fa, vcf], capture_output=True, text=True)
    assert r.returncode == 1 and "ERROR: VCF samples subset (code: 2)" in r.stderr
    r = subprocess.run([cli, "signatures", "-s", str(tmp_path / "missing.txt"), fa, vcf], capture_output=True, text=True)
    assert r.returncode == 1 and "ERROR: VCF samples subset" in r.stderr
    a, b = tmp_path / "a.txt", tmp_path / "b.txt"
    a.write_text("S7\nS2\nS9\nS3\n")
    b.write_text("S2\nS3\nS7\nS9\n")
    out = [subprocess.run([cli, "signatures", "-s", str(f), fa, vcf], capture_output=True, text=True, check=True).stdout
           for f in (a, b)]
    assert out[0] == out[1] and out[0].count("\n") > 500
    all_samples = subprocess.run([cli, "signatures", fa, vcf], capture_output=True, text=True, check=True).stdout
    assert all_samples != out[0]      # the subset really changes the haplotypes seen


@pytest.mark.parametrize("haploid", [False, True])
def test_signatures_many_samples(cli, ref_or_none, tmp_path, haploid):
    """400 panel samples (hundreds of distinct genotype patterns per block: the sample-class hash set grows), dense
    variants, unphased and missing genotypes"""
    import random

    rng = random.Random(31337 + haploid)
    refs = synth.make_reference(rng, [("1", 12_000)], n_run_every=5000)
    recs = synth.make_variants(rng, refs, 9, 400, haploid, multi_frac=0.15, sym_frac=0.02, long_frac=0.01, k=35)
    for r in recs:                      # common variants: many different haplotypes among the samples
        r.af = [min(0.45, 0.1 + 0.35 * rng.random()) / max(1, len(r.af)) for _ in r.af]
    recs2 = []
    for r in recs:                      # redraw the genotypes with the new frequencies
        n_real = len([a for a in r.alts if not a.startswith("<")])
        gts = []
        for _ in range(400):
            def draw():
                u, acc = rng.random(), 0.0
                for i in range(n_real):
                    acc += r.af[i]
                    if u < acc:
                        return i + 1
                return 0
            if n_real == 0:
                gts.append("0" if haploid else "0|0")
            elif haploid:
                gts.append(str(draw()))
            else:
                gts.append(f"{draw()}{'|' if rng.random() < 0.8 else '/'}{draw()}")
        r.gts = gts
        recs2.append(r)
    fa, vcf = str(tmp_path / "r.fa"), str(tmp_path / "v.vcf")
    synth.write_fasta(fa, refs)
    synth.write_vcf(vcf, refs, recs2, 400, haploid, 0.02, rng)
    flags = ["-1"] if haploid else []
    for index_mode in (True, False):
        got, used = cli_signatures(cli, fa, vcf, flags, index_mode)
        assert_reference_enumeration(ref_or_none, f"many_samples/haploid={haploid}/index_mode={index_mode}", got, used,
                                     fa, vcf, 35, haploid, "AF", False, index_mode)
        assert sum(len(v) for b in got.values() for v in b.values()) > 2000


# ---- short cuts of the VCF reader (block-parallel BGZF inflate, fixed-stride GT columns) against its general paths --------

def _bgzf_bytes(data: bytes, rng, max_member=6000) -> bytes:
    """BGZF as bgzip writes it: gzip members with a 'BC' extra field holding their own size, cut at arbitrary byte
    positions (lines straddle members), a few empty members in between, the 28-byte EOF marker at the end."""
    import struct
    import zlib

    def member(chunk: bytes) -> bytes:
        c = zlib.compressobj(6, zlib.DEFLATED, -15)
        body = c.compress(chunk) + c.flush()
        bsize = 18 + len(body) + 8
        assert bsize <= 65536
        return (b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", bsize - 1) + body +
                struct.pack("<II", zlib.crc32(chunk) & 0xFFFFFFFF, len(chunk)))

    out, pos = [], 0
    while pos < len(data):
        n = rng.randrange(1, max_member)
        out.append(member(data[pos:pos + n]))
        pos += n
        if rng.random() < 0.05:
            out.append(member(b""))
    out.append(member(b""))
    return b"".join(out)


def _signatures_text(cli, fa, vcf, flags, general, threads=None):
    env = dict(os.environ)
    env.pop("MALVA_GENERAL_DECODE", None)
    if general:
        env["MALVA_GENERAL_DECODE"] = "1"
    cmd = [cli, "signatures"] + list(flags) + (["--threads", str(threads)] if threads else []) + [fa, vcf]
    return subprocess.run(cmd, capture_output=True, text=True, env=env)


def test_bgzf_reader_equals_gzip_reader(cli, tmp_path):
    """the block-parallel BGZF source hands out the same bytes as zlib's gzread (the general path, which also reads
    BGZF as concatenated gzip members) and as the plain file; a damaged member is an error, not silent garbage"""
    import random

    rng = random.Random(4242)
    refs = synth.make_reference(rng, [("1", 20_000), ("2", 9_000)], n_run_every=5000)
    recs = synth.make_variants(rng, refs, 12, 60, False, multi_frac=0.15, sym_frac=0.02, long_frac=0.01, k=35)
    fa, vcf = str(tmp_path / "r.fa"), str(tmp_path / "v.vcf")
    synth.write_fasta(fa, refs)
    synth.write_vcf(vcf, refs, recs, 60, False, 0.02, rng)
    plain = open(vcf, "rb").read()
    want = _signatures_text(cli, fa, vcf, [], general=True)
    assert want.returncode == 0 and want.stdout.count("\n") > 500
    for trial, max_member in enumerate((300, 6000, 60000)):
        bg = str(tmp_path / f"v{trial}.vcf.gz")
        blob = _bgzf_bytes(plain, rng, max_member)
        open(bg, "wb").write(blob)
        for general in (False, True):
            for threads in (1, 4):
                got = _signatures_text(cli, fa, bg, [], general, threads)
                assert got.returncode == 0, got.stderr
                assert got.stdout == want.stdout, (trial, general, threads)
    # one flipped byte inside a member's deflate stream / a truncated file
    bad = bytearray(blob)
    bad[len(bad) // 2] ^= 0x55
    open(str(tmp_path / "bad.vcf.gz"), "wb").write(bytes(bad))
    r = _signatures_text(cli, fa, str(tmp_path / "bad.vcf.gz"), [], general=False)
    assert r.returncode != 0 and "BGZF" in r.stderr
    open(str(tmp_path / "cut.vcf.gz"), "wb").write(blob[: len(blob) // 2])
    r = _signatures_text(cli, fa, str(tmp_path / "cut.vcf.gz"), [], general=False)
    assert r.returncode != 0 and "BGZF" in r.stderr


@pytest.mark.parametrize("haploid", [False, True])
@pytest.mark.parametrize("n_samples", [1, 2, 3, 5, 17, 64, 131])
def test_fixed_stride_gt_columns_equal_general_decode(cli, ref_or_none, tmp_path, haploid, n_samples):
    """FORMAT = GT with one-symbol alleles takes the fixed-stride decode (vcf_io.hpp fast_gt_columns); the result is
    what the general decode gives and what the reference's Variant / VB::extract_kmers give (variant.hpp:158-211),
    for every mix the short cut has to get right or hand back: phased / unphased / mostly-unphased rows, missing
    entries, single-entry diploid columns, ten or more alleles (two-symbol indices), a FORMAT with a second field"""
    import random

    rng = random.Random(977 * n_samples + haploid)
    refs = synth.make_reference(rng, [("1", 9_000)], n_run_every=5000)
    recs = synth.make_variants(rng, refs, 10, n_samples, haploid, multi_frac=0.3, sym_frac=0.02, long_frac=0.01, k=35)
    for i, r in enumerate(recs):
        n_real = len([a for a in r.alts if not a.startswith("<")])
        mode = i % 6
        gts = []
        for s in range(n_samples):
            a, b = (rng.randrange(0, n_real + 1) if rng.random() < 0.3 else 0 for _ in range(2))
            if haploid:
                gts.append("." if rng.random() < 0.05 else str(a))
                continue
            sep = {0: "|", 1: "/", 2: "|" if rng.random() < 0.8 else "/", 3: "/" if rng.random() < 0.8 else "|",
                   4: "|", 5: "|"}[mode]
            g = f"{a}{sep}{b}"
            if mode == 4 and rng.random() < 0.1:
                g = "." + sep + (str(b) if rng.random() < 0.5 else ".")
            if mode == 5 and s == n_samples // 2:
                g = str(a)                 # one column of another width: the whole row goes the general way
            gts.append(g)
        r.gts = gts
    fa, vcf = str(tmp_path / "r.fa"), str(tmp_path / "v.vcf")
    synth.write_fasta(fa, refs)
    synth.write_vcf(vcf, refs, recs, n_samples, haploid, 0.02, rng)
    flags = ["-1"] if haploid else []
    fast = _signatures_text(cli, fa, vcf, flags, general=False)
    slow = _signatures_text(cli, fa, vcf, flags, general=True)
    assert fast.returncode == 0 and slow.returncode == 0, fast.stderr + slow.stderr
    assert fast.stdout == slow.stdout
    if haploid:     # one-symbol columns read WITHOUT -1 (the next sample's symbol stands in for the second allele)
        fast2 = _signatures_text(cli, fa, vcf, [], general=False)
        slow2 = _signatures_text(cli, fa, vcf, [], general=True)
        assert fast2.returncode == 0 and slow2.returncode == 0 and fast2.stdout == slow2.stdout
        assert n_samples < 3 or fast2.stdout != fast.stdout
    # kept-sample subsets (-s): the short cut decodes the kept columns only
    subsets = {"half": [i for i in range(n_samples) if rng.random() < 0.5], "first": [0], "last": [n_samples - 1],
               "but_last": list(range(n_samples - 1)), "but_first": list(range(1, n_samples))}
    for name, cols in subsets.items():
        if not cols:
            continue
        lst = tmp_path / f"{name}.txt"
        lst.write_text("".join(f"S{i}\n" for i in cols))
        for fl in ([flags] if not haploid else [flags, []]):
            a = _signatures_text(cli, fa, vcf, fl + ["-s", str(lst)], general=False)
            b = _signatures_text(cli, fa, vcf, fl + ["-s", str(lst)], general=True)
            assert a.returncode == 0 and b.returncode == 0, a.stderr + b.stderr
            assert a.stdout == b.stdout, (name, fl)
        if name in ("half", "but_first"):   # and what the reference's own enumeration gives for the kept columns
            got, used = cli_signatures(cli, fa, vcf, flags + ["-s", str(lst)], False)
            assert_reference_enumeration(ref_or_none, f"fixed_stride/haploid={haploid}/n_samples={n_samples}/{name}",
                                         got, used, fa, vcf, 35, haploid, "AF", False, False, sample_cols=cols)
    tr = subprocess.run([cli, "signatures", "--trace"] + flags + [fa, vcf], capture_output=True, text=True, check=True).stderr
    took, rows = map(int, re.search(r"fixed-stride GT decode: (\d+) of (\d+) rows", tr).groups())
    assert 0.8 * len(recs) <= rows <= len(recs) and took < rows
    assert n_samples < 5 or took >= rows // 3             # both ways are exercised by the file
    got, used = cli_signatures(cli, fa, vcf, flags, False)
    assert_reference_enumeration(ref_or_none, f"fixed_stride/haploid={haploid}/n_samples={n_samples}/all", got, used,
                                 fa, vcf, 35, haploid, "AF", False, False)


def test_sars_cov2_panel_fast_and_general_decode_agree(cli):
    """BASELINE config 1's real VCF (BGZF, 15,154 records x 27,934 one-symbol haploid columns): both decodes give the
    same signatures, byte for byte"""
    src = os.path.join(os.path.dirname(GOLD), "sars")
    fa, vcf = os.path.join(src, "reference_sarsCov2.fasta"), os.path.join(src, "sars_cov2.vcf.gz")
    fast = _signatures_text(cli, fa, vcf, ["-1"], general=False)
    slow = _signatures_text(cli, fa, vcf, ["-1"], general=True)
    assert fast.returncode == 0 and slow.returncode == 0
    assert fast.stdout == slow.stdout and fast.stdout.count("\n") > 10_000


def test_format_short_cuts_equal_the_library_calls(cli):
    """the integer and QUAL formatting of the output stage (malva_geno.cpp format_variant) against std::to_string and
    "%g" over 4.7e6 values (whole numbers, fractions, -0, inf, nan, denormals, random bit patterns)"""
    r = subprocess.run([cli, "format-selftest"], capture_output=True, text=True)
    assert r.returncode == 0 and " 0 differ" in r.stdout, r.stdout + r.stderr


def test_small_containers_equal_std_vector(cli):
    """InlineVec (a record's short lists) and Chain (signatures.hpp) against std::vector over 800,000 random
    operations: growth past the inline capacity, copies and moves in both states, strings beyond the SSO size"""
    r = subprocess.run([cli, "container-selftest"], capture_output=True, text=True)
    assert r.returncode == 0 and " 0 differ" in r.stdout, r.stdout + r.stderr


def test_sars_cov2_panel_against_the_reference_enumeration(cli, ref_or_none, tmp_path):
    """BASELINE config 1's real VCF -- 15,154 records in ONE var_block (every other base of the genome has a variant:
    chains of ~19 members) -- with 400 of its 27,934 haploid samples (the reference's own enumeration needs ~12 s for
    these; 5 minutes for all): malva-geno signatures == VB::extract_kmers, block by block, allele by allele"""
    import gzip
    import random

    src = os.path.join(os.path.dirname(GOLD), "sars")
    fa, vcf = os.path.join(src, "reference_sarsCov2.fasta"), os.path.join(src, "sars_cov2.vcf.gz")
    with gzip.open(vcf, "rt") as fh:
        names = next(l for l in fh if l.startswith("#CHROM")).rstrip("\n").split("\t")[9:]
    assert len(names) == 27934
    cols = sorted(random.Random(11).sample(range(len(names)), 400))
    lst = tmp_path / "kept.txt"
    lst.write_text("".join(names[i] + "\n" for i in cols))
    got, used = cli_signatures(cli, fa, vcf, ["-1", "-s", str(lst)], False)
    assert_reference_enumeration(ref_or_none, "sars_cov2_panel_400", got, used, fa, vcf, 35, True, "AF", False, False,
                                 sample_cols=cols)
    assert sum(len(v) for b in got.values() for v in b.values()) > 30_000


def test_error_in_a_later_batch_ends_the_pipeline(cli, tmp_path):
    """a malformed record in the second batch (the reader thread is a block ahead, the first batch is already being
    enumerated): the program reports it and exits, no stage is left waiting for another"""
    import synth_fast

    fa, vcf, _, n = synth_fast.build(str(tmp_path), 4_000_000)
    lines = open(vcf).read().split("\n")
    assert len("\n".join(lines)) > 14_000_000        # more than one 12 MB batch of text
    lines.insert(len(lines) - 2000, "garbage line without tabs")
    bad = str(tmp_path / "bad.vcf")
    open(bad, "w").write("\n".join(lines))
    r = subprocess.run([cli, "signatures", "--threads", "4", fa, bad], capture_output=True, text=True, timeout=60)
    assert r.returncode == 1 and "malformed VCF record: garbage line" in r.stderr
    good = subprocess.run([cli, "signatures", "--threads", "4", fa, vcf], capture_output=True, text=True, timeout=60)
    assert good.returncode == 0 and good.stdout.count("\n") > n
