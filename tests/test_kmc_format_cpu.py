"""The KMC database boundary (SURVEY 8a X1; call sites main.cpp:444-449, 482-490), table-driven.

No `kmc` binary and no KMC-written database exist in the build image, so what is checked here is that the THREE
independent readers of this repository -- the Python reader (malva_b200/kmc.py), the C++ host reader
(csrc/host/kmc_db.hpp, through `malva-geno kmc-dump`) and the stand-in CKMCFile the reference's own main.cpp is
compiled against (oracle/shim/kmc_file.h, through the shim_kmc_list hook, driven exactly like main.cpp:482-490) --
agree with each other and with the semantics the KMC API documents, over every header variant the format allows:
counter_size 1-4, both_strands stored inverted, lut_prefix_len 1-9, KMC1 ("version 0") and KMC2/3 (0x200) headers,
one and several bins, min_count / max_count filtering in ReadNextKmer (a 64-bit max_count split over two header
words), and a prefix LUT with or without a trailing guard entry.  The device decoder sees the same tables in
tests/test_gpu_parity.py::test_kmc_records_decoded_on_device.

What NO test here can pin without a file written by the real tool (DESIGN.md section 4): the exact number of reserved
bytes between both_strands and the version word (readers locate the header through header_offset, so any size
works), whether KMC1 files carry a guard LUT entry, and the minimiser-signature map's contents (never read: the
listing does not need it)."""
import ctypes as C
import os
import random
import struct
import subprocess

import numpy as np
import pytest

from malva_b200 import build as mbuild
from malva_b200 import kmc


def _records(rng, k, n, counter_size, lo=1):
    vals = sorted(rng.sample(range(4 ** min(k, 14)), min(n, 4 ** min(k, 14) // 2)))  # distinct, low-entropy prefixes
    vals = sorted({(v * 0x9E3779B97F4A7C15) % (4 ** k) for v in vals})
    top = min(256 ** counter_size - 1, 70000)
    counts = [rng.choice([lo, 2, 3, 7, 254, 255, top]) if counter_size > 1 else rng.choice([1, 2, 3, 7, 254, 255])
              for _ in vals]
    return kmc.ints_to_packed(vals), np.array(counts, dtype=np.uint32)


def _dump_cli(cli, prefix):
    out = subprocess.run([cli, "kmc-dump", prefix], capture_output=True, text=True, check=True).stdout
    return [(l.split("\t")[0], int(l.split("\t")[1])) for l in out.splitlines()]


def _dump_shim(shim, prefix):
    cap = 1 << 24
    buf = C.create_string_buffer(cap)
    info = (C.c_uint64 * 8)()
    n = shim.shim_kmc_list(prefix.encode(), info, buf, cap)
    assert n >= 0, n
    lines = buf.value.decode().splitlines()
    return [(l.split("\t")[0], int(l.split("\t")[1])) for l in lines], list(info)


CASES = [
    # (k, lut_prefix_len, version, counter_size, both_strands, min_count, max_count)
    (43, 7, 0x200, 1, True, 2, 255),          # what `kmc -k43` writes for MALVA (MALVA:107)
    (43, 3, 0x200, 1, True, 2, 255),
    (43, 3, 0, 1, True, 2, 255),              # KMC1 header: no signature_len word
    (43, 7, 0, 2, False, 1, 65535),
    (43, 7, 0x200, 2, True, 2, 1000),         # -cs1000: two counter bytes, max_count cuts the top
    (43, 7, 0x200, 3, True, 3, 70000),
    (43, 7, 0x200, 4, False, 2, (1 << 33) + 5),   # max_count above 2^32: the high word of the KMC 3 header
    (39, 3, 0x200, 1, True, 2, 255),
    (35, 7, 0x200, 1, True, 1, 255),
    (21, 1, 0x200, 1, True, 2, 254),
    (21, 5, 0, 4, True, 2, 3),                # a narrow [min, max] window
    (41, 9, 0x200, 1, True, 2, 255),
    (63, 3, 0x200, 2, True, 2, 65535),
]


@pytest.fixture(scope="module")
def cli():
    mbuild.build()
    return mbuild.CLI


@pytest.fixture(scope="module")
def shim():
    from oracle import pyoracle

    pyoracle.build()
    return pyoracle.kmc_shim()


@pytest.mark.parametrize("k,p,version,csz,both,minc,maxc", CASES)
def test_three_readers_agree(cli, shim, tmp_path, k, p, version, csz, both, minc, maxc):
    rng = random.Random(k * 1000 + p * 10 + csz)
    packed, counts = _records(rng, k, 600, csz)
    prefix = str(tmp_path / "db")
    kmc.write_kmc_db(prefix, packed, counts, k, lut_prefix_len=p, version=version, counter_size=csz, min_count=minc,
                     max_count=maxc, both_strands=both)
    # expectation from the definition: ascending k-mers, records outside [min_count, max_count] skipped
    exp = [(kmc.unpack_kmer(v, k), int(c)) for v, c in sorted(zip(kmc.packed_to_ints(packed), counts)) if minc <= c <= maxc]
    assert 0 < len(exp) <= len(counts)
    got_py, cts_py, k_py = kmc.read_kmc_db(prefix)
    assert k_py == k
    assert list(zip(kmc.packed_to_strings(got_py, k), [int(c) for c in cts_py])) == exp
    assert _dump_cli(cli, prefix) == exp
    got_shim, info = _dump_shim(shim, prefix)
    assert got_shim == exp
    # CKMCFile::Info as main.cpp:446-449 reads it
    assert info[0] == k and info[2] == csz and info[3] == p and info[5] == minc and info[6] == maxc
    assert info[7] == len(counts)   # total_kmers counts every record of the file, filtered or not
    db = kmc.open_kmc_db(prefix)
    assert db["both_strands"] == both and db["max_count"] == maxc and db["record_bytes"] == (k - p) // 4 + csz
    assert db["version"] == version and len(db["lut"]) == 4 ** p


def test_inverted_both_strands_byte_and_header_words(tmp_path):
    """the header fields byte by byte: both_strands is stored INVERTED (0 = canonical counting), max_count is split
    into a low word before total_kmers and a high word after the both_strands byte"""
    packed, counts = _records(random.Random(1), 43, 50, 1)
    for both in (True, False):
        prefix = str(tmp_path / f"b{int(both)}")
        kmc.write_kmc_db(prefix, packed, counts, 43, lut_prefix_len=7, both_strands=both, max_count=(7 << 32) | 255)
        pre = open(prefix + ".kmc_pre", "rb").read()
        version, hoff = struct.unpack("<II", pre[-12:-4])
        h = pre[len(pre) - 8 - hoff:]
        assert struct.unpack("<7I", h[:28]) == (43, 0, 1, 7, 5, 2, 255)
        assert struct.unpack("<Q", h[28:36])[0] == len(counts)
        assert h[36] == (0 if both else 1)
        assert struct.unpack("<I", h[37:41])[0] == 7
        assert version == 0x200 and pre[:4] == b"KMCP" and pre[-4:] == b"KMCP"


def test_lut_without_guard_entry_and_several_bins(cli, shim, tmp_path):
    """real KMC2 files hold n_bins x 4^p LUT entries and no guard; the writer here appends one.  Both must list alike."""
    rng = random.Random(5)
    k, p = 43, 3
    packed, counts = _records(rng, k, 400, 1)
    a, b = str(tmp_path / "guard"), str(tmp_path / "noguard")
    kmc.write_kmc_db_binned(a, packed, counts, k, bin_of=lambda v: v % 3, n_bins=3, lut_prefix_len=p)
    pre = bytearray(open(a + ".kmc_pre", "rb").read())
    n_lut = 3 * 4 ** p
    del pre[4 + 8 * n_lut:4 + 8 * (n_lut + 1)]           # drop the guard entry
    open(b + ".kmc_pre", "wb").write(pre)
    os.link(a + ".kmc_suf", b + ".kmc_suf")
    la, lb = _dump_cli(cli, a), _dump_cli(cli, b)
    assert la == lb and len(la) == sum(1 for c in counts if 2 <= c <= 255)
    assert _dump_shim(shim, a)[0] == la and _dump_shim(shim, b)[0] == la
    pa, ca, _ = kmc.read_kmc_db(a)
    pb, cb, _ = kmc.read_kmc_db(b)
    assert list(zip(kmc.packed_to_strings(pa, k), ca.tolist())) == la == list(zip(kmc.packed_to_strings(pb, k), cb.tolist()))
    # several bins: sorted inside a bin, not globally
    assert [s for s, _ in la] != sorted(s for s, _ in la)


def test_broken_files_are_refused(cli, tmp_path):
    packed, counts = _records(random.Random(2), 43, 50, 1)
    prefix = str(tmp_path / "db")
    kmc.write_kmc_db(prefix, packed, counts, 43, lut_prefix_len=7)
    good = open(prefix + ".kmc_pre", "rb").read()
    for name, data in (("marker", b"XXXX" + good[4:]), ("tail", good[:-4] + b"XXXX"), ("short", good[:40]),
                       ("version", good[:-12] + struct.pack("<I", 0x300) + good[-8:])):
        bad = str(tmp_path / name)
        open(bad + ".kmc_pre", "wb").write(data)
        os.link(prefix + ".kmc_suf", bad + ".kmc_suf")
        r = subprocess.run([cli, "kmc-dump", bad], capture_output=True, text=True)
        assert r.returncode != 0, name
        with pytest.raises(Exception):
            kmc.read_kmc_db(bad)
