"""End-to-end golden: the reference's bundled haploid example through the GPU path.

Inputs/outputs are the committed fixtures of tests/golden/haploid (made by tests/golden/make_golden.py):
the GPU index + scan + genotype must reproduce COVS, GT, GQ and the printed GTS of every record of the
verbose golden (produced by the shim-built reference; its GT:GQ equal example/haploid.malva.vcf).
Signatures are enumerated by the reference's own VB::extract_kmers (oracle/_ref hook) where it is built, so this
pins kernels K1-K5 and the C ABI, not the (host-kept) enumeration; elsewhere by `malva-geno signatures`."""
import pytest

import golden_flow
from malva_b200 import MalvaGpu

pytestmark = pytest.mark.gpu


def test_haploid_example_golden_on_gpu(ref_or_none):
    g = MalvaGpu(k=35, ref_k=43, bf_bits=1 << 33)  # -b 1, as in the README command

    def genotype(batch):
        r = g.genotype(batch, 0.001, 200, True)
        out = []
        for i in range(batch.n_variants):
            o = int(r.lik_off[i])
            out.append((int(r.status[i]), int(r.best_gt[i]), int(r.gq[i]), r.lik[o:o + int(r.n_gts[i])]))
        return r.cov, out

    try:
        lines = golden_flow.run_haploid_example(g, ref_or_none, genotype)
        assert g.popcount(0) == 422 and g.kmap_size() == 679  # SURVEY 8: bundled example sizes
    finally:
        g.close()
    gold = golden_flow.gold_lines("haploid.malva.verbose.vcf")
    plain = golden_flow.gold_lines("haploid.malva.vcf")
    assert len(lines) == len(gold) == len(plain) == 418
    for got, exp, pl in zip(lines, gold, plain):
        assert got == exp, (got, exp)
        assert got.split("\t")[-1] == pl.split("\t")[-1]
    assert sum(1 for l in lines if not l.endswith("0:0")) > 5
