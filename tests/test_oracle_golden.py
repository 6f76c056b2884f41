"""The CPU oracle against the reference's golden (CPU suite): the same flow the GPU golden test runs,
with oracle/liboracle.so holding bf / context_bf / ref_bf.  Pins the oracle end to end."""
import golden_flow
from parity_util import OracleRun


def test_oracle_reproduces_haploid_golden(oracle_lib, ref_or_none):
    o = OracleRun(oracle_lib, 35, 43, 1 << 26)

    def genotype(batch):
        cov, res = o.genotype(batch, 0.001, 200, True)
        return cov, [(e["status"], e["best"], e["gq"], e["probs"]) for e in res]

    try:
        lines = golden_flow.run_haploid_example(o, ref_or_none, genotype)
        assert oracle_lib.mo_bf_popcount(o.bf) == 422 and o.kmap_size() == 679
    finally:
        o.close()
    gold = golden_flow.gold_lines("haploid.malva.verbose.vcf")
    assert lines == gold
