"""The final pass of the fused EM kernel (k_em_one: one read group per sample, <= 256 samples) against the CPU oracle on a
cohort whose deletion has more supporting read pairs than the kernel's shared list holds (SUPP_CAP = 1536 in pd_em.cu):
64 samples at 100x, most of them carriers, give 57 final passes with up to 2 885 supporting read pairs. Those windows take
the recount path of the supporting-pair percentiles; the others fill the shared list from both warps of the block."""
import numpy as np
import pytest

from popdel_b200 import simulate
from parity import compare_scan_with_oracle

pytestmark = pytest.mark.gpu


def test_final_pass_beyond_the_supporting_pair_list(oracle_lib):
    n = 64
    specs = [[simulate.ReadGroupSpec(name=f"rg{s}", coverage=100.0)] for s in range(n)]
    dels = [simulate.Deletion(20_000, 1500, np.random.default_rng(7).binomial(2, 0.7, size=n))]
    samples, _ = simulate.simulate_cohort(seed=41, n_samples=n, contig_len=45_000, n_dels=0, dels=dels, rg_specs=specs)
    stats = compare_scan_with_oracle(samples, oracle_lib)
    assert stats["n_calls"] > 20
