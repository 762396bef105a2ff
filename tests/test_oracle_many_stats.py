"""CPU (not gpu): the reference's statistical criterion for prodAppxMSGibbsS (rangeUnitTests, test/runtests.jl:167-201)
on the oracle at more than 16 densities, the shapes tests/test_gpu_gibbs_many.py runs on the GPU: |mean| < sqrt(1/M)
and every std within (0.66, 1.33) sqrt(1/M), at least 5 of 10 repetitions."""
import numpy as np
import pytest

from oracle import oracle as O
from tests import test_oracle_stats as STATS


@pytest.mark.parametrize("D,M", [(2, 20), (2, 32), (2, 64)])
def test_oracle_passes_range_criterion_beyond_16_densities(D, M):
    rng = np.random.default_rng(1234 + 17 * D + M)
    v = [STATS.test_prods(STATS.oracle_prod, O.OKDE.kde_lcv, rng, D=D, M=M) for _ in range(10)]
    assert sum(v) >= 5, v
