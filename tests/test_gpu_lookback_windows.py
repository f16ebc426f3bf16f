"""Split searches large enough that the decoupled look-back of every search kernel walks past its first window of 32 predecessor tiles.

A tile of a (cluster, dimension) segment looks back over at most 32 predecessors at a time; a segment of more than 33 tiles is needed before a
walk can find no inclusive prefix in its first window and move on to the next one.  At level 0 the segment is the whole problem:
  * the sweeps (k_sweep_ss, k_sweep_split_scafs) and k_partition2 take 8192 elements per tile, so N must exceed 33 * 8192;
  * k_flip_prefix takes 2048 flip-list entries per tile; the list holds the scaffolds that can flip (n >= T/2 + 1), of which there must be more
    than 33 * 2048.
The one-pass scan of the per-scaffold SCG flags covers all S scaffolds in tiles of 2048 and crosses windows as well."""
import numpy as np
import pytest

from golden_util import _random_problem, assert_search_matches_oracle

pytestmark = pytest.mark.gpu

WINDOW = 32            # predecessors per look-back window
SW_TILE = 8192         # elements per tile of the sweeps and the partition (search.cu)
FP_TILE = 2048         # flip-list entries per tile of k_flip_prefix


@pytest.fixture(scope="module")
def ctx():
    from abawaca_b200 import capi
    c = capi.Context(0)
    yield c
    c.close()


@pytest.mark.parametrize("seed,partial,strategy", [(21, False, 0), (22, True, 0), (23, False, 1)])
def test_search_across_lookback_windows_matches_oracle(ctx, oracle, seed, partial, strategy):
    from abawaca_b200 import capi, pipeline
    rng = np.random.default_rng(seed)
    S, D = 80000, 3
    vals, dp2scaf, T, length, mask = _random_problem(rng, S, D, partial=partial)
    assert dp2scaf.size > (WINDOW + 1) * SW_TILE
    if strategy == 0:
        n = np.bincount(dp2scaf, minlength=S)
        assert np.count_nonzero(n >= T // 2 + 1) > (WINDOW + 1) * FP_TILE
    orecs, odp, osc = oracle.Search(vals, dp2scaf, T, length, mask).run(strategy=strategy)
    p = capi.default_params()
    p.min_reported_score = 0.0
    res = pipeline.search(ctx, vals, dp2scaf, T, length, mask, params=p, strategy=strategy)
    assert_search_matches_oracle(orecs, odp, osc, res)
