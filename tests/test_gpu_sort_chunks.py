"""abw_search_create sorts the dimensions in chunks that fit ABW_SORT_SCRATCH_GB (default 16).  A budget of 1 GB splits a problem of
150 k datapoints in 400 dimensions into two chunks; the search must come out exactly as with all dimensions in one chunk."""
import ctypes

import numpy as np
import pytest

from golden_util import _random_problem

pytestmark = pytest.mark.gpu


def _fields(rec):
    """Every field of a record (nested structures expanded, doubles by bit pattern); the padding bytes between fields are not part of the result."""
    vals = (getattr(rec, name) for name, _ in rec._fields_)
    return tuple(_fields(v) if isinstance(v, ctypes.Structure) else v.hex() if isinstance(v, float) else v for v in vals)


@pytest.fixture(scope="module")
def ctx():
    from abawaca_b200 import capi
    c = capi.Context(0)
    yield c
    c.close()


# ties=True: exact thousandths, sorted on 32-bit keys; ties=False: arbitrary doubles, sorted on 64-bit keys
@pytest.mark.parametrize("ties", [True, False])
def test_chunked_sort_matches_one_chunk(ctx, monkeypatch, ties):
    from abawaca_b200 import capi, pipeline
    rng = np.random.default_rng(31 if ties else 32)
    S, D = 30000, 400
    vals, dp2scaf, T, length, mask = _random_problem(rng, S, D, ties=ties)
    N = dp2scaf.size
    assert D > (1 << 30) // (N * 25 + 4096), "the problem must need more than one chunk of a 1 GB budget (per_dim in search.cu)"
    p = capi.default_params()
    p.min_reported_score = 0.0
    one = pipeline.search(ctx, vals, dp2scaf, T, length, mask, params=p)
    monkeypatch.setenv("ABW_SORT_SCRATCH_GB", "1")
    chunked = pipeline.search(ctx, vals, dp2scaf, T, length, mask, params=p)
    assert len(one.recs) > 1
    assert [_fields(r) for r in chunked.recs] == [_fields(r) for r in one.recs]
    assert np.array_equal(chunked.dp2cluster, one.dp2cluster)
    assert np.array_equal(chunked.scaf2cluster, one.scaf2cluster)
