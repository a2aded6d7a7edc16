"""GPU parity of the flat scan at the boundaries of its CTA-pair layout: a pass holds up to 512 query rows, each CTA of
a pair takes 128 or 256 of them, the pairs share every DB tile, and the thresholds come from 2 x pairs maxima."""
import numpy as np
import pytest

from util import assert_topk_matches

pytestmark = pytest.mark.gpu


def _indexes(x):
    from nafp_b200.eval.utils.get_index import Index
    from oracle.flat_index import FlatL2
    g, o = Index(0, 128), FlatL2(128)
    g.add(x)
    o.add(x)
    return g, o


def _rows(query, nq):
    return query[:nq] if nq <= len(query) else np.concatenate([query] * (nq // len(query) + 1))[:nq]


def _check_passes(st, nq):
    assert st["fallback_rows"] == 0, st
    if st["fallback_overflow"] == 0 and st["fallback_bound"] == 0:     # no row needed the retry pass
        assert st["passes"] == -(-nq // 512), st


@pytest.fixture(scope="module")
def set_200k():
    from nafp_b200 import synth
    dummy, db, query = synth.synth_search_set(200000, 5900, seed=21)
    x = np.concatenate([dummy, db])
    g, o = _indexes(x)
    return x, query, g, o


@pytest.mark.parametrize("nq", [129, 256, 257, 511, 512, 513, 1100])
def test_pass_boundaries(set_200k, nq):
    x, query, g, o = set_200k
    q = _rows(query, nq)
    Dg, Ig = g.search(q, 20)
    Do, Io = o.search(q, 20)
    assert_topk_matches(Dg, Ig, Do, Io, x, q)
    _check_passes(g.last_search_stats(), nq)


def test_k64(set_200k):
    x, query, g, o = set_200k
    q = _rows(query, 300)
    Dg, Ig = g.search(q, 64)
    Do, Io = o.search(q, 64)
    assert_topk_matches(Dg, Ig, Do, Io, x, q)
    _check_passes(g.last_search_stats(), 300)


def test_fewer_tiles_than_pairs():
    """8,300 rows are 33 tiles of 256: fewer tiles than CTA pairs on a B200.  The scan runs 33 pairs, whose 66 maxima give
    kg = 48 a loose threshold, so rows whose top-k the bound cannot prove may go to the exact fallback here."""
    from nafp_b200 import synth
    dummy, db, query = synth.synth_search_set(7710, 590, seed=22)
    x = np.concatenate([dummy, db])
    g, o = _indexes(x)
    for nq in (40, 300):
        q = _rows(query, nq)
        Dg, Ig = g.search(q, 20)
        Do, Io = o.search(q, 20)
        assert_topk_matches(Dg, Ig, Do, Io, x, q)
        assert g.last_search_stats()["passes"] >= -(-nq // 512)       # the tensor-core scan ran


def test_rows_limit_inside_last_tile():
    """set_search_rows(m) with m inside the last tile the scan reads: the rows of that tile beyond m are never returned."""
    from nafp_b200 import synth
    dummy, db, query = synth.synth_search_set(99410, 590, seed=23)
    x = np.concatenate([dummy, db])               # 100,000 rows; the last tile holds rows 99,840 ..
    g, _ = _indexes(x)
    m = 99900
    g.set_search_rows(m)
    from oracle.flat_index import FlatL2
    o = FlatL2(128)
    o.add(x[:m])
    q = np.concatenate([x[m - 40:m + 40], _rows(query, 400)])
    Dg, Ig = g.search(q, 20)
    Do, Io = o.search(q, 20)
    assert Ig.max() < m
    assert_topk_matches(Dg, Ig, Do, Io, x[:m], q)
    _check_passes(g.last_search_stats(), len(q))
