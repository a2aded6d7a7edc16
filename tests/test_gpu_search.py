"""GPU parity: exact flat index (SURVEY §8 a5) and the sequence matcher (a7) against the oracle.
Everything goes through the C ABI (ctypes) exactly as the CLI does."""
import numpy as np
import pytest

from util import assert_topk_matches

pytestmark = pytest.mark.gpu


def _oracle_index(parts):
    from oracle.flat_index import FlatL2
    idx = FlatL2(128)
    for p in parts:
        idx.add(p)
    return idx


def _gpu_index(parts):
    from nafp_b200.eval.utils.get_index import Index
    idx = Index(0, 128)
    for p in parts:
        idx.add(p)
    return idx


@pytest.mark.parametrize("n_dummy,n_db,nq,k", [
    (50000, 2950, 19, 20),      # tensor-core scan, one pass, ragged query count
    (200000, 5900, 300, 20),    # two passes (256 + 44 rows)
    (3000, 590, 7, 20),         # small database -> exact fp32 scan
    (30000, 590, 1, 5),         # single row, small k
    (120000, 590, 64, 33),      # larger k
])
def test_flat_search_matches_oracle(n_dummy, n_db, nq, k):
    from nafp_b200 import synth
    dummy, db, query = synth.synth_search_set(n_dummy, n_db, seed=3)
    g = _gpu_index([dummy, db])
    o = _oracle_index([dummy, db])
    assert g.ntotal == o.ntotal == n_dummy + n_db
    q = query[:nq] if nq <= len(query) else np.concatenate([query] * (nq // len(query) + 1))[:nq]
    Dg, Ig = g.search(q, k)
    Do, Io = o.search(q, k)
    x_all = np.concatenate([dummy, db])
    assert_topk_matches(Dg, Ig, Do, Io, x_all, q)
    st = g.last_search_stats()
    assert st["rows"] == nq


def test_flat_search_unnormalised_rows():
    """IndexFlatL2 semantics for rows that are not unit norm (|x|^2 matters for the ranking)."""
    rng = np.random.default_rng(5)
    x = (rng.standard_normal((40000, 128)) * rng.uniform(0.2, 3.0, (40000, 1))).astype(np.float32)
    q = (rng.standard_normal((33, 128)) * 1.5).astype(np.float32)
    g, o = _gpu_index([x]), _oracle_index([x])
    Dg, Ig = g.search(q, 20)
    Do, Io = o.search(q, 20)
    assert_topk_matches(Dg, Ig, Do, Io, x, q, dtol=2e-3)


def test_flat_search_zero_rows_and_ragged_adds():
    """The scan's prefilter uses each 256-row tile's min 0.5|x|^2: all-zero rows (silence), mixed norms
    inside a tile and add() calls that straddle tile boundaries / grow the allocation must not change
    the answer."""
    rng = np.random.default_rng(15)
    x = rng.standard_normal((70001, 128)).astype(np.float32)
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    x[::977] = 0.0                                   # silent segments
    x[5000:5300] *= rng.uniform(0.3, 2.0, (300, 1)).astype(np.float32)
    q = x[rng.integers(0, len(x), 140)] + 0.05 * rng.standard_normal((140, 128)).astype(np.float32)
    cuts = [0, 100, 1133, 1134, 20000, 20255, 45001, 70001]
    g = _gpu_index([x[a:b] for a, b in zip(cuts[:-1], cuts[1:])])      # no reserve(): grows by doubling
    o = _oracle_index([x])
    for nq in (140, 129, 128, 1):                    # two query halves (second mostly padding), one half, one row
        Dg, Ig = g.search(q[:nq], 20)
        Do, Io = o.search(q[:nq], 20)
        assert_topk_matches(Dg, Ig, Do, Io, x, q[:nq], dtol=2e-3)


def test_flat_search_rows_limit_excludes_halo():
    """set_search_rows(m): rows >= m are stored (sequence scoring reads them) but never returned."""
    from nafp_b200 import synth
    dummy, db, query = synth.synth_search_set(30000, 590, seed=4)
    x = np.concatenate([dummy, db])
    g = _gpu_index([x])
    m = 30000 + 300 + 7                              # inside a tile
    g.set_search_rows(m)
    o = _oracle_index([x[:m]])
    Dg, Ig = g.search(query[:50], 20)
    Do, Io = o.search(query[:50], 20)
    assert Ig.max() < m
    assert_topk_matches(Dg, Ig, Do, Io, x[:m], query[:50])


def test_flat_search_fewer_rows_than_k():
    rng = np.random.default_rng(6)
    x = rng.standard_normal((7, 128)).astype(np.float32)
    q = rng.standard_normal((3, 128)).astype(np.float32)
    g, o = _gpu_index([x]), _oracle_index([x])
    Dg, Ig = g.search(q, 20)
    Do, Io = o.search(q, 20)
    assert (Ig[:, 7:] == -1).all() and np.isinf(Dg[:, 7:]).all()
    np.testing.assert_array_equal(Ig, Io)
    np.testing.assert_allclose(Dg[:, :7], Do[:, :7], atol=1e-4)


def test_flat_search_duplicates_fall_back_to_exact():
    """Hundreds of identical rows defeat the bf16 bound; the fp32 fallback must answer (and say so)."""
    from nafp_b200 import synth
    dummy, db, query = synth.synth_search_set(40000, 590, seed=9)
    dup = np.repeat(db[:1], 400, axis=0)
    x = np.concatenate([dummy, dup, db])
    g, o = _gpu_index([x]), _oracle_index([x])
    q = np.concatenate([db[:1], query[:4]])
    Dg, Ig = g.search(q, 20)
    Do, Io = o.search(q, 20)
    np.testing.assert_allclose(Dg, Do, atol=2e-5)
    assert set(Ig[0]) <= set(range(40000, 40400)) | {40400}
    assert g.last_search_stats()["fallback_rows"] >= 1
    assert_topk_matches(Dg[1:], Ig[1:], Do[1:], Io[1:], x, q[1:])


def test_reconstruct_roundtrip():
    rng = np.random.default_rng(1)
    x = rng.standard_normal((1000, 128)).astype(np.float32)
    g = _gpu_index([x[:300], x[300:]])
    np.testing.assert_array_equal(g.reconstruct_n(250, 100), x[250:350])


def test_self_query_property_large():
    """Size-independent property at ~1M rows: every stored row is its own nearest neighbour (d=0)."""
    from nafp_b200 import synth
    dummy = synth.synth_fp_db(1000000, seed=11)
    g = _gpu_index([dummy])
    rows = np.random.default_rng(0).integers(0, len(dummy), 256)
    D, I = g.search(dummy[rows], 20)
    assert (I[:, 0] == rows).all()
    assert np.abs(D[:, 0]).max() < 1e-5
    assert (np.diff(D, axis=1) >= -1e-7).all()
    # spot-check three rows against a blocked exact numpy scan
    for r in range(3):
        d = ((dummy.astype(np.float64) - dummy[rows[r]].astype(np.float64)) ** 2).sum(1)
        ref = np.lexsort((np.arange(len(d)), d))[:20]
        mism = I[r] != ref
        assert np.abs(d[I[r]] - d[ref]).max() <= 4e-6 and mism.sum() <= 2
    assert g.last_search_stats()["fallback_rows"] == 0


@pytest.mark.parametrize("n_dummy", [60000, 2000])
def test_seq_match_matches_oracle(n_dummy):
    from nafp_b200 import synth
    from oracle import seq_match
    dummy, db, query = synth.synth_search_set(n_dummy, 2950, seed=4)
    g, o = _gpu_index([dummy, db]), _oracle_index([dummy, db])
    recon = np.concatenate([dummy, db])
    rng = np.random.default_rng(2)
    test_ids = np.concatenate([rng.integers(0, 2950 - 19, 60), [2950 - 5, 2950 - 19, 2950 - 1, 0]]).astype(np.int64)
    seq_lens = [1, 3, 5, 9, 11, 19]
    pred_g, score_g = g.seq_match(query, test_ids, seq_lens, k_probe=20)
    raw_o, pred_o = seq_match.evaluate(o, query, recon, n_dummy, test_ids, seq_lens, k_probe=20)
    # hit flags from the GPU predictions, computed the reference's way
    raw_g = np.zeros_like(raw_o)
    n_len = len(seq_lens)
    for ti, tid in enumerate(test_ids):
        for si in range(n_len):
            p = pred_g[ti, si]
            p = p[p >= 0]
            f = seq_match.hit_flags(p, tid + n_dummy)
            for b in range(4):
                raw_g[ti, b * n_len + si] = f[b]
    diff = np.argwhere(pred_g != pred_o)
    # any disagreement must be a score tie (fp32 summation order), never a different candidate set
    for ti, si, r in diff:
        assert abs(score_g[ti, si, r] - score_g[ti, si, max(r - 1, 0)]) < 1e-5 or \
               abs(score_g[ti, si, r] - score_g[ti, si, min(r + 1, 9)]) < 1e-5
    assert len(diff) <= 4
    assert np.abs(seq_match.hit_rates(raw_g, n_len) - seq_match.hit_rates(raw_o, n_len)).max() <= 0.1 + 100.0 * 2 / len(test_ids)
    np.testing.assert_array_equal(raw_g[:, :n_len], raw_o[:, :n_len]) if len(diff) == 0 else None


@pytest.mark.parametrize("seed", [3, 4])
def test_flat_search_fuzz(seed):
    """Random sizes, query counts, k, norms and ragged adds against the fp64 oracle, nine cases per seed."""
    rng = np.random.default_rng(seed)
    for case in range(9):
        n = int(rng.integers(8200, 260000))
        nq = int(rng.choice([1, 2, 31, 32, 33, 127, 128, 129, 255, 256, 257, 300, 511, 512, 513, 600, 1100]))
        k = int(rng.choice([1, 5, 20, 33, 64]))
        x = rng.standard_normal((n, 128)).astype(np.float32)
        mode = case % 3
        if mode == 0:
            x /= np.linalg.norm(x, axis=1, keepdims=True)
        elif mode == 1:
            x *= rng.uniform(0.5, 1.5, (n, 1)).astype(np.float32)
        else:
            x /= np.linalg.norm(x, axis=1, keepdims=True)
            x[rng.integers(0, n, 50)] = 0.0
        q = x[rng.integers(0, n, nq)] * rng.uniform(0.8, 1.2) + 0.3 / 128 ** 0.5 * rng.standard_normal((nq, 128)).astype(np.float32)
        cuts = np.unique(np.concatenate([[0, n], rng.integers(0, n, 3)]))
        g = _gpu_index([x[a:b] for a, b in zip(cuts[:-1], cuts[1:])])
        o = _oracle_index([x])
        Dg, Ig = g.search(q, k)
        Do, Io = o.search(q, k)
        assert_topk_matches(Dg, Ig, Do, Io, x, q, dtol=3e-3 if mode == 1 else 1e-4)


@pytest.mark.parametrize("nq", [1, 300])
def test_flat_search_edge_tile_hits(nq):
    """Hits inside the tile that holds the search_rows limit: only the exact per-column path of such a tile
    (rows < m of it may be returned) sees them.  Each query has an exact copy just past m, which must never come
    back, and a near copy just before m, which must come back first.  The tile also ends in padding rows."""
    rng = np.random.default_rng(21)
    n_base = 48
    m = 156 * 256 + 128 + 7                          # inside a tile, with n_base rows on either side
    n = m + n_base + 12                              # not a multiple of 256: the same tile ends in padding
    x = rng.standard_normal((n + n_base, 128)).astype(np.float32)
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    x, base = x[:n], x[n:]
    near = base + 0.01 * rng.standard_normal(base.shape).astype(np.float32)
    x[m - n_base:m] = near / np.linalg.norm(near, axis=1, keepdims=True)
    x[m:m + n_base] = base                           # halo: distance 0, never returnable
    which = np.arange(nq) % n_base
    q = base[which]
    g = _gpu_index([x])
    g.set_search_rows(m)
    o = _oracle_index([x[:m]])
    Dg, Ig = g.search(q, 20)
    Do, Io = o.search(q, 20)
    assert Ig.max() < m
    np.testing.assert_array_equal(Ig[:, 0], m - n_base + which)
    assert_topk_matches(Dg, Ig, Do, Io, x[:m], q)
    assert g.last_search_stats()["fallback_rows"] == 0
