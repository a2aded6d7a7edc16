"""GPU parity: IVF-PQ (SURVEY §8 a6).  With the SAME quantizers the CUDA index must agree with the
oracle id for id (codes, lists, ADC distances); with its own k-means training the contract is the
top-1 hit rate (within 0.1 pt of the oracle trained on the same data is a statistical statement, so
the test uses a generous margin at this tiny scale and the exact comparison carries the parity)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def test_ivfpq_same_quantizers_matches_oracle():
    from nafp_b200 import synth
    from nafp_b200.eval.utils.get_index import IVFPQ, Index
    from oracle.ivfpq_index import IVFPQ as OracleIVFPQ
    dummy, db, query = synth.synth_search_set(30000, 1180, seed=7)
    g = Index(IVFPQ, 128, nlist=256, pq_m=64, pq_nbits=8)
    assert not g.is_trained
    g.train(dummy, seed=1234)
    assert g.is_trained
    coarse, pq = g.ivfpq_params()
    assert np.isfinite(coarse).all() and np.isfinite(pq).all()
    g.add(dummy)
    g.add(db)
    g.nprobe = 40
    o = OracleIVFPQ(128, 256, 64, 8)
    o.set_params(coarse, pq)
    o.add(dummy)
    o.add(db)
    o.nprobe = 40
    q = query[:64]
    Dg, Ig = g.search(q, 20)
    Do, Io = o.search(q, 20)
    np.testing.assert_allclose(Dg, Do, rtol=0, atol=2e-5)
    bad = np.argwhere(Ig != Io)
    for r, c in bad:          # only permutations among (near-)equal ADC distances are tolerated
        assert abs(Do[r, c] - Dg[r, c]) < 2e-5 and abs(Do[r, list(Io[r]).index(Ig[r, c])] - Dg[r, c]) < 2e-5 if Ig[r, c] in Io[r] else False
    assert len(bad) <= 0.02 * Ig.size
    # the hit-rate contract: sequence matcher on top of the approximate segment search
    from oracle import seq_match
    ids = np.arange(0, 1100, 37, dtype=np.int64)
    lens = [1, 3, 5, 9]
    pred_g, _ = g.seq_match(query, ids, lens, 20)
    raw_o, pred_o = seq_match.evaluate(o, query, np.concatenate([dummy, db]), len(dummy), ids, lens, 20)
    top1_g = (pred_g[:, :, 0] == (ids + len(dummy))[:, None]).mean(0) * 100
    top1_o = seq_match.hit_rates(raw_o, len(lens))[0]
    assert np.abs(top1_g - top1_o).max() <= 100.0 / len(ids) + 1e-9


@pytest.mark.parametrize("nprobe,k", [(1, 20), (3, 5), (40, 40)])
def test_ivfpq_fallback_and_fast_path_agree_with_oracle(nprobe, k):
    """Few probed lists, or k = 40 (two slices per probed list): the default search -- the list-major scan, with the
    LUT kernel for the rows its proof cannot settle -- gives the oracle's answers with the same quantizers."""
    from nafp_b200 import synth
    from nafp_b200.eval.utils.get_index import IVFPQ, Index
    from oracle.ivfpq_index import IVFPQ as OracleIVFPQ
    dummy, db, query = synth.synth_search_set(12000, 590, seed=17)
    g = Index(IVFPQ, 128, nlist=256, pq_m=64, pq_nbits=8)
    g.train(dummy, seed=7)
    g.add(dummy)
    g.add(db)
    g.nprobe = nprobe
    o = OracleIVFPQ(128, 256, 64, 8)
    o.set_params(*g.ivfpq_params())
    o.add(dummy)
    o.add(db)
    o.nprobe = nprobe
    q = query[:48]
    Dg, Ig = g.search(q, k)
    Do, Io = o.search(q, k)
    fin = np.isfinite(Do)
    assert (np.isfinite(Dg) == fin).all() and ((Ig < 0) == (Io < 0)).all()
    np.testing.assert_allclose(Dg[fin], Do[fin], rtol=0, atol=2e-5)
    same = Ig == Io
    assert same.mean() >= 0.98
    for r, c in np.argwhere(~same):            # only permutations among (near-)equal ADC distances
        assert Ig[r, c] in Io[r] or abs(Dg[r, c] - Do[r, min(c + 1, k - 1)]) < 2e-5 or abs(Dg[r, c] - Do[r, c]) < 2e-5


def test_ivfpq_own_training_hit_rate_within_a_tenth_of_a_point():
    """The IVF-PQ gate of north_star -- top-1 hit rate within 0.1 pt of the reference index -- at a scale where 0.1 pt
    is resolvable: 200,000 + 2,360 rows, 2,360 query rows, three training seeds, BOTH sides running their OWN k-means
    (GPU: csrc/ivfpq.cu; oracle: the C restatement oracle/csrc/oracle.c) on the same seeded training subset.
    Measured: segment-level top-1 recall against the exact search and sequence-level top-1 hit rate of the
    evaluation loop; the averages over the seeds must agree to 0.1 pt, every single seed to 0.3 pt."""
    from nafp_b200 import synth
    from nafp_b200.eval.utils.get_index import IVFPQ, Index
    from oracle import native, seq_match
    dummy, db, query = synth.synth_search_set(200_000, 2360, seed=31)
    recon = np.concatenate([dummy, db])
    flat = native.FlatL2C(128)
    flat.add(dummy)
    flat.add(db)
    _, Ie = flat.search(query, 1)
    ids = np.arange(0, 2360 - 19, 4)                       # 586 sequences x 3 lengths
    lens = [1, 3, 5]
    gt = ids + len(dummy)
    rec, hit = [], []
    for seed in (1234, 7, 99):
        g = Index(IVFPQ, 128, nlist=256, pq_m=64, pq_nbits=8)
        g.train(dummy[:100_000], seed=seed)
        g.add(dummy)
        g.add(db)
        g.nprobe = 40
        o = native.IVFPQC(128, 256, 64, 8)
        o.train(dummy[:100_000], seed=seed)
        o.add(dummy)
        o.add(db)
        o.nprobe = 40
        cg, pg = g.ivfpq_params()
        # same algorithm, same rows, same fp32 rounding of the assignment distances: the two trainings agree
        print("seed", seed, "mean |coarse diff|", float(np.abs(cg - o.coarse).mean()), "mean |pq diff|", float(np.abs(pg - o.pq).mean()))
        assert np.abs(cg - o.coarse).mean() < 1e-2 and np.abs(pg - o.pq).mean() < 2e-2
        _, Ig = g.search(query, 20)
        _, Io = o.search(query, 20)
        rec.append(((Ig[:, 0] == Ie[:, 0]).mean(), (Io[:, 0] == Ie[:, 0]).mean()))
        pred_g, _ = g.seq_match(query, ids, lens, 20)
        _, pred_o = seq_match.evaluate(o, query, recon, len(dummy), ids, lens, 20, fast_scores=True, batch_search=True)
        hit.append(((pred_g[:, :, 0] == gt[:, None]).mean(0), (pred_o[:, :, 0] == gt[:, None]).mean(0)))
        del g
    rec, hit = np.array(rec), np.array(hit)
    print("segment top-1 recall (gpu, oracle) per seed:", rec.tolist())
    print("sequence top-1 hit rate (gpu, oracle) per seed:", hit.tolist())
    assert 0.5 < rec[:, 1].mean() < 0.999                  # the approximation is visible: the comparison means something
    assert np.abs(rec[:, 0] - rec[:, 1]).max() <= 0.003 and abs(rec[:, 0].mean() - rec[:, 1].mean()) <= 0.001
    assert np.abs(hit[:, 0] - hit[:, 1]).max() <= 0.003 and np.abs(hit[:, 0].mean(0) - hit[:, 1].mean(0)).max() <= 0.001


def test_ivfpq_untrained_add_is_refused():
    from nafp_b200._lib import NafpError
    from nafp_b200.eval.utils.get_index import IVFPQ, Index
    g = Index(IVFPQ, 128)
    with pytest.raises(NafpError):
        g.add(np.zeros((4, 128), np.float32))


@pytest.mark.parametrize("nlist,nprobe,k", [(400, 40, 20), (400, 2, 20), (64, 64, 5), (100, 10, 40)])
def test_ivf_flat_same_centroids_matches_oracle(nlist, nprobe, k):
    """index_type 'ivf' (faiss.IndexIVFFlat, nlist 400, nprobe 40): with the same coarse centroids the CUDA index
    returns the oracle's rows -- through the scan + probed-list filter (most rows at nprobe 40), through the
    exact list scan (few probes: most rows lack k probed rows among their 64 nearest) and for k above the fast
    path's limit."""
    from nafp_b200 import synth
    from nafp_b200.eval.utils.get_index import IVF_FLAT, Index
    from oracle.ivf_flat_index import IVFFlat
    dummy, db, query = synth.synth_search_set(20000, 590, seed=27)
    g = Index(IVF_FLAT, 128, nlist=nlist)
    assert not g.is_trained
    g.train(dummy, seed=99)
    assert g.is_trained
    g.add(dummy)
    g.add(db)
    g.nprobe = nprobe
    o = IVFFlat(128, nlist)
    o.set_coarse(g.ivf_coarse())
    o.add(dummy)
    o.add(db)
    o.nprobe = nprobe
    q = query[:96]
    Dg, Ig = g.search(q, k)
    Do, Io = o.search(q, k)
    fin = np.isfinite(Do)
    assert (np.isfinite(Dg) == fin).all() and ((Ig < 0) == (Io < 0)).all()
    np.testing.assert_allclose(Dg[fin], Do[fin], rtol=0, atol=2e-5)
    same = Ig == Io
    assert same.mean() >= 0.99
    for r, c in np.argwhere(~same):            # only permutations among (near-)equal distances
        assert abs(Dg[r, c] - Do[r, c]) < 2e-5 and Ig[r, c] in Io[r]


def test_ivf_flat_through_get_index_and_matcher():
    """get_index('ivf', ...) trains nlist 400 on the dummy rows, nprobe 40; the sequence matcher on top of it
    agrees with the oracle index holding the same centroids."""
    from nafp_b200 import synth
    from nafp_b200.eval.utils.get_index import get_index
    from oracle import seq_match
    from oracle.ivf_flat_index import IVFFlat
    dummy, db, query = synth.synth_search_set(30000, 1180, seed=31)
    g = get_index('ivf', dummy, dummy.shape, True, 1e7)
    assert g.nlist == 400 and g.nprobe == 40 and g.is_trained
    g.add(dummy)
    g.add(db)
    o = IVFFlat(128, 400)
    o.set_coarse(g.ivf_coarse())
    o.add(dummy)
    o.add(db)
    o.nprobe = 40
    ids = np.arange(0, 1100, 37, dtype=np.int64)
    lens = [1, 3, 5, 9]
    pred_g, _ = g.seq_match(query, ids, lens, 20)
    raw_o, pred_o = seq_match.evaluate(o, query, np.concatenate([dummy, db]), len(dummy), ids, lens, 20)
    assert (pred_g[:, :, 0] == np.asarray(pred_o)[:, :, 0]).all()


def test_ivf_flat_untrained_add_is_refused():
    from nafp_b200._lib import NafpError
    from nafp_b200.eval.utils.get_index import IVF_FLAT, Index
    g = Index(IVF_FLAT, 128, nlist=400)
    with pytest.raises(NafpError):
        g.add(np.zeros((4, 128), np.float32))


def test_ivfpq_rr_same_quantizers_matches_oracle():
    """index_type 'ivfpq-rr' (faiss.IndexIVFPQR, get_index_faiss.py:75-85): with the GPU-trained quantizers of both levels
    handed to the oracle, codes, refinement codes and re-ranked answers agree; own training on both sides (same seed)
    gives the same top-1 recall."""
    from nafp_b200 import synth
    from nafp_b200.eval.utils.get_index import IVFPQR, Index, get_index
    from oracle.flat_index import FlatL2
    from oracle.ivfpq_index import IVFPQR as OracleIVFPQR
    dummy, db, query = synth.synth_search_set(20000, 590, seed=41)
    g = Index(IVFPQR, 128, nlist=64, pq_m=64, pq_nbits=8)
    g.train(dummy[:16000], seed=77)
    g.add(dummy)
    g.add(db)
    g.nprobe = 16
    o = OracleIVFPQR(128, 64, 64, 8)
    o.set_params(*g.ivfpq_params())
    o.set_refine(g.ivfpqr_refine())
    o.add(dummy)
    o.add(db)
    o.nprobe = 16
    q = query[:64]
    Dg, Ig = g.search(q, 20)
    Do, Io = o.search(q, 20)
    assert ((Ig < 0) == (Io < 0)).all()
    fin = np.isfinite(Do)
    np.testing.assert_allclose(Dg[fin], Do[fin], rtol=0, atol=3e-5)
    same = Ig == Io
    assert same.mean() >= 0.97, same.mean()
    for r, c in np.argwhere(~same):            # only permutations among near-equal refined distances / first-level ties at rank 80
        assert abs(Dg[r, c] - Do[r, c]) < 3e-5 or Ig[r, c] in Io[r]
    # the sequence matcher runs on it like on the other index types
    ids = np.arange(0, 560, 20)
    pred, _ = g.seq_match(query, ids, [1, 3, 5], 20)
    assert (pred[:, 2, 0] == ids + len(dummy)).mean() > 0.9
    # own training: oracle vs GPU
    o2 = OracleIVFPQR(128, 64, 64, 8)
    o2.train(dummy[:16000], seed=77)
    o2.add(dummy)
    o2.add(db)
    o2.nprobe = 16
    flat = FlatL2(128)
    flat.add(dummy)
    flat.add(db)
    _, Ie = flat.search(query[:300], 1)
    _, Ig2 = g.search(query[:300], 20)
    _, Io2 = o2.search(query[:300], 20)
    rg, ro = (Ig2[:, 0] == Ie[:, 0]).mean(), (Io2[:, 0] == Ie[:, 0]).mean()
    assert abs(rg - ro) <= 0.02 and rg > 0.6, (rg, ro)
    # factory + the reference's error for the CPU-only types
    idx = get_index('ivfpq-rr', dummy[:8000], (8000, 128), True, 1e7)
    assert idx.is_trained and idx.nprobe == 40
    for mode in ('hnsw', 'ivfpq-ondisk'):
        with pytest.raises(NotImplementedError, match='only available in CPU'):
            get_index(mode, dummy[:100], (100, 128), True, 1e7)


# ------------------------------------------------------------------------------------------ list-major path (ivfpq_lm.cu)
def _ivfpq_with_path(monkeypatch, path, params, parts, nprobe, nlist=256):
    """An IVF-PQ index searched through `path` (NAFP_IVFPQ_PATH is read when the index is created)."""
    from nafp_b200.eval.utils.get_index import IVFPQ, Index
    monkeypatch.setenv("NAFP_IVFPQ_PATH", path)
    g = Index(IVFPQ, 128, nlist=nlist, pq_m=64, pq_nbits=8)
    g.set_ivfpq_params(*params)
    for p in parts:
        g.add(p)
    g.nprobe = nprobe
    return g


def _trained_params(train, nlist=256, seed=5):
    from nafp_b200.eval.utils.get_index import IVFPQ, Index
    t = Index(IVFPQ, 128, nlist=nlist, pq_m=64, pq_nbits=8)
    t.train(train, seed=seed)
    return t.ivfpq_params()


def test_ivfpq_search_paths_agree(monkeypatch):
    """The default list-major tensor-core scan and the LUT kernel answer alike: the list-major path re-scores its
    survivors with the LUT kernel's fp32 arithmetic, so its distances are bit-identical to the LUT path's and its ids
    equal; none of its rows needed the fallback."""
    from nafp_b200 import synth
    dummy, db, query = synth.synth_search_set(60000, 1180, seed=23)
    params = _trained_params(dummy[:40000])
    idx = {p: _ivfpq_with_path(monkeypatch, p, params, (dummy, db), 40) for p in ("lm", "lut")}
    q = query[:700]
    res = {p: g.search(q, 20) for p, g in idx.items()}
    st = idx["lm"].last_search_stats()
    assert st["rows"] == len(q) and st["fallback_rows"] == 0 and st["passes"] > 0, st      # passes = list-major work items
    assert idx["lut"].last_search_stats()["fallback_rows"] == len(q)
    np.testing.assert_array_equal(res["lm"][0], res["lut"][0])
    np.testing.assert_array_equal(res["lm"][1], res["lut"][1])


@pytest.mark.parametrize("n_rows,nlist,nprobe,k,nq", [(300, 64, 64, 5, 1), (300, 64, 1, 24, 3), (5000, 256, 40, 1, 130),
                                                      (5000, 16, 16, 20, 257), (40, 8, 3, 24, 19)])
def test_ivfpq_list_major_ragged_shapes(monkeypatch, n_rows, nlist, nprobe, k, nq):
    """Empty and tiny lists, lists shorter than one tile, fewer rows than k, one query row, more than one block of query
    rows per list: identical to the LUT kernel, and to the oracle within its tolerance."""
    from nafp_b200 import synth
    from oracle.ivfpq_index import IVFPQ as OracleIVFPQ
    dummy, db, query = synth.synth_search_set(max(n_rows, 3000), 590, seed=29)
    params = _trained_params(dummy[:3000], nlist=nlist)
    rows = dummy[:n_rows]
    a = _ivfpq_with_path(monkeypatch, "lm", params, (rows,), nprobe, nlist)
    b = _ivfpq_with_path(monkeypatch, "lut", params, (rows,), nprobe, nlist)
    q = query[:nq]
    Da, Ia = a.search(q, k)
    Db, Ib = b.search(q, k)
    np.testing.assert_array_equal(Da, Db)
    np.testing.assert_array_equal(Ia, Ib)
    o = OracleIVFPQ(128, nlist, 64, 8)
    o.set_params(*params)
    o.add(rows)
    o.nprobe = nprobe
    Do, Io = o.search(q, k)
    fin = np.isfinite(Do)
    assert (np.isfinite(Da) == fin).all() and ((Ia < 0) == (Io < 0)).all()
    np.testing.assert_allclose(Da[fin], Do[fin], rtol=0, atol=2e-5)
    assert (Ia == Io).mean() >= 0.97


def test_ivfpq_list_major_duplicates_go_to_the_lut_kernel(monkeypatch):
    """60 identical rows next to a query: the 32-entry candidate list of their list ends in a tie, the proof fails, the
    row is answered by the LUT kernel -- same ids (ties to the lower id) as the LUT path."""
    from nafp_b200 import synth
    dummy, db, query = synth.synth_search_set(20000, 590, seed=31)
    params = _trained_params(dummy[:12000])
    dup = np.repeat(db[7:8], 60, axis=0)
    parts = (dummy, dup, db)
    a = _ivfpq_with_path(monkeypatch, "lm", params, parts, 40)
    b = _ivfpq_with_path(monkeypatch, "lut", params, parts, 40)
    q = np.concatenate([db[7:8], query[:40]])
    Da, Ia = a.search(q, 20)
    Db, Ib = b.search(q, 20)
    np.testing.assert_array_equal(Da, Db)
    np.testing.assert_array_equal(Ia, Ib)
    assert (Ia[0] == np.arange(20000, 20020)).all()           # the 20 lowest ids of the 61 tied rows
    assert a.last_search_stats()["fallback_rows"] >= 1


def test_ivfpq_list_major_respects_search_rows(monkeypatch):
    """Rows past search_rows (the halo of a row-sharded index) are stored but never returned."""
    from nafp_b200 import synth
    dummy, db, query = synth.synth_search_set(20000, 590, seed=37)
    params = _trained_params(dummy[:12000])
    a = _ivfpq_with_path(monkeypatch, "lm", params, (dummy, db), 40)
    b = _ivfpq_with_path(monkeypatch, "lut", params, (dummy, db), 40)
    full = a.search(query[:64], 20)[1]
    assert (full >= 20000).any()
    for g in (a, b):
        g.set_search_rows(20000)
    Da, Ia = a.search(query[:64], 20)
    Db, Ib = b.search(query[:64], 20)
    assert (Ia < 20000).all()
    np.testing.assert_array_equal(Da, Db)
    np.testing.assert_array_equal(Ia, Ib)
    a.set_search_rows(-1)
    np.testing.assert_array_equal(a.search(query[:64], 20)[1], full)


def test_ivfpq_add_after_search_rebuilds_lists_from_released_codes(monkeypatch):
    """The row-order copy of the codes is released once the lists are built (76 B per row stay); a later add regenerates
    it from the lists.  Same answers as an index that received all rows before its first search."""
    from nafp_b200 import synth
    dummy, db, query = synth.synth_search_set(30000, 1180, seed=43)
    params = _trained_params(dummy[:20000])
    a = _ivfpq_with_path(monkeypatch, "lm", params, (dummy[:17000],), 40)
    first = a.search(query[:32], 20)[1]
    assert (first < 17000).all()
    a.add(dummy[17000:])
    a.search(query[:8], 5)
    a.add(db)
    b = _ivfpq_with_path(monkeypatch, "lm", params, (dummy, db), 40)
    Da, Ia = a.search(query[:200], 20)
    Db, Ib = b.search(query[:200], 20)
    np.testing.assert_array_equal(Da, Db)
    np.testing.assert_array_equal(Ia, Ib)
    assert a.ntotal == b.ntotal == 31180


def test_ivfpq_list_major_more_query_rows_than_one_launch_group(monkeypatch):
    """33,000 query rows (> LM_CHUNK_Q = 32,768): the search runs in two launch groups; every row equals the LUT path's."""
    from nafp_b200 import synth
    dummy, db, query = synth.synth_search_set(6000, 590, seed=47)
    params = _trained_params(dummy[:4000], nlist=64)
    a = _ivfpq_with_path(monkeypatch, "lm", params, (dummy, db), 6, nlist=64)
    b = _ivfpq_with_path(monkeypatch, "lut", params, (dummy, db), 6, nlist=64)
    rng = np.random.default_rng(3)
    q = query[rng.integers(0, len(query), 33000)] + 0.05 * rng.standard_normal((33000, 128)).astype(np.float32)
    q = (q / np.linalg.norm(q, axis=1, keepdims=True)).astype(np.float32)
    Da, Ia = a.search(q, 10)
    Db, Ib = b.search(q, 10)
    np.testing.assert_array_equal(Ia, Ib)
    np.testing.assert_array_equal(Da, Db)
