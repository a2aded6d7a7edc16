"""GPU: the list-major IVF-PQ scan for 24 < k <= 128 (ceil(k / 24) slices per probed list), IVFPQR ('ivfpq-rr') on it, the
LUT kernel's two-round merge for nprobe * k > 4096, and row-sharded IVFPQR."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

WIDE_K = [25, 32, 64, 80, 128]


def _index(monkeypatch, path, params, parts, nprobe, nlist=256, itype=None, refine=None):
    """An IVF-PQ (or IVFPQR) index searched through `path` (NAFP_IVFPQ_PATH is read when the index is created)."""
    from nafp_b200.eval.utils.get_index import IVFPQ, Index
    monkeypatch.setenv("NAFP_IVFPQ_PATH", path)
    g = Index(IVFPQ if itype is None else itype, 128, nlist=nlist, pq_m=64, pq_nbits=8)
    g.set_ivfpq_params(*params)
    if refine is not None:
        g.set_ivfpqr_refine(refine)
    for p in parts:
        g.add(p)
    g.nprobe = nprobe
    return g


def _trained_params(train, nlist=256, seed=5):
    from nafp_b200.eval.utils.get_index import IVFPQ, Index
    t = Index(IVFPQ, 128, nlist=nlist, pq_m=64, pq_nbits=8)
    t.train(train, seed=seed)
    return t.ivfpq_params()


def _same(a, b, q, k):
    Da, Ia = a.search(q, k)
    Db, Ib = b.search(q, k)
    np.testing.assert_array_equal(Da, Db)
    np.testing.assert_array_equal(Ia, Ib)
    return Da, Ia


@pytest.mark.parametrize("k", WIDE_K)
@pytest.mark.parametrize("n_rows,nlist,nprobe,nq", [(300, 64, 64, 1), (300, 64, 1, 3), (5000, 256, 40, 130),
                                                    (5000, 16, 16, 257), (40, 8, 3, 19)])
def test_wide_k_ragged_shapes_equal_the_lut_kernel(monkeypatch, k, n_rows, nlist, nprobe, nq):
    """Lists shorter than S tiles (empty slices), fewer rows than k, nprobe 1 / 40 / 64, more than one block of query
    rows per list: bit-identical to the LUT kernel, and to the oracle within its tolerance."""
    from nafp_b200 import synth
    from oracle.ivfpq_index import IVFPQ as OracleIVFPQ
    dummy, db, query = synth.synth_search_set(max(n_rows, 3000), 590, seed=29)
    params = _trained_params(dummy[:3000], nlist=nlist)
    rows = dummy[:n_rows]
    a = _index(monkeypatch, "lm", params, (rows,), nprobe, nlist)
    b = _index(monkeypatch, "lut", params, (rows,), nprobe, nlist)
    q = query[:nq]
    Da, Ia = _same(a, b, q, k)
    assert a.last_search_stats()["passes"] > 0
    o = OracleIVFPQ(128, nlist, 64, 8)
    o.set_params(*params)
    o.add(rows)
    o.nprobe = nprobe
    Do, Io = o.search(q, k)
    fin = np.isfinite(Do)
    assert (np.isfinite(Da) == fin).all() and ((Ia < 0) == (Io < 0)).all()
    np.testing.assert_allclose(Da[fin], Do[fin], rtol=0, atol=2e-5)
    assert (Ia == Io).mean() >= 0.97


@pytest.mark.parametrize("k", WIDE_K)
def test_wide_k_duplicates_go_to_the_lut_kernel(monkeypatch, k):
    """k + 40 identical rows next to a query: the slices' candidate lists end in ties, the proof fails, the row is
    answered by the LUT kernel -- the k lowest ids of the tied rows, as on the LUT path."""
    from nafp_b200 import synth
    dummy, db, query = synth.synth_search_set(20000, 590, seed=31)
    params = _trained_params(dummy[:12000])
    dup = np.repeat(db[7:8], k + 40, axis=0)
    parts = (dummy, dup, db)
    a = _index(monkeypatch, "lm", params, parts, 40)
    b = _index(monkeypatch, "lut", params, parts, 40)
    q = np.concatenate([db[7:8], query[:40]])
    _, Ia = _same(a, b, q, k)
    assert (Ia[0] == np.arange(20000, 20000 + k)).all()
    assert a.last_search_stats()["fallback_rows"] >= 1


@pytest.mark.parametrize("k", WIDE_K)
def test_wide_k_respects_search_rows(monkeypatch, k):
    """Rows past search_rows (the halo of a row-sharded index) are never returned by any slice."""
    from nafp_b200 import synth
    dummy, db, query = synth.synth_search_set(20000, 590, seed=37)
    params = _trained_params(dummy[:12000])
    a = _index(monkeypatch, "lm", params, (dummy, db), 40)
    b = _index(monkeypatch, "lut", params, (dummy, db), 40)
    assert (a.search(query[:64], k)[1] >= 20000).any()
    for g in (a, b):
        g.set_search_rows(20000)
    _, Ia = _same(a, b, query[:64], k)
    assert (Ia < 20000).all()


def test_wide_k_more_query_rows_than_one_launch_group(monkeypatch):
    """k = 128 (6 slices): a launch group holds 32,768 / 6 = 5,461 query rows; 12,000 rows run in three groups, every row
    equal to the LUT path's."""
    from nafp_b200 import synth
    dummy, db, query = synth.synth_search_set(6000, 590, seed=47)
    params = _trained_params(dummy[:4000], nlist=64)
    a = _index(monkeypatch, "lm", params, (dummy, db), 6, nlist=64)
    b = _index(monkeypatch, "lut", params, (dummy, db), 6, nlist=64)
    rng = np.random.default_rng(3)
    q = query[rng.integers(0, len(query), 12000)] + 0.05 * rng.standard_normal((12000, 128)).astype(np.float32)
    q = (q / np.linalg.norm(q, axis=1, keepdims=True)).astype(np.float32)
    _same(a, b, q, 128)


def test_wide_k_fallback_rows_on_the_search_paths_set(monkeypatch):
    """The 60,000-row set of test_ivfpq_search_paths_agree at k = 80: the list-major path answers (passes > 0),
    bit-identical to the LUT kernel, with at most 1 % of the rows sent to the LUT kernel."""
    from nafp_b200 import synth
    dummy, db, query = synth.synth_search_set(60000, 1180, seed=23)
    params = _trained_params(dummy[:40000])
    a = _index(monkeypatch, "lm", params, (dummy, db), 40)
    b = _index(monkeypatch, "lut", params, (dummy, db), 40)
    q = query[:700]
    _same(a, b, q, 80)
    st = a.last_search_stats()
    print(f"k 80: {st}")
    assert st["rows"] == len(q) and st["passes"] > 0 and st["fallback_rows"] <= 0.01 * len(q), st


def test_lut_kernel_merges_in_two_rounds_when_nprobe_k_exceeds_4096(monkeypatch):
    """nprobe 64 x k 128 = 8,192 partial keys per row (two rounds of the 4,096-key merge) give the oracle's answer."""
    from nafp_b200 import synth
    from oracle.ivfpq_index import IVFPQ as OracleIVFPQ
    dummy, db, query = synth.synth_search_set(8000, 590, seed=53)
    params = _trained_params(dummy[:6000], nlist=128)
    b = _index(monkeypatch, "lut", params, (dummy,), 64, nlist=128)
    q = query[:20]
    for k in (65, 100, 128):
        Db, Ib = b.search(q, k)
        o = OracleIVFPQ(128, 128, 64, 8)
        o.set_params(*params)
        o.add(dummy)
        o.nprobe = 64
        Do, Io = o.search(q, k)
        np.testing.assert_allclose(Db, Do, rtol=0, atol=2e-5)
        assert (Ib == Io).mean() >= 0.97


# ------------------------------------------------------------------------------------------ ivfpq-rr
def _ivfpqr_params(train, nlist=256, seed=77):
    from nafp_b200.eval.utils.get_index import IVFPQR, Index
    t = Index(IVFPQR, 128, nlist=nlist, pq_m=64, pq_nbits=8)
    t.train(train, seed=seed)
    return t.ivfpq_params(), t.ivfpqr_refine()


@pytest.mark.parametrize("k_probe", [20, 32])
def test_ivfpq_rr_list_major_first_level_equals_lut(monkeypatch, k_probe):
    """ivfpq-rr at nprobe 40: its 4 k first-level candidates come from the list-major scan; the answer equals the LUT
    path's (k_probe 32: 128 candidates, whose LUT merge takes two rounds), and the oracle's within the gates of
    test_ivfpq_rr_same_quantizers_matches_oracle."""
    from nafp_b200 import synth
    from nafp_b200.eval.utils.get_index import IVFPQR
    from oracle.ivfpq_index import IVFPQR as OracleIVFPQR
    dummy, db, query = synth.synth_search_set(30000, 590, seed=41)
    params, rpq = _ivfpqr_params(dummy[:20000])
    a = _index(monkeypatch, "lm", params, (dummy, db), 40, itype=IVFPQR, refine=rpq)
    b = _index(monkeypatch, "lut", params, (dummy, db), 40, itype=IVFPQR, refine=rpq)
    q = query[:200]
    Da, Ia = _same(a, b, q, k_probe)
    st = a.last_search_stats()
    assert st["passes"] > 0 and st["fallback_rows"] <= 0.05 * len(q), st
    o = OracleIVFPQR(128, 256, 64, 8)
    o.set_params(*params)
    o.set_refine(rpq)
    o.add(dummy)
    o.add(db)
    o.nprobe = 40
    Do, Io = o.search(q[:64], k_probe)
    assert ((Ia[:64] < 0) == (Io < 0)).all()
    fin = np.isfinite(Do)
    np.testing.assert_allclose(Da[:64][fin], Do[fin], rtol=0, atol=3e-5)
    same = Ia[:64] == Io
    assert same.mean() >= 0.97, same.mean()
    for r, c in np.argwhere(~same):
        assert abs(Da[r, c] - Do[r, c]) < 3e-5 or Ia[r, c] in Io[r]


def test_ivfpq_rr_k_probe_32_through_eval_search(tmp_path):
    """`eval_search -i ivfpq-rr -k 32` (nprobe 40, 128 first-level candidates) runs end to end, unsharded and as a
    one-rank row-sharded index, and finds the query segments."""
    from nafp_b200 import synth
    from nafp_b200.eval.eval_search import run_eval
    dummy, db, query = synth.synth_search_set(30000, 590, seed=59)
    for name, arr in (("dummy_db", dummy), ("db", db), ("query", query)):
        mm = np.memmap(str(tmp_path / f"{name}.mm"), dtype="float32", mode="w+", shape=arr.shape)
        mm[:] = arr
        mm.flush()
        np.save(str(tmp_path / f"{name}_shape.npy"), np.asarray(arr.shape))
    ids = str(tmp_path / "ids.npy")
    np.save(ids, np.arange(0, 560, 7))
    rates = {}
    for sharded in (False, True):
        rates[sharded] = np.asarray(run_eval(str(tmp_path) + "/", index_type="ivfpq-rr", test_ids=ids, test_seq_len="1 3 5 9",
                                             k_probe=32, display_interval=5, live=False, sharded=sharded), dtype=float)
        raw = np.load(str(tmp_path / "raw_score.npy"))
        assert raw.shape == (80, 16) and raw[:, 12:].mean() > 0.9          # top-10 exact
    assert np.abs(rates[False] - rates[True]).max() <= 5.0


# ------------------------------------------------------------------------------------------ row-sharded ivfpq-rr
class _OneGpuComm:
    """broadcast between ShardedFlatIndex objects of one process: rank 0's tensors are recorded in call order and
    handed to rank 1 in the same order."""

    def __init__(self, log):
        self.log = log

    def broadcast(self, t, src=0):
        if not self.log["replay"]:
            self.log["sent"].append(t.clone())
        else:
            t.copy_(self.log["sent"].pop(0))
        return t


def test_ivfpqr_shard_train_broadcasts_the_refinement_codebooks():
    """ShardedFlatIndex.train of an IVFPQR index: rank 0 trains; coarse centroids, PQ codebooks AND the (4, 16, 32)
    refinement codebooks reach rank 1, whose codes then equal rank 0's."""
    from nafp_b200 import synth
    from nafp_b200.dist import ShardedFlatIndex
    from nafp_b200.eval.utils.get_index import IVFPQR
    dummy, db, _ = synth.synth_search_set(20000, 590, seed=61)
    log = {"sent": [], "replay": False}
    s0 = ShardedFlatIndex(len(dummy) + len(db), 0, 2, max_len=9, device=0, comm=_OneGpuComm(log), index_type=IVFPQR)
    s0.train(dummy, seed=3)
    assert len(log["sent"]) == 3
    log["replay"] = True
    s1 = ShardedFlatIndex(len(dummy) + len(db), 1, 2, max_len=9, device=0, comm=_OneGpuComm(log), index_type=IVFPQR)
    s1.train(None)
    assert not log["sent"]
    np.testing.assert_array_equal(s1.index.ivfpqr_refine(), s0.index.ivfpqr_refine())
    for a, b in zip(s1.index.ivfpq_params(), s0.index.ivfpq_params()):
        np.testing.assert_array_equal(a, b)
    assert s0.index.nprobe == s1.index.nprobe == 40


def test_two_ivfpqr_shards_equal_the_unsharded_index():
    """Two IVFPQR shards on one GPU (the collectives replaced by their definitions): the merged first level, then the
    merged per-shard re-ranks, give exactly the unsharded index's D / I; predictions as the other IVF shard tests."""
    import torch
    from nafp_b200 import synth
    from nafp_b200.dist import ShardedFlatIndex
    from nafp_b200.eval.utils.get_index import IVFPQR, Index
    dummy, db, query = synth.synth_search_set(30000, 1180, seed=16)
    plain = Index(IVFPQR, 128, nlist=256)
    plain.train(dummy, seed=5)
    plain.add(dummy)
    plain.add(db)
    plain.nprobe = 40
    shards = []
    for r in range(2):
        s = ShardedFlatIndex(len(dummy) + len(db), r, 2, max_len=9, device=0, index_type=IVFPQR)
        s.index.set_ivfpq_params(*plain.ivfpq_params())
        s.index.set_ivfpqr_refine(plain.ivfpqr_refine())
        s.index.nprobe = 40
        s.add_from([dummy, db])
        shards.append(s)
    dev = torch.device("cuda", 0)
    k = 20
    ids = np.arange(0, 1150, 29, dtype=np.int64)
    lens = [1, 3, 5, 9]
    ops = [s.ops(len(query)) for s in shards]
    assert all(hasattr(o, "refine") for o in ops)
    q = torch.from_numpy(np.ascontiguousarray(query, np.float32)).to(dev)
    t_ids = torch.from_numpy(ids).to(dev)
    t_sl = torch.from_numpy(np.asarray(lens, np.int32)).to(dev)
    plans = [o.plan(q, t_ids) for o in ops]
    first = [o.local_topk(p.qrows, k) for o, p in zip(ops, plans)]
    assert first[0][1].shape[1] == 4 * k
    _, Ic = ops[0].merge(torch.stack([d for d, _ in first]), torch.stack([i for _, i in first]))
    ref = [o.refine(p.qrows, Ic, k) for o, p in zip(ops, plans)]
    D, I = ops[0].merge(torch.stack([d for d, _ in ref]), torch.stack([i for _, i in ref]))
    torch.cuda.synchronize()
    Dp, Ip = plain.search(plans[0].qrows.cpu().numpy(), k)
    np.testing.assert_array_equal(I.cpu().numpy(), Ip)
    np.testing.assert_array_equal(D.cpu().numpy(), Dp)
    cs = [o.cand_scores(q, p, t_ids, t_sl, k, I) for o, p in zip(ops, plans)]
    scores = torch.maximum(cs[0][1], cs[1][1])
    pid, _ = ops[0].top(cs[0][0], scores, cs[0][2], len(lens))
    got = pid.cpu().numpy()
    want, _ = plain.seq_match(query, ids, lens, k)
    np.testing.assert_array_equal(got[:, :, 0], want[:, :, 0])
    assert (got == want).mean() >= 0.995
