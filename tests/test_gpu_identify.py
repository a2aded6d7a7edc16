"""GPU: the clip matcher (nafp_clip_match) against nafp_seq_match and the oracle, its edge cases, and `run.py identify`
end to end on a WAV corpus."""
import json
import os

import numpy as np
import pytest
import yaml

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAFP_ERR_INVALID = -1


@pytest.fixture(scope="module")
def small_db():
    from nafp_b200 import synth
    from nafp_b200.eval.utils.get_index import Index
    dummy, db, query = synth.synth_search_set(20000, 2950, seed=5)
    g = Index(0, 128)
    g.add(dummy)
    g.add(db)
    return g, dummy, db, query


def _clips(query, starts_lens):
    rows = np.concatenate([query[s:s + L] for s, L in starts_lens])
    off = np.concatenate([[0], np.cumsum([L for _, L in starts_lens])]).astype(np.int64)
    return rows, off


# 1. a clip of L <= 32 rows is what nafp_seq_match computes for seq_lens = [L], bit for bit
@pytest.mark.parametrize("k_probe", [1, 20, 51])
def test_agrees_bit_for_bit_with_seq_match(small_db, k_probe):
    g, _, _, query = small_db
    lens = [L for L in (1, 7, 19, 32) if L * k_probe <= 1024]        # nafp_seq_match's candidate table
    starts = {L: np.arange(3 + L, len(query) - 40, 397) for L in lens}
    mixed = [(int(s), L) for i in range(max(len(v) for v in starts.values())) for L in lens if i < len(starts[L])
             for s in [starts[L][i]]]                                    # clips of every length interleaved
    rows, off = _clips(query, mixed)
    pred, sc = g.clip_match(rows, off, k_probe=k_probe, n_top=10)
    for L in lens:
        sel = [i for i, (_, l) in enumerate(mixed) if l == L]
        ids = np.array([mixed[i][0] for i in sel], np.int64)
        p_ref, s_ref = g.seq_match(query, ids, [L], k_probe)
        assert np.array_equal(pred[sel], p_ref[:, 0]), L
        assert np.array_equal(sc[sel].view(np.uint32), s_ref[:, 0].view(np.uint32)), L


def _scores_banded(q, recon, cand, L):
    """seq_scores of oracle.seq_match for many candidates of a long clip: per block of database rows one product
    Q X^T (fp32), whose diagonals summed in fp64 are the candidates' sums; rows past the end add nothing (the clamp)."""
    from numpy.lib.stride_tricks import as_strided
    n, blk = len(recon), 4096
    out = np.empty(len(cand))
    for b0 in range(0, n, blk):
        sel = (cand >= b0) & (cand < b0 + blk)
        if not sel.any():
            continue
        G = np.zeros((L, blk + L), np.float64)
        x = recon[b0:min(n, b0 + blk + L)]
        G[:, :len(x)] = np.asarray(q, np.float32) @ np.asarray(x, np.float32).T
        diag = as_strided(G, shape=(blk, L), strides=(G.strides[1], G.strides[0] + G.strides[1])).sum(1)
        cs = cand[sel]
        out[sel] = diag[cs - b0] / np.minimum(L, n - cs)
    return out


def _oracle_match(index, query, recon, tid, L, k_probe, table_rows=None, n_pred=10):
    """oracle.seq_match.match_one for one clip; where its one-shot scoring would not fit in memory, its candidates
    scored by _scores_banded and ordered as match_one orders them."""
    from oracle import seq_match
    q = np.asarray(query[tid:tid + L])
    if table_rows is None:
        _, table_rows = index.search(q, k_probe)
    table_rows = np.asarray(table_rows, np.int64)
    table = np.full((len(query), k_probe), -1, np.int64)
    table[tid:tid + L] = table_rows
    I = table_rows - np.arange(L)[:, None]
    cand = np.unique(I[I >= 0])
    if len(cand) * L <= 1 << 22:
        p, s = seq_match.match_one(index, query, recon, tid, L, k_probe, n_pred=n_pred, fast_scores=True, table=table)
        return p, s, len(cand)
    scores = _scores_banded(q, recon, cand, L)
    order = np.argsort(-scores, kind="stable")[:n_pred]
    return cand[order], scores[order], len(cand)


def _assert_same_outside_ties(p, s, p_ref, s_ref, q, recon, L, tol=1e-6):
    from oracle import seq_match
    n = len(p_ref)
    assert (p[n:] == -1).all()
    np.testing.assert_allclose(s[:n], s_ref, rtol=0, atol=1e-5)
    for r in np.nonzero(p[:n] != p_ref)[0]:          # a different id only where two candidates score the same
        mine = seq_match.seq_scores_fast(np.asarray(q), recon, np.array([p[r]]), L)[0]
        assert abs(mine - s_ref[r]) <= tol, (r, p[r], p_ref[r], mine, s_ref[r])


# 2. long clips against the oracle: more than 1,024 and more than 65,536 candidates
def test_long_clips_against_the_oracle():
    from nafp_b200 import synth
    from nafp_b200.eval.utils.get_index import Index
    from oracle.flat_index import FlatL2
    dummy, db, query = synth.synth_search_set(100000, 5900, seed=9)
    recon = np.concatenate([dummy, db])
    g = Index(0, 128)
    g.add(recon)
    o = FlatL2(128)
    o.add(recon)
    cases = [(33, 20, 100), (33, 128, 700), (100, 20, 1500), (100, 128, 40), (600, 20, 2000), (600, 128, 5000),
             (4096, 20, 0), (4096, 128, 1700)]
    n_cands = []
    for k in (20, 128):
        sel = [i for i, (_, kk, _) in enumerate(cases) if kk == k]
        rows, off = _clips(query, [(cases[i][2], cases[i][0]) for i in sel])
        pred, sc = g.clip_match(rows, off, k_probe=k, n_top=10)
        for j, i in enumerate(sel):
            L, _, tid = cases[i]
            p_ref, s_ref, n_c = _oracle_match(o, query, recon, tid, L, k)
            n_cands.append(n_c)
            print(f"L={L} k={k}: {n_c} candidates")
            _assert_same_outside_ties(pred[j], sc[j], p_ref, s_ref, query[tid:tid + L], recon, L)
    assert max(n_cands) > 65536 and sorted(n_cands)[-3] > 1024


# 3. edge cases
def test_c_abi_refuses_bad_arguments(small_db):
    from nafp_b200._lib import lib, ptr
    g, _, _, query = small_db
    q = np.ascontiguousarray(query[:8])
    pid = np.zeros(8 * 101, np.int64)
    psc = np.zeros(8 * 101, np.float32)

    def call(off, k=20, n_top=10, n_rows=8):
        off = np.asarray(off, np.int64)
        return lib.nafp_clip_match(g.h, ptr(q), n_rows, ptr(off), len(off) - 1, k, n_top, ptr(pid), ptr(psc))

    assert call([0, 4, 8]) == 0
    assert call([0, 5, 3, 8]) == NAFP_ERR_INVALID          # unsorted
    assert call([0, 0, 8]) == NAFP_ERR_INVALID             # L = 0
    big = np.ascontiguousarray(np.resize(query, (4097, 128)))
    off = np.array([0, 4097], np.int64)
    assert lib.nafp_clip_match(g.h, ptr(big), 4097, ptr(off), 1, 20, 10, ptr(pid), ptr(psc)) == NAFP_ERR_INVALID
    assert call([0, 8], k=129) == NAFP_ERR_INVALID
    assert call([0, 8], k=0) == NAFP_ERR_INVALID
    assert call([0, 8], n_top=101) == NAFP_ERR_INVALID
    assert call([0, 8], n_top=0) == NAFP_ERR_INVALID
    assert call([0, 8], n_rows=9) == NAFP_ERR_INVALID      # offsets must end at n_rows


def test_dev_entry_point_checks_the_offsets_on_the_device(small_db):
    """nafp_clip_match_dev cannot read its offsets on the host: with offsets out of range or out of order every clip
    reports -1 / -inf (and no query row outside the buffer is read); with good offsets it is nafp_clip_match."""
    import ctypes
    from nafp_b200._lib import check, lib
    g, _, _, query = small_db
    q = np.ascontiguousarray(query[:100])
    ctx = g.ctx
    q_dev = ctx.malloc(q.nbytes)
    off_dev = ctx.malloc(8 * 4)
    pid_dev = ctx.malloc(3 * 10 * 8)
    psc_dev = ctx.malloc(3 * 10 * 4)
    try:
        ctx.h2d(q_dev, q)

        def run(off):
            off = np.asarray(off, np.int64)
            ctx.h2d(off_dev, off)
            check(lib.nafp_clip_match_dev(g.h, q_dev, 100, off_dev, len(off) - 1, 20, 10, pid_dev, psc_dev))
            pid = np.empty((len(off) - 1, 10), np.int64)
            psc = np.empty((len(off) - 1, 10), np.float32)
            ctx.d2h(pid, pid_dev)
            ctx.d2h(psc, psc_dev)
            ctx.sync()
            return pid, psc

        good = [0, 30, 70, 100]
        p_ref, s_ref = g.clip_match(q, np.array(good), k_probe=20, n_top=10)
        pid, psc = run(good)
        assert (p_ref[:, 0] >= 0).all()
        assert np.array_equal(pid, p_ref) and np.array_equal(psc.view(np.uint32), s_ref.view(np.uint32))
        for bad in ([0, 4096], [0, 30, 4126], [0, 50, 30, 100], [-10, 30, 70], [0, 30, 30, 100], [0, 4097]):
            pid, psc = run(bad)
            assert (pid == -1).all() and np.isneginf(psc).all(), bad
        pid, _ = run(good)                                  # and the next good call is unaffected
        assert np.array_equal(pid, p_ref)
    finally:
        for p in (q_dev, off_dev, pid_dev, psc_dev):
            ctx.free(p)


def test_clips_past_the_end_of_the_database():
    """Candidates whose sequence runs past the last row are scored over the rows that exist (the clamp)."""
    from nafp_b200 import synth
    from nafp_b200.eval.utils.get_index import Index
    from oracle.flat_index import FlatL2
    dummy, db, query = synth.synth_search_set(3000, 590, seed=3)
    recon = np.concatenate([dummy, db])
    g, o = Index(0, 128), FlatL2(128)
    g.add(recon)
    o.add(recon)
    n_q = len(query)
    cases = [(n_q - 10, 40), (n_q - 3, 3), (n_q - 60, 200)]     # clips cut from the end of the query set, so
    qx = np.concatenate([query, synth.synth_fp_db(300, seed=77)])  # their true match runs past the database end
    rows, off = _clips(qx, [(t, L) for t, L in cases])
    pred, sc = g.clip_match(rows, off, k_probe=20, n_top=10)
    for j, (t, L) in enumerate(cases):
        p_ref, s_ref, _ = _oracle_match(o, qx, recon, t, L, 20)
        _assert_same_outside_ties(pred[j], sc[j], p_ref, s_ref, qx[t:t + L], recon, L)


def test_duplicated_rows_tie_to_the_lower_id():
    from nafp_b200 import synth
    from nafp_b200.eval.utils.get_index import Index
    a = synth.synth_fp_db(400, seed=21)
    g = Index(0, 128)
    g.add(a)
    g.add(a)                                             # rows i and i + 400 are equal
    rows, off = _clips(a, [(100, 12), (7, 1)])
    pred, sc = g.clip_match(rows, off, k_probe=4, n_top=10)
    for j, t in enumerate((100, 7)):
        assert pred[j, 0] == t and pred[j, 1] == t + 400
        assert sc[j, 0] == sc[j, 1]


def test_k_probe_larger_than_the_database_and_a_single_row():
    from nafp_b200 import synth
    from nafp_b200.eval.utils.get_index import Index
    from oracle.flat_index import FlatL2
    x = synth.synth_fp_db(5, seed=31)[:5]
    q = np.concatenate([x, synth.synth_fp_db(10, seed=32)[:10]])
    g, o = Index(0, 128), FlatL2(128)
    g.add(x)
    o.add(x)
    rows, off = _clips(q, [(0, 5), (2, 7), (5, 10)])
    pred, sc = g.clip_match(rows, off, k_probe=20, n_top=10)
    for j, (t, L) in enumerate([(0, 5), (2, 7), (5, 10)]):
        p_ref, s_ref, _ = _oracle_match(o, q, x, t, L, 20)
        assert len(p_ref) <= 5
        _assert_same_outside_ties(pred[j], sc[j], p_ref, s_ref, q[t:t + L], x, L)
        assert (pred[j, len(p_ref):] == -1).all() and np.isneginf(sc[j, len(p_ref):]).all()
    one = Index(0, 128)
    one.add(x[:1])
    pred, sc = one.clip_match(q[:3], np.array([0, 3]), k_probe=5, n_top=4)
    assert pred.tolist() == [[0, -1, -1, -1]]
    assert sc[0, 0] == np.float32(np.dot(q[0], x[0])) or abs(sc[0, 0] - np.dot(q[0], x[0])) < 1e-6


# 4. IVF-PQ: the matcher fed with the index's own search table is match_one fed with the same table
def test_ivfpq_against_match_one_on_the_gpu_table():
    from nafp_b200 import synth
    from nafp_b200.eval.utils.get_index import IVFPQ, Index
    dummy, db, query = synth.synth_search_set(20000, 2950, seed=6)
    recon = np.concatenate([dummy, db])
    gi = Index(IVFPQ, 128, nlist=64, pq_m=64, pq_nbits=8)
    gi.train(dummy[:8000], seed=1234)
    gi.add(recon)
    gi.nprobe = 16
    cases = [(10, 19), (500, 100), (2000, 600), (37, 1)]
    rows, off = _clips(query, cases)
    pred, sc = gi.clip_match(rows, off, k_probe=20, n_top=10)
    for j, (t, L) in enumerate(cases):
        _, I = gi.search(query[t:t + L], 20)
        p_ref, s_ref, _ = _oracle_match(gi, query, recon, t, L, 20, table_rows=I)
        _assert_same_outside_ties(pred[j], sc[j], p_ref, s_ref, query[t:t + L], recon, L)


# 5. end to end: `run.py identify` on WAV excerpts of the database
@pytest.fixture(scope="module")
def corpus(tmp_path_factory):
    from nafp_b200 import synth
    from nafp_b200.model.generate import generate_fingerprint
    root = tmp_path_factory.mktemp("corpus")
    src = root / "music"
    for sub in ("test-dummy-db-100k-full/a", "test-query-db-500-30s/query/a", "test-query-db-500-30s/db/a"):
        os.makedirs(src / sub)
    for i in range(12):                                    # dummy: 12 x 12 s
        synth.write_wav(str(src / "test-dummy-db-100k-full/a" / f"d{i:03d}.wav"), synth.synth_track(100 + i, 96000))
    tracks = []
    # db / query: 5 x 30 s.  No query comes from the last db track: its final rows end the database, where a candidate
    # is scored over the one or two rows that exist, and segments of one synthetic track resemble each other
    for i in range(5):
        x = synth.synth_track(200 + i, 240000)
        tracks.append(x)
        synth.write_wav(str(src / "test-query-db-500-30s/db/a" / f"s{i:03d}.wav"), x)
        synth.write_wav(str(src / "test-query-db-500-30s/query/a" / f"s{i:03d}.wav"), synth.add_noise_snr(x, 5.0, i))
    cfg = yaml.safe_load(open(os.path.join(ROOT, "config", "default.yaml")))
    cfg['DIR']['SOURCE_ROOT_DIR'] = str(src) + "/"
    cfg['DIR']['LOG_ROOT_DIR'] = str(root / "logs") + "/"
    cfg['DIR']['OUTPUT_ROOT_DIR'] = str(root / "logs" / "emb") + "/"
    cfg['DATA_SEL']['TEST_DUMMY_DB'] = '100k_full_icassp'
    cfg['BSZ']['TS_BATCH_SZ'] = 25
    generate_fingerprint(cfg, 'random-init:7', None, None, None, False)
    # queries: excerpts of db tracks starting on the 0.5 s grid, 5 s or 20 s long, noise at 5 dB SNR
    qdir = root / "queries"
    os.makedirs(qdir)
    expect = {}
    for i, (start, dur) in enumerate([(3.0, 5), (7.5, 20), (0.5, 5), (9.0, 20)]):
        x = tracks[i][int(start * 8000):int((start + dur) * 8000)]
        name = f"q{i}.wav"
        synth.write_wav(str(qdir / name), synth.add_noise_snr(x, 5.0, 50 + i))
        expect[name] = (f"s{i:03d}.wav", start)
    # two tracks in one recording: 10 s of s000 from 2 s, then 10 s of s002 from 15 s
    mix = np.concatenate([tracks[0][2 * 8000:12 * 8000], tracks[2][15 * 8000:25 * 8000]])
    mdir = root / "mixed"
    os.makedirs(mdir)
    synth.write_wav(str(mdir / "mix.wav"), synth.add_noise_snr(mix, 5.0, 60))
    return cfg, root, qdir, mdir, expect


def _cfg_file(cfg, root):
    path = str(root / "cfg.yaml")
    with open(path, "w") as f:
        yaml.safe_dump(cfg, f)
    return path


@pytest.mark.parametrize("index_type", ["l2", "ivfpq"])
def test_identify_excerpts(corpus, index_type):
    from click.testing import CliRunner
    from nafp_b200.run import cli
    cfg, root, qdir, _, expect = corpus
    out = str(root / f"matches_{index_type}.json")
    r = CliRunner().invoke(cli, ["identify", "random-init:7", "-c", _cfg_file(cfg, root), "--query", str(qdir),
                                 "-i", index_type, "-o", out])
    assert r.exit_code == 0, (r.output[-3000:], r.exception)
    res = json.load(open(out))
    assert len(res) == len(expect)
    for clip in res:
        name = os.path.basename(clip["query"])
        top = clip["matches"][0]
        print(name, expect[name], os.path.basename(top["file"]), top["offset_s"], top["score"])
        assert clip["start_s"] == 0.0
        assert (os.path.basename(top["file"]), top["offset_s"]) == expect[name], clip["matches"][:3]
        assert top["key"] == "db"


def test_query_fingerprints_equal_generate_source(corpus, tmp_path):
    from nafp_b200.eval.identify import fingerprint_sequence, query_sequence
    from nafp_b200.model.fp import build_fp
    from nafp_b200.model.generate import generate_fingerprint, load_checkpoint
    cfg, root, qdir, _, _ = corpus
    generate_fingerprint(cfg, 'random-init:7', None, str(qdir), str(tmp_path), True)
    emb_dir = str(tmp_path) + '/random-init:7/0/'
    shape = np.load(emb_dir + 'custom_source_shape.npy')
    ref = np.fromfile(emb_dir + 'custom_source.mm', np.float32).reshape(tuple(shape))
    _, m_fp = build_fp(cfg)
    load_checkpoint(cfg['DIR']['LOG_ROOT_DIR'] + 'checkpoint/', 'random-init:7', None, m_fp)
    got = fingerprint_sequence(m_fp, query_sequence(cfg, str(qdir)))
    assert got.shape == ref.shape and np.array_equal(got.view(np.uint32), ref.view(np.uint32))


def test_identify_window_finds_both_tracks(corpus):
    from nafp_b200.eval.identify import run_identify
    cfg, root, _, mdir, _ = corpus
    res = run_identify(cfg, 'random-init:7', None, str(mdir / "mix.wav"), index_type='l2', window=10.0)
    assert [c["start_s"] for c in res] == [0.0, 10.0]
    got = [(os.path.basename(c["matches"][0]["file"]), c["matches"][0]["offset_s"]) for c in res]
    assert got == [("s000.wav", 2.0), ("s002.wav", 15.0)], [c["matches"][:3] for c in res]
