"""GPU: the polyphase resampler (nafp_resample_pcm16_dev) against the fp64 oracle, the argument checks of both
resampling entry points, the fused any-rate fingerprint path against resample-then-fingerprint, and `run.py identify`
on recordings at 44.1 kHz stereo and 48 kHz mono."""
import json
import os

import numpy as np
import pytest
import yaml

from oracle import resample as R

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RATES = [4000, 11025, 16000, 22050, 32000, 44100, 48000, 96000, 192000]
NAFP_ERR_INVALID, NAFP_ERR_UNSUPPORTED = -1, -4


@pytest.fixture(scope="module")
def ctx():
    from nafp_b200._lib import Context
    return Context.get(0)


def _device_resample(ctx, x, fs_in, m0=0, n_out=None, frame0=0, n_frames=None, fs_out=8000):
    """nafp_resample_pcm16_dev over frames frame0 .. frame0+n_frames-1 of x ((N,) or (N, C) int16)."""
    from nafp_b200._lib import check, lib
    x = np.ascontiguousarray(x, np.int16)
    ch = 1 if x.ndim == 1 else x.shape[1]
    n = len(x)
    n_frames = n - frame0 if n_frames is None else n_frames
    n_out = R.out_length(n, fs_in, fs_out) - m0 if n_out is None else n_out
    win = np.ascontiguousarray(x[frame0:frame0 + n_frames])
    out = np.empty(n_out, np.int16)
    xd, od = ctx.malloc(max(win.nbytes, 2)), ctx.malloc(max(out.nbytes, 2))
    try:
        ctx.h2d(xd, win)
        check(lib.nafp_resample_pcm16_dev(ctx.h, xd, frame0, n_frames, ch, fs_in, fs_out, m0, n_out, od))
        ctx.d2h(out, od)
        ctx.sync()
    finally:
        ctx.free(xd)
        ctx.free(od)
    return out


def _assert_matches_oracle(got, x, fs_in, label):
    want, exact = R.resample_pcm16(x, fs_in, 8000)
    assert got.shape == want.shape, label
    diff = got.astype(np.int32) - want
    near_half = np.abs(np.abs(exact - np.floor(exact)) - 0.5) < 1e-7
    bad = (diff != 0) & ~(near_half & (np.abs(diff) == 1))
    assert not bad.any(), (label, np.flatnonzero(bad)[:10], got[bad][:10], want[bad][:10])
    n_ties = int((diff != 0).sum())
    print(f"{label}: {len(got)} samples, {n_ties} half-integer ties off by one")
    return want


def _signals(fs, ch, seed):
    from nafp_b200 import synth
    rng = np.random.default_rng(seed)
    n = fs + 37                                               # ~1 s
    noise = rng.integers(-20000, 20000, (n, ch)).astype(np.int16)
    music = R.resample_pcm16(synth.synth_track(seed, 8000 + 8000 // 4), 8000, fs)[0][:n]
    music = np.stack([music // (c + 1) for c in range(ch)], axis=1).astype(np.int16)
    period = max(2, fs // 441)
    square = np.where((np.arange(n) // (period // 2 or 1)) % 2 == 0, 32767, -32768).astype(np.int16)
    square = np.repeat(square[:, None], ch, axis=1)
    return {"noise": noise, "music": music, "square": square}


@pytest.mark.parametrize("fs_in", RATES)
@pytest.mark.parametrize("ch", [1, 2, 6])
def test_device_resampler_equals_the_oracle(ctx, fs_in, ch):
    for name, x in _signals(fs_in, ch, fs_in + ch).items():
        xx = x[:, 0] if ch == 1 else x
        got = _device_resample(ctx, xx, fs_in)
        whole = _assert_matches_oracle(got, xx, fs_in, f"{fs_in} Hz x{ch} {name}")
        if name == "square":
            assert whole.max() == 32767 and whole.min() == -32768          # the filter overshoots: saturation
        # a sub-range from the window the header comment gives equals the matching slice of the whole track
        up, down, hl = R.ratio(fs_in, 8000)
        m0, k = len(got) // 3, len(got) // 4
        lo = max(0, -(-(m0 * down - hl) // up))
        hi = min(len(xx) - 1, ((m0 + k - 1) * down + hl) // up)
        part = _device_resample(ctx, xx, fs_in, m0, k, lo, hi - lo + 1)
        np.testing.assert_array_equal(part, got[m0:m0 + k])


def test_equal_rates_copy_and_downmix(ctx):
    rng = np.random.default_rng(1)
    x = rng.integers(-32768, 32768, (50000, 2)).astype(np.int16)
    np.testing.assert_array_equal(_device_resample(ctx, x[:, 0], 8000), x[:, 0])
    np.testing.assert_array_equal(_device_resample(ctx, x, 8000), R.resample_pcm16(x, 8000, 8000)[0])


def test_argument_checks_before_device_work(ctx):
    from nafp_b200._lib import lib
    from nafp_b200.model.fp import FingerPrinter
    from nafp_b200.model.weights import init_weights
    buf = ctx.malloc(1 << 16)
    try:
        def dev(frame0=0, n_frames=100, ch=2, fs_in=44100, fs_out=8000, m0=0, n_out=10):
            return lib.nafp_resample_pcm16_dev(ctx.h, buf, frame0, n_frames, ch, fs_in, fs_out, m0, n_out, buf)
        assert dev() == 0
        assert dev(ch=0) == NAFP_ERR_INVALID
        assert dev(ch=9) == NAFP_ERR_UNSUPPORTED
        assert dev(fs_in=0) == NAFP_ERR_INVALID and dev(fs_out=-8000) == NAFP_ERR_INVALID
        assert dev(fs_in=44056) == NAFP_ERR_UNSUPPORTED
        assert "needs up 1000 / down 5507" in lib.nafp_last_error().decode()
        for kw in ("frame0", "n_frames", "m0", "n_out"):
            assert dev(**{kw: -1}) == NAFP_ERR_INVALID, kw
        ctx.sync()
    finally:
        ctx.free(buf)

    m_fp = FingerPrinter(ctx).load(init_weights(7))
    pcm = np.zeros(44100 * 2, np.int16)

    def src(runs, off=(0,), valid=(8000,), n_pcm=len(pcm)):
        runs = np.ascontiguousarray(runs, np.int64).reshape(-1, 7)
        off, valid = np.asarray(off, np.int64), np.asarray(valid, np.int32)
        emb = np.empty((len(off), 128), np.float32)
        return lib.nafp_fingerprint_pcm16_sources_host(ctx.h, pcm.ctypes.data, n_pcm, runs.ctypes.data, len(runs),
                                                       off.ctypes.data, valid.ctypes.data, len(off), 1, emb.ctypes.data)
    good = [0, 0, 44100, 2, 44100, 0, 8000]
    assert src(good) == 0
    for i, v, status in [(3, 0, NAFP_ERR_INVALID), (3, 9, NAFP_ERR_UNSUPPORTED), (4, 0, NAFP_ERR_INVALID),
                         (4, -44100, NAFP_ERR_INVALID), (4, 44056, NAFP_ERR_UNSUPPORTED), (0, -1, NAFP_ERR_INVALID),
                         (1, -1, NAFP_ERR_INVALID), (2, -1, NAFP_ERR_INVALID), (5, -1, NAFP_ERR_INVALID),
                         (6, -1, NAFP_ERR_INVALID), (0, 2, NAFP_ERR_INVALID)]:            # last: reads past n_pcm
        bad = list(good)
        bad[i] = v
        assert src(bad) == status, (i, v, lib.nafp_last_error())
    assert src(good, off=(1,)) == NAFP_ERR_INVALID                      # a segment past the resampled track
    assert src(good, valid=(8001,)) == NAFP_ERR_INVALID
    assert src([good, good], off=(8000,)) == 0
    assert src(good, n_pcm=len(pcm) - 1) == NAFP_ERR_INVALID
    ctx.sync()
    del m_fp


def _cfg(root, bsz):
    cfg = yaml.safe_load(open(os.path.join(ROOT, "config", "default.yaml")))
    cfg['DIR']['LOG_ROOT_DIR'] = str(root / "logs") + "/"
    cfg['DIR']['OUTPUT_ROOT_DIR'] = str(root / "logs" / "emb") + "/"
    cfg['BSZ']['TS_BATCH_SZ'] = bsz
    return cfg


def _read_wav(path):
    import wave
    with wave.open(path) as w:
        x = np.frombuffer(w.readframes(w.getnframes()), np.int16).reshape(-1, w.getnchannels())
        return x, w.getframerate()


def test_fused_sources_path_equals_resample_then_fingerprint(ctx, tmp_path):
    from nafp_b200 import synth
    from nafp_b200.model.generate import generate_fingerprint
    src, conv = tmp_path / "src", tmp_path / "conv"
    os.makedirs(src)
    os.makedirs(conv)
    rng = np.random.default_rng(9)
    for i in range(3):
        x = R.resample_pcm16(synth.synth_track(30 + i, 8000 * (9 + 4 * i)), 8000, 44100)[0]
        st = np.stack([x, (x.astype(np.int32) * 3 // 5).astype(np.int16)], axis=1)
        synth.write_wav(str(src / f"a{i}.wav"), st, 44100)
        y = R.resample_pcm16(synth.synth_track(40 + i, 8000 * (7 + 3 * i)), 8000, 22050)[0]
        synth.write_wav(str(src / f"b{i}.wav"), y, 22050)
        synth.write_wav(str(src / f"c{i}.wav"), synth.synth_track(50 + i, 8000 * (5 + i) + int(rng.integers(4000))))
    synth.write_wav(str(src / "d.wav"), rng.integers(-3000, 3000, (5000, 2)).astype(np.int16), 44100)   # < 1 segment
    for p in sorted(os.listdir(src)):
        x, fs = _read_wav(str(src / p))
        synth.write_wav(str(conv / p), _device_resample(ctx, x if x.shape[1] > 1 else x[:, 0], fs))
    cfg = _cfg(tmp_path, 25)
    out = {}
    for name, d in (("src", src), ("conv", conv)):
        generate_fingerprint(cfg, 'random-init:7', None, str(d), str(tmp_path / f"out_{name}"), True, batches_per_call=2)
        emb_dir = str(tmp_path / f"out_{name}") + '/random-init:7/0/'
        out[name] = open(emb_dir + 'custom_source.mm', 'rb').read()
        assert tuple(np.load(emb_dir + 'custom_source_shape.npy'))[1] == 128
    assert len(out["src"]) == len(out["conv"]) and out["src"] == out["conv"]


# end to end: `run.py identify` on recordings at 44.1 kHz stereo and 48 kHz mono against an 8 kHz database
@pytest.fixture(scope="module")
def corpus(tmp_path_factory):
    from nafp_b200 import synth
    from nafp_b200.model.generate import generate_fingerprint
    root = tmp_path_factory.mktemp("rs_corpus")
    src = root / "music"
    for sub in ("test-dummy-db-100k-full/a", "test-query-db-500-30s/query/a", "test-query-db-500-30s/db/a"):
        os.makedirs(src / sub)
    for i in range(12):
        synth.write_wav(str(src / "test-dummy-db-100k-full/a" / f"d{i:03d}.wav"), synth.synth_track(100 + i, 96000))
    tracks = []
    for i in range(5):
        x = synth.synth_track(200 + i, 240000)
        tracks.append(x)
        synth.write_wav(str(src / "test-query-db-500-30s/db/a" / f"s{i:03d}.wav"), x)
        synth.write_wav(str(src / "test-query-db-500-30s/query/a" / f"s{i:03d}.wav"), synth.add_noise_snr(x, 5.0, i))
    cfg = _cfg(root, 25)
    cfg['DIR']['SOURCE_ROOT_DIR'] = str(src) + "/"
    cfg['DATA_SEL']['TEST_DUMMY_DB'] = '100k_full_icassp'
    generate_fingerprint(cfg, 'random-init:7', None, None, None, False)
    qdir = root / "queries"
    os.makedirs(qdir)
    expect = {}
    for i, (start, dur, fs, gains) in enumerate([(3.0, 5, 44100, (0.9, 0.4)), (7.5, 20, 48000, None),
                                                 (0.5, 5, 48000, None), (9.0, 20, 44100, (0.3, 1.0))]):
        x = synth.add_noise_snr(tracks[i][int(start * 8000):int((start + dur) * 8000)], 5.0, 50 + i)
        y = R.resample_pcm16(x, 8000, fs)[0]
        if gains:
            y = np.stack([np.round(y * g).astype(np.int16) for g in gains], axis=1)
        name = f"q{i}.wav"
        synth.write_wav(str(qdir / name), y, fs)
        expect[name] = (f"s{i:03d}.wav", start)
    return cfg, root, qdir, expect


@pytest.mark.parametrize("index_type", ["l2", "ivfpq"])
def test_identify_recordings_at_other_rates(corpus, index_type):
    from click.testing import CliRunner
    from nafp_b200.run import cli
    cfg, root, qdir, expect = corpus
    path = str(root / "cfg.yaml")
    with open(path, "w") as f:
        yaml.safe_dump(cfg, f)
    out = str(root / f"matches_{index_type}.json")
    r = CliRunner().invoke(cli, ["identify", "random-init:7", "-c", path, "--query", str(qdir), "-i", index_type,
                                 "-o", out])
    assert r.exit_code == 0, (r.output[-3000:], r.exception)
    assert "Resampling to 8000 Hz mono on the GPU" in r.output and "44100 Hz 2 ch" in r.output
    res = json.load(open(out))
    assert len(res) == len(expect)
    for clip in res:
        name = os.path.basename(clip["query"])
        top = clip["matches"][0]
        print(name, expect[name], os.path.basename(top["file"]), top["offset_s"], top["score"])
        assert (os.path.basename(top["file"]), top["offset_s"]) == expect[name], clip["matches"][:3]
        assert top["key"] == "db"
