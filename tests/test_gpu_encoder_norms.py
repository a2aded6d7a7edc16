"""GPU parity of the encoder for MODEL.BN 'layer_norm1d' and 'batch_norm' (moving statistics calibrated on the
reference's own activations, perturbed by 10 %) against the fp64 reference of
tests/util_norms.py (gates as for 'layer_norm2d': cosine >= 0.9999, max abs error <= 1e-3), the fused entry points,
multi-pass runs, the melspec_maxnorm branch, weight reloads on one context and `run.py generate`."""
import glob
import os
import subprocess
import sys

import numpy as np
import pytest
import yaml

from util_norms import fingerprinter, weights

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ["layer_norm1d", "batch_norm"]


def _audio(n, seed=1, hop=700):
    from nafp_b200 import synth
    tr = synth.synth_track(seed).astype(np.float32) / 32768.0
    return np.stack([tr[i * hop:i * hop + 8000] for i in range(n)]).astype(np.float32)


def _mel(x, group_size, segment_norm=False):
    from oracle import melspec
    return melspec.melspec_layer(x[:, None, :], group_size=group_size, segment_norm=segment_norm, dtype=np.float32)


def _gate(emb, ref):
    cos, err = (emb * ref).sum(1).min(), np.abs(emb - ref).max()
    assert cos >= 0.9999 and err <= 1e-3, (cos, err)
    return cos, err


_CAL = {}


def _weights(norm, seed):
    if (norm, seed) not in _CAL:
        _CAL[(norm, seed)] = weights(norm, seed, _mel(_audio(16, seed=50 + seed, hop=3000), 16))
    return _CAL[(norm, seed)]


@pytest.mark.parametrize("seed", [7, 8, 9])
@pytest.mark.parametrize("norm", NEW)
def test_encoder_matches_reference_layer_by_layer(ctx, norm, seed):
    from nafp_b200.model.fp import FingerPrinter
    w = _weights(norm, seed)
    m_fp = FingerPrinter(ctx, norm=norm).load(w)
    mel = _mel(_audio(9, seed=seed), 9)
    emb = m_fp(mel)
    ref, acts = fingerprinter(mel, w, norm, return_all=True)
    for l in range(16):
        a = m_fp.activation(l, 9)
        assert a.shape == acts[l].shape
        err = np.abs(a - acts[l])
        assert err.mean() < 3e-3 and err.max() < 3e-2, (l, err.mean(), err.max())
    cos, err = _gate(emb, ref)
    print(f"{norm} seed {seed}: min cosine {cos:.7f}, max abs err {err:.3e}")
    assert np.allclose(np.linalg.norm(emb, axis=1), 1.0, atol=1e-5)


@pytest.mark.parametrize("norm", NEW)
def test_fused_entry_points(ctx, norm, tmp_path):
    from nafp_b200 import synth
    from nafp_b200.model import dataset
    from nafp_b200.model.fp import FingerPrinter, Melspec
    w = _weights(norm, 7)
    m_fp = FingerPrinter(ctx, norm=norm).load(w)
    pcm = np.stack([synth.synth_track(5)[i * 4000:i * 4000 + 8000] for i in range(13)])
    x = (pcm / 2 ** 15).astype(np.float32)
    ref = fingerprinter(_mel(x, 5), w, norm)
    ef, ep = m_fp.fingerprint(x[:, None, :], group_size=5), m_fp.fingerprint(pcm, group_size=5)
    _gate(ef, ref)
    np.testing.assert_array_equal(ef, ep)
    _gate(m_fp(Melspec(ctx)(x[:, None, :], group_size=5)), ef)      # encoder_forward on the standalone log-mel
    paths = []
    for i, n in enumerate([30000, 8000, 5000, 44123]):
        p = str(tmp_path / f"t{i}.wav")
        synth.write_wav(p, synth.synth_track(i, n_samples=n))
        paths.append(p)
    seq = dataset.SegmentSequence(paths, bsz=7)
    rows = m_fp.fingerprint(seq.get_pcm_range(0, len(seq)), group_size=7)
    np.testing.assert_array_equal(m_fp.fingerprint_tracks(*seq.get_track_block(0, len(seq)), group_size=7), rows)


@pytest.mark.parametrize("norm", NEW)
def test_two_encoder_passes_equal_single_calls(ctx, norm):
    from nafp_b200.model.fp import FingerPrinter
    m_fp = FingerPrinter(ctx, norm=norm).load(_weights(norm, 8))
    x = _audio(125, seed=3, hop=1000)
    big = np.tile(x, (34, 1))[:4200]               # two encoder passes (4,000 + 200 segments)
    emb = m_fp.fingerprint(big, group_size=125)
    one = m_fp.fingerprint(x, group_size=125)
    for g in range(33):
        np.testing.assert_array_equal(emb[g * 125:(g + 1) * 125], one)
    np.testing.assert_array_equal(emb[4125:], one[:75])


@pytest.mark.parametrize("norm", NEW)
def test_melspec_maxnorm_branch(ctx, norm):
    from nafp_b200.model.fp import FingerPrinter
    w = _weights(norm, 9)
    x = _audio(23, seed=4)
    m_fp = FingerPrinter(ctx, segment_norm=True, norm=norm).load(w)
    _gate(m_fp.fingerprint(x, group_size=10), fingerprinter(_mel(x, 10, segment_norm=True), w, norm))


@pytest.mark.parametrize("norm", NEW)
def test_layer_norm2d_after_another_norm_is_unchanged(ctx, norm):
    from nafp_b200._lib import Context
    from nafp_b200.model import weights as W
    from nafp_b200.model.fp import FingerPrinter
    x = _audio(40, seed=6)
    w2 = W.init_weights(7, randomize_affine=True)
    FingerPrinter(ctx, norm=norm).load(_weights(norm, 7)).fingerprint(x, group_size=10)
    got = FingerPrinter(ctx).load(w2).fingerprint(x, group_size=10)
    fresh = Context(0)
    np.testing.assert_array_equal(got, FingerPrinter(fresh).load(w2).fingerprint(x, group_size=10))


@pytest.mark.parametrize("norm", NEW)
def test_run_generate_with_model_bn(norm, tmp_path):
    from nafp_b200 import synth
    from nafp_b200._lib import Context
    from nafp_b200.model import dataset, weights as W
    from nafp_b200.model.fp import FingerPrinter
    src = tmp_path / "music"
    for sub in ("test-dummy-db-100k-full/a", "test-query-db-500-30s/query/a", "test-query-db-500-30s/db/a"):
        os.makedirs(src / sub)
    for i in range(3):
        synth.write_wav(str(src / "test-dummy-db-100k-full/a" / f"d{i:03d}.wav"), synth.synth_track(100 + i, 48000))
    for i in range(2):
        x = synth.synth_track(200 + i, 40000)
        synth.write_wav(str(src / "test-query-db-500-30s/db/a" / f"s{i:03d}.wav"), x)
        synth.write_wav(str(src / "test-query-db-500-30s/query/a" / f"s{i:03d}.wav"), synth.add_noise_snr(x, 5.0, i))
    cfg = yaml.safe_load(open(os.path.join(ROOT, "config", "default.yaml")))
    cfg['DIR']['SOURCE_ROOT_DIR'] = str(src) + "/"
    cfg['DIR']['LOG_ROOT_DIR'] = str(tmp_path / "logs") + "/"
    cfg['DATA_SEL']['TEST_DUMMY_DB'] = '100k_full_icassp'
    cfg['BSZ']['TS_BATCH_SZ'] = 25
    cfg['MODEL']['BN'] = norm
    cfg_path = str(tmp_path / "cfg.yaml")
    with open(cfg_path, "w") as f:
        yaml.safe_dump(cfg, f)
    out = str(tmp_path / "out") + "/"
    r = subprocess.run([sys.executable, "-m", "nafp_b200.run", "generate", "random-init:7", "-c", cfg_path, "-o", out],
                       env=dict(os.environ, PYTHONPATH=ROOT), cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout + r.stderr)[-2000:]
    m_fp = FingerPrinter(Context.get(0), norm=norm).load(W.init_weights(7, norm=norm))
    for key, sub in (("dummy_db", "test-dummy-db-100k-full/"), ("query", "test-query-db-500-30s/query/"),
                     ("db", "test-query-db-500-30s/db/")):
        shape = tuple(np.load(f"{out}random-init:7/0/{key}_shape.npy"))
        got = np.fromfile(f"{out}random-init:7/0/{key}.mm", np.float32).reshape(shape)
        files = sorted(glob.glob(str(src / sub) + '/**/*.wav', recursive=True))
        seq = dataset.SegmentSequence(files, 25)
        want = m_fp.fingerprint_tracks(*seq.get_track_block(0, len(seq)), group_size=25)
        np.testing.assert_array_equal(got, want)
