"""Seeded synthetic inputs of the shapes BASELINE.json names (datasets are unavailable offline).

* ``synth_track``       -- 30 s of 8 kHz int16 "music-like" audio (SURVEY §8 d, config 1).
* ``synth_fp_db``       -- unit-norm 128-d fingerprint rows with AR(1) correlation inside 59-row
                           tracks (what 0.5 s-hop segments of one song look like), config 2/4.
* ``synth_fp_queries``  -- noisy copies of db rows with a per-track noise level, so that
                           length-1 top-1 hit rate lands mid-range and saturates by length 19.
* ``write_wav``         -- 16-bit PCM writer for the generate-CLI tests.
Everything is a pure function of its seed so any rank can regenerate its own slice.
"""
from __future__ import annotations

import wave

import numpy as np

SEGS_PER_TRACK = 59     # 30 s at 1 s window / 0.5 s hop (reference audio_utils.py:173-177)


def synth_track(seed, n_samples=240000, fs=8000):
    rng = np.random.default_rng(1000 + int(seed))
    t = np.arange(n_samples, dtype=np.float64) / fs
    n_tones = int(rng.integers(8, 17))
    x = np.zeros(n_samples)
    for _ in range(n_tones):
        f = rng.uniform(300.0, 3800.0)
        am_f = rng.uniform(0.2, 4.0)
        am = 0.6 + 0.4 * np.sin(2 * np.pi * am_f * t + rng.uniform(0, 2 * np.pi))
        x += rng.uniform(0.3, 1.0) * am * np.sin(2 * np.pi * f * t + rng.uniform(0, 2 * np.pi))
    x /= np.sqrt(np.mean(x * x))
    x += 0.1 * rng.standard_normal(n_samples)          # white noise at -20 dB
    x *= 0.5 / np.max(np.abs(x))
    return np.round(x * 32767.0).astype(np.int16)


def add_noise_snr(x_int16, snr_db, seed):
    rng = np.random.default_rng(int(seed))
    x = x_int16.astype(np.float64)
    p = np.mean(x * x)
    n = rng.standard_normal(x.shape) * np.sqrt(p / (10 ** (snr_db / 10.0)))
    return np.clip(np.round(x + n), -32768, 32767).astype(np.int16)


def write_wav(path, x_int16, fs=8000):
    """16-bit PCM WAV of x: (n,) mono or (n, channels) frames."""
    x_int16 = np.asarray(x_int16)
    with wave.open(path, "w") as w:
        w.setnchannels(1 if x_int16.ndim == 1 else x_int16.shape[1])
        w.setsampwidth(2)
        w.setframerate(fs)
        w.writeframes(np.asarray(x_int16, dtype="<i2").tobytes())


def _normalize(x):
    return (x / np.linalg.norm(x, axis=1, keepdims=True)).astype(np.float32)


def synth_fp_db(n_rows, seed=11, dim=128, rho=0.5, track_len=SEGS_PER_TRACK, start_track=0):
    """(n_rows, dim) float32 unit-norm.  Each block of 4096 tracks depends only on
    (seed, id of its first track), so shards aligned to 4096 tracks regenerate independently."""
    n_tracks = -(-n_rows // track_len)
    out = np.empty((n_tracks * track_len, dim), dtype=np.float32)
    blk = 4096
    for t0 in range(0, n_tracks, blk):
        nt = min(blk, n_tracks - t0)
        rng = np.random.default_rng([int(seed), int(start_track + t0)])
        eps = rng.standard_normal((nt, track_len, dim), dtype=np.float32)
        r = np.empty_like(eps)
        r[:, 0] = eps[:, 0]
        c = np.float32(np.sqrt(1.0 - rho * rho))
        for j in range(1, track_len):
            r[:, j] = np.float32(rho) * r[:, j - 1] + c * eps[:, j]
        out[t0 * track_len:(t0 + nt) * track_len] = _normalize(r.reshape(-1, dim))
    return out[:n_rows]


def synth_fp_queries(db, seed=12, sigma_lo=0.8, sigma_hi=2.2, track_len=SEGS_PER_TRACK):
    """query[i] = normalise(db[i] + sigma_track * eps / sqrt(dim)); cos(q, db) ~ 1/sqrt(1+sigma^2)."""
    n, dim = db.shape
    rng = np.random.default_rng(int(seed))
    n_tracks = -(-n // track_len)
    sigma = np.repeat(rng.uniform(sigma_lo, sigma_hi, n_tracks), track_len)[:n].astype(np.float32)
    eps = rng.standard_normal((n, dim), dtype=np.float32)
    return _normalize(db + sigma[:, None] * eps / np.float32(np.sqrt(dim)))


def synth_search_set(n_dummy, n_db=29500, seed=11):
    """(dummy_db, db, query) for the search configs; dummy and db come from disjoint tracks."""
    n_dummy_tracks = -(-n_dummy // SEGS_PER_TRACK)
    dummy = synth_fp_db(n_dummy, seed)
    db = synth_fp_db(n_db, seed, start_track=n_dummy_tracks + 1)
    query = synth_fp_queries(db, seed + 1)
    return dummy, db, query
