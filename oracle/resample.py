"""fp64 numpy restatement of the resampling contract of ``nafp_resample_pcm16_dev`` (include/nafp.h).

For 16-bit PCM with C channels at fs_in, to fs_out: g = gcd, up = fs_out / g, down = fs_in / g,
hl = 10 max(up, down); h = firwin(2 hl + 1, 1 / max(up, down), window=('kaiser', 5.0)) * up (``resample_poly``'s
default filter); x[n] = mean of the channels of frame n; y[m] = sum_n x[n] h[hl + m down - n up] for
m < ceil(N up / down); int16 = rint (half to even), saturated.  Equal rates: a copy / round(mean).
"""
from __future__ import annotations

import math

import numpy as np


def ratio(fs_in, fs_out):
    g = math.gcd(int(fs_in), int(fs_out))
    up, down = int(fs_out) // g, int(fs_in) // g
    return up, down, (0 if up == down else 10 * max(up, down))


def out_length(n_frames, fs_in, fs_out):
    up, down, _ = ratio(fs_in, fs_out)
    return -(-int(n_frames) * up // down)


def kaiser_firwin(numtaps, cutoff, beta=5.0):
    """``scipy.signal.firwin(numtaps, cutoff, window=('kaiser', beta))``: windowed sinc scaled to unit DC gain."""
    alpha = 0.5 * (numtaps - 1)
    m = np.arange(numtaps, dtype=np.float64) - alpha
    h = cutoff * np.sinc(cutoff * m)
    w = np.i0(beta * np.sqrt(np.maximum(0.0, 1.0 - (m / alpha) ** 2))) / np.i0(beta) if numtaps > 1 else np.ones(1)
    h = h * w
    return h / h.sum()


def filter_taps(fs_in, fs_out):
    up, down, hl = ratio(fs_in, fs_out)
    if hl == 0:
        return np.ones(1)
    return kaiser_firwin(2 * hl + 1, 1.0 / max(up, down)) * up


def resample_exact(x, fs_in, fs_out, m0=0, n_out=None):
    """fp64 outputs m0 .. m0 + n_out - 1 (before rounding) of the track x: (N,) or (N, C) int16/float."""
    x = np.asarray(x, np.float64)
    x = x.mean(axis=1) if x.ndim == 2 else x
    n = len(x)
    up, down, hl = ratio(fs_in, fs_out)
    h = filter_taps(fs_in, fs_out)
    if n_out is None:
        n_out = out_length(n, fs_in, fs_out) - m0
    y = np.empty(n_out)
    K = 2 * hl // up + 1                     # taps of the longest phase
    block = max(256, (1 << 21) // K)
    for b0 in range(0, n_out, block):
        m = np.arange(m0 + b0, m0 + min(n_out, b0 + block), dtype=np.int64)
        nh = (hl + m * down) // up           # frame of tap 0; tap k reads frame nh - k
        k = np.arange(K - 1, -1, -1)         # ascending frames
        nn = nh[:, None] - k[None, :]
        j = hl + m[:, None] * down - nn * up
        ok = (j >= 0) & (j <= 2 * hl) & (nn >= 0) & (nn < n)
        terms = np.where(ok, x[np.clip(nn, 0, max(n - 1, 0))] * h[np.clip(j, 0, 2 * hl)], 0.0) if n else np.zeros(nn.shape)
        y[b0:b0 + len(m)] = terms.sum(axis=1)
    return y


def to_int16(y):
    return np.clip(np.rint(y), -32768, 32767).astype(np.int16)


def resample_pcm16(x, fs_in, fs_out, m0=0, n_out=None):
    """int16 outputs (what the device writes) and the fp64 values they round."""
    y = resample_exact(x, fs_in, fs_out, m0, n_out)
    return to_int16(y), y
