"""Resampling throughput: the polyphase kernel alone, and the any-rate fingerprint path against the 8 kHz path.

    python scripts/bench_resample.py [--hours 1] [--reps 10] [--out FILE]

1. Kernel: nafp_resample_pcm16_dev over --hours of seeded noise (larger than the 126 MB L2) at 44.1 kHz stereo,
   48 kHz stereo and 22.05 kHz mono, timed with CUDA events on the ctx stream.  Reported: seconds of audio per second,
   input GB/s, fp64 multiply-adds per second (the nonzero filter taps, (2 hl + 1) / up per output), and the share of the
   least time the card could take: the larger of bytes (int16 in + out) over 7.7 TB/s of HBM3e and multiply-adds over
   the fp64 rate, 37 TFLOP/s (NVIDIA's HGX B200 data sheet prints 296 TFLOP/s FP64 for eight GPUs).
2. Fingerprints/s of one generate-sized block (8,000 segments, 136 tracks of 30 s) through
   nafp_fingerprint_pcm16_sources_host from pinned 44.1 kHz stereo, and through nafp_fingerprint_pcm16_tracks_host on
   the same audio already at 8 kHz (pinned), the two alternated; host wall clock around calls that return synchronised.
3. For scale, a CPU figure: scipy.signal.resample_poly on one core for 300 s of 44.1 kHz mono.
The card's name and power limit are read in the same run.  Prints one JSON line (and writes it to --out).
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_BPS = 7.7e12
FP64_FLOPS = 37e12


def gpu_info():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (s.strip() for s in out.split(","))
    return {"gpu": name, "power_limit": power}


def pinned(ctx, lib, check, shape, dtype):
    p = ctypes.c_void_p()
    n = int(np.prod(shape)) * np.dtype(dtype).itemsize
    check(lib.nafp_malloc_host(ctx.h, n, ctypes.byref(p)))
    buf = (ctypes.c_byte * n).from_address(p.value)
    return np.frombuffer(buf, dtype=dtype).reshape(shape), p


def kernel_leg(ctx, lib, check, fs, ch, hours, reps):
    from nafp_b200.model.dataset import resample_ratio, resampled_length
    up, down, hl = resample_ratio(fs, 8000)
    n = int(hours * 3600 * fs)
    n_out = resampled_length(n, fs, 8000)
    rng = np.random.default_rng(fs + ch)
    x = rng.integers(-20000, 20000, n * ch, dtype=np.int16)
    xd, od = ctx.malloc(x.nbytes), ctx.malloc(n_out * 2)
    try:
        ctx.h2d(xd, x)
        call = lambda: check(lib.nafp_resample_pcm16_dev(ctx.h, xd, 0, n, ch, fs, 8000, 0, n_out, od))
        for _ in range(2):
            call()
        ctx.sync()
        times = []
        for _ in range(reps):
            ctx.timer_start()
            call()
            times.append(ctx.timer_stop() / 1e3)
    finally:
        ctx.free(xd)
        ctx.free(od)
    t = float(np.median(times))
    fma = n_out * (2 * hl + 1) / up
    nbytes = x.nbytes + n_out * 2
    t_hbm, t_fp64 = nbytes / HBM_BPS, 2 * fma / FP64_FLOPS
    return {"fs_in": fs, "channels": ch, "audio_s": n / fs, "kernel_ms_median": t * 1e3,
            "kernel_ms_min": min(times) * 1e3, "audio_s_per_s": n / fs / t, "input_GBps": x.nbytes / t / 1e9,
            "fp64_fma_per_s": fma / t, "taps_per_output": (2 * hl + 1) / up,
            "bound": "fp64" if t_fp64 > t_hbm else "hbm", "share_of_bound": max(t_hbm, t_fp64) / t}


def pipeline_leg(ctx, lib, check, reps):
    from nafp_b200 import synth
    from nafp_b200.model.dataset import n_segments, source_window
    from nafp_b200.model.fp import FingerPrinter
    from nafp_b200.model.weights import init_weights
    from oracle import resample as R
    m_fp = FingerPrinter(ctx).load(init_weights(7))
    n_tracks, fs, ch, T8 = 136, 44100, 2, 240000
    n8_total = n_tracks * T8
    src, _ = pinned(ctx, lib, check, (n_tracks * 1323000 * ch,), np.int16)
    base = synth.synth_track(1, T8)
    up8 = R.resample_pcm16(base, 8000, fs)[0]                  # 30 s at 44.1 kHz, reused for every track
    for i in range(n_tracks):
        g = 0.5 + 0.5 * (i % 7) / 7
        src[i * 1323000 * ch:(i + 1) * 1323000 * ch] = np.repeat((up8 * g).astype(np.int16), ch)
    runs, offs, valid = [], [], []
    nseg = n_segments(T8)
    starts = np.floor(np.arange(nseg) * 4000).astype(np.int64)
    for i in range(n_tracks):
        first, last = 0, min(int(starts[-1]) + 8000, T8)
        f0, cnt = source_window(first, last - first, 1323000, fs, 8000)
        runs.append((i * 1323000 * ch + f0 * ch, f0, cnt, ch, fs, first, last - first))
        offs.append(starts + i * T8)
        valid.append(np.minimum(8000, T8 - starts).astype(np.int32))
    runs = np.asarray(runs, np.int64)
    offs, valid = np.concatenate(offs)[:8000], np.concatenate(valid)[:8000]
    n_seg = len(offs)
    # the same audio at 8 kHz: the device resampler's output, pinned
    trk, _ = pinned(ctx, lib, check, (n8_total,), np.int16)
    xd, od = ctx.malloc(1323000 * ch * 2), ctx.malloc(T8 * 2)
    for i in range(n_tracks):
        ctx.h2d(xd, src[i * 1323000 * ch:(i + 1) * 1323000 * ch])
        check(lib.nafp_resample_pcm16_dev(ctx.h, xd, 0, 1323000, ch, fs, 8000, 0, T8, od))
        ctx.d2h(trk[i * T8:(i + 1) * T8], od)
    ctx.sync()
    ctx.free(xd)
    ctx.free(od)
    emb_a, emb_b = np.empty((n_seg, 128), np.float32), np.empty((n_seg, 128), np.float32)

    def sources():
        check(lib.nafp_fingerprint_pcm16_sources_host(ctx.h, src.ctypes.data, len(src), runs.ctypes.data, len(runs),
                                                       offs.ctypes.data, valid.ctypes.data, n_seg, 125,
                                                       emb_a.ctypes.data))

    def tracks():
        check(lib.nafp_fingerprint_pcm16_tracks_host(ctx.h, trk.ctypes.data, len(trk), offs.ctypes.data,
                                                     valid.ctypes.data, n_seg, 125, emb_b.ctypes.data))
    for _ in range(2):
        sources()
        tracks()
    ts, tt = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        sources()
        ts.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        tracks()
        tt.append(time.perf_counter() - t0)
    same = bool(np.array_equal(emb_a.view(np.uint32), emb_b.view(np.uint32)))
    return {"segments": n_seg, "tracks": n_tracks, "source": "44100 Hz stereo, pinned",
            "sources_host_fp_per_s": n_seg / float(np.median(ts)), "tracks_host_8k_fp_per_s": n_seg / float(np.median(tt)),
            "sources_host_ms_median": float(np.median(ts)) * 1e3, "tracks_host_ms_median": float(np.median(tt)) * 1e3,
            "source_bytes": int(runs[:, 2].sum() * ch * 2), "track_bytes_8k": int(n8_total * 2),
            "fingerprints_bit_identical": same}


def scipy_leg():
    import scipy.signal
    x = np.random.default_rng(0).integers(-20000, 20000, 300 * 44100).astype(np.float64)
    scipy.signal.resample_poly(x[:44100], 80, 441)
    t0 = time.perf_counter()
    scipy.signal.resample_poly(x, 80, 441)
    t = time.perf_counter() - t0
    return {"what": "CPU, one core: scipy.signal.resample_poly, 300 s of 44.1 kHz mono", "seconds": t,
            "audio_s_per_s": 300.0 / t}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--hours", type=float, default=1.0)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from nafp_b200._lib import Context, check, lib
    ctx = Context.get(0)
    rec = {"bench": "resample", **gpu_info(),
           "peaks": {"hbm_Bps": HBM_BPS, "fp64_flops": FP64_FLOPS,
                     "fp64_source": "NVIDIA HGX B200 data sheet: 296 TFLOPS FP64 for 8 GPUs"}}
    rec["kernel"] = [kernel_leg(ctx, lib, check, fs, ch, args.hours, args.reps)
                     for fs, ch in ((44100, 2), (48000, 2), (22050, 1))]
    rec["pipeline"] = pipeline_leg(ctx, lib, check, max(3, args.reps // 2))
    rec["cpu_reference"] = scipy_leg()
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
