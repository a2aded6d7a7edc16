"""Encoder throughput and accuracy per MODEL.BN ('layer_norm2d', 'layer_norm1d', 'batch_norm').

    python scripts/bench_encoder_norms.py [--segments 4000] [--passes 10] [--rounds 3] [--check 16] [--out FILE]

Seeded synthetic int16 audio, `--segments` per call of the fused device entry point (nafp_fingerprint: log-mel +
encoder, one 4,000-segment encoder pass at the default), groups of 125.  Each mode has its own context and weights
(random, seed 7, random affine parameters; 'batch_norm' with moving statistics calibrated on the reference's own
activations, perturbed by 10 %), is warmed up, and the modes are timed in alternation, `--rounds` times
`--passes` calls each, host clock around device-synchronised work.  The error is the largest absolute difference
and the smallest cosine against the fp64 reference (tests/util_norms.py) on the first `--check` segments.  One JSON
line (stdout, and --out if given) with segments/s per mode, the card's name and power limit, and per mode the device
time of each kernel over one pass (torch.profiler, CUDA activities, in a separate untimed pass).  Nothing is written
into the tree.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

NORMS = ("layer_norm2d", "layer_norm1d", "batch_norm")


def _card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as e:       # (the numbers are still printed; the card is then unknown)
        return {"gpu": f"unknown ({e})", "power_limit": "unknown"}


def _audio(n):
    from nafp_b200 import synth
    tracks, have = [], 0
    seed = 0
    while have < n:
        tr = synth.synth_track(1000 + seed, 8000 * 60)
        rows = np.stack([tr[i * 4000:i * 4000 + 8000] for i in range((len(tr) - 8000) // 4000 + 1)])
        tracks.append(rows)
        have += len(rows)
        seed += 1
    return np.ascontiguousarray(np.concatenate(tracks)[:n], dtype=np.int16)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--segments", type=int, default=4000)
    ap.add_argument("--passes", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--check", type=int, default=16)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    from nafp_b200._lib import Context, check, lib
    from nafp_b200.model import weights as W
    from nafp_b200.model.fp import FingerPrinter
    from oracle import melspec
    import util_norms

    pcm = _audio(a.segments)
    x = (pcm / 2 ** 15).astype(np.float32)
    calib = melspec.melspec_layer(x[:64:4, None, :], group_size=16, dtype=np.float32)
    models, bufs = {}, {}
    for norm in NORMS:
        w = W.init_weights(7, randomize_affine=True, norm=norm)
        if norm == "batch_norm":
            w = util_norms.calibrate_batch_norm(calib, w, seed=7)
        ctx = Context(0)
        models[norm] = (ctx, FingerPrinter(ctx, norm=norm).load(w), w)
        xd, ed = ctx.malloc(x.nbytes), ctx.malloc(a.segments * 128 * 4)
        ctx.h2d(xd, x)
        bufs[norm] = (xd, ed)

    def run(norm, passes):
        ctx = models[norm][0]
        xd, ed = bufs[norm]
        for _ in range(passes):
            check(lib.nafp_fingerprint(ctx.h, xd, a.segments, 125, ed))
        ctx.sync()

    for norm in NORMS:                      # warm-up: modules, arena, every kernel of every mode
        run(norm, 2)
    times = {n: [] for n in NORMS}
    for _ in range(a.rounds):
        for norm in NORMS:
            t0 = time.perf_counter()
            run(norm, a.passes)
            times[norm].append(time.perf_counter() - t0)

    kernels = {}
    try:                                    # per-kernel device time of one pass per mode (separate from the timing)
        import torch
        from torch.profiler import ProfilerActivity, profile
        for norm in NORMS:
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                run(norm, 1)
            per = {}
            for e in prof.events():
                if e.device_type.name == "CUDA":
                    name = e.name.split("(")[0].replace("void ", "").replace("nafp::", "")
                    per[name] = per.get(name, 0.0) + e.device_time_total / 1e3
            kernels[norm] = {k: round(v, 3) for k, v in sorted(per.items(), key=lambda kv: -kv[1])}
    except Exception as e:                  # the rates above stand without the breakdown
        kernels = {"error": repr(e)[:200]}

    res = {"bench": "encoder_norms", "segments_per_call": a.segments, "passes": a.passes, "rounds": a.rounds}
    res.update(_card())
    for norm in NORMS:
        ctx, m_fp, w = models[norm]
        rates = [a.segments * a.passes / t for t in times[norm]]
        n = a.check
        mel = melspec.melspec_layer(x[:n, None, :], group_size=125, dtype=np.float32)
        ref = util_norms.fingerprinter(mel, w, norm)
        emb = m_fp.fingerprint(pcm[:n], group_size=125)
        res[norm] = {"seg_per_s": round(float(np.median(rates))), "seg_per_s_all": [round(r) for r in rates],
                     "ms_per_4000": round(4000 / float(np.median(rates)) * 1e3, 3),
                     "max_abs_err": float(np.abs(emb - ref).max()), "min_cosine": float((emb * ref).sum(1).min())}
    res["kernel_ms_per_pass"] = kernels
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
