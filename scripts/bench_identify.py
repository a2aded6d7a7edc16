"""Identify throughput: clips of 10 s, 30 s, 60 s and 300 s against seeded synthetic databases (flat 'l2' index).

    python scripts/bench_identify.py [--rows 1000000,56000000] [--k 20] [--clips 64] [--out FILE]

The database rows come from nafp_synth_fp_rows (unit-norm, AR(1)-correlated inside 59-row tracks); every clip is a run
of consecutive database rows, regenerated from the same seed, with noise added (cos ~ 0.6 to its source row), so the
right answer is known.  Per clip length one nafp_clip_match_dev call identifies all clips.  CUDA events time that call
(and, for reference, the segment search of the same rows alone).  A separate profiled pass (torch.profiler, CUDA
activities) then splits the call's device time by kernel: the matcher's kernels (clip_*) against the search's kernels,
each summed from the kernels' own durations, so the matcher figure does not depend on subtracting two noisy timings.
The card's name and power limit are read in the same run.  Prints one JSON line (and writes it to --out).
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SEED = 13
TRACK = 59
CLIP_SECONDS = (10, 30, 60, 300)


def gpu_info():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (s.strip() for s in out.split(","))
    return {"gpu": name, "power_limit": power}


def kernel_ms(torch, fn, reps):
    """(matcher, search) device ms per call of ``fn``: the durations of its kernels in a profiled pass, the clip_*
    kernels counted as the matcher and every other kernel as the search (memsets and copies in neither)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    match = search = 0.0
    for a in prof.key_averages():
        us = getattr(a, "self_device_time_total", None)
        if us is None:
            us = a.self_cuda_time_total
        name = a.key
        if "clip_" in name:
            match += us
        elif not name.lower().startswith(("memset", "memcpy")):
            search += us
    if match == 0.0 or search == 0.0:
        raise RuntimeError("the profiler recorded no matcher or no search kernels")
    return match / 1000.0 / reps, search / 1000.0 / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", default="1000000,56000000")
    ap.add_argument("--k", type=int, default=20)
    ap.add_argument("--clips", type=int, default=64, help="clips per length")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--prof-reps", type=int, default=5, help="calls in the profiled pass")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from nafp_b200._lib import Context, check, lib
    from nafp_b200.eval.utils.get_index import FLAT_L2, Index
    info = gpu_info()
    ctx = Context.get(0)
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)
    torch.cuda.set_stream(stream)
    rng = np.random.default_rng(SEED)
    results = []
    for n_rows in (int(r) for r in args.rows.split(",")):
        idx = Index(FLAT_L2, 128, ctx=ctx)
        idx.reserve(n_rows)
        buf = torch.empty((min(4_000_000, n_rows), 128), dtype=torch.float32, device=dev)
        for r in range(0, n_rows, len(buf)):
            n = min(len(buf), n_rows - r)
            check(lib.nafp_synth_fp_rows(ctx.h, SEED, r, n, TRACK, 0.5, ctypes.c_void_p(buf.data_ptr())))
            idx.add_dev(buf.data_ptr(), n)
        del buf
        torch.cuda.synchronize(dev)
        for seconds in CLIP_SECONDS:
            L = (seconds - 1) * 2 + 1                      # 1 s segments every 0.5 s
            starts = np.sort(rng.choice(n_rows - L, args.clips, replace=False))
            clip = torch.empty((L, 128), dtype=torch.float32, device=dev)
            rows = []
            for s in starts:
                check(lib.nafp_synth_fp_rows(ctx.h, SEED, int(s), L, TRACK, 0.5, ctypes.c_void_p(clip.data_ptr())))
                x = clip.cpu().numpy()
                x = x + 1.3 * rng.standard_normal(x.shape).astype(np.float32) / np.sqrt(128, dtype=np.float32)
                rows.append(x / np.linalg.norm(x, axis=1, keepdims=True))
            q = torch.from_numpy(np.concatenate(rows)).to(dev)
            off = torch.from_numpy(np.arange(args.clips + 1, dtype=np.int64) * L).to(dev)
            n_q = len(q)
            D = torch.empty((n_q, args.k), dtype=torch.float32, device=dev)
            I = torch.empty((n_q, args.k), dtype=torch.int64, device=dev)
            pid = torch.empty((args.clips, 10), dtype=torch.int64, device=dev)
            psc = torch.empty((args.clips, 10), dtype=torch.float32, device=dev)

            def search():
                idx.search_dev(q.data_ptr(), n_q, args.k, D.data_ptr(), I.data_ptr())

            def identify():
                check(lib.nafp_clip_match_dev(idx.h, ctypes.c_void_p(q.data_ptr()), n_q, ctypes.c_void_p(off.data_ptr()),
                                              args.clips, args.k, 10, ctypes.c_void_p(pid.data_ptr()),
                                              ctypes.c_void_p(psc.data_ptr())))

            def timed(fn):
                for _ in range(args.warmup):
                    fn()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for _ in range(args.reps):
                    fn()
                e1.record(stream)
                e1.synchronize()
                return e0.elapsed_time(e1) / args.reps

            ms_search = timed(search)
            ms_call = timed(identify)
            k_match, k_search = kernel_ms(torch, identify, args.prof_reps)
            hit = float((pid[:, 0].cpu().numpy() == starts).mean())
            rec = dict(db_rows=n_rows, clip_s=seconds, segments=L, clips=args.clips, k_probe=args.k,
                       call_ms=round(ms_call, 3), search_alone_ms=round(ms_search, 3),
                       search_kernels_ms=round(k_search, 3), matcher_kernels_ms=round(k_match, 3),
                       ms_per_clip=round(ms_call / args.clips, 4),
                       search_kernels_ms_per_clip=round(k_search / args.clips, 4),
                       matcher_kernels_ms_per_clip=round(k_match / args.clips, 4),
                       clips_per_s=round(1000.0 * args.clips / ms_call, 1), top1_exact=hit)
            print(json.dumps(rec), file=sys.stderr)
            results.append(rec)
        del idx
        torch.cuda.synchronize(dev)
    line = json.dumps({"bench": "identify", **info, "index": "l2",
                       "timing": f"call_ms / search_alone_ms: CUDA events, mean of {args.reps} calls after "
                                 f"{args.warmup} warm-up calls; *_kernels_ms: summed kernel durations per call from a "
                                 f"torch.profiler pass of {args.prof_reps} calls (matcher = clip_* kernels)",
                       "results": results})
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
