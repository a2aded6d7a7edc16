"""Throughput of 'ivfpq-rr' (IVFPQR) and of 'ivfpq' at wide k_probe on the bench's seeded synthetic data.

    python scripts/bench_ivfpqr.py [--rows 1000000 56000000] [--steps 3] [--warmup 1] [--rounds 2]
    torchrun --nproc_per_node N scripts/bench_ivfpqr.py ...        (row-sharded form, ShardedFlatIndex)

Database [dummy (seed 11); db (seed 13)], queries and the 2,000 ICASSP test ids x 6 sequence lengths are bench.py's. Per
database size it times one evaluation step (the sequence matcher over every test id, host arrays in and out on one
GPU, device tensors across ranks) of:
  * ivfpq-rr at k_probe 20 through the list-major first level (80 candidates = 4 slices per probed list) and through
    NAFP_IVFPQ_PATH=lut, alternating, `--rounds` times each;
  * ivfpq (the same coarse / PQ quantizers) at k_probe 20 and 32.
It reports queries/s, top-1 hit rates, and the rows the LUT kernel answered per step, with the card's name and power
limit, as one JSON line (stdout, and --out if given).  Nothing is written into the tree.
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

import bench  # noqa: E402  (seeded data, test ids, timing helper)


def _card(local_rank):
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(local_rank), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as e:       # (the numbers are still printed; the card is then unknown)
        return {"gpu": f"unknown ({e})", "power_limit": "unknown"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, nargs="+", default=[1_000_000, bench.N_DUMMY_FULL], help="dummy rows per database")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--rounds", type=int, default=2, help="alternations of the list-major and LUT first levels")
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    args = ap.parse_args()

    import torch
    import torch.distributed as dist
    from nafp_b200._lib import Context, check, lib
    from nafp_b200.dist import ShardedFlatIndex, TorchComm
    from nafp_b200.eval.utils.get_index import IVFPQ, IVFPQR, Index

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    comm = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
        comm = TorchComm()
    barrier = dist.barrier if world > 1 else (lambda: None)
    ctx = Context.get(local_rank)
    torch.cuda.set_stream(torch.cuda.ExternalStream(ctx.stream, device=dev))

    test_ids = bench._test_ids()
    sl_host = np.asarray(bench.SEQ_LENS, np.int32)
    n_queries = len(test_ids) * len(bench.SEQ_LENS)
    dbt = torch.empty((bench.N_DB, 128), dtype=torch.float32, device=dev)
    check(lib.nafp_synth_fp_rows(ctx.h, 13, 0, bench.N_DB, 59, 0.5, ctypes.c_void_p(dbt.data_ptr())))
    query_host = bench._make_queries(dbt.cpu().numpy())
    q_dev = torch.from_numpy(query_host).to(dev)
    ids_dev = torch.from_numpy(test_ids).to(dev)
    sl_dev = torch.from_numpy(sl_host).to(dev)

    def make(itype, path, n_dummy, params):
        """One index over [dummy; db] with the given quantizers (None: train them as bench.py's ivfpq leg does); on
        torchrun every rank holds its row block."""
        os.environ["NAFP_IVFPQ_PATH"] = path
        try:
            if world == 1:
                idx = Index(itype, 128, nlist=256, pq_m=64, pq_nbits=8, device=local_rank)
                target = idx
            else:
                sidx = ShardedFlatIndex(n_dummy + bench.N_DB, rank, world, max_len=max(bench.SEQ_LENS), device=local_rank,
                                        comm=comm, index_type=itype, nlist=256)
                idx = sidx.index
        finally:
            del os.environ["NAFP_IVFPQ_PATH"]
        if params is None:
            buf = torch.empty((min(4_000_000, n_dummy), 128), dtype=torch.float32, device=dev)
            check(lib.nafp_synth_fp_rows(ctx.h, 11, 0, len(buf), 59, 0.5, ctypes.c_void_p(buf.data_ptr())))
            train_rows = buf[:: max(1, len(buf) // 100_000)].contiguous().cpu().numpy()
            del buf
            if world == 1:
                idx.train(train_rows, seed=1234)
            else:
                sidx.train(train_rows if rank == 0 else None, seed=1234)
        else:
            idx.set_ivfpq_params(*params[:2])
            if itype == IVFPQR:
                idx.set_ivfpqr_refine(params[2])
            if world > 1:
                sidx.index.nprobe = 40
        if world == 1:
            idx.reserve(n_dummy + bench.N_DB)
            buf = torch.empty((min(4_000_000, n_dummy), 128), dtype=torch.float32, device=dev)
            r = 0
            while r < n_dummy:
                n = min(len(buf), n_dummy - r)
                check(lib.nafp_synth_fp_rows(ctx.h, 11, r, n, 59, 0.5, ctypes.c_void_p(buf.data_ptr())))
                idx.add_dev(buf.data_ptr(), n)
                r += n
            del buf
            idx.add_dev(dbt.data_ptr(), bench.N_DB)
            idx.nprobe = 40
        else:
            bench.build_sharded_index(ctx, torch, sidx, n_dummy, dev)
            target = sidx
        torch.cuda.synchronize(dev)
        return target, idx

    def leg(target, idx, n_dummy, k_probe, steps):
        result = {}
        if world == 1:
            def step():
                result["pid"] = target.seq_match(query_host, test_ids, sl_host, k_probe)[0]
        else:
            def step():
                result["pid"] = target.seq_match_dev(q_dev, ids_dev, sl_dev, k_probe)[0]
        idx.last_search_stats()
        ms = bench.time_steps(torch, dev, step, steps, args.warmup, barrier)
        st = idx.last_search_stats()
        n_run = steps + args.warmup
        pid = result["pid"] if world == 1 else result["pid"].cpu().numpy()
        return {"k_probe": k_probe, "queries_per_s": n_queries / (ms * 1e-3), "ms_per_step": ms,
                "query_rows_per_step": st["rows"] / n_run, "lut_kernel_rows_per_step": st["fallback_rows"] / n_run,
                "list_major_work_items_per_step": st["passes"] / n_run,
                "top1_hit_rate": [round(float(100.0 * np.mean(pid[:, si, 0] == test_ids + n_dummy)), 2)
                                  for si in range(len(bench.SEQ_LENS))]}

    res = {"script": "scripts/bench_ivfpqr.py", **_card(local_rank), "world": world,
           "form": "host API, one GPU" if world == 1 else "row-sharded (ShardedFlatIndex, NCCL)",
           "queries_per_step": n_queries, "seq_lens": bench.SEQ_LENS, "nlist": 256, "nprobe": 40, "steps": args.steps,
           "warmup": args.warmup, "sizes": []}
    for n_dummy in args.rows:
        t0 = time.time()
        rr_lm, idx_lm = make(IVFPQR, "lm", n_dummy, None)
        params = (*idx_lm.ivfpq_params(), idx_lm.ivfpqr_refine())
        rr_lut, idx_lut = make(IVFPQR, "lut", n_dummy, params)
        t_build = time.time() - t0
        size = {"db_rows": n_dummy + bench.N_DB, "build_s_two_ivfpqr_indexes": t_build, "ivfpq_rr_list_major": [],
                "ivfpq_rr_lut": []}
        for _ in range(args.rounds):
            size["ivfpq_rr_list_major"].append(leg(rr_lm, idx_lm, n_dummy, 20, args.steps))
            size["ivfpq_rr_lut"].append(leg(rr_lut, idx_lut, n_dummy, 20, args.steps))
        del rr_lut, idx_lut
        pq, idx_pq = make(IVFPQ, "lm", n_dummy, params)
        size["ivfpq"] = [leg(pq, idx_pq, n_dummy, kp, args.steps) for kp in (20, 32)]
        del pq, idx_pq, rr_lm, idx_lm
        size["ivfpq_rr_lm_top1_equals_lut"] = all(
            a["top1_hit_rate"] == b["top1_hit_rate"] for a, b in zip(size["ivfpq_rr_list_major"], size["ivfpq_rr_lut"]))
        res["sizes"].append(size)
        torch.cuda.empty_cache()
    if rank == 0:
        line = json.dumps(res)
        print(line)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
