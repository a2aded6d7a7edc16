#!/usr/bin/env python
"""bench.py -- the driver-facing benchmark of the B200 fingerprint-retrieval hot path.

Headline (BASELINE.json `metric`): search queries/s at the full-scale ~56 M-fingerprint database,
where a "query" is one (test id, sequence length) evaluation -- the unit of the reference's own
"ms/query" (eval/eval_faiss.py:246-258).  One step = the whole evaluation job of the reference CLI:
2,000 query sequences (the ICASSP test ids) x sequence lengths 1 3 5 9 11 19 (12,000 queries),
k_probe 20, against [dummy_db; db] = 56,000,000 + 29,500 unit-norm 128-d rows generated on the device
(BASELINE configs[3]).  With N GPUs the same database is row-sharded (strong scaling) and the per-rank
top-k / candidate scores are combined with an NCCL all-gather and a max all-reduce.

  value        device-resident: queries already in HBM, CUDA events around the kernels + collectives
  e2e          the plugin call a user makes -- N = 1: the C-ABI host entry nafp_seq_match (pinned host queries in,
               predictions out); N > 1: the sharded matcher fed from pinned host memory -- every step
  roofline     the flat scan kernel: rows_local x 256 B (and 2 x rows x 128 x query rows flop) per launch /
               CUDA-event launch time vs the measured HBM copy bandwidth and sustained bf16 rate
               (MEASURED_PEAKS.json); the nearer bound leads, the other is under "other_bound";
               `traffic` = DRAM bytes of one launch parsed from the committed ncu capture under profiles/
  fingerprint  BASELINE configs[2] per GPU: log-mel + encoder segments/s (tensor roofline), its own e2e, a `logmel`
               sub-record (HBM roofline of logmel_kernel alone) and a torch-CPU `cpu_baseline`
  mini_1M      BASELINE configs[1]; ivfpq_1M / ivfpq_full: BASELINE configs[4] at 1 M rows (with the CPU oracle's hit
               rates beside the GPU's) and at the full 56 M rows (every N); config0: BASELINE configs[0] as stated
  cpu_baseline the C oracle (oracle/csrc/oracle.c: faiss-flat semantics, fp32 SIMD, all host threads) + the reference's
               matching loop, timed at three database sizes, fitted a + b x rows and extrapolated to the full size;
               rank 0 at N = 1 only

`--impl reference` times that CPU implementation alone (no GPU work at all), --steps / --warmup honoured.
`--dump-outputs DIR` writes what each timed GPU path returned in its last step (predictions and scores of every search
leg, the fingerprints) as DIR/<name>.npy, float32 / float64, under 64 MB in all.
"""
from __future__ import annotations

import argparse
import csv
import glob
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_DUMMY_FULL = 56_000_000
N_DB = 29_500
SEQ_LENS = [1, 3, 5, 9, 11, 19]
K_PROBE = 20
FP_SEGS_PER_STEP = 4000          # 32 groups of TS_BATCH_SZ = 125 = one full encoder pass (ENC_CHUNK_MAX)
FP_E2E_SEGS = 8000               # host-API step: what one generate.py call hands over (64 batches)
FLOPS_PER_SEGMENT = 607_199_232  # model/arch.py (conv + div-enc)
LOGMEL_BYTES_PER_SEGMENT = 64_768    # SURVEY 8(d): 32,000 B of samples in + 32,768 B of log-mel out
CPU_FIT = [(250_000, 200), (1_000_000, 200), (4_000_000, 40)]      # (database rows, test ids) of the CPU baseline fit
REF_STEP_ROWS, REF_STEP_IDS = 1_000_000, 24                          # one step of the --impl reference arm
DUMP_MAX_BYTES = 64 << 20


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 6650.0, 1590.0, 1400.0, "fallback"


def _test_ids():
    return np.load(os.path.join(ROOT, "neural-audio-fp_b200", "eval", "test_ids_icassp2021.npy")).astype(np.int64)


def _make_queries(db, seed=12):
    from nafp_b200 import synth
    return synth.synth_fp_queries(db, seed)


def ncu_traffic(kernel_substr, pattern):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of `kernel_substr` from the newest committed ncu
    summary under profiles/ matching `pattern` (header row, unit row, one row per launch).  Returns (bytes, file, rows_note)."""
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", pattern)), key=lambda f: (os.path.basename(f)[:2], os.path.getmtime(f)), reverse=True):
        try:
            rows = list(csv.reader(open(path)))
            hdr, units = rows[0], rows[1]
            ir, iw = hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum")
            for r in rows[2:]:
                if kernel_substr in r[0]:
                    return float(r[ir]) * unit[units[ir]] + float(r[iw]) * unit[units[iw]], os.path.relpath(path, ROOT)
        except (ValueError, IndexError, KeyError, OSError):
            continue
    return None, None


# ----------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        self.gpu = gpu
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=open(self.path, "w"),
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
            rows = [r.strip().split(", ") for r in open(self.path) if r.strip()]
            rows = [r for r in rows if len(r) >= 8]
            sm = sorted(float(r[0]) for r in rows)
            if sm:
                out["sm_mhz"] = sm[len(sm) // 2]
                out["sm_max_mhz"] = float(rows[0][1])
                out["samples"] = len(sm)
                names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
                for i, nm in enumerate(names):
                    if any(r[4 + i].strip().lower().startswith("active") for r in rows):
                        out["reasons"].append(nm)
        except Exception as e:  # clocks are evidence, not a reason to lose the number
            out["error"] = str(e)
        finally:
            try:
                os.unlink(self.path)
            except OSError:
                pass
        return out


# ----------------------------------------------------------------------------------------------
# CPU implementation (oracle) -- cpu_baseline legs and the --impl reference arm
# ----------------------------------------------------------------------------------------------
def _cpu_rows(n, seed):
    """Host copy of the synthetic database rows [0, n) (numpy generator of nafp_b200.synth: same distribution as the
    device generator, AR(1) tracks of 59 rows)."""
    from nafp_b200 import synth
    return synth.synth_fp_db(n, seed=seed)


def cpu_search_once(index, recon, n_dummy, query, ids):
    """One pass of the reference's evaluation loop (eval_faiss.py:204-243) over `ids` on the CPU index; seconds."""
    from oracle import seq_match
    t0 = time.perf_counter()
    seq_match.evaluate(index, query, recon, n_dummy, ids, SEQ_LENS, K_PROBE, fast_scores=True)
    return time.perf_counter() - t0


def cpu_search_fit(db, query, test_ids, n_full_rows, sizes=CPU_FIT, big=None):
    """Seconds per query of the CPU implementation at several database sizes -> least-squares a + b x rows ->
    queries/s at the full database (extrapolation, labelled as such).  `big`: host rows of the synthetic database
    (generated here when not given)."""
    from oracle import native
    pts = []
    if big is None:
        big = _cpu_rows(max(r for r, _ in sizes), 11)
    for rows, n_ids in sizes:
        idx = native.FlatL2C(128)
        idx.add(big[:rows])
        idx.add(db)
        recon = idx._data()
        ids = test_ids[:n_ids]
        cpu_search_once(idx, recon, rows, query, ids[:2])                       # warm (page faults, thread pool)
        sec = cpu_search_once(idx, recon, rows, query, ids)
        pts.append({"rows": rows + len(db), "test_ids": int(n_ids), "sec_per_query": sec / (n_ids * len(SEQ_LENS))})
        del idx, recon
    x = np.array([p["rows"] for p in pts], np.float64)
    y = np.array([p["sec_per_query"] for p in pts], np.float64)
    b, a = np.polyfit(x, y, 1)
    full = a + b * n_full_rows
    return dict(value=1.0 / full, unit="queries/s", cores=native.threads(), kind="port",
                implementation="oracle/csrc/oracle.c orc_flat_search (faiss IndexFlatL2 semantics for nq < 20: fp32 SIMD "
                               "(q - x)^2, OpenMP over the database) + the reference's matching loop (oracle/seq_match.py)",
                fit={"sec_per_query = a + b * rows": {"a": float(a), "b": float(b)}, "points": pts},
                sample=f"measured at {[p['rows'] for p in pts]} rows on {[p['test_ids'] for p in pts]} of the "
                       f"{len(test_ids)} test ids x {len(SEQ_LENS)} lengths; value = 1 / (a + b x {n_full_rows:,}) "
                       f"-- an EXTRAPOLATION of the fitted line to the full database, which does not fit the sample budget")


def cpu_generate(n_seg=250, group=125, seed=5):
    """The extractor on torch-CPU fp32, all host threads (oracle/torch_ref.py): segments/s."""
    import torch
    from nafp_b200 import synth
    from nafp_b200.model import weights as W
    from oracle import torch_ref
    tr = synth.synth_track(seed, 8000 + 4000 * (n_seg - 1)).astype(np.float32) / 32768.0
    x = np.stack([tr[i * 4000:i * 4000 + 8000] for i in range(n_seg)])[:, None, :]
    fp = torch_ref.TorchFingerPrinter(W.init_weights(7))
    fp(torch_ref.melspec_torch(x[:group], group))                                  # warm-up
    t0 = time.perf_counter()
    for s in range(0, n_seg, group):
        fp(torch_ref.melspec_torch(x[s:s + group], group))
    sec = time.perf_counter() - t0
    return dict(value=n_seg / sec, unit="segments/s", cores=torch.get_num_threads(), kind="port",
                implementation="oracle/torch_ref.py: torch-CPU fp32 stft + mel + conv2d / layer_norm (what the reference's "
                               "TensorFlow-CPU generate runs through oneDNN), batches of TS_BATCH_SZ 125",
                sample=f"{n_seg} one-second segments ({n_seg // group} batches) after one warm-up batch")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import native
    native.lib().orc_set_threads(os.cpu_count() or 1)      # torchrun exports OMP_NUM_THREADS=1: this arm owns the host
    threads = native.threads()
    n_full = args.db_rows + N_DB
    db = _cpu_rows(N_DB, 13)
    query = _make_queries(db)
    test_ids = _test_ids()
    # calibration (untimed): slope and intercept of seconds per query against database rows
    big = _cpu_rows(2_000_000, 11)
    fit = cpu_search_fit(db, query, test_ids, n_full, sizes=[(250_000, 24), (1_000_000, 24), (2_000_000, 12)], big=big)
    a, b = fit["fit"]["sec_per_query = a + b * rows"]["a"], fit["fit"]["sec_per_query = a + b * rows"]["b"]
    rows = min(REF_STEP_ROWS, args.db_rows)
    idx = native.FlatL2C(128)
    idx.add(big[:rows])
    del big
    idx.add(db)
    recon = idx._data()
    times = []
    for s in range(args.warmup + args.steps):
        ids = test_ids[(s * REF_STEP_IDS) % 1900:(s * REF_STEP_IDS) % 1900 + REF_STEP_IDS]
        dt = cpu_search_once(idx, recon, rows, query, ids)
        if s >= args.warmup:
            times.append(dt)
    sec_q_sample = float(np.mean(times)) / (REF_STEP_IDS * len(SEQ_LENS))
    # the measured per-query time at the sample size, moved to the full size along the calibrated slope
    sec_q_full = sec_q_sample + b * (n_full - (rows + N_DB))
    value = 1.0 / sec_q_full
    cb = dict(value=value, unit="queries/s", cores=threads, kind="port", implementation=fit["implementation"],
              measured_queries_per_s_on_sample=1.0 / sec_q_sample, sec_per_step=float(np.mean(times)),
              calibration=fit["fit"],
              sample=f"each step: {REF_STEP_IDS} test ids x {len(SEQ_LENS)} lengths against a {rows + N_DB:,}-row sample; "
                     f"value = 1 / (measured s/query + b x (full rows - sample rows)), b = {b:.3e} s/query/row from the "
                     f"three-size calibration -- an EXTRAPOLATION to the {n_full:,}-row database")
    line = {"impl": "reference", "metric": "search_queries_per_s", "value": value, "unit": "queries/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(np.mean(times)) * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": _config(args, 1), "cpu_baseline": cb,
            "e2e": {"value": value, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))
    return 0


def _config(args, world):
    return {"workload": f"exact flat-L2 search + sequence rescoring: 2,000 query sequences x lengths {SEQ_LENS}, "
                        f"k_probe {K_PROBE}, vs {args.db_rows + N_DB:,}-row 128-d database "
                        f"(BASELINE configs[3]; configs[0] / [1] / [2] / [4] ride along as config0 / mini_1M / fingerprint / ivfpq_*)",
            "db_rows": args.db_rows + N_DB, "n_test_ids": 2000, "seq_lens": SEQ_LENS, "k_probe": K_PROBE,
            "parallelism": f"db-row-shard x{world}" if world > 1 else "single GPU",
            "l2_policy": "inputs larger than L2 (bf16 scan copy >= 1.8 GB per GPU is streamed every pass)"}


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
def build_sharded_index(ctx, torch, sidx, n_dummy, dev):
    """Fill this rank's block of [dummy (seed 11); db (seed 13)] on the device, chunk by chunk."""
    from nafp_b200._lib import check, lib
    import ctypes
    lo, hi = sidx.local_rows_needed()
    chunk = 4_000_000
    buf = torch.empty((min(chunk, hi - lo), 128), dtype=torch.float32, device=dev)
    r = lo
    while r < hi:
        if r < n_dummy:
            n = min(chunk, min(hi, n_dummy) - r)
            check(lib.nafp_synth_fp_rows(ctx.h, 11, r, n, 59, 0.5, ctypes.c_void_p(buf.data_ptr())))
        else:
            n = min(chunk, hi - r)
            check(lib.nafp_synth_fp_rows(ctx.h, 13, r - n_dummy, n, 59, 0.5, ctypes.c_void_p(buf.data_ptr())))
        sidx.add_local_dev(buf.data_ptr(), n)
        r += n
    torch.cuda.synchronize(dev)
    del buf


def dump_outputs(outputs, out_dir):
    """--dump-outputs: each array as out_dir/<name>.npy.  The inputs are seeded, so two builds run with the same
    arguments can be compared output for output."""
    assert sum(a.nbytes for a in outputs.values()) <= DUMP_MAX_BYTES
    os.makedirs(out_dir, exist_ok=True)
    for name, a in outputs.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def time_steps(torch, dev, fn, steps, warmup, barrier):
    for _ in range(warmup):
        fn()
    barrier()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize(dev)
    barrier()
    return e0.elapsed_time(e1) / steps


def run_gpu(args):
    import ctypes
    import torch
    import torch.distributed as dist
    from nafp_b200._lib import Context, check, lib
    from nafp_b200.dist import ShardedFlatIndex, TorchComm
    from nafp_b200.model import weights as W
    from nafp_b200.model.fp import FingerPrinter

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

    def barrier():
        if world > 1:
            dist.barrier()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    ctx = Context.get(local_rank)
    # all torch work (copies, NCCL, CUDA events) on the stream the library launches its kernels on
    torch.cuda.set_stream(torch.cuda.ExternalStream(ctx.stream, device=dev))
    hbm_peak, tf_burst, tf_sustained, peak_src = _peaks()
    n_dummy = args.db_rows
    n_total = n_dummy + N_DB
    test_ids = _test_ids()
    n_queries = len(test_ids) * len(SEQ_LENS)
    sl_host = np.asarray(SEQ_LENS, np.int32)

    # ---- database shard + queries
    t_build = time.time()
    sidx = ShardedFlatIndex(n_total, rank, world, max_len=max(SEQ_LENS), device=local_rank, comm=comm)
    build_sharded_index(ctx, torch, sidx, n_dummy, dev)
    dbt = torch.empty((N_DB, 128), dtype=torch.float32, device=dev)
    check(lib.nafp_synth_fp_rows(ctx.h, 13, 0, N_DB, 59, 0.5, ctypes.c_void_p(dbt.data_ptr())))
    db_host = dbt.cpu().numpy()
    query_host = _make_queries(db_host)
    t_build = time.time() - t_build

    q_pin = torch.from_numpy(query_host).pin_memory()
    ids_pin = torch.from_numpy(test_ids).pin_memory()
    sl_pin = torch.tensor(SEQ_LENS, dtype=torch.int32).pin_memory()
    q_dev, ids_dev, sl_dev = q_pin.to(dev), ids_pin.to(dev), sl_pin.to(dev)
    result = {}

    def step_resident():
        result["pid"], result["psc"] = sidx.seq_match_dev(q_dev, ids_dev, sl_dev, K_PROBE)

    if world == 1:
        q_pin_np = q_pin.numpy()               # the same pinned pages, handed to the C ABI as a plain host pointer

        def step_e2e():                        # the advertised plugin call: host buffers in, host buffers out
            result["pid_host"], result["psc_host"] = sidx.index.seq_match(q_pin_np, test_ids, sl_host, K_PROBE)
        e2e_through = "nafp_seq_match (C-ABI host entry: pinned host queries + ids in, predictions out)"
    else:
        def step_e2e():
            q = q_pin.to(dev, non_blocking=True)
            ids = ids_pin.to(dev, non_blocking=True)
            sl = sl_pin.to(dev, non_blocking=True)
            pid, psc = sidx.seq_match_dev(q, ids, sl, K_PROBE)
            result["pid_host"] = pid.to("cpu")
            result["psc_host"] = psc.to("cpu")
        e2e_through = "ShardedFlatIndex.seq_match_dev fed from pinned host memory (H2D queries, NCCL, D2H predictions)"

    # ---- headline: resident
    sampler = ClockSampler(local_rank)
    sampler.start()                       # nvidia-smi needs a few hundred ms to start; warm-up runs under load too
    for _ in range(args.warmup):
        step_resident()
    torch.cuda.synchronize(dev)
    sidx.index.profile_scans(True)
    sidx.index.last_search_stats()
    launches0 = ctx.launches
    ms_res = max_over_ranks(time_steps(torch, dev, step_resident, args.steps, 0, barrier))
    clocks = sampler.stop()
    # what each timed path returned in its last step, for --dump-outputs (ids as float64: exact below 2**53)
    outputs = {"search_pred_ids": result["pid"].cpu().numpy().astype(np.float64),
               "search_pred_scores": result["psc"].cpu().numpy()}
    launches = ctx.launches - launches0
    scan_ms, n_scans = sidx.index.profile_scans(False)
    stats = sidx.index.last_search_stats()
    # ---- e2e
    ms_e2e = max_over_ranks(time_steps(torch, dev, step_e2e, args.steps, max(3, args.warmup // 2), barrier))

    pid = result["pid"].cpu().numpy()
    gt = test_ids + n_dummy
    top1 = [float(100.0 * np.mean(pid[:, si, 0] == gt)) for si in range(len(SEQ_LENS))]
    e2e_same = bool((np.asarray(result["pid_host"])[:, :, 0] == pid[:, :, 0]).all())

    # ---- roofline of the scan kernel (this rank's rows; all ranks launch the same count).
    # One launch streams the rank's bf16 rows once (rows x 256 B) and multiplies them with up to 256 query
    # rows (2 x rows x 128 x query rows flop).  With 256-row passes the two bounds are within 15 % of each
    # other on B200; the line reports the bound the kernel is closer to, the other one rides along.
    rows_local = sidx.hi - sidx.lo
    scan_avg_ms = scan_ms / max(n_scans, 1)
    alg_bytes = rows_local * 256.0
    q_rows_per_launch = stats["rows"] / max(stats["passes"], 1) if stats.get("passes") else 256.0
    alg_flops = 2.0 * rows_local * 128.0 * q_rows_per_launch
    gbs = alg_bytes / (scan_avg_ms * 1e-3) / 1e9 if n_scans else 0.0
    tfs = alg_flops / (scan_avg_ms * 1e-3) / 1e12 if n_scans else 0.0
    hbm_part = {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
                "peak_source": f"{peak_src} (MEASURED_PEAKS.json hbm_gbs)", "algorithmic_bytes_per_launch": alg_bytes}
    tensor_part = {"bound": "tensor", "achieved": tfs, "peak": tf_sustained, "unit": "TFLOP/s", "frac": tfs / tf_sustained,
                   "peak_source": f"{peak_src} (MEASURED_PEAKS.json bf16_tflops_sustained: kernel timed inside a long step)",
                   "algorithmic_flops_per_launch": alg_flops}
    first, second = (tensor_part, hbm_part) if tensor_part["frac"] >= hbm_part["frac"] else (hbm_part, tensor_part)
    # DRAM bytes of ONE launch, parsed from the committed ncu --set full capture of this kernel (56,029,500-row shard);
    # a smaller shard streams proportionally fewer rows (the capture is 1.02 x the algorithmic bytes)
    cap_bytes, cap_file = ncu_traffic("flat_scan_kernel", "r*_prof_scan*summary.csv")
    traffic, traffic_note = None, None
    if cap_bytes is not None:
        full_rows = N_DUMMY_FULL + N_DB
        traffic = cap_bytes if rows_local == full_rows else cap_bytes * rows_local / full_rows
        traffic_note = ("dram__bytes_read.sum + dram__bytes_write.sum of one launch" if rows_local == full_rows else
                        f"the captured launch ({full_rows:,} rows) scaled to this rank's {rows_local:,} rows")
    roofline = {"kernel": "flat_scan_kernel", **first, "traffic": traffic, "traffic_source": cap_file, "traffic_note": traffic_note,
                "other_bound": second, "launches": n_scans,
                "avg_launch_ms": scan_avg_ms, "scan_share_of_step": scan_ms / max(ms_res * args.steps, 1e-9),
                "query_rows_per_launch": q_rows_per_launch}

    # ---- secondary: fingerprint generation (every rank runs its own batches, no collective) -- BASELINE configs[2]
    fp = None
    if not args.no_fp:
        m_fp = FingerPrinter(ctx).load(W.init_weights(7))
        x_dev = torch.empty((FP_SEGS_PER_STEP, 8000), dtype=torch.float32, device=dev)
        check(lib.nafp_synth_audio(ctx.h, 5, rank * FP_SEGS_PER_STEP, FP_SEGS_PER_STEP, ctypes.c_void_p(x_dev.data_ptr())))
        emb_dev = torch.empty((FP_SEGS_PER_STEP, 128), dtype=torch.float32, device=dev)
        mel_dev = torch.empty((FP_SEGS_PER_STEP, 8192), dtype=torch.float32, device=dev)
        # e2e: int16 PCM segments from pinned host memory (the / 2**15 of audio_utils.py:243-244 runs on the GPU),
        # fingerprints back to host memory; one e2e step = one call of generate.py's size (batches_per_call 64 x
        # TS_BATCH_SZ 125 = two encoder passes: the upload of the second runs under the kernels of the first)
        x_pin = (x_dev.clamp(-1.0, 1.0) * 32767.0).round().to(torch.int16).cpu().repeat(FP_E2E_SEGS // FP_SEGS_PER_STEP, 1).pin_memory()
        emb_host = np.empty((FP_E2E_SEGS, 128), np.float32)

        def fp_resident():
            check(lib.nafp_fingerprint(ctx.h, ctypes.c_void_p(x_dev.data_ptr()), FP_SEGS_PER_STEP, 125,
                                       ctypes.c_void_p(emb_dev.data_ptr())))

        def fp_e2e():
            check(lib.nafp_fingerprint_pcm16_host(ctx.h, ctypes.c_void_p(x_pin.data_ptr()), FP_E2E_SEGS, 125,
                                                  emb_host.ctypes.data_as(ctypes.c_void_p)))

        def logmel_only():
            check(lib.nafp_logmel_forward_raw(ctx.h, ctypes.c_void_p(x_dev.data_ptr()), FP_SEGS_PER_STEP, 125,
                                              ctypes.c_void_p(mel_dev.data_ptr()), None))

        l0 = ctx.launches
        ms_fp = max_over_ranks(time_steps(torch, dev, fp_resident, args.steps, args.warmup, barrier))
        fp_launches = (ctx.launches - l0) // (args.steps + args.warmup)
        outputs["fingerprints"] = emb_dev.cpu().numpy()
        ms_fp_e2e = max_over_ranks(time_steps(torch, dev, fp_e2e, args.steps, 3, barrier))
        ms_mel = max_over_ranks(time_steps(torch, dev, logmel_only, args.steps, 3, barrier))
        segs = FP_SEGS_PER_STEP * world
        tfl = segs / (ms_fp * 1e-3) * FLOPS_PER_SEGMENT / 1e12 / world
        mel_gbs = FP_SEGS_PER_STEP * LOGMEL_BYTES_PER_SEGMENT / (ms_mel * 1e-3) / 1e9
        mel_traffic, mel_file = ncu_traffic("logmel_kernel", "r*_prof_logmel*summary.csv")
        fp = {"metric": "fp_segments_per_s", "value": segs / (ms_fp * 1e-3), "unit": "segments/s", "ms_per_step": ms_fp,
              "segments_per_step": segs, "dtype": "fp16 operands (split hi + lo from L4a on), fp32 accumulate",
              "workload": "BASELINE configs[2] per GPU: log-mel + FingerPrinter over device-resident synthetic 1 s segments, "
                          "groups of TS_BATCH_SZ 125; ranks run independent batches (no collective)",
              "e2e": {"value": FP_E2E_SEGS * world / (ms_fp_e2e * 1e-3), "unit": "segments/s", "segments_per_step": FP_E2E_SEGS * world,
                      "h2d_bytes_per_step": FP_E2E_SEGS * 16000, "d2h_bytes_per_step": FP_E2E_SEGS * 512,
                      "through": "nafp_fingerprint_pcm16_host ((n, 8000) int16 rows from pinned host memory; model/generate.py's "
                                 "track-window entry point uploads half as many samples)"},
              "gpu_launches_per_step": int(fp_launches),
              "roofline": {"kernel": "conv_gemm_kernel (encoder, whole step)", "bound": "tensor", "achieved": tfl,
                           "peak": tf_sustained, "unit": "TFLOP/s", "frac": tfl / tf_sustained, "traffic": None,
                           "peak_source": f"{peak_src} (bf16_tflops_sustained, per GPU)"},
              "logmel": {"value": FP_SEGS_PER_STEP / (ms_mel * 1e-3), "unit": "segments/s per GPU", "ms_per_step": ms_mel,
                         "through": "nafp_logmel_forward_raw (logmel_kernel + the 2 us group-maximum fill, as the fused path runs it)",
                         "roofline": {"kernel": "logmel_kernel", "bound": "hbm", "achieved": mel_gbs, "peak": hbm_peak,
                                      "unit": "GB/s", "frac": mel_gbs / hbm_peak, "traffic": mel_traffic,
                                      "traffic_source": mel_file,
                                      "algorithmic_bytes_per_launch": FP_SEGS_PER_STEP * LOGMEL_BYTES_PER_SEGMENT,
                                      "peak_source": f"{peak_src} (MEASURED_PEAKS.json hbm_gbs)",
                                      "note": "~1 MFLOP of fp32 FFT butterflies per segment: the kernel is bound by the FP32 / "
                                              "shared-memory pipes, not by HBM (DESIGN 4.2); it is 6 % of the generation step"}}}
        if world == 1 and not args.no_cpu:
            fp["cpu_baseline"] = cpu_generate()
        del x_dev, emb_dev, mel_dev, x_pin

    # ---- mini scale (BASELINE configs[1]): same job against a 1 M-row database, N = 1 only
    mini = None
    if world == 1 and not args.no_mini and n_dummy > 1_000_000:
        midx = ShardedFlatIndex(1_000_000 + N_DB, 0, 1, max_len=max(SEQ_LENS), device=local_rank)
        build_sharded_index(ctx, torch, midx, 1_000_000, dev)

        def mini_step():
            result["mini"] = midx.seq_match_dev(q_dev, ids_dev, sl_dev, K_PROBE)

        ms_mini = time_steps(torch, dev, mini_step, args.steps, args.warmup, barrier)
        mp = result["mini"][0].cpu().numpy()
        outputs["mini_1M_pred_ids"] = mp.astype(np.float64)
        outputs["mini_1M_pred_scores"] = result["mini"][1].cpu().numpy()
        mini = {"db_rows": 1_000_000 + N_DB, "value": n_queries / (ms_mini * 1e-3), "unit": "queries/s",
                "ms_per_step": ms_mini,
                "top1_hit_rate": [float(100.0 * np.mean(mp[:, si, 0] == test_ids + 1_000_000)) for si in range(len(SEQ_LENS))]}
        del midx

    # ---- IVF-PQ (SURVEY 8 a6, BASELINE configs[4]): the approximate index the reference builds for index_type "ivfpq"
    # (nlist 256, M 64, 8 bit, nprobe 40), host API incl. H2D / D2H
    def ivfpq_leg(rows_dummy, name, keep=False):
        """Index build (k-means on a 1-in-N sample of the dummy rows, encoding of every row) and the timed
        evaluation job through the host API; the database is generated chunk by chunk on the device."""
        from nafp_b200.eval.utils.get_index import IVFPQ, Index
        t_ivf = time.time()
        iidx = Index(IVFPQ, 128, nlist=256, pq_m=64, pq_nbits=8, device=local_rank)
        chunk = min(4_000_000, rows_dummy)
        buf = torch.empty((chunk, 128), dtype=torch.float32, device=dev)
        check(lib.nafp_synth_fp_rows(ctx.h, 11, 0, chunk, 59, 0.5, ctypes.c_void_p(buf.data_ptr())))
        # 100,000 training rows from the first chunk (<= 256 per centroid is what faiss samples anyway)
        train_rows = buf[:: max(1, chunk // 100_000)].contiguous().cpu().numpy()
        iidx.train(train_rows, seed=1234)
        t_train = time.time() - t_ivf
        iidx.reserve(rows_dummy + N_DB)
        r = 0
        while r < rows_dummy:
            n = min(chunk, rows_dummy - r)
            if r:
                check(lib.nafp_synth_fp_rows(ctx.h, 11, r, n, 59, 0.5, ctypes.c_void_p(buf.data_ptr())))
            iidx.add_dev(buf.data_ptr(), n)
            r += n
        iidx.add_dev(dbt.data_ptr(), N_DB)
        iidx.nprobe = 40
        torch.cuda.synchronize(dev)
        t_add = time.time() - t_ivf - t_train
        del buf

        def ivf_step():
            result["ivf"] = iidx.seq_match(query_host, test_ids, sl_host, K_PROBE)

        iidx.last_search_stats()
        ms_ivf = time_steps(torch, dev, ivf_step, args.steps, args.warmup, barrier)
        st = iidx.last_search_stats()
        ip = result["ivf"][0]
        outputs[f"{name}_pred_ids"] = ip.astype(np.float64)
        outputs[f"{name}_pred_scores"] = result["ivf"][1]
        n_run = args.steps + args.warmup             # the statistics cover the warm-up steps too
        tiles = st["reranked"] / n_run               # (for an IVF-PQ index: 128 x 128 tiles of the list-major scan)
        out = {"index": "IVFPQ nlist 256, M 64, 8 bit, nprobe 40", "db_rows": rows_dummy + N_DB,
               "value": n_queries / (ms_ivf * 1e-3), "unit": "queries/s", "ms_per_step": ms_ivf, "train_s": t_train,
               "add_s": t_add,
               "through": "host API (nafp_seq_match: H2D queries, D2H predictions inside the timed region)",
               "path": "list-major compressed-domain tensor-core scan (csrc/ivfpq_lm.cu): codes decoded tile by tile in shared "
                       "memory, bf16 tcgen05 scores, exact fp32 ADC re-rank + proof, LUT kernel for what is not proven",
               "index_bytes_per_row": 76,            # 64 B codes (list order, tile-transposed) + row id + h + list id; the row-order
                                                     # staging copy of the codes is released when the lists are built
               "search_stats_per_step": {"query_rows": st["rows"] / n_run, "rows_answered_by_lut_kernel": st["fallback_rows"] / n_run,
                                         "work_items": st["passes"] / n_run, "tiles_128x128": tiles},
               "mma_tflops_over_whole_step": tiles * 2 * 128 * 128 * 128 / (ms_ivf * 1e-3) / 1e12,
               "top1_hit_rate": [float(100.0 * np.mean(ip[:, si, 0] == test_ids + rows_dummy)) for si in range(len(SEQ_LENS))]}
        if keep:
            return out, iidx, train_rows
        del iidx
        return out

    def ivfpq_oracle_hit_rates(train_rows, rows_dummy):
        """The CPU oracle's IVF-PQ (C restatement, own k-means with the SAME seed and the same seeded training subset)
        on the same 1 M-row database: top-1 hit rates of the same 2,000 x 6 queries, so that "within 0.1 pt" is a number."""
        from oracle import native, seq_match
        t0 = time.time()
        o = native.IVFPQC(128, 256, 64, 8)
        o.train(train_rows, seed=1234)
        dummy_host = torch.empty((rows_dummy, 128), dtype=torch.float32, device=dev)
        check(lib.nafp_synth_fp_rows(ctx.h, 11, 0, rows_dummy, 59, 0.5, ctypes.c_void_p(dummy_host.data_ptr())))
        dummy_np = dummy_host.cpu().numpy()
        del dummy_host
        o.add(dummy_np)
        o.add(db_host)
        o.nprobe = 40
        recon = np.concatenate([dummy_np, db_host])
        raw, pred = seq_match.evaluate(o, query_host, recon, rows_dummy, test_ids, SEQ_LENS, K_PROBE, fast_scores=True,
                                       batch_search=True)
        return {"top1_hit_rate": [float(100.0 * np.mean(pred[:, si, 0] == test_ids + rows_dummy)) for si in range(len(SEQ_LENS))],
                "implementation": "oracle/csrc/oracle.c (k-means, PQ encode, LUT + ADC list scan) + oracle/seq_match.py; "
                                  "trained on the same 100,000 rows with the same seed as the GPU index",
                "cores": native.threads(), "seconds": time.time() - t0}

    def ivfpq_lut_leg(iidx):
        """The kernel north_star names -- per (query row, probed list) a 64 x 256 fp32 look-up table in shared memory and
        an ADC scan of the list's codes (ivfpq_scan_kernel, the fallback of the list-major path) -- timed alone on 256
        query rows of the same 1 M-row index; algorithmic bytes = SURVEY 8(d): 68 B per (query row, probed row)."""
        from nafp_b200.eval.utils.get_index import IVFPQ, Index
        os.environ["NAFP_IVFPQ_PATH"] = "lut"
        try:
            lidx = Index(IVFPQ, 128, nlist=256, pq_m=64, pq_nbits=8, device=local_rank)
        finally:
            del os.environ["NAFP_IVFPQ_PATH"]
        lidx.set_ivfpq_params(*iidx.ivfpq_params())
        rows = 1_000_000
        buf = torch.empty((rows, 128), dtype=torch.float32, device=dev)
        check(lib.nafp_synth_fp_rows(ctx.h, 11, 0, rows, 59, 0.5, ctypes.c_void_p(buf.data_ptr())))
        lidx.add_dev(buf.data_ptr(), rows)
        lidx.add_dev(dbt.data_ptr(), N_DB)
        lidx.nprobe = 40
        del buf
        nq = 256
        qd = q_dev[:nq].contiguous()
        Dd = torch.empty((nq, K_PROBE), dtype=torch.float32, device=dev)
        Id = torch.empty((nq, K_PROBE), dtype=torch.int64, device=dev)

        def lut_step():
            lidx.search_dev(qd.data_ptr(), nq, K_PROBE, Dd.data_ptr(), Id.data_ptr())

        ms = time_steps(torch, dev, lut_step, args.steps, 3, barrier)
        Dl, Il = iidx.search(qd.cpu().numpy(), K_PROBE)
        probed_rows = 40.0 / 256.0 * (rows + N_DB)
        return {"kernel": "ivfpq_scan_kernel (shared-memory LUT ADC scan, one CTA per (query row, probed list))",
                "query_rows": nq, "ms_per_search": ms, "value": nq / (ms * 1e-3), "unit": "query rows/s",
                "algorithmic_GBps": nq * probed_rows * 68 / (ms * 1e-3) / 1e9,
                "lut_lookups_per_s": nq * probed_rows * 64 / (ms * 1e-3),
                "ids_identical_to_list_major_path": bool((Il == Id.cpu().numpy()).all()),
                "distances_identical_to_list_major_path": bool((Dl == Dd.cpu().numpy()).all())}

    ivf = None
    if world == 1 and not args.no_mini and not args.no_ivfpq and n_dummy >= 1_000_000:
        if args.no_cpu:
            ivf, iidx_keep, train_rows = ivfpq_leg(1_000_000, "ivfpq_1M", keep=True)
            ivf["lut_kernel"] = ivfpq_lut_leg(iidx_keep)
            del iidx_keep
        else:
            ivf, iidx_keep, train_rows = ivfpq_leg(1_000_000, "ivfpq_1M", keep=True)
            ivf["lut_kernel"] = ivfpq_lut_leg(iidx_keep)
            del iidx_keep
            orc = ivfpq_oracle_hit_rates(train_rows, 1_000_000)
            ivf["oracle"] = orc
            ivf["top1_hit_rate_minus_oracle_pt"] = [g - o for g, o in zip(ivf["top1_hit_rate"], orc["top1_hit_rate"])]

    # the flat index (43 GB at N = 1) makes room for the full-size IVF-PQ index
    del sidx
    torch.cuda.empty_cache()

    # BASELINE configs[4] at full size: one GPU holds it (4.3 GB of index next to the 28.7 GB of exact rows the sequence
    # scoring reads); N > 1 row-shards it like the flat index (quantizers trained on rank 0 and broadcast, codes / lists
    # local), same all-gather + merge + max all-reduce
    ivf_full = None
    if world == 1 and not args.no_ivfpq_full and n_dummy > 1_000_000:
        ivf_full = ivfpq_leg(n_dummy, "ivfpq_full")
    if world > 1 and not args.no_ivfpq_full:
        from nafp_b200.eval.utils.get_index import IVFPQ
        t_ivf = time.time()
        sivf = ShardedFlatIndex(n_total, rank, world, max_len=max(SEQ_LENS), device=local_rank, comm=comm, index_type=IVFPQ)
        tr = torch.empty((min(4_000_000, n_dummy), 128), dtype=torch.float32, device=dev)
        check(lib.nafp_synth_fp_rows(ctx.h, 11, 0, tr.shape[0], 59, 0.5, ctypes.c_void_p(tr.data_ptr())))
        sivf.train(tr[:: max(1, tr.shape[0] // 100_000)].contiguous().cpu().numpy())
        del tr
        t_train = time.time() - t_ivf
        build_sharded_index(ctx, torch, sivf, n_dummy, dev)
        t_add = time.time() - t_ivf - t_train

        def sivf_step():
            result["sivf"] = sivf.seq_match_dev(q_dev, ids_dev, sl_dev, K_PROBE)

        ms_sivf = max_over_ranks(time_steps(torch, dev, sivf_step, args.steps, args.warmup, barrier))
        sp = result["sivf"][0].cpu().numpy()
        outputs["ivfpq_full_pred_ids"] = sp.astype(np.float64)
        outputs["ivfpq_full_pred_scores"] = result["sivf"][1].cpu().numpy()
        ivf_full = {"index": "IVFPQ nlist 256, M 64, 8 bit, nprobe 40, row-sharded", "db_rows": n_total,
                    "value": n_queries / (ms_sivf * 1e-3), "unit": "queries/s", "ms_per_step": ms_sivf, "train_s": t_train,
                    "add_s": t_add, "through": "device-resident queries (seq_match_dev), NCCL all-gather + max all-reduce",
                    "path": "list-major compressed-domain tensor-core scan (csrc/ivfpq_lm.cu) on every rank's row block",
                    "top1_hit_rate": [float(100.0 * np.mean(sp[:, si, 0] == test_ids + n_dummy)) for si in range(len(SEQ_LENS))]}
        del sivf

    # ---- BASELINE configs[0] as stated: default.yaml, 200 synthetic 30 s tracks, generate + evaluate, seq lens 1 3 5 9 11
    cfg0 = None
    if world == 1 and not args.no_config0:
        cfg0 = config0_leg(ctx, torch, dev, lib, check, cpu=not args.no_cpu)

    # ---- CPU baseline of the headline (rank 0, N = 1)
    cpu = None
    if world == 1 and not args.no_cpu:
        n_big = max(r for r, _ in CPU_FIT)
        big = torch.empty((n_big, 128), dtype=torch.float32, device=dev)           # the device generator is the faster one
        check(lib.nafp_synth_fp_rows(ctx.h, 11, 0, n_big, 59, 0.5, ctypes.c_void_p(big.data_ptr())))
        big_host = big.cpu().numpy()
        del big
        cpu = cpu_search_fit(db_host, query_host, test_ids, n_total, big=big_host)
        del big_host

    if rank == 0:
        line = {"metric": "search_queries_per_s", "value": n_queries / (ms_res * 1e-3), "unit": "queries/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_res,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "bf16 scan, f32 re-rank", "data": "synthetic", "config": _config(args, world),
                "clocks": clocks,
                "e2e": {"value": n_queries / (ms_e2e * 1e-3), "unit": "queries/s", "ms_per_step": ms_e2e,
                        "h2d_bytes_per_step": int(query_host.nbytes + test_ids.nbytes + 4 * len(SEQ_LENS)),
                        "d2h_bytes_per_step": int(len(test_ids) * len(SEQ_LENS) * 10 * 12),
                        "through": e2e_through, "top1_identical_to_resident_path": e2e_same},
                "gpu_launches": int(launches),
                "roofline": roofline, "cpu_baseline": cpu,
                "top1_hit_rate": dict(zip(map(str, SEQ_LENS), top1)),
                "search_stats_per_step": {k: v / args.steps for k, v in stats.items()},
                "fingerprint": fp, "mini_1M": mini, "ivfpq_1M": ivf, "ivfpq_full": ivf_full, "config0": cfg0,
                "db_build_s": t_build}
        if args.dump_outputs:
            dump_outputs(outputs, args.dump_outputs)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def config0_leg(ctx, torch, dev, lib, check, cpu=True, n_tracks=200, n_sec=30, n_ids=500):
    """BASELINE configs[0]: "default.yaml: generate.py fingerprints for 200 synthetic 30 s 8 kHz tracks + eval_faiss
    IndexFlat, test_seq_len 1 3 5 9 11" through the product's host API -- int16 tracks in pinned host memory ->
    nafp_fingerprint_pcm16_tracks_host (the call model/generate.py makes) -> flat index -> nafp_seq_match -- with the CPU
    implementation of both halves timed beside it on a bounded sample (SURVEY 8(d) config 1: db = all 11,800
    fingerprints, query = the same audio + white noise at 5 dB SNR, 500 seeded ids; dummy_db = 100 MORE tracks -- the
    survey's "first 100 tracks" would put an exact copy of half the db in front of it and turn every such query into a
    tie that the lower label wins)."""
    import ctypes
    from nafp_b200.eval.utils.get_index import Index
    from nafp_b200.model import weights as W
    from nafp_b200.model.fp import FingerPrinter
    seq_lens = [1, 3, 5, 9, 11]
    spt = (n_sec * 8000 - 8000 + 4000) // 4000                  # 59 segments per 30 s track (audio_utils.py:173-177)
    n_seg = n_tracks * spt
    # synthetic tracks: n_sec one-second pieces of the device generator back to back, as int16 PCM
    x = torch.empty((n_tracks * n_sec, 8000), dtype=torch.float32, device=dev)
    check(lib.nafp_synth_audio(ctx.h, 1000, 0, n_tracks * n_sec, ctypes.c_void_p(x.data_ptr())))
    clean = x.reshape(n_tracks, n_sec * 8000)
    g = torch.Generator(device=dev)
    g.manual_seed(0)
    p_sig = (clean * clean).mean(1, keepdim=True)
    noisy = clean + torch.randn(clean.shape, device=dev, generator=g) * torch.sqrt(p_sig / (10 ** 0.5))     # 5 dB SNR
    to_pcm = lambda t: (t.clamp(-1.0, 1.0) * 32767.0).round().to(torch.int16).cpu().pin_memory()
    pcm_db, pcm_q = to_pcm(clean), to_pcm(noisy)
    del x, clean, noisy
    seg_off = (np.arange(n_tracks)[:, None] * (n_sec * 8000) + np.arange(spt)[None, :] * 4000).reshape(-1).astype(np.int64)
    seg_valid = np.full(n_seg, 8000, np.int32)
    m_fp = FingerPrinter(ctx).load(W.init_weights(7))

    def gen(pcm):
        return m_fp.fingerprint_tracks(pcm.numpy().reshape(-1), seg_off, seg_valid, group_size=125)

    emb_dummy = gen(pcm_db)[:(n_tracks // 2) * spt]               # warm-up (arena, clocks) ...
    x = torch.empty(((n_tracks // 2) * n_sec, 8000), dtype=torch.float32, device=dev)      # ... and the dummy tracks
    check(lib.nafp_synth_audio(ctx.h, 2000, 0, (n_tracks // 2) * n_sec, ctypes.c_void_p(x.data_ptr())))
    pcm_dummy = to_pcm(x.reshape(n_tracks // 2, n_sec * 8000))
    del x
    n_dummy = (n_tracks // 2) * spt
    emb_dummy = m_fp.fingerprint_tracks(pcm_dummy.numpy().reshape(-1), seg_off[:n_dummy], seg_valid[:n_dummy], group_size=125)
    t0 = time.perf_counter()
    emb_db = gen(pcm_db)
    emb_q = gen(pcm_q)
    ctx.sync()
    sec_gen = time.perf_counter() - t0
    rng = np.random.default_rng(0)
    ids = np.sort(rng.permutation(n_seg - max(seq_lens))[:n_ids]).astype(np.int64)
    index = Index(0, 128, ctx=ctx)
    index.add(emb_dummy)
    index.add(emb_db)
    sl = np.asarray(seq_lens, np.int32)
    index.seq_match(emb_q, ids, sl, K_PROBE)                      # warm-up
    t0 = time.perf_counter()
    pred, _ = index.seq_match(emb_q, ids, sl, K_PROBE)
    sec_eval = time.perf_counter() - t0
    gt = ids + n_dummy
    out = {"workload": f"{n_tracks} synthetic {n_sec} s tracks x 2 (db + noisy query) = {2 * n_seg:,} segments generated, "
                       f"{n_dummy + n_seg:,}-row flat index, {n_ids} ids x lengths {seq_lens}",
           "generate": {"value": 2 * n_seg / sec_gen, "unit": "segments/s", "seconds": sec_gen,
                        "through": "nafp_fingerprint_pcm16_tracks_host (int16 tracks in pinned host memory -> fingerprints on the host)"},
           "evaluate": {"value": n_ids * len(seq_lens) / sec_eval, "unit": "queries/s", "seconds": sec_eval,
                        "through": "nafp_seq_match (host queries in, predictions out)"},
           "top1_hit_rate": [float(100.0 * np.mean(pred[:, si, 0] == gt)) for si in range(len(seq_lens))]}
    if cpu:
        from oracle import native, seq_match
        out["generate"]["cpu_baseline"] = cpu_generate()
        o = native.FlatL2C(128)
        o.add(emb_dummy)
        o.add(emb_db)
        t0 = time.perf_counter()
        _, pred_o = seq_match.evaluate(o, emb_q, o._data(), n_dummy, ids, seq_lens, K_PROBE, fast_scores=True)
        sec_cpu = time.perf_counter() - t0
        out["evaluate"]["cpu_baseline"] = dict(value=n_ids * len(seq_lens) / sec_cpu, unit="queries/s", cores=native.threads(),
                                               kind="port", sample="the whole evaluation job (no sampling needed at this size)")
        out["evaluate"]["predictions_identical_to_cpu"] = float(np.mean(pred[:, :, 0] == pred_o[:, :, 0]))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="nafp", choices=["nafp", "reference"])
    ap.add_argument("--db-rows", type=int, default=N_DUMMY_FULL, help="dummy_db rows (full scale: 56,000,000)")
    ap.add_argument("--no-fp", action="store_true")
    ap.add_argument("--no-mini", action="store_true")
    ap.add_argument("--no-ivfpq", action="store_true")
    ap.add_argument("--no-ivfpq-full", action="store_true", help="skip IVF-PQ on the full-size database (BASELINE configs[4])")
    ap.add_argument("--no-config0", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what each timed path returned in its last step as DIR/<name>.npy (float32 / float64)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU arm")
    args.warmup = max(args.warmup, 3)              # timing rule: at least three warm-up steps
    if args.impl == "reference":
        return run_reference(args)
    return run_gpu(args)


if __name__ == "__main__":
    sys.exit(main())
