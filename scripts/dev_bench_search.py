"""Developer micro-benchmark of the flat scan (not the contract bench): device-resident queries."""
import sys, os, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from nafp_b200 import synth
from nafp_b200._lib import Context
from nafp_b200.eval.utils.get_index import Index

n = int(sys.argv[1]) if len(sys.argv) > 1 else 1000000
ctx = Context.get(0)
t0 = time.time(); dummy = synth.synth_fp_db(n, seed=11); db = synth.synth_fp_db(29500, 11, start_track=n // 59 + 2)
query = synth.synth_fp_queries(db, 12); print("synth", time.time() - t0)
idx = Index(0, 128); idx.add(dummy); idx.add(db)
N = idx.ntotal
for nq in (19, 64, 128, 247, 256, 512, 1024):
    q = np.concatenate([query[i * 59: i * 59 + 19] for i in range(60)])[:nq]
    qd = ctx.malloc(q.nbytes); ctx.h2d(qd, q)
    Dd = ctx.malloc(nq * 20 * 4); Id = ctx.malloc(nq * 20 * 8)
    for _ in range(3): idx.search_dev(qd.value, nq, 20, Dd.value, Id.value)
    ctx.sync(); idx.last_search_stats()
    reps = 20
    ctx.timer_start()
    for _ in range(reps): idx.search_dev(qd.value, nq, 20, Dd.value, Id.value)
    ms = ctx.timer_stop() / reps
    st = idx.last_search_stats()
    passes = (nq + 511) // 512
    print(f"N={N} nq={nq}: {ms*1e3:.1f} us/search  scan-bytes {N*256*passes/ms/1e6:.0f} GB/s-equivalent  "
          f"{nq/ms*1e3:.0f} rows/s  {2*nq*N*128/ms/1e9:.1f} TFLOP/s stats/rep={ {k: v/reps for k, v in st.items()} }")

from nafp_b200._lib import lib, check, ptr
for nq in (19, 256, 512):
    q = np.concatenate([query[i * 59: i * 59 + 19] for i in range(60)])[:nq]
    D, I = idx.search(q, 20)
    fl = np.zeros(512, np.int32); th = np.zeros(512, np.float32); tot = np.zeros(512, np.int32)
    check(lib.nafp_index_debug_last_pass(idx.h, ptr(fl), ptr(th), ptr(tot)))
    print("nq", nq, "flags", fl[:nq].tolist())
    print("thr", np.round(th[:nq], 3).tolist()[:64])
    print("tot", tot[:nq].tolist()[:64])
    print("s20", np.round(0.5 - 0.5 * D[:nq, 19] - 0.0, 3).tolist()[:64])
