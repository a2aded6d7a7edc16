import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, ctypes
from nafp_b200 import synth
from nafp_b200._lib import Context, lib, check, ptr
from nafp_b200.eval.utils.get_index import Index
n = int(sys.argv[1]) if len(sys.argv) > 1 else 1000000
ctx = Context.get(0)
dummy = synth.synth_fp_db(n, seed=11); db = synth.synth_fp_db(29500, 11, start_track=n // 59 + 2); query = synth.synth_fp_queries(db, 12)
idx = Index(0, 128); idx.add(dummy); idx.add(db)
for nq in (512, 256, 32):
    q = np.concatenate([query[i * 59: i * 59 + 19] for i in range(60)])[:nq]
    idx.search(q, 20)
    g = ctypes.c_int32()
    check(lib.nafp_index_debug_enable(idx.h, None, None, ctypes.byref(g)))
    G = g.value
    idx.search(q, 20)
    cnt = np.zeros((G, 512), np.int32); first = np.zeros((G, 512), np.int32)
    check(lib.nafp_index_debug_enable(idx.h, ptr(cnt), ptr(first), None))
    np.set_printoptions(linewidth=250)
    print("nq", nq, "G", G)
    for qq in (0, 5, 31, 32, 40, 100, 200, 255, 256, 511):
        if qq >= nq: continue
        print(" q", qq, "first-thr tile hist", np.bincount(np.clip(first[:, qq], -1, 12) + 1, minlength=14).tolist(), "cnt hist(0,1-8,9-64,65-127,128)",
              [(cnt[:, qq] == 0).sum(), ((cnt[:, qq] > 0) & (cnt[:, qq] <= 8)).sum(), ((cnt[:, qq] > 8) & (cnt[:, qq] <= 64)).sum(), ((cnt[:, qq] > 64) & (cnt[:, qq] < 128)).sum(), (cnt[:, qq] >= 128).sum()])
    print(" cta0 first", first[0, :nq].tolist()[:80])
    print(" cta100 first", first[100, :nq].tolist()[:80])
