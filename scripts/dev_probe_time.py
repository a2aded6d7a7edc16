"""Developer probe: in-kernel timestamps of the flat scan (ns since the CTA started)."""
import ctypes, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from nafp_b200._lib import Context, check, lib, ptr
from nafp_b200.eval.utils.get_index import Index

n = int(sys.argv[1]) if len(sys.argv) > 1 else 1_000_000
nq = int(sys.argv[2]) if len(sys.argv) > 2 else 200
ctx = Context.get(0)
dev = torch.device("cuda", 0)
torch.cuda.set_stream(torch.cuda.ExternalStream(ctx.stream, device=dev))
idx = Index(0, 128); idx.reserve(n + 29500)
buf = torch.empty((min(n, 4_000_000), 128), dtype=torch.float32, device=dev)
r = 0
while r < n:
    m = min(4_000_000, n - r)
    check(lib.nafp_synth_fp_rows(ctx.h, 11, r, m, 59, 0.5, ctypes.c_void_p(buf.data_ptr()))); idx.add_dev(buf.data_ptr(), m); r += m
check(lib.nafp_synth_fp_rows(ctx.h, 13, 0, 29500, 59, 0.5, ctypes.c_void_p(buf.data_ptr()))); idx.add_dev(buf.data_ptr(), 29500)
q = torch.nn.functional.normalize(buf[:29500][torch.arange(nq, device=dev) * 23 % 29500] + 0.03 * torch.randn((nq, 128), device=dev), dim=1).contiguous()
D = torch.empty((nq, 20), dtype=torch.float32, device=dev); I = torch.empty((nq, 20), dtype=torch.int64, device=dev)
idx.search_dev(q.data_ptr(), nq, 20, D.data_ptr(), I.data_ptr()); torch.cuda.synchronize()
g = ctypes.c_int32(); check(lib.nafp_index_debug_enable(idx.h, None, None, ctypes.byref(g))); G = g.value
for rep in range(2):
    idx.search_dev(q.data_ptr(), nq, 20, D.data_ptr(), I.data_ptr()); torch.cuda.synchronize()
    cnt = np.zeros((G, 512), np.int32); first = np.zeros((G, 512), np.int32)
    check(lib.nafp_index_debug_enable(idx.h, ptr(cnt), ptr(first), None))
    t = first[:, 504:512]
    print("rep", rep, "G", G, "ns since start: tile0 done / thresholds ok / first thresholded tile done / own tiles done / end / item 16 done / item 32 done / item 96 done")
    print(" median", np.median(t, 0).tolist(), " min", t.min(0).tolist(), " max", t.max(0).tolist())
    print(" survivors per CTA-query: mean", cnt[:, :nq].sum() / (nq * G // 2), "max", cnt[:, :nq].max())   # G / 2 CTAs hold each row
    own = t[:, 3]
    order = np.argsort(own)
    print(" own-tiles-done ns by CTA (sorted): fastest", [(int(c), int(own[c])) for c in order[:6]], "slowest", [(int(c), int(own[c])) for c in order[-10:]])
    print(" survivors per CTA (sum over queries): slowest", [int(cnt[c, :nq].sum()) for c in order[-10:]], "fastest", [int(cnt[c, :nq].sum()) for c in order[:6]], "corr", float(np.corrcoef(own, cnt[:, :nq].sum(1))[0, 1]))
