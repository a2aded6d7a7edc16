"""Developer helper: fingerprint error against the fp64 oracle (max |err|, rms, min cosine) and throughput of the
encoder.  usage: dev_encoder_err.py [n_segments]"""
import ctypes, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from nafp_b200 import synth
from nafp_b200._lib import Context, lib, check
from nafp_b200.model import weights as W, fp as FP
from oracle import fingerprinter as ofp, melspec

n = int(sys.argv[1]) if len(sys.argv) > 1 else 120
ctx = Context.get(0)
out = []
for wseed, affine in ((7, True), (11, True), (7, False)):
    w = W.init_weights(wseed, randomize_affine=affine)
    m_fp = FP.FingerPrinter(ctx).load(w)
    tr = np.concatenate([synth.synth_track(20 + i).astype(np.float32) / 32768.0 for i in range(3)])
    x = np.stack([tr[i * 4000:i * 4000 + 8000] for i in range(n)])[:, None, :]
    emb = m_fp.fingerprint(x, group_size=40)
    ref = ofp.fingerprinter(melspec.melspec_layer(x, group_size=40), w)
    err = np.abs(emb - ref)
    out.append((wseed, affine, float(err.max()), float(np.sqrt((err ** 2).mean())), float((emb * ref).sum(1).min())))
xd = ctx.malloc(4000 * 32000)
check(lib.nafp_synth_audio(ctx.h, 5, 0, 4000, xd))
ed = ctx.malloc(4000 * 512)
for _ in range(3):
    check(lib.nafp_fingerprint(ctx.h, xd, 4000, 125, ed))
ms = ctypes.c_float()
check(lib.nafp_timer_start(ctx.h))
for _ in range(10):
    check(lib.nafp_fingerprint(ctx.h, xd, 4000, 125, ed))
check(lib.nafp_timer_stop(ctx.h, ctypes.byref(ms)))
print(f"{4000 / (ms.value / 10) * 1e3:,.0f} seg/s; " +
      "; ".join(f"w{s}{'a' if a else ''}: max {mx:.2e} rms {r:.2e} cos {c:.7f}" for s, a, mx, r, c in out))
