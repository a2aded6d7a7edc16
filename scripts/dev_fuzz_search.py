"""Developer fuzz of the flat search against the fp64 oracle: random sizes, query counts, k, norms, ragged adds."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import numpy as np
from util import assert_topk_matches
from nafp_b200.eval.utils.get_index import Index
from oracle.flat_index import FlatL2

rng = np.random.default_rng(int(sys.argv[1]) if len(sys.argv) > 1 else 0)
n_cases = int(sys.argv[2]) if len(sys.argv) > 2 else 25
for case in range(n_cases):
    n = int(rng.integers(8200, 260000))
    nq = int(rng.choice([1, 2, 31, 32, 33, 127, 128, 129, 255, 256, 257, 300, 511, 512, 513, 600, 1100]))
    k = int(rng.choice([1, 5, 20, 33, 64]))
    x = rng.standard_normal((n, 128)).astype(np.float32)
    mode = case % 3
    if mode == 0:
        x /= np.linalg.norm(x, axis=1, keepdims=True)
    elif mode == 1:
        x *= rng.uniform(0.5, 1.5, (n, 1)).astype(np.float32)
    else:
        x /= np.linalg.norm(x, axis=1, keepdims=True)
        x[rng.integers(0, n, 50)] = 0.0
    q = x[rng.integers(0, n, nq)] * rng.uniform(0.8, 1.2) + 0.3 / 128 ** 0.5 * rng.standard_normal((nq, 128)).astype(np.float32)
    cuts = np.unique(np.concatenate([[0, n], rng.integers(0, n, 3)]))
    g = Index(0, 128)
    for a, b in zip(cuts[:-1], cuts[1:]):
        g.add(x[a:b])
    o = FlatL2(128)
    o.add(x)
    Dg, Ig = g.search(q, k)
    Do, Io = o.search(q, k)
    assert_topk_matches(Dg, Ig, Do, Io, x, q, dtol=3e-3 if mode == 1 else 1e-4)
    st = g.last_search_stats()
    print(f"case {case}: n={n} nq={nq} k={k} mode={mode} ok  passes={st['passes']} fallback={st['fallback_rows']}", flush=True)
print("fuzz ok")
