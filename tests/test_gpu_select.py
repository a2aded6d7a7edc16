"""GPU: the selection rules every search shares (csrc/topk.cuh and the coarse probe) checked directly: the top-k merge
at its key limit, and the lower-id tie rule of the coarse quantizer in `add` and in `search`."""
import numpy as np
import pytest
from util import assert_topk_matches

pytestmark = pytest.mark.gpu

MERGE_KEYS = 4096         # keys one merge block sorts (TOPK_MERGE_KEYS)


def _merge(ctx, D_all, I_all):
    from nafp_b200._lib import check, lib
    W, nq, k = D_all.shape
    bufs = [ctx.malloc(D_all.nbytes), ctx.malloc(I_all.nbytes), ctx.malloc(nq * k * 4), ctx.malloc(nq * k * 8)]
    try:
        ctx.h2d(bufs[0], D_all)
        ctx.h2d(bufs[1], I_all)
        check(lib.nafp_topk_merge_dev(ctx.h, bufs[0], bufs[1], W, nq, k, bufs[2], bufs[3]))
        D = np.empty((nq, k), np.float32)
        I = np.empty((nq, k), np.int64)
        ctx.d2h(D, bufs[2])
        ctx.d2h(I, bufs[3])
        ctx.sync()
        return D, I
    finally:
        for b in bufs:
            ctx.free(b)


def test_topk_merge_at_the_key_limit_orders_by_distance_then_label(ctx):
    """W * k = 4096 per-shard entries per row, many equal distances, shards padded with (+inf, -1): the merge returns
    the k smallest by (distance, label), padding last, exactly as numpy's lexsort does."""
    rng = np.random.default_rng(41)
    W, k, nq = 32, MERGE_KEYS // 32, 3
    D_all = rng.integers(0, 40, (W, nq, k)).astype(np.float32) * 0.25          # few distinct values: ties everywhere
    I_all = rng.permutation(10 * W * nq * k)[:W * nq * k].reshape(W, nq, k).astype(np.int64)
    pad = rng.random((W, nq, k)) < 0.2
    pad[:, 2, :] = True
    pad[5, 2, :3] = False                        # row 2: three real entries, the rest of its answer is padding
    D_all[pad] = np.inf
    I_all[pad] = -1
    D, I = _merge(ctx, D_all, I_all)
    for q in range(nq):
        d, i = D_all[:, q, :].reshape(-1), I_all[:, q, :].reshape(-1)
        real = i >= 0
        order = np.lexsort((i[real], d[real]))[:k]
        want_D = np.full(k, np.inf, np.float32)
        want_I = np.full(k, -1, np.int64)
        want_D[:len(order)] = d[real][order]
        want_I[:len(order)] = i[real][order]
        np.testing.assert_array_equal(I[q], want_I)
        np.testing.assert_array_equal(D[q], want_D)
    assert (I[2, :3] >= 0).all() and (I[2, 3:] == -1).all() and np.isinf(D[2, 3:]).all()


def test_topk_merge_refuses_more_keys_than_one_block_sorts(ctx):
    from nafp_b200._lib import NafpError
    D_all = np.zeros((1, 1, MERGE_KEYS + 1), np.float32)
    I_all = np.zeros((1, 1, MERGE_KEYS + 1), np.int64)
    with pytest.raises(NafpError):
        _merge(ctx, D_all, I_all)


@pytest.mark.parametrize("nlist", [200, 400])       # the shared-memory probe (nlist <= 256) and the global one
def test_ivf_flat_add_and_search_break_centroid_ties_alike(nlist):
    """Duplicated coarse centroids: the stored rows nearest a duplicated pair are equally near both copies.  `add` and
    `search` both send such a row to the LOWER list id, so a copy of it searched with nprobe = 1 finds itself at rank 0,
    distance 0 -- both through the flat scan + filter (k <= 32) and through the exact list scan (k > 32).  The answers
    also equal the oracle's id for id, outside ties of the oracle's own distances."""
    from nafp_b200.eval.utils.get_index import IVF_FLAT, Index
    from oracle.ivf_flat_index import IVFFlat
    rng = np.random.default_rng(nlist)
    coarse = rng.standard_normal((nlist, 128)).astype(np.float32)
    lo = rng.choice(nlist // 2, 16, replace=False)
    hi = nlist // 2 + rng.choice(nlist // 2, 16, replace=False)
    coarse[hi] = coarse[lo]                                                  # 16 duplicated pairs, copies at higher ids
    near = np.repeat(lo, 12)                                                 # 12 stored rows next to every pair
    rows_near = coarse[near] + 0.05 * rng.standard_normal((len(near), 128)).astype(np.float32)
    rows_far = coarse[rng.integers(0, nlist, 4000)] + 0.3 * rng.standard_normal((4000, 128)).astype(np.float32)
    x = np.concatenate([rows_far[:2000], rows_near, rows_far[2000:]]).astype(np.float32)
    ids = np.arange(2000, 2000 + len(rows_near))
    idx = Index(IVF_FLAT, 128, nlist=nlist)
    idx.set_ivf_coarse(coarse)
    idx.add(x)
    idx.nprobe = 1
    o = IVFFlat(128, nlist)
    o.set_coarse(coarse)
    o.add(x)
    o.nprobe = 1
    q = x[ids]
    s = float((q * q).sum(1).max())       # rows are not unit-norm here: rounding and ties scale with |q|^2
    for k in (10, 40):
        D, I = idx.search(q, k)
        np.testing.assert_array_equal(I[:, 0], ids)
        if k > 32:                                   # exact list scan: sum of (q - x)^2
            assert (D[:, 0] == 0).all()
        else:
            assert (D[:, 0] <= 2e-5 * s).all()
        oD, oI = o.search(q, k)
        assert_topk_matches(D, I, oD, oI, x, q, tie=1e-6 * s, dtol=2e-5 * s)
