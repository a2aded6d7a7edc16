"""world_size-2 gloo test of the row-sharded IVFPQR ('ivfpq-rr') orchestration of nafp_b200.dist.sharded_seq_match: the
first level's per-rank top 4k are merged, every rank re-ranks the merged candidates it owns, the per-rank top-k are
merged again.  The rank-local work is done by a numpy stand-in built on oracle.ivfpq_index.IVFPQR; the result must
equal the unsharded oracle's evaluation."""
import os
import socket

import numpy as np
import pytest

from nafp_b200 import synth
from nafp_b200.dist import TorchComm, sharded_seq_match
from oracle import seq_match
from oracle.ivfpq_index import IVFPQ, IVFPQR
from test_dist_gloo import SEQ_LENS, TEST_IDS, CpuOps

N_DUMMY, N_DB, K, NLIST, M, NPROBE = 3000, 590, 20, 16, 16, 4


def _oracle_params(x):
    o = IVFPQR(128, NLIST, M, 8)
    o.train(x[:3000], seed=11)
    return o.coarse, o.pq, o.rpq


def _oracle_index(params, rows):
    o = IVFPQR(128, NLIST, M, 8)
    o.set_params(params[0], params[1])
    o.set_refine(params[2])
    o.add(rows)
    o.nprobe = NPROBE
    return o


class RefineCpuOps(CpuOps):
    """CpuOps with the IVFPQR contracts of nafp_b200.dist.GpuRefineOps: ``local_topk`` returns the first level's top 4k
    of the rank's searched rows, ``refine`` re-ranks the merged candidates whose labels the rank owns."""

    def __init__(self, x_all, rank, world, query, params):
        super().__init__(x_all, rank, world, query)
        self.index = _oracle_index(params, self.x[:self.hi - self.lo])

    def local_topk(self, qrows, k):
        D, I = IVFPQ.search(self.index, qrows.numpy(), k * IVFPQR.K_FACTOR)      # the first level alone
        I = np.where(I >= 0, I + self.lo, -1)
        return self.torch.from_numpy(D), self.torch.from_numpy(I)

    def refine(self, qrows, cand_I, k):
        q, cand = qrows.numpy(), cand_I.numpy()
        o = self.index
        D = np.full((len(q), k), np.inf, np.float32)
        I = np.full((len(q), k), -1, np.int64)
        for i in range(len(q)):
            ids = cand[i][(cand[i] >= self.lo) & (cand[i] < self.hi)]
            if len(ids) == 0:
                continue
            loc = ids - self.lo
            rec = o.reconstruct(loc) + o.rpq[np.arange(o.M_REFINE)[None, :], o.rcodes[loc]].reshape(len(loc), o.d)
            d = ((q[i][None] - rec) ** 2).sum(1, dtype=np.float32)
            order = np.lexsort((ids, d))[:k]
            D[i, :len(order)] = d[order]
            I[i, :len(order)] = ids[order]
        return self.torch.from_numpy(D), self.torch.from_numpy(I)


def _worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    dummy, db, query = synth.synth_search_set(N_DUMMY, N_DB, seed=8)
    params = _oracle_params(dummy)
    ops = RefineCpuOps(np.concatenate([dummy, db]), rank, world, query, params)
    pred, _ = sharded_seq_match(ops, TorchComm(), query, TEST_IDS, SEQ_LENS, K)
    if rank == 0:
        np.save(out, pred)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.timeout(600)
def test_two_rank_sharded_ivfpqr_match_equals_unsharded_oracle(tmp_path):
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    out = str(tmp_path / "pred.npy")
    mp.spawn(_worker, args=(2, port, out), nprocs=2, join=True)
    pred = np.load(out)
    dummy, db, query = synth.synth_search_set(N_DUMMY, N_DB, seed=8)
    x_all = np.concatenate([dummy, db])
    idx = _oracle_index(_oracle_params(dummy), x_all)
    _, ref = seq_match.evaluate(idx, query, x_all, N_DUMMY, TEST_IDS, SEQ_LENS, K)
    np.testing.assert_array_equal(pred, ref)
    assert (pred[:, :, 0] == (TEST_IDS + N_DUMMY)[:, None]).mean() > 0.5       # the index finds the query segments
