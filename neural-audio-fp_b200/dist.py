"""Row-sharded database across the GPUs of one node (SURVEY §8 e).

One process per GPU (``torch.distributed``, NCCL over NVLink).  The database [dummy_db; db] is split
into contiguous row blocks; rank r additionally keeps a copy of the ``halo`` rows that follow its
block (max sequence length - 1), so every candidate sequence that STARTS in its block can be scored
locally.  Queries are replicated.  Per batch of test ids:

    local top-k per query row  ->  all-gather (W, rows, k)  ->  merge to the global top-k
    ->  every rank scores the candidates it owns (-inf elsewhere)  ->  max all-reduce  ->  top-10

The two collectives move k*12 bytes per query row per rank and 4 bytes per candidate score; they are
the only exchange steps of the path.  An index with a second level (IVFPQR, ``ops.refine``) exchanges twice
before the candidates are scored: the merged first-level top-kc (kc = 4k) is re-ranked by every rank over the
labels it owns, and the per-rank top-k are all-gathered and merged again, which gives exactly the answer of one
index over all rows.  The orchestration below is backend-agnostic (``ops`` does the
local work, ``comm`` the collectives) so that the host logic is testable with gloo on CPU.
"""
from __future__ import annotations

import ctypes

import numpy as np

SEQ_MAXC = 1024
N_PRED = 10


def shard_bounds(n_total, rank, world):
    """Contiguous, balanced row block [lo, hi) of rank ``rank``."""
    per, rem = divmod(int(n_total), int(world))
    lo = rank * per + min(rank, rem)
    return lo, lo + per + (1 if rank < rem else 0)


def shard_with_halo(n_total, rank, world, halo):
    lo, hi = shard_bounds(n_total, rank, world)
    return lo, hi, min(hi + int(halo), int(n_total))


class TorchComm:
    """The two collectives of the path on torch tensors (NCCL on GPU, gloo on CPU)."""

    def __init__(self, group=None):
        import torch.distributed as dist
        self.dist = dist
        self.group = group
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)

    def all_gather(self, t):
        import torch
        out = torch.empty((self.world,) + tuple(t.shape), dtype=t.dtype, device=t.device)
        self.dist.all_gather_into_tensor(out.view(-1), t.contiguous().view(-1), group=self.group) \
            if t.is_cuda else self.dist.all_gather(list(out.unbind(0)), t.contiguous(), group=self.group)
        return out

    def all_reduce_max(self, t):
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX, group=self.group)
        return t

    def broadcast(self, t, src=0):
        """Quantizers of an IVF index trained on rank ``src`` (not on the search path)."""
        self.dist.broadcast(t, src=src, group=self.group)
        return t


def sharded_seq_match(ops, comm, query, test_ids, seq_lens, k_probe):
    """Backend-agnostic orchestration; see the module docstring.  ``query`` is the whole query set
    (every rank holds it); returns (pred_ids, pred_scores)."""
    plan = ops.plan(query, test_ids)               # unique query rows + (test id, offset) -> row map
    D_loc, I_loc = ops.local_topk(plan.qrows, k_probe)        # (with ops.refine: the first level's top-kc)
    if comm is not None:
        D_all = comm.all_gather(D_loc)
        I_all = comm.all_gather(I_loc)
        _, I = ops.merge(D_all, I_all)
    else:
        I = I_loc
    if hasattr(ops, "refine"):
        D_loc, I_loc = ops.refine(plan.qrows, I, k_probe)
        if comm is not None:
            _, I = ops.merge(comm.all_gather(D_loc), comm.all_gather(I_loc))
        else:
            I = I_loc
    cand_ids, cand_scores, n_cand = ops.cand_scores(query, plan, test_ids, seq_lens, k_probe, I)
    if comm is not None:
        # a test id has at most k_probe x max_len distinct candidates (380 of the table's 1,024 columns at k_probe 20,
        # length 19): only that part of the score table is live and crosses NVLink (18 instead of 49 MB per step)
        live = getattr(ops, "live_candidates", lambda k: cand_scores.shape[-1])(k_probe)
        if live < cand_scores.shape[-1]:
            part = cand_scores[..., :live].contiguous()
            cand_scores[..., :live] = comm.all_reduce_max(part)
        else:
            cand_scores = comm.all_reduce_max(cand_scores)
    return ops.top(cand_ids, cand_scores, n_cand, len(seq_lens))


class SeqPlan:
    """Overlapping query sequences share rows: ``qrows`` (n_uniq, d) are the distinct query rows the
    test ids need, ``rowmap`` (n_test*max_len) maps (test id, offset) to its row of ``qrows`` (-1 past
    the end of the query set)."""

    def __init__(self, qrows, rowmap, uniq_rows):
        self.qrows, self.rowmap, self.uniq_rows = qrows, rowmap, uniq_rows


class GpuOps:
    """Local work of ``sharded_seq_match`` on this rank's GPU through the C ABI (torch CUDA tensors
    carry the memory; libnafp runs on torch's current stream)."""

    def __init__(self, index, n_query_rows, n_rows_global, owned_lo, owned_hi, max_len):
        import torch
        from ._lib import check, lib
        self.torch, self.lib, self.check = torch, lib, check
        self.index = index
        self.n_query_rows = int(n_query_rows)
        self.n_rows_global = int(n_rows_global)
        self.owned = (int(owned_lo), int(owned_hi))
        self.max_len = int(max_len)
        self.dev = torch.device('cuda', index.ctx.device)
        # torch work (allocations, copies, NCCL, events) must be ordered with libnafp's kernels: make
        # the library's stream torch's current stream (torch's default stream handle is 0, which the
        # C ABI cannot adopt, so the adoption goes this way round)
        self.stream = torch.cuda.ExternalStream(index.ctx.stream, device=self.dev)
        torch.cuda.set_stream(self.stream)

    def _p(self, t):
        return ctypes.c_void_p(t.data_ptr())

    def plan(self, q_dev, test_ids_dev):
        t = self.torch
        n_test = test_ids_dev.numel()
        pairs = n_test * self.max_len
        scratch = t.empty((2 * self.n_query_rows + 1,), dtype=t.int32, device=self.dev)
        rowmap = t.empty((pairs,), dtype=t.int32, device=self.dev)
        uniq = t.empty((max(pairs, 1),), dtype=t.int32, device=self.dev)
        n_uniq = ctypes.c_int64(0)
        self.check(self.lib.nafp_seq_plan_dev(self.index.ctx.h, self._p(test_ids_dev), n_test, self.max_len,
                                              self.n_query_rows, self._p(scratch), self._p(rowmap), self._p(uniq),
                                              ctypes.byref(n_uniq)))
        n_uniq = int(n_uniq.value)
        qrows = t.empty((n_uniq, 128), dtype=t.float32, device=self.dev)
        self.check(self.lib.nafp_seq_gather_rows_dev(self.index.ctx.h, self._p(q_dev), self._p(uniq), n_uniq, self._p(qrows)))
        return SeqPlan(qrows, rowmap, uniq[:n_uniq])

    def local_topk(self, qrows, k):
        n = qrows.shape[0]
        D = self.torch.empty((n, k), dtype=self.torch.float32, device=self.dev)
        I = self.torch.empty((n, k), dtype=self.torch.int64, device=self.dev)
        self.check(self.lib.nafp_index_search_dev(self.index.h, self._p(qrows), n, k, self._p(D), self._p(I)))
        return D, I

    def merge(self, D_all, I_all):
        W, n, k = D_all.shape
        D = self.torch.empty((n, k), dtype=self.torch.float32, device=self.dev)
        I = self.torch.empty((n, k), dtype=self.torch.int64, device=self.dev)
        self.check(self.lib.nafp_topk_merge_dev(self.index.ctx.h, self._p(D_all), self._p(I_all), W, n, k, self._p(D), self._p(I)))
        return D, I

    def cand_scores(self, q_dev, plan, test_ids_dev, seq_lens_dev, k, I):
        n_test, n_len = test_ids_dev.numel(), seq_lens_dev.numel()
        cid = self.torch.empty((n_test, SEQ_MAXC), dtype=self.torch.int64, device=self.dev)
        csc = self.torch.empty((n_test, n_len, SEQ_MAXC), dtype=self.torch.float32, device=self.dev)
        nc = self.torch.empty((n_test,), dtype=self.torch.int32, device=self.dev)
        self.check(self.lib.nafp_seq_cand_dev(self.index.h, self._p(q_dev), self.n_query_rows, self._p(test_ids_dev), n_test,
                                              self._p(seq_lens_dev), n_len, self.max_len, k, self._p(I),
                                              self._p(plan.rowmap), self.n_rows_global,
                                              self.owned[0], self.owned[1], self._p(cid), self._p(csc), self._p(nc)))
        return cid, csc, nc

    def live_candidates(self, k):
        """Columns of the candidate tables that can hold a candidate: k results per query row x max_len rows."""
        return min(SEQ_MAXC, -(-k * self.max_len // 64) * 64)

    def top(self, cand_ids, cand_scores, n_cand, n_len):
        n_test = cand_ids.shape[0]
        pid = self.torch.empty((n_test, n_len, N_PRED), dtype=self.torch.int64, device=self.dev)
        psc = self.torch.empty((n_test, n_len, N_PRED), dtype=self.torch.float32, device=self.dev)
        self.check(self.lib.nafp_seq_top_dev(self.index.ctx.h, n_test, n_len, self._p(cand_ids), self._p(cand_scores),
                                             self._p(n_cand), self._p(pid), self._p(psc)))
        return pid, psc


class GpuRefineOps(GpuOps):
    """``GpuOps`` of an IVFPQR shard: ``local_topk`` returns the first level's top 4k, ``refine`` re-ranks the merged
    candidates this rank owns."""

    K_FACTOR = 4                    # faiss IndexIVFPQR.k_factor

    def local_topk(self, qrows, k):
        n, kc = qrows.shape[0], k * self.K_FACTOR
        D = self.torch.empty((n, kc), dtype=self.torch.float32, device=self.dev)
        I = self.torch.empty((n, kc), dtype=self.torch.int64, device=self.dev)
        self.check(self.lib.nafp_index_ivfpqr_first_level_dev(self.index.h, self._p(qrows), n, kc, self._p(D), self._p(I)))
        return D, I

    def refine(self, qrows, cand_I, k):
        n, kc = cand_I.shape
        cand_I = cand_I.contiguous()
        D = self.torch.empty((n, k), dtype=self.torch.float32, device=self.dev)
        I = self.torch.empty((n, k), dtype=self.torch.int64, device=self.dev)
        self.check(self.lib.nafp_index_ivfpqr_rerank_dev(self.index.h, self._p(qrows), n, self._p(cand_I), kc, k,
                                                         self._p(D), self._p(I)))
        return D, I


class ShardedFlatIndex:
    """Rank-local block (+ halo) of a row-sharded index and the collective sequence matcher.

    ``index_type`` FLAT_L2 (default), IVFPQ, IVF_FLAT or IVFPQR (``eval/utils/get_index.py``).  The IVF types shard
    their codes / lists by the same row blocks with the quantizers replicated (SURVEY §8 e, the equivalent of
    faiss.IndexShards over one trained index): ``train`` runs on rank 0 and the centroids / codebooks (IVFPQR: also
    the refinement codebooks) are broadcast, after which every rank adds its own rows.  IVFPQR re-ranks in a second
    exchange (``GpuRefineOps``), so its answers equal one index's, unlike faiss.IndexShards over IVFPQR shards."""

    def __init__(self, n_rows_global, rank, world, max_len=19, device=None, comm=None, index_type=0, nlist=None,
                 pq_m=64, pq_nbits=8):
        from .eval.utils.get_index import FLAT_L2, IVF_FLAT, IVFPQ, IVFPQR, Index
        self.rank, self.world = int(rank), int(world)
        self.n_rows_global = int(n_rows_global)
        self.max_len = int(max_len)
        self.index_type = int(index_type)
        self.lo, self.hi, self.hi_halo = shard_with_halo(n_rows_global, rank, world, max_len - 1)
        if nlist is None:
            nlist = 400 if self.index_type == IVF_FLAT else 256          # get_index_faiss.py:65,71
        self.index = Index(self.index_type, 128, nlist=nlist, pq_m=pq_m, pq_nbits=pq_nbits,
                           device=self.rank if device is None else device)
        self._ivf = self.index_type in (IVFPQ, IVF_FLAT, IVFPQR)
        self._ivfpq = self.index_type in (IVFPQ, IVFPQR)
        self._refine = self.index_type == IVFPQR
        if not self._ivf:
            self.index.reserve(self.hi_halo - self.lo)
        self.index.set_label_offset(self.lo)
        self.comm = comm
        self._ops = None

    def train(self, x, seed=1234, nprobe=40):
        """IVF types: k-means on rank 0, quantizers broadcast to the other ranks (no-op for the flat index)."""
        if not self._ivf:
            return
        import torch
        if self.rank == 0:
            self.index.train(x, seed=seed)
        if self.world > 1 and self.comm is None:
            raise ValueError("a row-sharded IVF index needs a communicator (comm=TorchComm()) to share its quantizers")
        if self.world > 1:
            dev = torch.device('cuda', self.index.ctx.device) if torch.cuda.is_available() else torch.device('cpu')
            coarse = torch.empty((self.index.nlist, 128), dtype=torch.float32, device=dev)
            pq = torch.empty((self.index.pq_m, 256, 128 // self.index.pq_m), dtype=torch.float32, device=dev) if self._ivfpq else None
            rpq = torch.empty((4, 16, 32), dtype=torch.float32, device=dev) if self._refine else None
            if self.rank == 0:
                if self._ivfpq:
                    c, p = self.index.ivfpq_params()
                    pq.copy_(torch.from_numpy(p))
                else:
                    c = self.index.ivf_coarse()
                coarse.copy_(torch.from_numpy(c))
                if self._refine:
                    rpq.copy_(torch.from_numpy(self.index.ivfpqr_refine()))
            self.comm.broadcast(coarse, 0)
            if self._ivfpq:
                self.comm.broadcast(pq, 0)
            if self._refine:
                self.comm.broadcast(rpq, 0)
            if self.rank != 0:
                if self._refine:
                    self.index.set_ivfpqr_refine(rpq.cpu().numpy())
                if self._ivfpq:
                    self.index.set_ivfpq_params(coarse.cpu().numpy(), pq.cpu().numpy())
                else:
                    self.index.set_ivf_coarse(coarse.cpu().numpy())
        self.index.reserve(self.hi_halo - self.lo)
        self.index.nprobe = nprobe

    @property
    def ntotal(self):
        return self.n_rows_global

    def local_rows_needed(self):
        """Global row range [lo, hi_halo) this rank must add, in order."""
        return self.lo, self.hi_halo

    def add_local(self, x):
        self.index.add(x)
        self._finish_if_complete()

    def add_local_dev(self, dev_ptr, n):
        self.index.add_dev(dev_ptr, n)
        self._finish_if_complete()

    def _finish_if_complete(self):
        if self.index.ntotal == self.hi_halo - self.lo:
            self.index.set_search_rows(self.hi - self.lo)

    def add_from(self, parts):
        """``parts``: row-indexable arrays (e.g. the dummy_db and db memmaps) forming the global database."""
        base = 0
        for p in parts:
            n = len(p)
            a, b = max(self.lo, base), min(self.hi_halo, base + n)
            if a < b:
                self.index.add(p[a - base:b - base])
            base += n
        assert base == self.n_rows_global, (base, self.n_rows_global)
        self._finish_if_complete()

    def ops(self, n_query_rows):
        if self._ops is None or self._ops.n_query_rows != n_query_rows:
            cls = GpuRefineOps if self._refine else GpuOps
            self._ops = cls(self.index, n_query_rows, self.n_rows_global, self.lo, self.hi, self.max_len)
        return self._ops

    def seq_match_dev(self, q_dev, test_ids_dev, seq_lens_dev, k_probe=20):
        """Everything on device tensors (torch); returns device tensors."""
        ops = self.ops(q_dev.shape[0])
        comm = self.comm if (self.world > 1 or self.comm is not None) else None
        return sharded_seq_match(ops, comm, q_dev, test_ids_dev, seq_lens_dev, k_probe)

    def seq_match(self, query, test_ids, seq_lens, k_probe=20):
        """Host arrays in, host arrays out (includes H2D / D2H)."""
        import torch
        dev = torch.device('cuda', self.index.ctx.device)
        query = np.ascontiguousarray(query, dtype=np.float32)
        if not query.flags.writeable:          # read-only memmaps: torch wants a writable buffer
            query = query.copy()
        q = torch.from_numpy(query).to(dev, non_blocking=True)
        ids = torch.from_numpy(np.ascontiguousarray(test_ids, dtype=np.int64)).to(dev, non_blocking=True)
        sl = torch.from_numpy(np.ascontiguousarray(seq_lens, dtype=np.int32)).to(dev, non_blocking=True)
        pid, psc = self.seq_match_dev(q, ids, sl, k_probe)
        return pid.cpu().numpy(), psc.cpu().numpy()


ShardedIndex = ShardedFlatIndex      # the class serves every index type; the old name stays for its callers
