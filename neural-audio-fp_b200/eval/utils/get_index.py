"""Index factory: the reference's ``get_index`` (``eval/utils/get_index_faiss.py:10-121``) over
libnafp instead of faiss.

``get_index(index_type, train_data, train_data_shape, use_gpu, max_nitem_train)`` returns an object
with the faiss surface the reference uses: ``train(x)``, ``add(x)``, ``ntotal``, ``nprobe``
(attribute), ``search(q, k) -> (D, I)`` (squared-L2 ascending, int64 labels, -1 padding),
``reconstruct_n(i0, n)``.  Built: 'l2', 'ivfpq' (the hot path), 'ivf' (IndexIVFFlat, nlist 400) and 'ivfpq-rr'
(IndexIVFPQR).  'ivfpq-ondisk' and 'hnsw' raise NotImplementedError("... only available in CPU"), which is what the
reference does for them whenever use_gpu is set (``get_index_faiss.py:86-98``).
"""
from __future__ import annotations

import ctypes
import time

import numpy as np

from ..._lib import Context, NafpError, check, lib, ptr

FLAT_L2, IVFPQ, IVF_FLAT, IVFPQR = 0, 1, 2, 3
_ADD_CHUNK = 1 << 20      # rows per host->device copy (memmaps are read chunk by chunk)
CLIP_MAXL = 4096          # rows of one clip (34 min at the 0.5 s hop), include/nafp.h
CLIP_NTOP = 100           # best matches per clip, at most
CLIP_CALL_ROWS = 1 << 16  # query rows per nafp_clip_match call: bounds its device workspace (~0.4 GB at k_probe 128)


def _f32c(x):
    return np.ascontiguousarray(x, dtype=np.float32)


class Index:
    """Device-resident index (nafp_index)."""

    def __init__(self, index_type=FLAT_L2, d=128, nlist=256, pq_m=64, pq_nbits=8, device=0, ctx=None):
        self.ctx = ctx or Context.get(device)
        self.d = int(d)
        self.index_type = index_type
        self.nlist, self.pq_m = int(nlist), int(pq_m)
        h = ctypes.c_void_p()
        check(lib.nafp_index_create(self.ctx.h, int(index_type), int(d), int(nlist), int(pq_m), int(pq_nbits),
                                    ctypes.byref(h)))
        self.h = h
        self._nprobe = 1

    def __del__(self):
        h = getattr(self, "h", None)
        if h:
            lib.nafp_index_destroy(h)
            self.h = None

    # ---- faiss-like surface
    @property
    def ntotal(self):
        return int(lib.nafp_index_ntotal(self.h))

    @property
    def is_trained(self):
        return bool(lib.nafp_index_is_trained(self.h))

    @property
    def nprobe(self):
        return self._nprobe

    @nprobe.setter
    def nprobe(self, v):
        check(lib.nafp_index_set_nprobe(self.h, int(v)))
        self._nprobe = int(v)

    def train(self, x, seed=1234):
        x = _f32c(x)
        check(lib.nafp_index_train(self.h, ptr(x), x.shape[0], int(seed)))

    def ivfpq_params(self):
        """(coarse (nlist,128), pq (M,256,128/M)) of a trained IVF-PQ index."""
        coarse = np.empty((self.nlist, 128), np.float32)
        pq = np.empty((self.pq_m, 256, 128 // self.pq_m), np.float32)
        check(lib.nafp_index_ivfpq_get_params(self.h, ptr(coarse), ptr(pq)))
        return coarse, pq

    def ivfpqr_refine(self):
        """(4, 16, 32) refinement codebooks of a trained IVFPQR index."""
        rpq = np.empty((4, 16, 32), np.float32)
        check(lib.nafp_index_ivfpqr_get_refine(self.h, ptr(rpq)))
        return rpq

    def set_ivfpqr_refine(self, rpq):
        rpq = _f32c(rpq)
        if rpq.shape != (4, 16, 32):
            raise ValueError("expected (4, 16, 32) refinement codebooks")
        check(lib.nafp_index_ivfpqr_set_refine(self.h, ptr(rpq)))

    def ivf_coarse(self):
        """(nlist,128) coarse centroids of a trained IVF-Flat / IVF-PQ index."""
        coarse = np.empty((self.nlist, 128), np.float32)
        check(lib.nafp_index_ivf_get_coarse(self.h, ptr(coarse)))
        return coarse

    def set_ivf_coarse(self, coarse):
        coarse = _f32c(coarse)
        if coarse.shape != (self.nlist, 128):
            raise ValueError(f"expected ({self.nlist}, 128) centroids")
        check(lib.nafp_index_ivf_set_coarse(self.h, ptr(coarse)))

    def set_ivfpq_params(self, coarse, pq):
        coarse, pq = _f32c(coarse), _f32c(pq)
        check(lib.nafp_index_ivfpq_set_params(self.h, ptr(coarse), ptr(pq)))

    def reserve(self, n_total):
        check(lib.nafp_index_reserve(self.h, int(n_total)))

    def add(self, x):
        n = len(x)
        if n and np.ndim(x) != 2 or (n and x.shape[1] != self.d):
            raise ValueError(f"add: expected (n, {self.d}) rows")
        self.reserve(self.ntotal + n)
        for s in range(0, n, _ADD_CHUNK):
            blk = _f32c(x[s:s + _ADD_CHUNK])
            check(lib.nafp_index_add(self.h, ptr(blk), blk.shape[0]))

    def add_dev(self, dev_ptr, n):
        check(lib.nafp_index_add_dev(self.h, ctypes.c_void_p(dev_ptr), int(n)))

    def search_dev(self, q_dev_ptr, nq, k, D_dev_ptr, I_dev_ptr):
        """Device-pointer search, asynchronous on the context stream."""
        check(lib.nafp_index_search_dev(self.h, ctypes.c_void_p(q_dev_ptr), int(nq), int(k),
                                        ctypes.c_void_p(D_dev_ptr), ctypes.c_void_p(I_dev_ptr)))

    def search(self, q, k):
        q = _f32c(q)
        if q.ndim != 2 or q.shape[1] != self.d:
            raise ValueError(f"search: expected (nq, {self.d}) queries")
        nq = q.shape[0]
        D = np.empty((nq, k), dtype=np.float32)
        I = np.empty((nq, k), dtype=np.int64)
        check(lib.nafp_index_search(self.h, ptr(q), nq, int(k), ptr(D), ptr(I)))
        return D, I

    def reconstruct_n(self, i0, n):
        out = np.empty((int(n), self.d), dtype=np.float32)
        check(lib.nafp_index_reconstruct_host(self.h, int(i0), int(n), ptr(out)))
        return out

    # ---- extensions
    def set_label_offset(self, off):
        check(lib.nafp_index_set_label_offset(self.h, int(off)))

    def set_search_rows(self, n):
        check(lib.nafp_index_set_search_rows(self.h, int(n)))

    def last_search_stats(self):
        out = np.zeros(8, dtype=np.int64)
        check(lib.nafp_index_last_search_stats(self.h, out.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))))
        return dict(rows=int(out[0]), fallback_rows=int(out[1]), passes=int(out[2]), reranked=int(out[3]),
                    fallback_overflow=int(out[5]), fallback_bound=int(out[6]))

    def profile_scans(self, enable=True):
        """(total ms, launches) of the scan kernel since the previous call; arms / disarms the timer."""
        ms = ctypes.c_double()
        n = ctypes.c_int64()
        check(lib.nafp_index_profile_scans(self.h, int(bool(enable)), ctypes.byref(ms), ctypes.byref(n)))
        return float(ms.value), int(n.value)

    def seq_match(self, query, test_ids, seq_lens, k_probe=20):
        """Batched body of the reference's evaluation loop (``eval/eval_faiss.py:204-232``).
        Returns pred_ids (n_test, n_len, 10) int64 (-1 padded) and their scores."""
        query = _f32c(query)
        test_ids = np.ascontiguousarray(test_ids, dtype=np.int64)
        seq_lens = np.ascontiguousarray(seq_lens, dtype=np.int32)
        n_test, n_len = len(test_ids), len(seq_lens)
        pred = np.full((n_test, n_len, 10), -1, dtype=np.int64)
        scores = np.full((n_test, n_len, 10), -np.inf, dtype=np.float32)
        check(lib.nafp_seq_match(self.h, ptr(query), query.shape[0], ptr(test_ids), n_test, ptr(seq_lens), n_len,
                                 int(k_probe), ptr(pred), ptr(scores)))
        return pred, scores

    def clip_match(self, rows, clip_off, k_probe=20, n_top=10):
        """Identify clips: clip i is ``rows[clip_off[i]:clip_off[i+1]]`` (1..CLIP_MAXL consecutive segment
        fingerprints); every clip is matched as one sequence of its own length (``nafp_clip_match``).
        Returns pred_ids (n_clips, n_top) int64 -- start rows of the best-matching sequences, -1 padded -- and their
        scores (float32, -inf padded).  Clips are sent in calls of at most CLIP_CALL_ROWS rows."""
        rows = _f32c(rows)
        clip_off = np.ascontiguousarray(clip_off, dtype=np.int64)
        if rows.ndim != 2 or rows.shape[1] != self.d:
            raise ValueError(f"clip_match: expected (n, {self.d}) rows")
        if clip_off.ndim != 1 or len(clip_off) < 1 or clip_off[0] != 0 or clip_off[-1] != len(rows):
            raise ValueError("clip_match: clip_off must run from 0 to len(rows)")
        n_clips = len(clip_off) - 1
        pred = np.full((n_clips, n_top), -1, dtype=np.int64)
        scores = np.full((n_clips, n_top), -np.inf, dtype=np.float32)
        c0 = 0
        while c0 < n_clips:
            c1 = c0 + 1               # as many whole clips as fit in one call (one clip always goes)
            while c1 < n_clips and clip_off[c1 + 1] - clip_off[c0] <= CLIP_CALL_ROWS:
                c1 += 1
            off = clip_off[c0:c1 + 1] - clip_off[c0]
            q = rows[clip_off[c0]:clip_off[c1]]
            p = np.empty((c1 - c0, n_top), dtype=np.int64)
            s = np.empty((c1 - c0, n_top), dtype=np.float32)
            check(lib.nafp_clip_match(self.h, ptr(q), len(q), ptr(off), c1 - c0, int(k_probe), int(n_top), ptr(p),
                                      ptr(s)))
            pred[c0:c1], scores[c0:c1] = p, s
            c0 = c1
        return pred, scores


def get_index(index_type, train_data, train_data_shape, use_gpu=True, max_nitem_train=2e7, device=0, seed=None):
    """Same contract as the reference factory.  ``use_gpu=False`` is refused: this build has no CPU
    path (the reference's ``--nogpu`` would run faiss-cpu)."""
    if not use_gpu:
        raise NafpError("use_gpu=False: nafp-b200 has no CPU search path (no fallback by design)")
    d = int(train_data_shape[1])
    mode = index_type.lower()
    print(f'Creating index: \033[93m{mode}\033[0m')
    if mode == 'l2':
        index = Index(FLAT_L2, d, device=device)
    elif mode == 'ivfpq':
        # reference: code_sz 64, n_centroids 256, nbits 8 (get_index_faiss.py:69-74)
        index = Index(IVFPQ, d, nlist=256, pq_m=64, pq_nbits=8, device=device)
    elif mode == 'ivf':
        # reference: IndexIVFFlat, nlist 400 (get_index_faiss.py:63-66)
        index = Index(IVF_FLAT, d, nlist=400, device=device)
    elif mode == 'ivfpq-rr':
        # reference: IndexIVFPQR, code_sz 64, n_centroids 256, nbits 8, M_refine 4, nbits_refine 4 (get_index_faiss.py:75-85)
        index = Index(IVFPQR, d, nlist=256, pq_m=64, pq_nbits=8, device=device)
    elif mode in ('ivfpq-ondisk', 'hnsw'):
        # get_index_faiss.py:86-98: both raise under use_gpu, and this build has no CPU path
        raise NotImplementedError(f'{mode} is only available in CPU.')
    else:
        raise ValueError(mode)

    start_time = time.time()
    max_nitem_train = int(max_nitem_train)
    if len(train_data) > max_nitem_train:
        print('Training index using {:>3.2f} % of data...'.format(100. * max_nitem_train / len(train_data)))
        rng = np.random.default_rng(seed)
        sel = np.sort(rng.permutation(len(train_data))[:max_nitem_train])
        index.train(train_data[sel, :])
    else:
        print('Training index...')
        if mode != 'l2':
            index.train(train_data)
    print('Elapsed time: {:.2f} seconds.'.format(time.time() - start_time))
    index.nprobe = 40
    return index
