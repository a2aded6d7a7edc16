"""ctypes binding of libnafp.so (the C ABI in include/nafp.h).

There is no CPU fallback: importing this module without the built library, or creating a
context without a B200, raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int, c_int16, c_int32, c_int64, c_void_p

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NAFP_LIBRARY") or os.path.join(_HERE, "csrc", "libnafp.so")   # override: A/B builds


class NafpError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise NafpError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). There is no CPU fallback for the hot path.")
    return ctypes.CDLL(LIB_PATH)


lib = _load()

_fp = POINTER(c_float)
_i64p = POINTER(c_int64)
_i32p = POINTER(c_int32)
_vpp = POINTER(c_void_p)

_SIGS = {
    "nafp_version": (c_int, []),
    "nafp_last_error": (c_char_p, []),
    "nafp_device_count": (c_int, []),
    "nafp_ctx_create": (c_int, [c_int, _vpp]),
    "nafp_ctx_destroy": (c_int, [c_void_p]),
    "nafp_sync": (c_int, [c_void_p]),
    "nafp_ctx_set_stream": (c_int, [c_void_p, c_void_p]),
    "nafp_ctx_stream": (c_void_p, [c_void_p]),
    "nafp_ctx_launch_count": (c_int64, [c_void_p]),
    "nafp_malloc": (c_int, [c_void_p, c_int64, _vpp]),
    "nafp_free": (c_int, [c_void_p, c_void_p]),
    "nafp_malloc_host": (c_int, [c_void_p, c_int64, _vpp]),
    "nafp_free_host": (c_int, [c_void_p, c_void_p]),
    "nafp_memcpy_h2d": (c_int, [c_void_p, c_void_p, c_void_p, c_int64]),
    "nafp_memcpy_d2h": (c_int, [c_void_p, c_void_p, c_void_p, c_int64]),
    "nafp_timer_start": (c_int, [c_void_p]),
    "nafp_timer_stop": (c_int, [c_void_p, _fp]),
    "nafp_synth_fp_rows": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_int32, c_float, c_void_p]),
    "nafp_synth_audio": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_void_p]),
    "nafp_weights_load": (c_int, [c_void_p, POINTER(_fp), POINTER(_fp), POINTER(_fp), POINTER(_fp), _fp, _fp, _fp, _fp]),
    "nafp_weights_load_norm": (c_int, [c_void_p, c_int32, POINTER(_fp), POINTER(_fp), POINTER(_fp), POINTER(_fp), POINTER(_fp),
                                       POINTER(_fp), _fp, _fp, _fp, _fp]),
    "nafp_logmel_forward": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p]),
    "nafp_logmel_forward_raw": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
    "nafp_logmel_set_segment_norm": (c_int, [c_void_p, c_int32]),
    "nafp_encoder_forward": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "nafp_fingerprint": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p]),
    "nafp_fingerprint_host": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p]),
    "nafp_fingerprint_pcm16_host": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p]),
    "nafp_fingerprint_pcm16_tracks_host": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_int64, c_void_p]),
    "nafp_resample_pcm16_dev": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int32, c_int32, c_int32, c_int64, c_int64,
                                        c_void_p]),
    "nafp_fingerprint_pcm16_sources_host": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_int64,
                                                    c_int64, c_void_p]),
    "nafp_encoder_activation_host": (c_int, [c_void_p, c_int, c_int64, c_void_p]),
    "nafp_index_create": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, _vpp]),
    "nafp_index_destroy": (c_int, [c_void_p]),
    "nafp_index_train": (c_int, [c_void_p, c_void_p, c_int64, c_int64]),
    "nafp_index_add": (c_int, [c_void_p, c_void_p, c_int64]),
    "nafp_index_add_dev": (c_int, [c_void_p, c_void_p, c_int64]),
    "nafp_index_ivfpq_get_params": (c_int, [c_void_p, c_void_p, c_void_p]),
    "nafp_index_ivfpq_set_params": (c_int, [c_void_p, c_void_p, c_void_p]),
    "nafp_index_ivfpqr_get_refine": (c_int, [c_void_p, c_void_p]),
    "nafp_index_ivfpqr_set_refine": (c_int, [c_void_p, c_void_p]),
    "nafp_index_ivfpqr_first_level_dev": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    "nafp_index_ivfpqr_rerank_dev": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "nafp_index_ivf_get_coarse": (c_int, [c_void_p, c_void_p]),
    "nafp_index_ivf_set_coarse": (c_int, [c_void_p, c_void_p]),
    "nafp_index_reserve": (c_int, [c_void_p, c_int64]),
    "nafp_index_ntotal": (c_int64, [c_void_p]),
    "nafp_index_is_trained": (c_int, [c_void_p]),
    "nafp_index_set_nprobe": (c_int, [c_void_p, c_int]),
    "nafp_index_set_label_offset": (c_int, [c_void_p, c_int64]),
    "nafp_index_set_search_rows": (c_int, [c_void_p, c_int64]),
    "nafp_index_search": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    "nafp_index_search_dev": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    "nafp_index_reconstruct_host": (c_int, [c_void_p, c_int64, c_int64, c_void_p]),
    "nafp_index_last_search_stats": (c_int, [c_void_p, _i64p]),
    "nafp_index_profile_scans": (c_int, [c_void_p, c_int, POINTER(ctypes.c_double), _i64p]),
    "nafp_seq_match": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int32, c_int32, c_void_p, c_void_p]),
    "nafp_seq_plan_dev": (c_int, [c_void_p, c_void_p, c_int64, c_int32, c_int64, c_void_p, c_void_p, c_void_p, _i64p]),
    "nafp_seq_gather_rows_dev": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "nafp_seq_cand_dev": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int32, c_int32, c_int32,
                                  c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_void_p, c_void_p]),
    "nafp_seq_top_dev": (c_int, [c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "nafp_clip_match": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_int32, c_int32, c_void_p, c_void_p]),
    "nafp_clip_match_dev": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_int32, c_int32, c_void_p, c_void_p]),
    "nafp_topk_merge_dev": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_int64, c_int32, c_void_p, c_void_p]),
    "nafp_pairwise_dists_host": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int64, c_int32, c_int32, c_void_p]),
    "nafp_conv_eye_host": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int32, c_void_p]),
    "nafp_mini_search_host": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int64, c_void_p, c_int32, c_int32,
                                      c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
}
for _name, (_res, _args) in _SIGS.items():
    _f = getattr(lib, _name)
    _f.restype = _res
    _f.argtypes = _args

EXPORTS = tuple(_SIGS)


def check(status):
    if status != 0:
        msg = lib.nafp_last_error()
        raise NafpError(f"libnafp status {status}: {msg.decode(errors='replace') if msg else ''}")


def ptr(a):
    """Raw pointer of a C-contiguous numpy array (or None)."""
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(c_void_p)


class Context:
    """One per (process, GPU).  Mirrors nafp_ctx."""
    _cache = {}

    def __init__(self, device=0):
        h = c_void_p()
        check(lib.nafp_ctx_create(int(device), ctypes.byref(h)))
        self.h = h
        self.device = int(device)

    @classmethod
    def get(cls, device=0):
        if device not in cls._cache:
            cls._cache[device] = cls(device)
        return cls._cache[device]

    def sync(self):
        check(lib.nafp_sync(self.h))

    def set_stream(self, cuda_stream_ptr):
        check(lib.nafp_ctx_set_stream(self.h, c_void_p(cuda_stream_ptr) if cuda_stream_ptr else None))

    @property
    def stream(self):
        return lib.nafp_ctx_stream(self.h)

    @property
    def launches(self):
        return int(lib.nafp_ctx_launch_count(self.h))

    def malloc(self, nbytes):
        p = c_void_p()
        check(lib.nafp_malloc(self.h, int(nbytes), ctypes.byref(p)))
        return p

    def free(self, p):
        check(lib.nafp_free(self.h, p))

    def h2d(self, dst, src_np):
        check(lib.nafp_memcpy_h2d(self.h, dst, ptr(src_np), src_np.nbytes))

    def d2h(self, dst_np, src):
        check(lib.nafp_memcpy_d2h(self.h, ptr(dst_np), src, dst_np.nbytes))

    def timer_start(self):
        check(lib.nafp_timer_start(self.h))

    def timer_stop(self):
        ms = c_float()
        check(lib.nafp_timer_stop(self.h, ctypes.byref(ms)))
        return float(ms.value)


def device_count():
    n = lib.nafp_device_count()
    return max(n, 0)
