"""Host-side handles of the extractor: the reference's ``m_pre`` (``Melspec_layer``,
``model/fp/melspec/melspectrogram.py``) and ``m_fp`` (``FingerPrinter``, ``model/fp/nnfp.py``), as thin
objects over libnafp.  ``build_fp(cfg)`` mirrors ``model/generate.py:16-23``.
"""
from __future__ import annotations

import ctypes

import numpy as np

from .._lib import Context, NafpError, check, lib, ptr
from . import arch
from .weights import init_weights, load_weights

_FP = ctypes.POINTER(ctypes.c_float)
def _check_norm(norm):
    if norm not in arch.NORMS:
        raise NotImplementedError(f"MODEL.BN={norm!r}: one of {arch.NORMS}")


def _check_model_cfg(cfg):
    m = cfg['MODEL']
    fixed = dict(FS=8000, STFT_WIN=1024, STFT_HOP=256, N_MELS=256, EMB_SZ=128)
    for k, v in fixed.items():
        if int(m[k]) != v:
            raise NotImplementedError(f"MODEL.{k}={m[k]}: the B200 kernels are built for {v} (all reference configs)")
    if float(m['DUR']) != 1.0 or float(m['F_MIN']) != 300.0 or float(m['F_MAX']) != 4000.0:
        raise NotImplementedError("MODEL.DUR/F_MIN/F_MAX other than 1 s / 300 Hz / 4000 Hz are not built")
    if m['FEAT'] not in ('melspec', 'melspec_maxnorm'):      # model/generate.py:17-20 raises for anything else, too
        raise NotImplementedError(m['FEAT'])
    _check_norm(m['BN'])


class Melspec:
    """``m_pre``: (B,1,8000) float32 -> (B,256,32,1) float32; rows are grouped in consecutive
    ``group_size`` batches that share the batch-global max (``melspectrogram.py:108``)."""

    def __init__(self, ctx=None, device=0, segment_norm=False):
        self.ctx = ctx or Context.get(device)
        self.segment_norm = bool(segment_norm)       # MODEL.FEAT == 'melspec_maxnorm' (melspectrogram.py:110-111)

    def __call__(self, x, group_size=None):
        x = np.ascontiguousarray(x, dtype=np.float32)
        if x.size != len(x) * 8000:
            raise ValueError("expected (B, 1, 8000) segments")
        x = x.reshape(len(x), 8000)
        n = x.shape[0]
        g = int(group_size) if group_size else max(n, 1)
        out = np.empty((n, 256, 32, 1), dtype=np.float32)
        if n == 0:
            return out
        xd = self.ctx.malloc(x.nbytes)
        od = self.ctx.malloc(out.nbytes)
        try:
            self.ctx.h2d(xd, x)
            check(lib.nafp_logmel_set_segment_norm(self.ctx.h, int(self.segment_norm)))
            check(lib.nafp_logmel_forward(self.ctx.h, xd, n, g, od))
            self.ctx.d2h(out, od)
            self.ctx.sync()
        finally:
            self.ctx.free(xd)
            self.ctx.free(od)
        return out


class FingerPrinter:
    """``m_fp`` (+ the fused ``test_step``).  Weights live on the device after ``load``; ``norm`` is MODEL.BN
    (``FingerPrinter(norm=...)``, nnfp.py:186) and decides which normalisation variables ``load`` expects."""

    def __init__(self, ctx=None, device=0, segment_norm=False, norm='layer_norm2d'):
        _check_norm(norm)
        self.ctx = ctx or Context.get(device)
        self.loaded = False
        self.segment_norm = bool(segment_norm)       # feature variant of the fused test_step entry points
        self.norm = norm

    def load(self, weights):
        specs = arch.conv_specs()
        keep = []

        def arr(name, shape):
            a = np.ascontiguousarray(weights[name], dtype=np.float32)
            if a.shape != tuple(shape):
                raise ValueError(f"weight {name}: shape {a.shape}, expected {tuple(shape)}")
            keep.append(a)
            return a.ctypes.data_as(_FP)

        cw, cb, lg, lb, lm, lv = [(_FP * 16)() for _ in range(6)]
        for l, s in enumerate(specs):
            kshape = (1, 3, s.c_in, s.c_out) if s.axis == "t" else (3, 1, s.c_in, s.c_out)
            ln = s.name.replace("conv", "ln")
            cw[l] = arr(f"{s.name}_w", kshape)
            cb[l] = arr(f"{s.name}_b", (s.c_out,))
            shapes = arch.norm_shapes(s, self.norm)
            lg[l] = arr(f"{ln}_g", shapes["g"])
            lb[l] = arr(f"{ln}_b", shapes["b"])
            if self.norm == 'batch_norm':
                lm[l] = arr(f"{ln}_mean", shapes["mean"])
                lv[l] = arr(f"{ln}_var", shapes["var"])
        div = (arr("div_w1", (128, 8, 32)), arr("div_b1", (128, 32)), arr("div_w2", (128, 32, 1)), arr("div_b2", (128, 1)))
        if self.norm == 'layer_norm2d':
            check(lib.nafp_weights_load(self.ctx.h, cw, cb, lg, lb, *div))
        else:
            bn = self.norm == 'batch_norm'
            check(lib.nafp_weights_load_norm(self.ctx.h, arch.NORMS.index(self.norm), cw, cb, lg, lb, lm if bn else None,
                                             lv if bn else None, *div))
        self.loaded = True
        return self

    def __call__(self, mel):
        """(B,256,32,1) float32 log-mel -> (B,128) unit-norm fingerprints."""
        mel = np.ascontiguousarray(mel, dtype=np.float32).reshape(len(mel), -1)
        if mel.shape[1] != 8192:
            raise ValueError("expected (B, 256, 32, 1) log-mel input")
        n = mel.shape[0]
        emb = np.empty((n, 128), dtype=np.float32)
        if n == 0:
            return emb
        md = self.ctx.malloc(mel.nbytes)
        ed = self.ctx.malloc(emb.nbytes)
        try:
            self.ctx.h2d(md, mel)
            check(lib.nafp_encoder_forward(self.ctx.h, md, n, ed))
            self.ctx.d2h(emb, ed)
            self.ctx.sync()
        finally:
            self.ctx.free(md)
            self.ctx.free(ed)
        return emb

    def fingerprint(self, x, group_size):
        """Fused ``m_fp(m_pre(X))`` on host buffers: float32 (B,1,8000) or int16 PCM (B,8000)."""
        x = np.asarray(x)
        n = x.shape[0]
        emb = np.empty((n, 128), dtype=np.float32)
        if n == 0:
            return emb
        if x.dtype == np.int16:
            x = np.ascontiguousarray(x).reshape(n, -1)
            fn = lib.nafp_fingerprint_pcm16_host
        else:
            x = np.ascontiguousarray(x, dtype=np.float32).reshape(n, -1)
            fn = lib.nafp_fingerprint_host
        if x.shape[1] != 8000:
            raise ValueError("expected 8000-sample segments")
        check(lib.nafp_logmel_set_segment_norm(self.ctx.h, int(self.segment_norm)))
        check(fn(self.ctx.h, ptr(x), n, int(group_size), ptr(emb)))
        return emb

    def fingerprint_tracks(self, pcm, seg_off, seg_valid, group_size):
        """``fingerprint`` for segments given as windows of whole-track int16 sample runs
        (``SegmentSequence.get_track_block``): the overlapping segments are cut on the GPU."""
        pcm = np.ascontiguousarray(pcm, dtype=np.int16)
        seg_off = np.ascontiguousarray(seg_off, dtype=np.int64)
        seg_valid = np.ascontiguousarray(seg_valid, dtype=np.int32)
        n = len(seg_off)
        if len(seg_valid) != n:
            raise ValueError("seg_off and seg_valid differ in length")
        emb = np.empty((n, 128), dtype=np.float32)
        if n == 0:
            return emb
        check(lib.nafp_logmel_set_segment_norm(self.ctx.h, int(self.segment_norm)))
        check(lib.nafp_fingerprint_pcm16_tracks_host(self.ctx.h, ptr(pcm), len(pcm), ptr(seg_off), ptr(seg_valid), n,
                                                     int(group_size), ptr(emb)))
        return emb

    def fingerprint_sources(self, pcm, seg_off, seg_valid, runs, group_size):
        """``fingerprint_tracks`` for source files at any rate and channel count (``SegmentSequence.get_source_block``):
        one launch resamples the runs to 8 kHz int16 on the GPU, which the segments then index."""
        pcm = np.ascontiguousarray(pcm, dtype=np.int16)
        runs = np.ascontiguousarray(runs, dtype=np.int64).reshape(-1, 7)
        seg_off = np.ascontiguousarray(seg_off, dtype=np.int64)
        seg_valid = np.ascontiguousarray(seg_valid, dtype=np.int32)
        n = len(seg_off)
        if len(seg_valid) != n:
            raise ValueError("seg_off and seg_valid differ in length")
        emb = np.empty((n, 128), dtype=np.float32)
        check(lib.nafp_logmel_set_segment_norm(self.ctx.h, int(self.segment_norm)))
        check(lib.nafp_fingerprint_pcm16_sources_host(self.ctx.h, ptr(pcm), len(pcm), ptr(runs), len(runs), ptr(seg_off),
                                                      ptr(seg_valid), n, int(group_size), ptr(emb)))
        return emb

    def fingerprint_block(self, block, group_size):
        """Fingerprints of a ``SegmentSequence.get_source_block`` block: blocks of 8 kHz mono files take the
        ``fingerprint_tracks`` path, any other through ``fingerprint_sources``."""
        pcm, seg_off, seg_valid, runs = block
        if runs is None:
            return self.fingerprint_tracks(pcm, seg_off, seg_valid, group_size)
        return self.fingerprint_sources(pcm, seg_off, seg_valid, runs, group_size)

    def activation(self, layer, n_seg):
        """Activation (n_seg, F, T, C) of conv ``layer`` after its normalisation, from the last encoder pass."""
        s = arch.conv_specs()[layer]
        out = np.empty((n_seg, s.f_out, s.t_out, s.c_out), dtype=np.float32)
        check(lib.nafp_encoder_activation_host(self.ctx.h, int(layer), int(n_seg), ptr(out)))
        return out


def build_fp(cfg, device=0):
    """(m_pre, m_fp) -- ``model/generate.py:16-23``."""
    _check_model_cfg(cfg)
    ctx = Context.get(device)
    seg_norm = cfg['MODEL']['FEAT'] == 'melspec_maxnorm'
    return Melspec(ctx, segment_norm=seg_norm), FingerPrinter(ctx, segment_norm=seg_norm, norm=cfg['MODEL']['BN'])


def test_step(X, m_pre, m_fp, group_size=None):
    """``model/generate.py:83-88``: one batch -> (BSZ, 128); the batch is one max-normalisation group."""
    n = len(X)
    return m_fp.fingerprint(X, group_size or max(n, 1))
