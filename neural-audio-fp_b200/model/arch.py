"""Geometry of the FingerPrinter encoder (host side).

Mirrors the constructor defaults of the reference's ``FingerPrinter``
(``model/fp/nnfp.py:186-222``): eight separable ConvLayers (1x3 then 3x1, TF 'SAME' padding)
with channels ``:193`` and strides ``:194-197``, followed by the divide-and-encode head.
Everything the CUDA library needs to size its buffers is derived here and passed through the
C ABI as plain integers.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Tuple

HIDDEN_CH = (128, 128, 256, 256, 512, 512, 1024, 1024)
# (stride of the 1x3 conv, stride of the 3x1 conv), each as (freq, time)
STRIDES = (((1, 2), (2, 1)), ((1, 2), (2, 1)), ((1, 2), (2, 1)), ((1, 2), (2, 1)),
           ((1, 1), (2, 1)), ((1, 2), (2, 1)), ((1, 1), (2, 1)), ((1, 2), (2, 1)))
EMB_SZ = 128
DIVENC_UNITS = (32, 1)
LN_EPS = 1e-3
L2_EPS = 1e-12
# MODEL.BN (nnfp.py:20-83, ConvLayer(norm=...)): LayerNormalization over (F,T,C), LayerNormalization over C, or
# BatchNormalization over C (inference mode); eps 1e-3 for all three (Keras defaults)
NORMS = ("layer_norm2d", "layer_norm1d", "batch_norm")


def norm_shapes(spec: "ConvSpec", norm: str = "layer_norm2d") -> dict:
    """Variables of the normalisation after conv ``spec``: suffix -> shape (``g``, ``b``; ``mean``, ``var`` for
    batch_norm -- Keras' moving statistics)."""
    if norm not in NORMS:
        raise ValueError(f"norm {norm!r}: one of {NORMS}")
    if norm == "layer_norm2d":
        shp = (spec.f_out, spec.t_out, spec.c_out)
        return {"g": shp, "b": shp}
    out = {"g": (spec.c_out,), "b": (spec.c_out,)}
    if norm == "batch_norm":
        out.update(mean=(spec.c_out,), var=(spec.c_out,))
    return out


def tf_same(n_in: int, k: int, s: int) -> Tuple[int, int, int]:
    """TensorFlow 'SAME' output size and (lo, hi) padding for one axis."""
    n_out = (n_in + s - 1) // s
    total = max((n_out - 1) * s + k - n_in, 0)
    return n_out, total // 2, total - total // 2


@dataclass(frozen=True)
class ConvSpec:
    name: str
    axis: str               # 't' for the 1x3 conv, 'f' for the 3x1 conv
    stride: int             # stride along ``axis``
    pad_lo: int
    f_in: int
    t_in: int
    c_in: int
    f_out: int
    t_out: int
    c_out: int

    @property
    def m_per_seg(self) -> int:
        return self.f_out * self.t_out

    @property
    def k(self) -> int:
        return 3 * self.c_in

    @property
    def flops_per_seg(self) -> int:
        return 2 * self.m_per_seg * self.c_out * self.k


def conv_specs(input_shape=(256, 32, 1)) -> List[ConvSpec]:
    f, t, c = input_shape
    specs = []
    for i, (ch, (sa, sb)) in enumerate(zip(HIDDEN_CH, STRIDES)):
        to, lo, _ = tf_same(t, 3, sa[1])
        assert sa[0] == 1
        specs.append(ConvSpec(f"conv{i}_a", "t", sa[1], lo, f, t, c, f, to, ch))
        t, c = to, ch
        fo, lo, _ = tf_same(f, 3, sb[0])
        assert sb[1] == 1
        specs.append(ConvSpec(f"conv{i}_b", "f", sb[0], lo, f, t, c, fo, t, ch))
        f = fo
    return specs


def n_params(input_shape=(256, 32, 1), norm="layer_norm2d") -> int:
    """Keras' ``count_params`` of the FingerPrinter (batch_norm's moving statistics included)."""
    n = 0
    specs = conv_specs(input_shape)
    for s in specs:
        n += 3 * s.c_in * s.c_out + s.c_out
        for shp in norm_shapes(s, norm).values():
            k = 1
            for d in shp:
                k *= d
            n += k
    last = specs[-1]
    flat = last.f_out * last.t_out * last.c_out
    sl = flat // EMB_SZ
    n += EMB_SZ * (sl * DIVENC_UNITS[0] + DIVENC_UNITS[0] + DIVENC_UNITS[0] * DIVENC_UNITS[1] + DIVENC_UNITS[1])
    return n


FLOPS_PER_SEGMENT = sum(s.flops_per_seg for s in conv_specs()) + 2 * EMB_SZ * (8 * 32 + 32)
