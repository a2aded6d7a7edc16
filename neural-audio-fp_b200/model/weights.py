"""FingerPrinter weights: seeded Keras-default initialisation and the ``.npz`` exchange format.

No trained checkpoints are available offline, so weights are random-initialised the way Keras
initialises the reference's layers (``model/fp/nnfp.py:48-61,135-137``): conv / dense kernels
``glorot_uniform`` (limit = sqrt(6 / (fan_in + fan_out))), biases zero, LayerNormalization
gamma = 1 / beta = 0, BatchNormalization moving mean = 0 / moving variance = 1.  ``randomize_affine=True``
additionally draws biases and the normalisation's gamma/beta at random so that affine bugs are visible in parity
tests (the moving statistics keep their defaults).

Exchange format (one ``.npz``; what a TF-checkpoint converter would also emit):
    conv{i}_a_w (1,3,Cin,Cout)  conv{i}_a_b (Cout)  ln{i}_a_g / ln{i}_a_b (F,T,C)     i = 0..7
    conv{i}_b_w (3,1,C,C)       conv{i}_b_b (C)     ln{i}_b_g / ln{i}_b_b (F,T,C)
    div_w1 (128,8,32)  div_b1 (128,32)  div_w2 (128,32,1)  div_b2 (128,1)
All float32; conv kernels HWIO as in Keras.  That is MODEL.BN 'layer_norm2d'; for 'layer_norm1d' and 'batch_norm'
``ln*_g`` / ``ln*_b`` have shape (C,), and 'batch_norm' adds ``ln{i}_{a,b}_mean`` / ``ln{i}_{a,b}_var`` (C,).
"""
from __future__ import annotations

import numpy as np

from .arch import DIVENC_UNITS, EMB_SZ, conv_specs, norm_shapes


def _glorot(rng, shape, fan_in, fan_out):
    lim = np.sqrt(6.0 / (fan_in + fan_out))
    return rng.uniform(-lim, lim, size=shape).astype(np.float32)


def init_weights(seed=7, randomize_affine=False, input_shape=(256, 32, 1), norm="layer_norm2d"):
    rng = np.random.default_rng(seed)
    w = {}
    specs = conv_specs(input_shape)
    for s in specs:
        kshape = (1, 3, s.c_in, s.c_out) if s.axis == "t" else (3, 1, s.c_in, s.c_out)
        w[f"{s.name}_w"] = _glorot(rng, kshape, 3 * s.c_in, 3 * s.c_out)
        ln = s.name.replace("conv", "ln")
        shapes = norm_shapes(s, norm)
        shp = shapes["g"]
        if "mean" in shapes:
            w[f"{ln}_mean"] = np.zeros(shapes["mean"], np.float32)
            w[f"{ln}_var"] = np.ones(shapes["var"], np.float32)
        if randomize_affine:
            w[f"{s.name}_b"] = rng.normal(0, 0.1, s.c_out).astype(np.float32)
            w[f"{ln}_g"] = (1.0 + 0.2 * rng.standard_normal(shp)).astype(np.float32)
            w[f"{ln}_b"] = (0.2 * rng.standard_normal(shp)).astype(np.float32)
        else:
            w[f"{s.name}_b"] = np.zeros(s.c_out, np.float32)
            w[f"{ln}_g"] = np.ones(shp, np.float32)
            w[f"{ln}_b"] = np.zeros(shp, np.float32)
    last = specs[-1]
    sl = last.f_out * last.t_out * last.c_out // EMB_SZ
    u0, u1 = DIVENC_UNITS
    w["div_w1"] = _glorot(rng, (EMB_SZ, sl, u0), sl, u0)
    w["div_w2"] = _glorot(rng, (EMB_SZ, u0, u1), u0, u1)
    if randomize_affine:
        w["div_b1"] = rng.normal(0, 0.1, (EMB_SZ, u0)).astype(np.float32)
        w["div_b2"] = rng.normal(0, 0.1, (EMB_SZ, u1)).astype(np.float32)
    else:
        w["div_b1"] = np.zeros((EMB_SZ, u0), np.float32)
        w["div_b2"] = np.zeros((EMB_SZ, u1), np.float32)
    return w


def save_weights(path, weights):
    np.savez(path, **weights)


def load_weights(path):
    with np.load(path) as z:
        return {k: np.ascontiguousarray(z[k], dtype=np.float32) for k in z.files}
