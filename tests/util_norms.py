"""TEST INFRASTRUCTURE: fp64 reference of the FingerPrinter for every MODEL.BN (model/fp/nnfp.py:20-83,
``ConvLayer(norm=...)``), in TF 2.4 Keras semantics, eps 1e-3 throughout:

* 'layer_norm2d': LayerNormalization(axis=(1,2,3)), gamma / beta (F,T,C) -- ``oracle.fingerprinter`` itself;
* 'layer_norm1d': LayerNormalization(axis=-1): mean / biased variance over the C channels of each (segment, f, t),
  gamma / beta (C,);
* 'batch_norm': BatchNormalization(axis=-1) in inference mode (``test_step`` sets ``m_fp.trainable = False``):
  gamma (x - moving_mean) / sqrt(moving_variance + eps) + beta, all (C,).

conv -> ELU -> norm twice per ConvLayer, then the unchanged DivEnc head and L2 normalisation, reusing the pieces of
``oracle/fingerprinter.py``."""
import numpy as np

from oracle import fingerprinter as ofp

EPS = 1e-3
NORMS = ("layer_norm2d", "layer_norm1d", "batch_norm")


def normalise(y, w, ln, norm):
    """The normalisation ``ln`` (e.g. 'ln3_b') of the ELU output y (B,F,T,C)."""
    g, b = w[f"{ln}_g"], w[f"{ln}_b"]
    if norm == "layer_norm2d":
        return ofp.layer_norm_ftc(y, g, b, EPS)
    if norm == "layer_norm1d":
        mu = y.mean(axis=-1, keepdims=True)
        var = ((y - mu) ** 2).mean(axis=-1, keepdims=True)
        return (y - mu) / np.sqrt(var + EPS) * g + b
    if norm == "batch_norm":
        return (y - w[f"{ln}_mean"]) / np.sqrt(w[f"{ln}_var"] + EPS) * g + b
    raise ValueError(norm)


def _layers():
    for i, (s_a, s_b) in enumerate(ofp.FRONT_STRIDES):
        yield f"conv{i}_a", f"ln{i}_a", s_a
        yield f"conv{i}_b", f"ln{i}_b", s_b


def fingerprinter(mel, weights, norm="layer_norm2d", dtype=np.float64, return_all=False):
    """mel (B,256,32,1) -> (B,128) unit-norm fingerprints; ``return_all`` also returns every normalised activation."""
    w = {k: np.asarray(v, dtype=dtype) for k, v in weights.items()}
    x = np.asarray(mel, dtype=dtype)
    acts = []
    for conv, ln, stride in _layers():
        x = normalise(ofp._elu(ofp.conv2d_same_nhwc(x, w[f"{conv}_w"], w[f"{conv}_b"], stride)), w, ln, norm)
        acts.append(x)
    emb = ofp.l2_normalize(ofp.div_enc(x.reshape(x.shape[0], -1), w))
    return (emb, acts) if return_all else emb


def calibrate_batch_norm(mel, weights, perturb=0.1, seed=0):
    """'batch_norm' weights whose moving statistics are the per-channel mean / variance of a calibration batch, layer by
    layer through the network being calibrated, each scaled by a factor drawn from [1 - perturb, 1 + perturb] (a
    trained model's statistics describe its activations; arbitrary ones let them drift through 16 layers)."""
    rng = np.random.default_rng(seed)
    w = dict(weights)
    x = np.asarray(mel, dtype=np.float64)
    for conv, ln, stride in _layers():
        y = ofp._elu(ofp.conv2d_same_nhwc(x, w[f"{conv}_w"].astype(np.float64), w[f"{conv}_b"].astype(np.float64), stride))
        c = y.shape[-1]
        mean, var = y.mean(axis=(0, 1, 2)), y.var(axis=(0, 1, 2))
        w[f"{ln}_mean"] = (mean * rng.uniform(1 - perturb, 1 + perturb, c)).astype(np.float32)
        w[f"{ln}_var"] = (var * rng.uniform(1 - perturb, 1 + perturb, c)).astype(np.float32)
        x = normalise(y, {k: np.asarray(v, np.float64) for k, v in w.items() if k.startswith(ln)}, ln, "batch_norm")
    return w


def weights(norm, seed, mel_calib=None):
    """Random weights with random affine parameters for ``norm``; 'batch_norm' is calibrated on ``mel_calib``."""
    from nafp_b200.model import weights as W
    w = W.init_weights(seed, randomize_affine=True, norm=norm)
    if norm == "batch_norm":
        w = calibrate_batch_norm(mel_calib, w, seed=seed)
    return w
