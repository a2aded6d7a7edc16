"""MODEL.BN 'layer_norm1d' and 'batch_norm' on the host side: the fp64 reference against torch.nn.functional, parameter
counts, the config check, the TensorFlow-checkpoint mapping and the .npz exchange format."""
import numpy as np
import pytest

from nafp_b200.model import arch, tf_checkpoint as T
from nafp_b200.model import weights as W
from util_norms import NORMS, calibrate_batch_norm, fingerprinter
from util_tf_bundle import reference_variable_names, write_bundle

SUF = "/.ATTRIBUTES/VARIABLE_VALUE"


def _mel(n, seed=0):
    rng = np.random.default_rng(seed)
    return np.clip(rng.normal(-30, 15, (n, 256, 32, 1)), -80, 0)


def _torch_layer(x, w, conv, ln, stride, norm):
    """conv (TF SAME) -> ELU -> norm through torch.nn.functional, NHWC in and out, fp64."""
    import torch
    import torch.nn.functional as F
    from oracle.fingerprinter import same_pad
    t = torch.from_numpy(x).permute(0, 3, 1, 2)
    k = torch.from_numpy(w[f"{conv}_w"].astype(np.float64)).permute(3, 2, 0, 1)      # HWIO -> OIHW
    _, flo, fhi = same_pad(t.shape[2], k.shape[2], stride[0])
    _, tlo, thi = same_pad(t.shape[3], k.shape[3], stride[1])
    y = F.elu(F.conv2d(F.pad(t, (tlo, thi, flo, fhi)), k, torch.from_numpy(w[f"{conv}_b"].astype(np.float64)), stride))
    g, b = (torch.from_numpy(w[f"{ln}_{s}"].astype(np.float64)) for s in ("g", "b"))
    if norm == "layer_norm1d":
        return F.layer_norm(y.permute(0, 2, 3, 1), (y.shape[1],), g, b, eps=1e-3).numpy()
    mean, var = (torch.from_numpy(w[f"{ln}_{s}"].astype(np.float64)) for s in ("mean", "var"))
    return F.batch_norm(y, mean, var, g, b, training=False, eps=1e-3).permute(0, 2, 3, 1).numpy()


@pytest.mark.parametrize("norm", ["layer_norm1d", "batch_norm"])
def test_reference_matches_torch_layer_by_layer(norm):
    from oracle.fingerprinter import FRONT_STRIDES
    mel = _mel(2)
    w = W.init_weights(5, randomize_affine=True, norm=norm)
    if norm == "batch_norm":
        w = calibrate_batch_norm(mel, w, seed=5)
    emb, acts = fingerprinter(mel, w, norm, return_all=True)
    x = mel
    for l in range(16):
        i, half = divmod(l, 2)
        got = _torch_layer(x, w, f"conv{i}_{'ab'[half]}", f"ln{i}_{'ab'[half]}", FRONT_STRIDES[i][half], norm)
        np.testing.assert_allclose(acts[l], got, rtol=1e-9, atol=1e-9)
        x = acts[l]
    assert np.allclose(np.linalg.norm(emb, axis=1), 1.0)
    # the last ConvLayer's output is one position: 'layer_norm1d' there is 'layer_norm2d' with (1, 1, C) parameters
    if norm == "layer_norm1d":
        from oracle.fingerprinter import layer_norm_ftc
        from util_norms import normalise
        y = np.random.default_rng(1).normal(0, 2, (3, 1, 1, 1024))
        g, b = w["ln7_b_g"].astype(np.float64), w["ln7_b_b"].astype(np.float64)
        np.testing.assert_allclose(normalise(y, {"ln7_b_g": g, "ln7_b_b": b}, "ln7_b", norm),
                                   layer_norm_ftc(y, g.reshape(1, 1, -1), b.reshape(1, 1, -1)), rtol=1e-12, atol=1e-12)


def test_reference_layer_norm2d_is_the_oracle():
    from oracle import fingerprinter as ofp
    mel = _mel(2, 1)
    w = W.init_weights(3, randomize_affine=True)
    np.testing.assert_array_equal(fingerprinter(mel, w, "layer_norm2d"), ofp.fingerprinter(mel, w))


def test_parameter_counts():
    assert arch.n_params(norm="layer_norm2d") == arch.n_params() == 16_939_008        # nnfp.py:270-274
    assert arch.n_params(norm="layer_norm1d") == 14_662_656
    assert arch.n_params(norm="batch_norm") == 14_678_016                             # moving statistics included
    for norm in NORMS:
        assert sum(v.size for v in W.init_weights(1, norm=norm).values()) == arch.n_params(norm=norm)


def test_check_model_cfg_accepts_the_three_norms():
    import yaml
    import os
    from nafp_b200.model.fp import FingerPrinter, _check_model_cfg
    cfg = yaml.safe_load(open(os.path.join(os.path.dirname(os.path.dirname(__file__)), "config", "default.yaml")))
    for norm in NORMS:
        cfg["MODEL"]["BN"] = norm
        _check_model_cfg(cfg)
    cfg["MODEL"]["BN"] = "foo"
    with pytest.raises(NotImplementedError):
        _check_model_cfg(cfg)
    with pytest.raises(NotImplementedError):
        FingerPrinter(ctx=object(), norm="foo")


def test_init_weights_layer_norm2d_draws_are_unchanged():
    a, b = W.init_weights(7, randomize_affine=True), W.init_weights(7, randomize_affine=True, norm="layer_norm2d")
    assert set(a) == set(b) and all((a[k] == b[k]).all() for k in a)
    bn = W.init_weights(7, norm="batch_norm")
    assert (bn["ln3_b_g"] == 1).all() and (bn["ln3_b_b"] == 0).all() and (bn["ln3_b_mean"] == 0).all()
    assert (bn["ln3_b_var"] == 1).all() and bn["ln3_b_var"].shape == (256,)
    assert W.init_weights(7, norm="layer_norm1d")["ln0_a_g"].shape == (128,)


def _bundle(w, norm):
    tensors = reference_variable_names(w)
    if norm == "batch_norm":
        for i in range(8):
            for half, tag in (("a", "1x3"), ("b", "3x1")):
                base = f"model/front_conv/layer_with_weights-{i}/BN_{tag}/"
                tensors[f"{base}moving_mean{SUF}"] = w[f"ln{i}_{half}_mean"]
                tensors[f"{base}moving_variance{SUF}"] = w[f"ln{i}_{half}_var"]
    return tensors


@pytest.mark.parametrize("norm", ["layer_norm1d", "batch_norm"])
def test_checkpoint_round_trip(tmp_path, norm):
    rng = np.random.default_rng(2)
    w = W.init_weights(2, randomize_affine=True, norm=norm)
    if norm == "batch_norm":
        for k in [k for k in w if k.endswith("_mean")]:
            w[k] = rng.normal(0, 0.3, w[k].shape).astype(np.float32)
            w[k.replace("_mean", "_var")] = rng.uniform(0.2, 2.0, w[k].shape).astype(np.float32)
    tensors = _bundle(w, norm)
    assert sum(v.size for v in tensors.values()) == arch.n_params(norm=norm)
    prefix = str(tmp_path / "ckpt-3")
    write_bundle(prefix, tensors)
    got = T.load_tf_checkpoint(prefix, norm=norm)
    assert set(got) == set(w) and all((got[k] == w[k]).all() for k in w)
    # .npz exchange format: convert, load back, and the host loader accepts the shapes
    back = W.load_weights(T.convert(prefix, str(tmp_path / "w.npz"), norm=norm))
    assert set(back) == set(w) and all((back[k] == w[k]).all() for k in w)
    W.save_weights(str(tmp_path / "again.npz"), back)
    again = W.load_weights(str(tmp_path / "again.npz"))
    assert all((again[k] == w[k]).all() for k in w)


def test_checkpoint_of_another_norm_raises_and_names_the_variables(tmp_path):
    bn = W.init_weights(2, randomize_affine=True, norm="batch_norm")
    prefix = str(tmp_path / "ckpt-1")
    write_bundle(prefix, _bundle(bn, "batch_norm"))
    with pytest.raises(ValueError) as e:                          # moving statistics are not layer_norm1d variables
        T.load_tf_checkpoint(prefix, norm="layer_norm1d")
    assert "BN_1x3/moving_mean" in str(e.value) and "layer_norm1d" in str(e.value)
    with pytest.raises(ValueError) as e:                          # (C,) gammas are not (F,T,C)
        T.load_tf_checkpoint(prefix, norm="layer_norm2d")
    assert "layer_with_weights-0/BN_1x3/gamma" in str(e.value) and "expected (256, 16, 128)" in str(e.value)
    ln1 = W.init_weights(2, randomize_affine=True, norm="layer_norm1d")
    prefix = str(tmp_path / "ckpt-2")
    write_bundle(prefix, _bundle(ln1, "layer_norm1d"))
    with pytest.raises(ValueError) as e:                          # no moving statistics for batch_norm
        T.load_tf_checkpoint(prefix, norm="batch_norm")
    assert "missing ln0_a_mean" in str(e.value) and "missing ln7_b_var" in str(e.value)
    ln2 = W.init_weights(2, randomize_affine=True)
    prefix = str(tmp_path / "ckpt-4")
    write_bundle(prefix, reference_variable_names(ln2))
    with pytest.raises(ValueError) as e:
        T.load_tf_checkpoint(prefix, norm="batch_norm")
    assert "expected (128,)" in str(e.value)
