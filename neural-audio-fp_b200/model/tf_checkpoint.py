"""TensorFlow checkpoint -> FingerPrinter weights, without TensorFlow (SURVEY §8 f2).

The reference restores ``tf.train.Checkpoint(model=m_fp)`` files (``model/generate.py:26-51``:
``{LOG_ROOT_DIR}/checkpoint/{name}/ckpt-{index}.index`` + ``.data-00000-of-00001``).  This module reads that
on-disk format directly -- the *tensor bundle*: an SSTable (``.index``: prefix-compressed key blocks, restart
arrays, 5-byte block trailers, 48-byte footer with magic 0xdb4775248b80fb57) whose values are
``BundleEntryProto`` messages (dtype, shape, shard, offset, size, crc32c) pointing into the raw ``.data`` shards
-- and maps the object-graph keys of the reference's model (``model/fp/nnfp.py``) onto the ``.npz`` exchange
format of ``model/weights.py``:

    model/front_conv/layer_with_weights-{i}/conv2d_1x3/{kernel,bias}     -> conv{i}_a_w, conv{i}_a_b
    model/front_conv/layer_with_weights-{i}/BN_1x3/{gamma,beta}          -> ln{i}_a_g,  ln{i}_a_b
    model/front_conv/layer_with_weights-{i}/conv2d_3x1/{kernel,bias}     -> conv{i}_b_w, conv{i}_b_b
    model/front_conv/layer_with_weights-{i}/BN_3x1/{gamma,beta}          -> ln{i}_b_g,  ln{i}_b_b
    model/front_conv/layer_with_weights-{i}/BN_*/{moving_mean,moving_variance} -> ln{i}_*_mean, ln{i}_*_var
                                                                            (MODEL.BN 'batch_norm' only)
    model/div_enc/split_fc_layers/{q}/layer_with_weights-{0,1}/{kernel,bias} -> div_w1/div_b1, div_w2/div_b2 [q]

(each followed by ``/.ATTRIBUTES/VARIABLE_VALUE``; the same variables reached through ``.../forward/
layer_with_weights-{0..3}`` are accepted too; optimizer slots are ignored).  Every tensor is checked against the
shape ``model/arch.py`` derives for it under the configured MODEL.BN (gamma / beta (F,T,C) for 'layer_norm2d', (C,)
otherwise), and against its stored crc32c.

STATUS: the file format is restated from TensorFlow's published sources (tensorflow/core/util/tensor_bundle,
tensorflow/core/lib/io/table*) -- no TensorFlow and no reference checkpoint exist in the build container, so the
reader is verified against a writer of the same restatement (``tests/test_tf_checkpoint.py``), not against a file
TensorFlow wrote: PARITY UNPINNED until one is available.
"""
from __future__ import annotations

import glob
import os
import re
import struct

import numpy as np

from .arch import DIVENC_UNITS, EMB_SZ, conv_specs, norm_shapes

TABLE_MAGIC = 0xdb4775248b80fb57
FOOTER_LEN = 48
_SUFFIX = "/.ATTRIBUTES/VARIABLE_VALUE"
# tensorflow/core/framework/types.proto
_DTYPES = {1: np.float32, 2: np.float64, 3: np.int32, 4: np.uint8, 5: np.int16, 6: np.int8, 9: np.int64, 10: np.bool_,
           17: np.uint16, 19: np.float16, 22: np.uint32, 23: np.uint64}


# ------------------------------------------------------------------------------------------ crc32c (Castagnoli)
def _make_crc_table():
    tab = []
    for n in range(256):
        c = n
        for _ in range(8):
            c = (c >> 1) ^ 0x82F63B78 if c & 1 else c >> 1
        tab.append(c)
    return np.array(tab, dtype=np.uint32)


_CRC_TABLE = _make_crc_table()


def crc32c(data, crc=0):
    """CRC-32C of ``data`` (bytes-like); ``crc`` continues a previous value."""
    tab = _CRC_TABLE
    c = int(crc) ^ 0xFFFFFFFF
    for b in bytes(data):
        c = int(tab[(c ^ b) & 0xFF]) ^ (c >> 8)
    return c ^ 0xFFFFFFFF


def crc32c_mask(crc):
    """The masked form TensorFlow / LevelDB store (rotate right 15, add a constant)."""
    return ((((crc >> 15) | (crc << 17)) & 0xFFFFFFFF) + 0xA282EAD8) & 0xFFFFFFFF


# ------------------------------------------------------------------------------------------ varints, protobuf
def _varint(buf, pos):
    out, shift = 0, 0
    while True:
        b = buf[pos]
        pos += 1
        out |= (b & 0x7F) << shift
        if not b & 0x80:
            return out, pos
        shift += 7
        if shift > 70:
            raise ValueError("malformed varint")


def _proto_fields(buf):
    """Yield (field number, wire type, value) of one protobuf message (values: int or bytes)."""
    pos, n = 0, len(buf)
    while pos < n:
        key, pos = _varint(buf, pos)
        field, wt = key >> 3, key & 7
        if wt == 0:
            v, pos = _varint(buf, pos)
        elif wt == 1:
            v = struct.unpack_from("<Q", buf, pos)[0]
            pos += 8
        elif wt == 2:
            ln, pos = _varint(buf, pos)
            v = bytes(buf[pos:pos + ln])
            pos += ln
        elif wt == 5:
            v = struct.unpack_from("<I", buf, pos)[0]
            pos += 4
        else:
            raise ValueError(f"unsupported protobuf wire type {wt}")
        yield field, wt, v


def _parse_entry(buf):
    """BundleEntryProto (tensorflow/core/protobuf/tensor_bundle.proto)."""
    e = dict(dtype=0, shape=[], shard_id=0, offset=0, size=0, crc32c=None, sliced=False)
    for field, _, v in _proto_fields(buf):
        if field == 1:
            e["dtype"] = v
        elif field == 2:                      # TensorShapeProto: repeated Dim dim = 2 { int64 size = 1 }
            for f2, _, dim in _proto_fields(v):
                if f2 == 2:
                    size = 0
                    for f3, _, s in _proto_fields(dim):
                        if f3 == 1:
                            size = s
                    e["shape"].append(size)
        elif field == 3:
            e["shard_id"] = v
        elif field == 4:
            e["offset"] = v
        elif field == 5:
            e["size"] = v
        elif field == 6:
            e["crc32c"] = v
        elif field == 7:
            e["sliced"] = True
    return e


# ------------------------------------------------------------------------------------------ snappy (raw format)
def _snappy_decompress(buf):
    n, pos = _varint(buf, 0)
    out = bytearray()
    while pos < len(buf):
        tag = buf[pos]
        pos += 1
        kind = tag & 3
        if kind == 0:
            ln = tag >> 2
            if ln >= 60:
                nb = ln - 59
                ln = int.from_bytes(buf[pos:pos + nb], "little")
                pos += nb
            ln += 1
            out += buf[pos:pos + ln]
            pos += ln
            continue
        if kind == 1:
            ln = ((tag >> 2) & 7) + 4
            off = ((tag >> 5) << 8) | buf[pos]
            pos += 1
        elif kind == 2:
            ln = (tag >> 2) + 1
            off = int.from_bytes(buf[pos:pos + 2], "little")
            pos += 2
        else:
            ln = (tag >> 2) + 1
            off = int.from_bytes(buf[pos:pos + 4], "little")
            pos += 4
        if off == 0 or off > len(out):
            raise ValueError("malformed snappy block")
        for _ in range(ln):
            out.append(out[-off])
    if len(out) != n:
        raise ValueError("snappy length mismatch")
    return bytes(out)


# ------------------------------------------------------------------------------------------ SSTable
def _read_block(data, offset, size, verify=True):
    raw = data[offset:offset + size]
    ctype = data[offset + size]
    stored = struct.unpack_from("<I", data, offset + size + 1)[0]
    if verify and crc32c_mask(crc32c(data[offset:offset + size + 1])) != stored:
        raise ValueError(f"index block at {offset}: checksum mismatch")
    if ctype == 0:
        return raw
    if ctype == 1:
        return _snappy_decompress(raw)
    raise ValueError(f"index block at {offset}: unknown compression type {ctype}")


def _block_entries(block):
    n_restarts = struct.unpack_from("<I", block, len(block) - 4)[0]
    end = len(block) - 4 - 4 * n_restarts
    pos, key = 0, b""
    while pos < end:
        shared, pos = _varint(block, pos)
        non_shared, pos = _varint(block, pos)
        vlen, pos = _varint(block, pos)
        key = key[:shared] + bytes(block[pos:pos + non_shared])
        pos += non_shared
        yield key, bytes(block[pos:pos + vlen])
        pos += vlen


def read_index(index_path, verify=True):
    """``{key: BundleEntryProto bytes}`` of a ``.index`` file (the header entry has key '')."""
    with open(index_path, "rb") as f:
        data = f.read()
    if len(data) < FOOTER_LEN:
        raise ValueError(f"{index_path}: too short for an SSTable")
    footer = data[-FOOTER_LEN:]
    lo, hi = struct.unpack_from("<II", footer, FOOTER_LEN - 8)
    if (hi << 32 | lo) != TABLE_MAGIC:
        raise ValueError(f"{index_path}: not a TensorFlow checkpoint index (bad magic)")
    pos = 0
    _, pos = _varint(footer, pos)          # metaindex handle
    _, pos = _varint(footer, pos)
    ioff, pos = _varint(footer, pos)
    isize, pos = _varint(footer, pos)
    out = {}
    for _, handle in _block_entries(_read_block(data, ioff, isize, verify)):
        boff, p = _varint(handle, 0)
        bsize, _ = _varint(handle, p)
        for key, value in _block_entries(_read_block(data, boff, bsize, verify)):
            out[key.decode("utf-8", errors="replace")] = value
    return out


def read_bundle(prefix, verify=True, only=None):
    """All numeric tensors of the checkpoint ``prefix`` (``prefix.index`` + data shards) as numpy arrays.
    ``only``: optional predicate on the key."""
    entries = read_index(prefix + ".index", verify)
    num_shards = 1
    if "" in entries:
        for field, _, v in _proto_fields(entries[""]):
            if field == 1:
                num_shards = v
            if field == 2 and v != 0:
                raise ValueError("big-endian checkpoints are not supported")
    shards = {}
    out = {}
    for key, raw in entries.items():
        if key == "" or (only is not None and not only(key)):
            continue
        e = _parse_entry(raw)
        if e["dtype"] not in _DTYPES:       # strings (object graph), resources ...
            continue
        if e["sliced"]:
            raise ValueError(f"{key}: partitioned (sliced) variables are not supported")
        sid = e["shard_id"]
        if sid not in shards:
            shards[sid] = np.memmap(f"{prefix}.data-{sid:05d}-of-{num_shards:05d}", dtype=np.uint8, mode="r")
        blob = shards[sid][e["offset"]:e["offset"] + e["size"]]
        dt = np.dtype(_DTYPES[e["dtype"]])
        n = int(np.prod(e["shape"])) if e["shape"] else 1
        if n * dt.itemsize != e["size"]:
            raise ValueError(f"{key}: {e['size']} bytes for shape {e['shape']} of {dt}")
        if verify and e["crc32c"] is not None:
            c = _crc32c_fast(blob)
            if e["crc32c"] not in (crc32c_mask(c), c):          # stored masked (crc32c::Mask) by BundleWriter
                raise ValueError(f"{key}: tensor checksum mismatch")
        out[key] = np.frombuffer(bytes(blob), dtype=dt).reshape(e["shape"])
    return out


def _gf2_times(mat, vec):
    out, i = 0, 0
    while vec:
        if vec & 1:
            out ^= mat[i]
        vec >>= 1
        i += 1
    return out


def _gf2_square(mat):
    return [_gf2_times(mat, mat[n]) for n in range(32)]


def _zeros_operator(n_bytes):
    """32x32 GF(2) matrix that advances a (pre/post-inverted) CRC-32C over ``n_bytes`` zero bytes -- the operator of
    zlib's crc32_combine, for the Castagnoli polynomial -- folded into ONE matrix."""
    odd = [0x82F63B78] + [1 << n for n in range(31)]       # one zero bit
    even = _gf2_square(odd)                                 # two
    odd = _gf2_square(even)                                 # four
    op = None
    n = n_bytes
    while n:
        even = _gf2_square(odd)                             # first round: 8 bits = one byte
        if n & 1:
            op = even if op is None else [_gf2_times(even, col) for col in op]
        n >>= 1
        if not n:
            break
        odd = _gf2_square(even)
        if n & 1:
            op = odd if op is None else [_gf2_times(odd, col) for col in op]
        n >>= 1
    return op


def _crc32c_fast(blob, lanes=1024):
    """CRC-32C of a large uint8 array: ``lanes`` equal chunks advance together (one vectorised table step per byte
    position), their CRCs are then chained with the zero-append operator (crc(A||B) = op_len(B)(crc(A)) ^ crc(B))."""
    b = np.ascontiguousarray(np.asarray(blob, dtype=np.uint8))
    n = len(b)
    if n < 1 << 16:
        return crc32c(b.tobytes())
    per = n // lanes
    cols = np.ascontiguousarray(b[:lanes * per].reshape(lanes, per).T)      # [byte position][lane]
    c = np.full(lanes, 0xFFFFFFFF, dtype=np.uint32)
    tab = _CRC_TABLE
    for j in range(per):
        c = tab[(c ^ cols[j]) & 0xFF] ^ (c >> 8)
    crcs = (c ^ 0xFFFFFFFF).tolist()
    op = _zeros_operator(per)
    total = crcs[0]
    for v in crcs[1:]:
        total = _gf2_times(op, total) ^ v
    return crc32c(b[lanes * per:].tobytes(), total)


# ------------------------------------------------------------------------------------------ name mapping
_CONV_RE = re.compile(r"front_conv/layer_with_weights-(\d+)/(?:forward/layer_with_weights-(\d)/|"
                      r"(conv2d_1x3|BN_1x3|conv2d_3x1|BN_3x1)/)(kernel|bias|gamma|beta|moving_mean|moving_variance)$")
_DIV_RE = re.compile(r"div_enc/split_fc_layers/(\d+)/layer_with_weights-(\d)/(kernel|bias)$")
_FORWARD_SLOTS = ("conv2d_1x3", "BN_1x3", "conv2d_3x1", "BN_3x1")        # nnfp.py:73-79 (ELU layers have no weights)


def is_model_variable(key):
    return key.endswith(_SUFFIX) and "/.OPTIMIZER_SLOT/" not in key and ("front_conv/" in key or "div_enc/" in key)


_BN_VARS = {"gamma": "g", "beta": "b", "moving_mean": "mean", "moving_variance": "var"}


def map_variables(tensors, input_shape=(256, 32, 1), norm="layer_norm2d"):
    """Bundle tensors (``read_bundle``) -> the weights dict of ``model/weights.py`` for MODEL.BN ``norm``; raises with
    the list of what is missing, has an unexpected shape or belongs to another MODEL.BN."""
    specs = conv_specs(input_shape)
    n_blocks = len(specs) // 2
    w = {}
    u0, u1 = DIVENC_UNITS
    last = specs[-1]
    sl = last.f_out * last.t_out * last.c_out // EMB_SZ
    div = {"w1": np.zeros((EMB_SZ, sl, u0), np.float32), "b1": np.zeros((EMB_SZ, u0), np.float32),
           "w2": np.zeros((EMB_SZ, u0, u1), np.float32), "b2": np.zeros((EMB_SZ, u1), np.float32)}
    div_seen = set()
    problems = []
    for key, arr in tensors.items():
        if not is_model_variable(key):
            continue
        name = key[:-len(_SUFFIX)]
        m = _CONV_RE.search(name)
        if m:
            blk = int(m.group(1))
            layer = m.group(3) or (_FORWARD_SLOTS[int(m.group(2))] if int(m.group(2)) < 4 else None)
            if blk >= n_blocks or layer is None:
                problems.append(f"unexpected variable {key}")
                continue
            half = "a" if layer.endswith("1x3") else "b"
            spec = specs[2 * blk + (0 if half == "a" else 1)]
            what = m.group(4)
            if layer.startswith("conv"):
                want = ((1, 3, spec.c_in, spec.c_out) if half == "a" else (3, 1, spec.c_in, spec.c_out)) if what == "kernel" \
                    else (spec.c_out,)
                dst = f"conv{blk}_{half}_{'w' if what == 'kernel' else 'b'}"
            else:
                shapes = norm_shapes(spec, norm)
                sfx = _BN_VARS.get(what)
                if sfx not in shapes:
                    problems.append(f"{key}: not a variable of MODEL.BN={norm!r}")
                    continue
                want = shapes[sfx]
                dst = f"ln{blk}_{half}_{sfx}"
            if what not in (("kernel", "bias") if layer.startswith("conv") else _BN_VARS) or tuple(arr.shape) != want:
                problems.append(f"{key}: shape {tuple(arr.shape)}, expected {want}")
                continue
            w[dst] = np.ascontiguousarray(arr, dtype=np.float32)
            continue
        m = _DIV_RE.search(name)
        if m:
            q, dense, what = int(m.group(1)), int(m.group(2)), m.group(3)
            dst = ("w" if what == "kernel" else "b") + str(dense + 1)
            if q >= EMB_SZ or dense > 1 or tuple(arr.shape) != div[dst].shape[1:]:
                problems.append(f"{key}: shape {tuple(arr.shape)}, expected {div[dst].shape[1:]}")
                continue
            div[dst][q] = arr
            div_seen.add((q, dst))
            continue
        problems.append(f"unrecognised model variable {key}")
    for s in specs:
        ln = s.name.replace("conv", "ln")
        for k in (f"{s.name}_w", f"{s.name}_b", *(f"{ln}_{sfx}" for sfx in norm_shapes(s, norm))):
            if k not in w:
                problems.append(f"missing {k}")
    for q in range(EMB_SZ):
        for dst in ("w1", "b1", "w2", "b2"):
            if (q, dst) not in div_seen:
                problems.append(f"missing div_enc slice {q} {dst}")
    if problems:
        raise ValueError(f"checkpoint does not match the FingerPrinter of model/fp/nnfp.py (MODEL.BN={norm!r}):\n  "
                         + "\n  ".join(problems[:40]))
    w.update({"div_w1": div["w1"], "div_b1": div["b1"], "div_w2": div["w2"], "div_b2": div["b2"]})
    return w


def load_tf_checkpoint(prefix, verify=True, input_shape=(256, 32, 1), norm="layer_norm2d"):
    """``prefix`` = path without extension (``.../ckpt-100``) -> weights dict for MODEL.BN ``norm``."""
    return map_variables(read_bundle(prefix, verify, only=is_model_variable), input_shape, norm)


def latest_checkpoint(checkpoint_dir):
    """(index, prefix) of the newest ``ckpt-N`` in a ``tf.train.CheckpointManager`` directory: the ``checkpoint``
    state file if it is there (``model_checkpoint_path: "ckpt-N"``), else the largest N on disk."""
    state = os.path.join(checkpoint_dir, "checkpoint")
    if os.path.exists(state):
        with open(state) as f:
            m = re.search(r'^model_checkpoint_path:\s*"(.*?ckpt-(\d+))"', f.read(), re.M)
        if m:
            p = m.group(1)
            p = p if os.path.isabs(p) else os.path.join(checkpoint_dir, os.path.basename(p))
            if os.path.exists(p + ".index"):
                return int(m.group(2)), p
    found = []
    for p in glob.glob(os.path.join(checkpoint_dir, "ckpt-*.index")):
        m = re.search(r"ckpt-(\d+)\.index$", p)
        if m:
            found.append((int(m.group(1)), p[:-len(".index")]))
    return max(found) if found else (None, None)


def convert(prefix, npz_path=None, norm="layer_norm2d"):
    """CLI helper: write the ``.npz`` exchange file next to the checkpoint (or to ``npz_path``); 'batch_norm' adds the
    moving statistics as ``ln*_mean`` / ``ln*_var``."""
    from .weights import save_weights
    w = load_tf_checkpoint(prefix, norm=norm)
    npz_path = npz_path or prefix + ".npz"
    save_weights(npz_path, w)
    return npz_path


if __name__ == "__main__":
    import sys
    if len(sys.argv) < 2:
        raise SystemExit("usage: python -m nafp_b200.model.tf_checkpoint CKPT_PREFIX [OUT.npz] [MODEL.BN]")
    print(convert(sys.argv[1], sys.argv[2] if len(sys.argv) > 2 and sys.argv[2] else None,
                  sys.argv[3] if len(sys.argv) > 3 else "layer_norm2d"))
