"""Weight import for the B200 executor: a trained ResNet (conv + batch-norm layers, as a PyTorch
`state_dict` or any mapping of numpy arrays) -> the canonical fp32 blob of DESIGN.md §5 (BN folded
into conv weights and biases) -> an NSBW file that `infer::B200::load(path)` reads.

The reference loads an external ONNX through TensorRT (reference src/infer/trt.cc:109-232), which
folds batch-norm itself while building the engine; this executor has no engine build step, so the
fold happens here, once, in fp64.  Only the tensor contract of the net is pinned by the reference
(trt.cc:144-150,193-227): `input` [B,86,9,9] -> `policy` 2187 logits (plane-major), `value`, `draw`
probabilities.  The layer naming below is this repo's (there is no model in the reference tree).

Expected keys (PyTorch naming; `bn` groups are optional - without them the conv must carry a bias):
    stem.conv.weight [C,86,3,3]   stem.conv.bias? [C]   stem.bn.{weight,bias,running_mean,running_var}?
    blocks.{i}.conv1.* / blocks.{i}.bn1.*   blocks.{i}.conv2.* / blocks.{i}.bn2.*      i = 0..blocks-1
    policy.conv.weight [27,C,1,1]  policy.conv.bias [27]
    value.conv.weight [1,C,1,1]    value.conv.bias? [1]  value.bn.*?
    value.fc1.weight [H,81]  value.fc1.bias [H]   value.fc2.weight [2,H]  value.fc2.bias [2]
"""
from __future__ import annotations

import struct
from typing import Mapping, Optional

import numpy as np

MAGIC = b"NSBW"
VERSION = 1
BN_EPS = 1e-5  # torch.nn.BatchNorm2d default


def _np(x) -> np.ndarray:
    if hasattr(x, "detach"):
        x = x.detach().cpu().numpy()
    return np.asarray(x, dtype=np.float64)


def fold_bn(weight, bias, bn: Optional[Mapping[str, object]], eps: float = BN_EPS):
    """conv(x) followed by inference-mode batch-norm == conv'(x):
    w' = w * gamma / sqrt(var + eps) per output channel, b' = (b - mean) * gamma / sqrt(var + eps) + beta."""
    w = _np(weight)
    b = np.zeros(w.shape[0]) if bias is None else _np(bias)
    if bn is None:
        return w, b
    gamma, beta = _np(bn["weight"]), _np(bn["bias"])
    mean, var = _np(bn["running_mean"]), _np(bn["running_var"])
    scale = gamma / np.sqrt(var + eps)
    return w * scale.reshape(-1, *([1] * (w.ndim - 1))), (b - mean) * scale + beta


def _group(state: Mapping[str, object], prefix: str) -> Optional[dict]:
    keys = ("weight", "bias", "running_mean", "running_var")
    if f"{prefix}.weight" not in state:
        return None
    missing = [k for k in keys if f"{prefix}.{k}" not in state]
    if missing:
        raise KeyError(f"batch-norm group {prefix!r} lacks {missing}")
    return {k: state[f"{prefix}.{k}"] for k in keys}


def blob_from_state(state: Mapping[str, object], channels: int, blocks: int, value_hidden: int = 256,
                    in_channels: int = 86, eps: float = BN_EPS) -> np.ndarray:
    """Canonical fp32 blob (DESIGN.md §5) from a state dict with the key names of the module docstring."""
    C, H = channels, value_hidden
    out = []

    def conv(prefix, bn_prefix, shape):
        w, b = fold_bn(state[f"{prefix}.weight"], state.get(f"{prefix}.bias"), _group(state, bn_prefix), eps)
        if w.shape != shape:
            raise ValueError(f"{prefix}.weight has shape {w.shape}, expected {shape}")
        out.extend([w.reshape(-1), b.reshape(-1)])

    conv("stem.conv", "stem.bn", (C, in_channels, 3, 3))
    for i in range(blocks):
        conv(f"blocks.{i}.conv1", f"blocks.{i}.bn1", (C, C, 3, 3))
        conv(f"blocks.{i}.conv2", f"blocks.{i}.bn2", (C, C, 3, 3))
    conv("policy.conv", "policy.bn", (27, C, 1, 1))
    conv("value.conv", "value.bn", (1, C, 1, 1))
    for name, shape in (("value.fc1", (H, 81)), ("value.fc2", (2, H))):
        w, b = _np(state[f"{name}.weight"]), _np(state[f"{name}.bias"])
        if w.shape != shape:
            raise ValueError(f"{name}.weight has shape {w.shape}, expected {shape}")
        out.extend([w.reshape(-1), b.reshape(-1)])
    return np.concatenate(out).astype(np.float32)


def pad_channels(blob: np.ndarray, desc, channels: int) -> np.ndarray:
    """The blob of the same net at trunk width `channels` >= desc.channels: the added channels get zero conv weights
    (as outputs and as inputs), zero biases and zero policy / value-conv weights, so they stay exactly zero through
    every layer and the net computes what it computed before.  `desc` has the attributes of binding.net_desc."""
    C, IN, H, NB = desc.channels, desc.in_channels, desc.value_hidden, desc.blocks
    W = channels
    if W < C:
        raise ValueError(f"pad_channels: cannot narrow a {C}-channel net to {W}")
    blob = np.asarray(blob, dtype=np.float32)
    out, o = [], 0

    def take(shape):
        nonlocal o
        n = int(np.prod(shape))
        a = blob[o:o + n].reshape(shape)
        o += n
        return a

    def padded(a, shape):
        z = np.zeros(shape, dtype=np.float32)
        z[tuple(slice(0, s) for s in a.shape)] = a
        out.append(z.reshape(-1))

    padded(take((C, IN, 3, 3)), (W, IN, 3, 3))
    padded(take((C,)), (W,))
    for _ in range(2 * NB):
        padded(take((C, C, 3, 3)), (W, W, 3, 3))
        padded(take((C,)), (W,))
    padded(take((27, C)), (27, W))
    out.append(take((27,)).reshape(-1))
    padded(take((C,)), (W,))
    rest = blob[o:]
    if rest.size != 1 + H * 81 + H + 2 * H + 2:
        raise ValueError(f"pad_channels: blob has {blob.size} floats, which does not match the net description")
    out.append(rest)
    return np.concatenate(out)


def write_nsbw(path: str, blob: np.ndarray, channels: int, blocks: int, value_hidden: int = 256, in_channels: int = 86):
    """File format read by infer::B200::load (host/infer_b200.h): "NSBW", u32 version, i32 channels,
    blocks, hidden, in_channels, then the blob."""
    blob = np.ascontiguousarray(blob, dtype="<f4")
    with open(path, "wb") as f:
        f.write(MAGIC + struct.pack("<Iiiii", VERSION, channels, blocks, value_hidden, in_channels))
        f.write(blob.tobytes())


def read_nsbw(path: str):
    with open(path, "rb") as f:
        head = f.read(24)
        if len(head) != 24 or head[:4] != MAGIC:
            raise ValueError(f"{path}: not an NSBW file")
        version, channels, blocks, hidden, in_channels = struct.unpack("<Iiiii", head[4:])
        if version != VERSION:
            raise ValueError(f"{path}: NSBW version {version}, expected {VERSION}")
        blob = np.frombuffer(f.read(), dtype="<f4").copy()
    return {"channels": channels, "blocks": blocks, "value_hidden": hidden, "in_channels": in_channels}, blob
