"""Weights shared by the golden generator and the tests: a deterministic, name-keyed fill (the same state-dict keys
always receive the same values, so no weights need to be stored) and a 4-bit packing for trained weights that are stored."""
import zlib

import torch


def det_tensor(key, shape, kind, seed=0):
    g = torch.Generator().manual_seed((zlib.crc32(key.encode()) + 7919 * seed) & 0x7FFFFFFF)
    if kind == "conv_w":
        fan_in = 1
        for s in shape[1:]:
            fan_in *= s
        return torch.randn(shape, generator=g) * (2.0 / max(fan_in, 1)) ** 0.5
    if kind == "bn_w":  # mostly positive, a few negative gammas (exercises the max/min pooling logic)
        w = 0.5 + torch.rand(shape, generator=g)
        sign = torch.where(torch.rand(shape, generator=g) < 0.1, -1.0, 1.0)
        return w * sign
    if kind == "var":
        return 0.5 + torch.rand(shape, generator=g)
    if kind == "small":
        return 0.1 * torch.randn(shape, generator=g)
    raise ValueError(kind)


def det_state_dict(reference_sd, seed=0):
    """Return a new state dict with the keys/shapes of `reference_sd` and deterministic values."""
    out = {}
    for k, v in reference_sd.items():
        if k.endswith("num_batches_tracked"):
            out[k] = torch.zeros_like(v)
        elif k.endswith("running_var"):
            out[k] = det_tensor(k, v.shape, "var", seed)
        elif k.endswith("running_mean"):
            out[k] = det_tensor(k, v.shape, "small", seed)
        elif ".bn." in k and k.endswith("weight") and v.dim() == 1:
            out[k] = det_tensor(k, v.shape, "bn_w", seed)
        elif k.endswith("bias"):
            out[k] = det_tensor(k, v.shape, "small", seed)
        elif v.dim() >= 2:
            out[k] = det_tensor(k, v.shape, "conv_w", seed)
        else:  # 1-D weights of plain nn.BatchNorm1d (M2-Track nets)
            out[k] = det_tensor(k, v.shape, "bn_w", seed)
    return out


def pack_state_4bit(sd):
    """Trained weights small enough to store: every floating tensor of two or more dimensions becomes symmetric 4-bit
    codes per output channel (two codes a byte, key ':q4') and float32 channel scales (':scale'); all other entries
    (BatchNorm statistics, biases, counters) are kept exactly.  `unpack_state_4bit` inverts it."""
    import numpy as np
    out = {}
    for k, v in sd.items():
        a = v.detach().cpu().numpy()
        if a.dtype != np.float32 or a.ndim < 2:
            out[k] = a
            continue
        rows = a.reshape(a.shape[0], -1)
        scale = np.abs(rows).max(axis=1, keepdims=True) / 7
        scale[scale == 0] = 1
        codes = (np.round(rows / scale) + 7).astype(np.uint8).ravel()
        codes = np.append(codes, np.zeros(codes.size % 2, np.uint8))
        out[k + ":q4"] = codes[0::2] | (codes[1::2] << 4)
        out[k + ":scale"] = scale.astype(np.float32)
        out[k + ":shape"] = np.array(a.shape, np.int64)
    return out


def unpack_state_4bit(packed):
    """The float32 state dict that `pack_state_4bit` stored (codes times scales, the same numbers on every machine)."""
    import numpy as np
    sd = {}
    for k in packed:
        if k.endswith((":scale", ":shape")):
            continue
        if k.endswith(":q4"):
            name = k[:-3]
            shape = tuple(int(s) for s in packed[name + ":shape"])
            b = packed[k]
            codes = np.stack([b & 15, b >> 4], axis=1).ravel()[:int(np.prod(shape))]
            rows = (codes.astype(np.float32) - 7).reshape(shape[0], -1) * packed[name + ":scale"]
            sd[name] = torch.from_numpy(np.ascontiguousarray(rows.reshape(shape)))
        else:
            sd[k] = torch.from_numpy(np.array(packed[k]))
    return sd
