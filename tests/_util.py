import numpy as np
import torch


def bf16_round(t):
    return t.to(torch.bfloat16).float()


def to_c8(x):
    """[N,C,D,H,W] float -> C8-planar bf16 tensor on x.device."""
    from fplplus_b200 import ops
    return ops.ncdhw_to_c8(x)


def from_c8(buf, channels=None):
    from fplplus_b200 import ops
    return ops.c8_to_ncdhw(buf, channels)


def rel_l2(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float((a - b).norm() / (b.norm() + 1e-30))


def max_rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).abs().max() / (b.abs().max() + 1e-30))


def rng(seed):
    return np.random.Generator(np.random.PCG64(seed))


def randn(seed, *shape, scale=1.0):
    return torch.from_numpy((rng(seed).standard_normal(shape) * scale).astype(np.float32))


def golden_voxels(out, g, key):
    """``out`` [N, C, ...] at the voxels a sampled golden array holds: g[key] is [N, C, M] at the flat voxel indices
    g[key + '_idx'] of an output of shape g[key + '_shape']."""
    assert tuple(out.shape) == tuple(int(s) for s in g[key + "_shape"]), (tuple(out.shape), g[key + "_shape"])
    idx = g[key + "_idx"].astype(np.int64)
    if torch.is_tensor(out):
        idx = torch.from_numpy(idx).to(out.device)
    return out.reshape(out.shape[0], out.shape[1], -1)[:, :, idx]
