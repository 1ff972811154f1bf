import numpy as np
import torch

DEV = "cuda:0"
SENTINEL = 7.0
FULL_SMS = 148


def cdiv(a, b):
    return -(-a // b)


def bitwise_equal(a, b):
    if a.dtype == torch.bfloat16:
        return torch.equal(a.view(torch.int16), b.view(torch.int16))
    return torch.equal(a.view(torch.int32), b.view(torch.int32))


def slice_buf(x, c8tot, c8off):
    """x [N,C,D,H,W] at channel group c8off of a C8-planar bf16 buffer of c8tot groups; other channels = SENTINEL."""
    n, c, d, h, w = x.shape
    full = torch.full((n, c8tot * 8, d, h, w), SENTINEL, device=x.device)
    full[:, c8off * 8:c8off * 8 + c] = x
    return to_c8(full.to(DEV))


def sentinel_buf(n, d, c8tot, h, w):
    return torch.full((n, d, c8tot, h, w, 8), SENTINEL, dtype=torch.bfloat16, device=DEV)


def read_slice(buf, c8off, c, device="cpu"):
    """The c channels at group c8off of a C8-planar buffer, after checking every other channel still holds SENTINEL."""
    full = from_c8(buf).to(device)
    lo, hi = c8off * 8, c8off * 8 + c
    assert torch.all(full[:, :lo] == SENTINEL) and torch.all(full[:, hi:] == SENTINEL), "write outside the target slice"
    return full[:, lo:hi]


def run_sm_budgets(fn):
    """[fn() under fpl_set_sm_budget(148), fn() under fpl_set_sm_budget(16)].  At 16 SMs the persistent grids are
    16-32 CTAs, so a CTA walks several tiles (TMEM accumulator ping-pong, barrier phase wrap) or items; the budget is
    always restored."""
    from fplplus_b200 import ops
    outs = []
    try:
        for sms in (FULL_SMS, 16):
            ops.call("fpl_set_sm_budget", sms)
            outs.append(fn())
            torch.cuda.synchronize()
    finally:
        ops.call("fpl_set_sm_budget", FULL_SMS)
    return outs


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


_M32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """Philox4x32-10 (Salmon et al., Random123) on the host, as csrc/common.cuh computes it.  ctr: integer array
    [..., 4] of 32-bit words, key: [..., 2]; returns uint64 [..., 4] holding the 32-bit output words."""
    ctr = np.asarray(ctr, dtype=np.uint64)
    key = np.asarray(key, dtype=np.uint64)
    x0, x1, x2, x3 = (ctr[..., i] for i in range(4))
    k0, k1 = key[..., 0], key[..., 1]
    m0, m1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
    w0, w1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
    s32 = np.uint64(32)
    for _ in range(10):
        p0, p1 = x0 * m0, x2 * m1                   # < 2^64: exact in uint64
        x0, x1, x2, x3 = (p1 >> s32) ^ x1 ^ k0, p1 & _M32, (p0 >> s32) ^ x3 ^ k1, p0 & _M32
        k0, k1 = (k0 + w0) & _M32, (k1 + w1) & _M32
    return np.stack([x0, x1, x2, x3], -1)


def dropout_keep_c8(seed, offset, n, c, d, h, w, p):
    """Keep mask bool [N,C,D,H,W] of the Philox dropout of csrc/common.cuh (dropout_keep8) for a layer of c channels:
    vector vec = ((n*D + d)*C8 + c8)*H*W + h*W + w over the layer's own channel groups, counters 2*vec + offset and
    2*vec + offset + 1 (mod 2^64) as (lo32, hi32, 0, 0), key (lo32(seed), hi32(seed)); the 8 output words feed channels
    0..7 of the group; keep iff (r >> 8) * 2^-24 >= float32(p), i.e. (r >> 8) >= ceil(float32(p) * 2^24) exactly."""
    assert c % 8 == 0
    c8 = c // 8
    seed, offset = int(seed) % (1 << 64), int(offset) % (1 << 64)
    vec = np.arange(n * d * c8 * h * w, dtype=np.uint64)
    ctr = vec * np.uint64(2) + np.uint64(offset)     # wraps mod 2^64 like the device's uint64
    key = np.array([seed & 0xFFFFFFFF, seed >> 32], dtype=np.uint64)
    zero = np.zeros_like(vec)
    words = [philox4x32_10(np.stack([cc & _M32, cc >> np.uint64(32), zero, zero], -1), key)
             for cc in (ctr, ctr + np.uint64(1))]
    r = np.concatenate(words, -1)                    # [vec, 8]: a.x..a.w, b.x..b.w
    thr = int(np.ceil(float(np.float32(p)) * 2.0 ** 24))
    keep = (r >> np.uint64(8)) >= np.uint64(thr)
    return torch.from_numpy(keep.reshape(n, d, c8, h, w, 8).transpose(0, 2, 5, 1, 3, 4).reshape(n, c, d, h, w).copy())


def golden_voxels(out, g, key):
    """``out`` [N, C, ...] at the voxels a sampled golden array holds: g[key] is [N, C, M] at the flat voxel indices
    g[key + '_idx'] of an output of shape g[key + '_shape']."""
    assert tuple(out.shape) == tuple(int(s) for s in g[key + "_shape"]), (tuple(out.shape), g[key + "_shape"])
    idx = g[key + "_idx"].astype(np.int64)
    if torch.is_tensor(out):
        idx = torch.from_numpy(idx).to(out.device)
    return out.reshape(out.shape[0], out.shape[1], -1)[:, :, idx]
