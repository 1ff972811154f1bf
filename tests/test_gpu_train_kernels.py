"""Per-kernel parity of the training step at multi-tile geometries: the BatchNorm statistics the conv kernels accumulate
and their finalize, the DSBN + PReLU + dropout + max-pool forward and backward in training and eval mode, and the data
and weight gradients.  Every kernel is compared with a float64 torch reference of the same operation on the bf16-rounded
operands it sees (computed on the device, so the full-resolution references fit); each bar names the rounding it allows.

The case lists are chosen with host restatements of the launch decisions (first section, no GPU needed) so that at the
full SM budget and at 16 SMs the persistent kernels walk several items / tiles per CTA, the DSBN walks wrap their chunk
index and cross sample boundaries, and the weight gradients run split-K with ragged slices as well as split = 1.
Outputs go into a channel slice of a wider buffer whose other groups hold SENTINEL; inputs come from a slice at a
non-zero group offset wherever the entry point takes one."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests._util import (DEV, FULL_SMS, SENTINEL, bitwise_equal, cdiv, dropout_keep_c8, from_c8, read_slice,
                         run_sm_budgets, sentinel_buf, slice_buf, to_c8)

EPS = 1e-5
EPS64 = float(np.float32(EPS))          # the kernels add eps as a float32
MOMENTUM = 0.1
RATIOS = (0.0, 3.0, 30.0)               # per-channel mean / std of the BatchNorm inputs, cycled over the channels


def _ops():
    from fplplus_b200 import ops
    return ops


def _lib():
    from fplplus_b200 import lib
    return lib


def _call(name, *a):
    _ops().call(name, *a)


_KEEP = []


def _p(t):
    # the C ABI borrows raw pointers: keep every tensor handed to it alive until the test ends
    if t is None:
        return None
    _KEEP.append(t)
    return _ops().ptr(t)


@pytest.fixture(autouse=True)
def _release_borrowed_tensors():
    yield
    if torch.cuda.is_available():
        torch.cuda.synchronize()
    del _KEEP[:]


def _st():
    return _ops().stream_ptr()


@pytest.fixture
def sm_budgets():
    """run(fn) -> [fn() under fpl_set_sm_budget(148), fn() under fpl_set_sm_budget(16)] (tests/_util.py)."""
    return run_sm_budgets


def _randn(seed, *shape):
    g = torch.Generator(device=DEV)
    g.manual_seed(seed)
    return torch.randn(shape, generator=g, device=DEV)


def _bf16(t):
    return t.to(torch.bfloat16).float()


def _chan(v):
    return v.view(1, -1, 1, 1, 1)


def _csum(t):
    return t.sum((0, 2, 3, 4))


def _ratios(c):
    return torch.tensor([RATIOS[i % len(RATIOS)] for i in range(c)], dtype=torch.float64, device=DEV)


def _ulp_bf16(r):
    """The spacing of bf16 numbers at |r| (0 where r == 0)."""
    a = r.abs()
    e = torch.floor(torch.log2(torch.where(a > 0, a, torch.ones_like(a))))
    return torch.where(a > 0, torch.exp2(e - 7), torch.zeros_like(a))


# ------------------------------------------------------------------------------------------
# host restatements of launch decisions (so that the case lists provably reach them)
# ------------------------------------------------------------------------------------------
def _dsbn_act_grid(sms, n, c, d, h, w, pool_kd):
    """act_fwd_launch (csrc/dsbn.cu): blocks per channel group and the work items (plane, chunk) they walk; chunks of
    2*256 vectors, or 256 pooled vectors for dsbn_act_pool_fwd_kernel."""
    if pool_kd:
        chunks = cdiv((h // 2) * (w // 2), 256)
        items = n * (d // pool_kd) * chunks
    else:
        chunks = cdiv(h * w, 2 * 256)
        items = n * d * chunks
    return max(1, min(cdiv(sms * 8, c // 8), items)), chunks, items


def _dsbn_bwd_grid(sms, n, c, d, h, w):
    """bwd_grid (csrc/dsbn.cu): 8 blocks per SM over the channel groups, at most one per item of kBwdV*256 vectors."""
    chunks = cdiv(h * w, 2 * 256)
    items = n * d * chunks
    return max(1, min(cdiv(sms * 8, c // 8), items)), chunks, items


def _stepped_wrap(bx, chunks, items):
    """A block walks more than one item and its chunk index steps by step_ch != 0 (so the `ch >= chunks` wrap runs)."""
    return items > bx and bx % chunks != 0


def _crosses_sample(bx, chunks, items, d):
    """Some block's next item is a plane of the next sample (the pooled (pn, pd) walk carries into pn)."""
    i = np.arange(max(items - bx, 0))
    return bool(np.any((i // chunks) // d != ((i + bx) // chunks) // d))


def _wgrad_plan(sms, cin, cout, kd, taps, n, d, h, w):
    """(kernel, split, tiles) of wgrad_tc_launch (csrc/conv_wgrad_tc.cu): the h-stacked and row-stacked kernels when
    eligible (csrc/conv_wgrad_hs.cu), else make_wg_cfg's M tiles x N chunks (`pairs`) and the split-K over voxel
    tiles, capped at tiles / 2."""
    if kd == 3 and taps == 9 and cin in (16, 32) and cout % 16 == 0 and d >= 2 and h >= 2 and w >= 16:
        g = cin // 8
        th = 8 if h >= 8 else (h + 1) // 2 * 2
        tw = 32 if (w >= 32 and g == 2) else 16
        tiles = cdiv(h, th) * cdiv(w, tw) * cdiv(d, 2) * n
        return "hs", max(1, min(sms // (cout // 16), tiles)), tiles
    if kd == 1 and taps == 9 and cin == 16 and cout == 8 and h >= 6 and w >= 16:
        th, tw, planes = (12 if h >= 12 else 6), (32 if w >= 32 else 16), (2 if d >= 2 else 1)
        tiles = cdiv(h, th) * cdiv(w, tw) * cdiv(d, planes) * n
        return "rs", min(sms, tiles), tiles
    tw = 32 if w >= 32 else (16 if w >= 16 else 8)
    th = 8 if h >= 8 else (h + 1) // 2 * 2
    g = cin // 8
    ndy = 1
    if d >= 2:
        if kd == 3 and g <= 4 and cout % 16 == 0:
            ndy = 2
        elif kd == 1 and cout == 8 and g <= 2:
            ndy = 4
        elif kd == 1 and cout == 8 and g <= 4:
            ndy = 2
        elif kd == 1 and cout == 16 and g <= 8:
            ndy = 2
    if ndy > 1 or kd * g <= 16:
        mtiles_kd, mtiles_c = 1, 1
    else:
        c8chunk = min(g, 16)
        mtiles_kd, mtiles_c = kd, g // c8chunk
    nb = 8 if cout == 8 else (32 if (cout % 32 == 0 and ndy == 1) else 16)
    pairs = mtiles_kd * mtiles_c * (cout // nb)
    tiles = cdiv(h, th) * cdiv(w, tw) * cdiv(d, ndy) * n
    return "tc", max(1, min(sms // pairs, tiles // 2)), tiles


def _convt_wgrad_split(sms, cin, cout, kd2, n, d, h, w):
    """convt_wgrad_launch (csrc/convt_tc.cu): M tiles of <= 16 channel groups x N chunks, split-K over the 16x8
    low-resolution tiles, capped at tiles / 4."""
    g = cin // 8
    mgroups = min(g, 16)
    m = 64 if mgroups <= 8 else 128
    nb = 32 if cout % 32 == 0 else 16
    plane = 16 * 8 * 16
    if 2 * (mgroups * plane + 4 * kd2 * (nb // 8) * plane) > 200 * 1024 - (m // 8) * plane:
        nb = 16
    pairs = (g // mgroups) * (cout // nb)
    tiles = cdiv(h, 16) * cdiv(w, 8) * d * n
    return max(1, min(sms // pairs, tiles // 4)), tiles


def _stem_wgrad_split(sms, n, d, h, w):
    """fpl_stem_wgrad_tc_launch (csrc/stem_tc.cu): one slice per CTA over the 16x32 tiles."""
    tiles = cdiv(h, 16) * cdiv(w, 32) * n * d
    return min(sms, tiles), tiles


# (n, c, d, h, w, pool_kd, dropout, g1): the bench levels (n = 2) and ragged ones; dropout None / "philox" / "mask";
# g1 False = the gradient arrives through the pool only
DSBN_CASES = [
    (2, 16, 32, 128, 128, 1, None, True),          # full resolution, pool (1,2,2): the pooled walk crosses samples
    (2, 16, 32, 128, 128, 0, "philox", True),      # full resolution, the first unit of a block (dropout, no pool)
    (2, 32, 32, 64, 64, 2, None, False),           # pool (2,2,2), pool-only gradient
    (2, 64, 32, 32, 32, 0, "philox", True),
    (2, 256, 4, 8, 8, 0, "philox", True),          # the deepest level
    (2, 8, 9, 60, 90, 1, None, True),              # W not a power of two, odd depth
    (2, 48, 13, 24, 56, 0, "mask", True),          # 6 channel groups, explicit uint8 mask
]

# (kind, cin, cout, kd, (n, d, h, w)): many tiles per CTA; one case of each kind at the bench's full-resolution level
STATS_CASES = [
    ("tc", 16, 16, 3, (2, 32, 128, 128)),          # N split 1
    ("tc", 16, 16, 1, (2, 16, 64, 64)),
    ("tc", 64, 64, 3, (2, 4, 16, 16)),             # N split 2
    ("tc", 128, 128, 3, (1, 4, 16, 16)),           # N split 4
    ("dfold", 32, 16, 3, (2, 32, 128, 128)),
    ("k311", 48, 16, 3, (2, 32, 128, 128)),        # the hi / lo stem: fpl_patch9_c8(split) + 48-channel k(3,1,1)
    ("stem", 1, 16, 3, (2, 32, 128, 128)),         # fpl_stem_conv_fwd (stem_tc.cu)
]

# (kind, cin, cout, kd or kd2, (n, d, h, w)) of the FORWARD layer; convt: cin low-resolution channels, (d, h, w) the
# low-resolution shape
DGRAD_CASES = [
    ("tc", 32, 16, 3, (2, 32, 128, 128)),
    ("tc", 64, 64, 3, (2, 8, 32, 32)),
    ("tc", 128, 128, 1, (2, 8, 16, 16)),
    ("tc", 256, 256, 3, (2, 4, 8, 8)),
    ("dfold", 16, 16, 3, (2, 32, 128, 128)),
    ("dfold", 64, 32, 3, (2, 32, 32, 32)),
    ("convt", 32, 16, 1, (2, 32, 64, 64)),
    ("convt", 64, 32, 1, (2, 32, 32, 32)),
    ("convt", 256, 128, 2, (2, 4, 8, 8)),
]

WGRAD_CASES = [
    ("conv", 16, 16, 3, (2, 32, 128, 128)),        # h-stacked (32-wide tiles), split 148 over 2048 tiles
    ("conv", 32, 32, 3, (2, 16, 64, 64)),          # h-stacked, four channel groups (16-wide tiles)
    ("conv", 16, 8, 1, (2, 32, 128, 128)),         # row-stacked (the head)
    ("conv", 64, 64, 3, (1, 9, 24, 32)),           # generic, split 13 / 2 over 27 tiles
    ("conv", 256, 256, 3, (2, 4, 8, 8)),           # generic, split 3 over 8 tiles / split 1
    ("conv", 256, 256, 3, (1, 2, 8, 8)),           # generic, split 1 (2 tiles)
    ("conv", 128, 128, 1, (2, 8, 16, 16)),         # generic, k(1,3,3), depth-stacked
    ("k311", 16, 16, 3, (2, 32, 128, 128)),        # fpl_conv3d_wgrad_tc_k311 (the stem's k(3,1,1) form)
    ("stem", 1, 16, 3, (2, 32, 128, 128)),         # fpl_stem_conv_wgrad
    ("convt", 32, 16, 1, (2, 32, 64, 64)),
    ("convt", 256, 128, 2, (2, 4, 8, 8)),
]


def test_case_lists_reach_the_launch_decisions():
    """At 148 and at 16 SMs the case lists run the stepped DSBN walks with a chunk wrap, a pooled backward walk that
    crosses from sample n to n + 1, pools with W a power of two and not, the generic / h-stacked / row-stacked wgrad
    kernels, split-K > 1 with ragged slices and split = 1, and a ConvTranspose wgrad with split > 1."""
    pool_w = {w & (w - 1) == 0 for _n, _c, _d, _h, w, pool_kd, _dr, _g in DSBN_CASES if pool_kd}
    assert pool_w == {True, False}
    assert {pool_kd for *_s, pool_kd, _dr, _g in DSBN_CASES} == {0, 1, 2}
    assert any(d % 2 for _n, _c, d, _h, _w, pool_kd, _dr, _g in DSBN_CASES if pool_kd == 1)
    kinds = {_wgrad_plan(FULL_SMS, ci, co, kd, 9, *shape)[0] for k, ci, co, kd, shape in WGRAD_CASES if k == "conv"}
    assert kinds == {"tc", "hs", "rs"}
    for sms in (FULL_SMS, 16):
        fwd = [_dsbn_act_grid(sms, n, c, d, h, w, 0) for n, c, d, h, w, pk, _dr, _g in DSBN_CASES if not pk]
        bwd = [_dsbn_bwd_grid(sms, n, c, d, h, w) for n, c, d, h, w, _pk, _dr, _g in DSBN_CASES]
        assert any(_stepped_wrap(*g) for g in fwd), sms
        assert any(_stepped_wrap(*g) for g in bwd), sms
        assert any(_crosses_sample(*_dsbn_bwd_grid(sms, n, c, d, h, w), d)
                   for n, c, d, h, w, pk, _dr, _g in DSBN_CASES if pk), sms
        assert any(_dsbn_act_grid(sms, n, c, d, h, w, pk)[0] < _dsbn_act_grid(sms, n, c, d, h, w, pk)[2]
                   for n, c, d, h, w, pk, _dr, _g in DSBN_CASES if pk), sms
        plans = [_wgrad_plan(sms, ci, co, kd, 9, *shape) for k, ci, co, kd, shape in WGRAD_CASES if k == "conv"]
        plans.append(_wgrad_plan(sms, 16, 16, 3, 1, 2, 32, 128, 128))        # the k311 case
        assert any(split > 1 and tiles % split != 0 for _k, split, tiles in plans), sms
        assert any(split == 1 for _k, split, _t in plans), sms
        assert any(kind == "tc" and split > 1 and tiles % split != 0 for kind, split, tiles in plans), sms
        ct = [_convt_wgrad_split(sms, ci, co, kd2, *shape) for k, ci, co, kd2, shape in WGRAD_CASES if k == "convt"]
        assert any(split > 1 for split, _t in ct), sms
        assert _stem_wgrad_split(sms, 2, 32, 128, 128)[0] == sms
    # the restatements against hand-derived values of the source
    assert _dsbn_bwd_grid(FULL_SMS, 2, 16, 32, 128, 128) == (592, 32, 2048)
    assert _wgrad_plan(FULL_SMS, 64, 64, 3, 9, 1, 9, 24, 32) == ("tc", 13, 27)
    assert _wgrad_plan(16, 256, 256, 3, 9, 2, 4, 8, 8) == ("tc", 1, 8)
    assert _wgrad_plan(FULL_SMS, 16, 16, 3, 9, 2, 32, 128, 128) == ("hs", 148, 2048)
    assert _wgrad_plan(16, 16, 8, 1, 9, 2, 32, 128, 128) == ("rs", 16, 1408)
    assert _convt_wgrad_split(FULL_SMS, 256, 128, 2, 2, 4, 8, 8) == (2, 8)


# ------------------------------------------------------------------------------------------
# 1. training BatchNorm statistics -> fpl_dsbn_finalize / fpl_dsbn_bn_act_fwd
# ------------------------------------------------------------------------------------------
def _tc_image(wt, cin, cout, kd, transpose):
    L = _lib().load()
    ci, co = (cout, cin) if transpose else (cin, cout)
    img = torch.empty(L.fpl_conv3d_weight_image_bytes(ci, co, kd) // 2, dtype=torch.bfloat16, device=DEV)
    _call("fpl_conv3d_prep_weight", _p(wt.contiguous()), cin, cout, kd, transpose, _p(img), _st())
    return img


def _dfold_image(wt, cin, cout, transpose):
    L = _lib().load()
    ci, co = (cout, cin) if transpose else (cin, cout)
    img = torch.empty(L.fpl_conv3d_dfold_image_bytes(ci, co) // 2, dtype=torch.bfloat16, device=DEV)
    _call("fpl_conv3d_dfold_prep_weight", _p(wt.contiguous()), cin, cout, transpose, _p(img), _st())
    return img


def _stats_setup(kind, cin, cout, kd, shape, seed):
    """(reference conv without bias [float64], launcher(bias, y, stats))."""
    n, d, h, w = shape
    if kind in ("tc", "dfold"):
        x = _bf16(_randn(seed, n, cin, d, h, w))
        wt = _bf16(_randn(seed + 1, cout, cin, kd, 3, 3) * 0.1)
        ref0 = F.conv3d(x.double(), wt.double(), None, padding=(kd // 2, 1, 1))
        xb = slice_buf(x, 2 * cin // 8, cin // 8)                     # the second half of a concat buffer
        if kind == "tc":
            img = _tc_image(wt, cin, cout, kd, 0)
            return ref0, lambda b, y, s: _call("fpl_conv3d_tc", _p(xb), 2 * cin // 8, cin // 8, _p(img), _p(b), _p(y),
                                               cout // 8, 0, _p(s), n, d, h, w, cin, cout, kd, _st())
        img = _dfold_image(wt, cin, cout, 0)
        return ref0, lambda b, y, s: _call("fpl_conv3d_tc_dfold", _p(xb), 2 * cin // 8, cin // 8, _p(img), _p(b), _p(y),
                                           cout // 8, 0, _p(s), n, d, h, w, cin, cout, _st())
    # the stem: a 1-channel fp32 image and fp32 weights, against the float64 conv of the UNROUNDED operands
    xf = _randn(seed, n, 1, d, h, w)
    wf = _randn(seed + 1, cout, 1, 3, 3, 3) * 0.2
    ref0 = F.conv3d(xf.double(), wf.double(), None, padding=1)
    if kind == "stem":
        return ref0, lambda b, y, s: _call("fpl_stem_conv_fwd", _p(xf), _p(wf), _p(b), _p(y), cout // 8, 0, _p(s), n, 1,
                                           d, h, w, cout, 3, _st())
    xs4 = torch.empty((n, d, 4, h, w, 8), dtype=torch.bfloat16, device=DEV)
    _call("fpl_patch9_c8", _p(xf), _p(xs4), 1, n, d, h, w, _st())
    wk = wf[:, 0].reshape(cout, 3, 9).permute(0, 2, 1)
    hi = _bf16(wk)
    w48 = torch.zeros(cout, 48, 3, device=DEV)
    w48[:, 0:9], w48[:, 16:25], w48[:, 32:41] = hi, hi, wk - hi
    img = torch.empty(48 * 3 * cout, dtype=torch.bfloat16, device=DEV)
    _call("fpl_conv3d_k311_prep_weight", _p(w48), 48, cout, _p(img), _st())
    return ref0, lambda b, y, s: _call("fpl_conv3d_tc_k311", _p(xs4), 4, 0, _p(img), _p(b), _p(y), cout // 8, 0, _p(s),
                                       n, d, h, w, 48, cout, 32, _st())


def _ulps(a, b):
    return int((a.view(torch.int32).long() - b.view(torch.int32).long()).abs().max())


@pytest.mark.gpu
@pytest.mark.parametrize("kind,cin,cout,kd,shape", STATS_CASES)
def test_training_statistics_and_finalize_match_float64(kind, cin, cout, kd, shape, sm_budgets, record_property):
    """Sum y and sum y^2 as the conv epilogues accumulate them (fp32 per warp / thread over all the tiles it walks, then
    fp64 atomics), with per-channel mean / std of 0, 3 and 30 set through the conv bias, and what fpl_dsbn_finalize and
    the fused fpl_dsbn_bn_act_fwd make of them (var = E[y^2] - mean^2)."""
    n, d, h, w = shape
    if kind == "tc":
        from tests.test_gpu_infer_kernels import _tc_nsub
        assert _tc_nsub(cin, cout, n, d, h, w) == {16: 1, 64: 2, 128: 4}[cout]
    ref0, launch = _stats_setup(kind, cin, cout, kd, shape, 601)
    bias = (_ratios(cout) * ref0.std((0, 2, 3, 4))).float()
    ref = ref0 + _chan(bias.double())
    cnt = n * d * h * w
    ref_s1, ref_abs1, ref_s2 = _csum(ref), _csum(ref.abs()), _csum(ref * ref)
    m64 = ref_s1 / cnt
    var64 = _csum((ref - _chan(m64)) ** 2) / cnt
    invstd64 = 1.0 / torch.sqrt(var64 + EPS64)
    del ref0, ref
    gamma, beta = (_randn(602, cout) * 0.3 + 1.0), _randn(603, cout) * 0.2
    rm0, rv0 = _randn(604, cout) * 0.1, _randn(605, cout).abs() + 0.5
    sl = torch.tensor([0.25], device=DEV)

    def run():
        y = torch.empty((n, d, cout // 8, h, w, 8), dtype=torch.bfloat16, device=DEV)
        stats = torch.zeros(2 * cout, dtype=torch.float64, device=DEV)
        launch(bias, y, stats)
        res = {"stats": stats}
        for fused in (0, 1):
            rm, rv, nbt = rm0.clone(), rv0.clone(), torch.tensor(5, dtype=torch.int64, device=DEV)
            out = [torch.empty(cout, device=DEV) for _ in range(4)]
            if fused:
                a = sentinel_buf(n, d, cout // 8 + 1, h, w)
                _call("fpl_dsbn_bn_act_fwd", _p(y), _p(stats), cnt, _p(gamma), _p(beta), _p(rm), _p(rv), _p(nbt), MOMENTUM,
                      EPS, 1, *[_p(t) for t in out], _p(sl), _p(a), cout // 8 + 1, 1, None, 0, 0, None, 0, 0.0, None, 0, 0,
                      None, n, d, h, w, cout, _st())
            else:
                _call("fpl_dsbn_finalize", _p(stats), cnt, _p(gamma), _p(beta), _p(rm), _p(rv), _p(nbt), MOMENTUM, EPS, 1,
                      *[_p(t) for t in out], cout, _st())
            res[fused] = out + [rm, rv, nbt]
        return res

    worst = 0.0
    for sms, res in zip((FULL_SMS, 16), sm_budgets(run)):
        s = res["stats"]
        # fp32 partial sums over many tiles, flushed into fp64: a few 2^-24 of the sum of magnitudes per term
        assert bool(((s[:cout] - ref_s1).abs() <= 1e-5 * ref_abs1).all()), (sms, ((s[:cout] - ref_s1).abs() / ref_abs1).max())
        assert bool(((s[cout:] - ref_s2).abs() <= 1e-5 * ref_s2).all()), (sms, ((s[cout:] - ref_s2).abs() / ref_s2).max())
        scale, shift, smean, sinv, rm, rv, nbt = res[0]
        inv_rel = ((sinv.double() - invstd64).abs() / invstd64)
        worst = max(worst, float(inv_rel.max()))
        record_property("invstd_rel_err_%d" % sms, float(inv_rel.max()))
        # var = E[y^2] - mean^2 magnifies the error of sum y^2 by 1 + (mean/std)^2 = 901 at mean/std = 30
        assert float(inv_rel.max()) <= 2e-5, (sms, inv_rel.tolist())
        mean_tol = 1e-5 * ref_abs1 / cnt + 2.0 ** -23 * m64.abs()
        assert bool(((smean.double() - m64).abs() <= mean_tol).all()), sms
        rm_ref = (1 - MOMENTUM) * rm0.double() + MOMENTUM * m64
        rv_ref = (1 - MOMENTUM) * rv0.double() + MOMENTUM * var64 * cnt / (cnt - 1)
        # fp32 momentum update (a few 2^-24) on top of the mean / variance errors allowed above
        assert bool(((rm.double() - rm_ref).abs() <= 4e-7 * (rm0.double().abs() + m64.abs()) + MOMENTUM * mean_tol).all())
        assert bool(((rv.double() - rv_ref).abs() <= 4e-7 * rv_ref + MOMENTUM * 4e-5 * var64 * cnt / (cnt - 1)).all())
        assert int(nbt) == 6
        # the fused prologue is the same arithmetic: 1 ulp of fp32 contraction
        for a, b in zip(res[0][:6], res[1][:6]):
            assert _ulps(a, b) <= 1
        assert int(res[1][6]) == 6
    record_property("invstd_rel_err_worst", worst)


# ------------------------------------------------------------------------------------------
# 2. DSBN + PReLU + dropout + max-pool, forward and backward, training and eval
# ------------------------------------------------------------------------------------------
def _dense_mask_c8(keep):
    """bool [N,C,D,H,W] -> uint8 in dense C8-planar element order."""
    n, c, d, h, w = keep.shape
    return keep.reshape(n, c // 8, 8, d, h, w).permute(0, 3, 1, 4, 5, 2).contiguous().to(torch.uint8)


def _windows(t, kd):
    """[N,C,D,H,W] -> [N,C,D/kd,H/2,W/2,kd*4], window position (dd*2 + hh)*2 + ww: the argmax code order."""
    n, c, d, h, w = t.shape
    return t.reshape(n, c, d // kd, kd, h // 2, 2, w // 2, 2).permute(0, 1, 2, 4, 6, 3, 5, 7).reshape(
        n, c, d // kd, h // 2, w // 2, kd * 4)


def _unwindow(t, kd):
    n, c, d2, h2, w2, _q = t.shape
    return t.reshape(n, c, d2, h2, w2, kd, 2, 2).permute(0, 1, 2, 5, 3, 6, 4, 7).reshape(n, c, d2 * kd, h2 * 2, w2 * 2)


def _codes_ncdhw(idx):
    n, d2, c8, h2, w2, _e = idx.shape
    return idx.permute(0, 2, 5, 1, 3, 4).reshape(n, c8 * 8, d2, h2, w2).long()


@pytest.mark.gpu
@pytest.mark.parametrize("training", [1, 0])
@pytest.mark.parametrize("n,c,d,h,w,pool_kd,drop,g1_on", DSBN_CASES)
def test_dsbn_fwd_bwd_match_float64_autograd(n, c, d, h, w, pool_kd, drop, g1_on, training, sm_budgets):
    """fpl_dsbn_bn_act_fwd -> fpl_dsbn_act_bwd_reduce -> fpl_dsbn_act_bwd_apply_fin (and fpl_dsbn_act_bwd_apply) against
    float64 autograd of batch_norm -> prelu -> dropout -> max_pool3d.  The pooled gradient is routed by the kernel's
    argmax codes, which are checked first against a first-max-wins argmax of the kernel's bf16 activations."""
    c8, cnt = c // 8, n * d * h * w
    d2, h2, w2 = (d // pool_kd, h // 2, w // 2) if pool_kd else (0, 0, 0)
    ratios = _ratios(c)
    std = (torch.rand(c, device=DEV, generator=torch.Generator(device=DEV).manual_seed(701)) + 0.5).double()
    y = _bf16((_randn(702, n, c, d, h, w).double() * _chan(std) + _chan(ratios * std)).float())
    y64 = y.double()
    yb = to_c8(y)
    stats = torch.cat([_csum(y64), _csum(y64 * y64)]).contiguous()
    gamma, beta = _randn(703, c) * 0.3 + 1.0, _randn(704, c) * 0.2
    rm0 = ((ratios + 0.1 * _randn(705, c).double()) * std).float()
    rv0 = (std * std * (0.8 + 0.4 * torch.rand(c, device=DEV, generator=torch.Generator(device=DEV).manual_seed(706)))).float()
    slope = 0.2
    sl = torch.tensor([slope], device=DEV)
    p, mask, seed, offset, seed_dev, keep = 0.0, None, 0, 0, None, None
    if drop == "philox":
        p, seed, offset = 0.3, 2 ** 63 + 12345, 3 * 2 ** 32 + 16
        seed_all = torch.tensor([3, 2 ** 40 + 7, 9], dtype=torch.int64, device=DEV)
        seed_dev = seed_all[1:2]
        keep = dropout_keep_c8((seed + 2 ** 40 + 7) % 2 ** 64, offset, n, c, d, h, w, p).to(DEV)
    elif drop == "mask":
        p = 0.4
        keep = torch.rand((n, c, d, h, w), device=DEV, generator=torch.Generator(device=DEV).manual_seed(707)) >= p
        mask = _dense_mask_c8(keep)
    keep_scale = float(np.float32(1.0) / (np.float32(1.0) - np.float32(p)))      # the kernels' fp32 1 / (1 - p)
    g1 = _bf16(_randn(708, n, c, d, h, w)) if g1_on else None
    g1b = slice_buf(g1, c8 + 3, 2) if g1_on else None
    gp = _bf16(_randn(709, n, c, d2, h2, w2)) if pool_kd else None
    gpb = slice_buf(gp, c8 + 2, 1) if pool_kd else None
    pre = [_randn(710 + i, c) for i in range(2)] + [_randn(712, 1), _randn(713, c)]   # dgamma, dbeta, dslope, dbias
    numel = n * d * c8 * h * w * 8
    state = {}

    def dy_buf():
        return torch.full((numel + 4096,), SENTINEL, dtype=torch.bfloat16, device=DEV)   # dense dy, then a guard tail

    def run():
        rm, rv, nbt = rm0.clone(), rv0.clone(), torch.tensor(3, dtype=torch.int64, device=DEV)
        aff = [torch.empty(c, device=DEV) for _ in range(4)]                  # scale, shift, save_mean, save_invstd
        a = sentinel_buf(n, d, c8 + 2, h, w)
        pooled = sentinel_buf(n, d2, c8 + 1, h2, w2) if pool_kd else None
        idx = torch.full((n, d2, c8, h2, w2, 8), 255, dtype=torch.uint8, device=DEV) if pool_kd else None
        _call("fpl_dsbn_bn_act_fwd", _p(yb), _p(stats), cnt, _p(gamma), _p(beta), _p(rm), _p(rv), _p(nbt), MOMENTUM, EPS,
              training, *[_p(t) for t in aff], _p(sl), _p(a), c8 + 2, 1, _p(pooled), c8 + 1, 1, _p(idx), pool_kd, p,
              _p(mask), seed, offset, _p(seed_dev), n, d, h, w, c, _st())
        common = (_p(yb), _p(g1b), c8 + 3, 2, _p(gpb), c8 + 2, 1, _p(idx), pool_kd, *[_p(t) for t in aff], _p(sl), p,
                  _p(mask), seed, offset, _p(seed_dev))
        red = torch.zeros(2 * c + 1, dtype=torch.float64, device=DEV)
        _call("fpl_dsbn_act_bwd_reduce", *common, _p(red), n, d, h, w, c, _st())
        dy = dy_buf()
        fin = [t.clone() for t in pre]
        _call("fpl_dsbn_act_bwd_apply_fin", *common, _p(red), training, _p(dy), n, d, h, w, c, _st(), *[_p(t) for t in fin])
        dy_same = None
        if "red" in state:                  # the apply pass under this budget, fed the other budget's reduction
            dy_same = dy_buf()
            _call("fpl_dsbn_act_bwd_apply", *common, _p(state["red"]), training, _p(dy_same), n, d, h, w, c, _st())
        else:
            state["red"] = red
        return dict(aff=aff, rm=rm, rv=rv, nbt=nbt, a=a, pooled=pooled, idx=idx, red=red, dy=dy, fin=fin, dy_same=dy_same)

    r148, r16 = sm_budgets(run)
    # elementwise forward: bit-identical whatever the grid; the apply pass too, given the same reduction
    for key in ("a", "pooled", "rm", "rv"):
        if r148[key] is not None:
            assert bitwise_equal(r148[key], r16[key]), key
    for t148, t16 in zip(r148["aff"], r16["aff"]):
        assert bitwise_equal(t148, t16)
    assert torch.equal(r148["nbt"], r16["nbt"]) and (not pool_kd or torch.equal(r148["idx"], r16["idx"]))
    assert bitwise_equal(r16["dy_same"], r148["dy"])
    for r in (r148, r16):
        assert bool((r["dy"][numel:] == SENTINEL).all())

    scale, shift, smean, sinv = (t.double() for t in r148["aff"])
    if training:
        m_used = stats[:c] / cnt
        var64 = stats[c:] / cnt - m_used * m_used
        inv_used = 1.0 / torch.sqrt(var64 + EPS64)
        assert bool(((smean - m_used).abs() <= 2.0 ** -24 * m_used.abs() + 1e-9 * std).all())
        assert bool(((sinv - inv_used).abs() <= 2.0 ** -23 * inv_used).all())
        rm_ref = (1 - MOMENTUM) * rm0.double() + MOMENTUM * m_used
        rv_ref = (1 - MOMENTUM) * rv0.double() + MOMENTUM * var64 * cnt / (cnt - 1)
        assert bool(((r148["rm"].double() - rm_ref).abs() <= 4e-7 * (rm0.double().abs() + m_used.abs())).all())
        assert bool(((r148["rv"].double() - rv_ref).abs() <= 4e-7 * rv_ref).all())
        assert int(r148["nbt"]) == 4
    else:
        m_used, inv_used = rm0.double(), 1.0 / torch.sqrt(rv0.double() + EPS64)
        assert torch.equal(smean.float(), rm0) and bool(((sinv - inv_used).abs() <= 2.0 ** -22 * inv_used).all())
        assert torch.equal(r148["rm"], rm0) and torch.equal(r148["rv"], rv0) and int(r148["nbt"]) == 3

    act = read_slice(r148["a"], 1, c, device=DEV)
    # the PReLU branch of each voxel as the kernel takes it: y*scale + shift with the kernel's fp32 scale / shift (the
    # float64 sum of the exact product rounds but never changes sign)
    pos = (y64 * _chan(scale) + _chan(shift)) > 0
    g_route = torch.zeros_like(y64) if g1 is None else g1.double()
    if pool_kd:
        win = _windows(act, pool_kd)
        eq = win == win.amax(-1, keepdim=True)
        first = (eq & (eq.cumsum(-1) == 1)).to(torch.uint8).argmax(-1)
        codes = _codes_ncdhw(r148["idx"])
        assert torch.equal(codes, first)                                  # first max wins, on the bf16 activations
        assert torch.equal(read_slice(r148["pooled"], 1, c, device=DEV), win.amax(-1))
        onehot = (codes.unsqueeze(-1) == torch.arange(pool_kd * 4, device=DEV)).double()
        g_route = g_route + _unwindow(onehot * gp.double().unsqueeze(-1), pool_kd)
    keepf = torch.ones_like(y64) if keep is None else keep.double() * keep_scale

    yv = y64.clone().requires_grad_(True)
    gv, bv = gamma.double().requires_grad_(True), beta.double().requires_grad_(True)
    sv = torch.tensor([slope], dtype=torch.float64, device=DEV, requires_grad=True)
    if training:
        z = F.batch_norm(yv, None, None, gv, bv, training=True, eps=EPS64)
    else:
        z = F.batch_norm(yv, rm0.double(), rv0.double(), gv, bv, training=False, eps=EPS64)
    a64 = torch.where(pos, z, sv * z) * keepf
    (a64 * g_route).sum().backward()
    a64 = a64.detach()
    # forward: the bf16 rounding of the output (half an ulp, <= 2^-8 relative) plus the fp32 affine map
    assert bool(((act.double() - a64).abs() <= 2.0 ** -8 * a64.abs() + 1e-5 * a64.abs().max()).all())

    dz = g_route * keepf * torch.where(pos, torch.ones_like(y64), torch.full_like(y64, slope))
    s_dz = _csum(dz.abs())
    # sum dz*xhat is formed as invstd * (sum dz*y - mean * sum dz): those are the terms the fp32 partials hold
    s_dzx = inv_used * (_csum((dz * y64).abs()) + m_used.abs() * s_dz)
    s_sl = float((z.detach().abs() * (g_route * keepf).abs() * (~pos)).sum())
    ref_red = [bv.grad, gv.grad, sv.grad]
    for r in (r148, r16):
        red = r["red"]
        # fp32 per-thread and per-block partials before the fp64 atomics: 1e-5 of the sum of the terms' magnitudes
        assert bool(((red[:c] - ref_red[0]).abs() <= 1e-5 * s_dz).all())
        assert bool(((red[c:2 * c] - ref_red[1]).abs() <= 1e-5 * s_dzx).all())
        assert abs(float(red[2 * c]) - float(ref_red[2])) <= 1e-5 * s_sl
    dg, db, dsl, dbias = (t.double() for t in r148["fin"])
    pg, pb, psl, pbias = (t.double() for t in pre)
    # accumulated into the pre-filled gradients: the reduction bar, 1e-4 of the same scale, plus the fp32 add
    assert bool(((dg - (pg + ref_red[1])).abs() <= 1e-4 * s_dzx + 2.0 ** -23 * pg.abs()).all())
    assert bool(((db - (pb + ref_red[0])).abs() <= 1e-4 * s_dz + 2.0 ** -23 * pb.abs()).all())
    assert abs(float(dsl - (psl + ref_red[2]))) <= 1e-4 * s_sl + 2.0 ** -23 * abs(float(psl))
    if training:
        assert torch.equal(r148["fin"][3], pre[3])            # the conv bias feeds BatchNorm: its gradient is 0
    else:
        assert bool(((dbias - (pbias + scale * ref_red[0])).abs() <= 1e-4 * scale.abs() * s_dz + 2.0 ** -23 * pbias.abs()).all())

    dy = from_c8(r148["dy"][:numel].view(n, d, c8, h, w, 8)).double()
    ref_dy = yv.grad
    # the bf16 rounding of dy plus the fp32 per-channel constants of the apply pass (which cancel at mean/std = 30)
    err = (dy - ref_dy).abs() - 2 * _ulp_bf16(ref_dy) - 1e-5 * ref_dy.abs().max()
    assert float(err.max()) <= 0, float(err.max())


# ------------------------------------------------------------------------------------------
# 3. data gradients
# ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind,cin,cout,kd,shape", DGRAD_CASES)
def test_dgrad_matches_float64_and_is_grid_independent(kind, cin, cout, kd, shape, sm_budgets, record_property):
    """dx of fpl_conv3d_tc (transpose image), fpl_conv3d_tc_dfold (transpose = 1) and fpl_convt_k2s2_dgrad_tc: dy read
    from a slice, dx written into a sentinel-guarded slice, each output written once (bitwise the same at 148 and 16
    SMs)."""
    n, d, h, w = shape
    if kind == "convt":
        wt = _bf16(_randn(801, cin, cout, kd, 2, 2) * 0.2)
        dy = _bf16(_randn(802, n, cout, d * kd, 2 * h, 2 * w))
        img = torch.empty(_lib().load().fpl_convt_weight_image_bytes(cin, cout, kd) // 2, dtype=torch.bfloat16, device=DEV)
        _call("fpl_convt_prep_weight", _p(wt), cin, cout, kd, 1, _p(img), _st())
        ref = F.conv3d(dy.double(), wt.double(), stride=(kd, 2, 2))
        bound = F.conv3d(dy.double().abs(), wt.double().abs(), stride=(kd, 2, 2))
    else:
        wt = _bf16(_randn(801, cout, cin, kd, 3, 3) * 0.1)
        dy = _bf16(_randn(802, n, cout, d, h, w))
        img = _tc_image(wt, cin, cout, kd, 1) if kind == "tc" else _dfold_image(wt, cin, cout, 1)
        ref = F.conv_transpose3d(dy.double(), wt.double(), padding=(kd // 2, 1, 1))
        bound = F.conv_transpose3d(dy.double().abs(), wt.double().abs(), padding=(kd // 2, 1, 1))
    dyb = slice_buf(dy, cout // 8 + 1, 1)

    def run():
        dx = sentinel_buf(n, d, cin // 8 + 2, h, w)
        if kind == "tc":
            _call("fpl_conv3d_tc", _p(dyb), cout // 8 + 1, 1, _p(img), None, _p(dx), cin // 8 + 2, 1, None, n, d, h, w, cout,
                  cin, kd, _st())
        elif kind == "dfold":
            _call("fpl_conv3d_tc_dfold", _p(dyb), cout // 8 + 1, 1, _p(img), None, _p(dx), cin // 8 + 2, 1, None, n, d, h, w,
                  cout, cin, _st())
        else:
            _call("fpl_convt_k2s2_dgrad_tc", _p(dyb), cout // 8 + 1, 1, _p(img), _p(dx), cin // 8 + 2, 1, n, d, h, w, cin, cout,
                  kd, _st())
        return dx

    dx148, dx16 = sm_budgets(run)
    assert bitwise_equal(dx148, dx16)
    got = read_slice(dx148, 1, cin, device=DEV).double()
    # bf16 output rounding (<= 2^-8 relative) plus fp32 accumulation, 2^-16 of the sum of the terms' magnitudes
    tol = 2.0 ** -8 * ref.abs() + 2.0 ** -16 * bound
    ratio = float(((got - ref).abs() / tol).max())
    record_property("dgrad_err_over_bar", ratio)
    assert ratio <= 1.0, ratio


# ------------------------------------------------------------------------------------------
# 4. weight gradients
# ------------------------------------------------------------------------------------------
def _wgrad_operands(kind, cin, cout, kd, shape, seed):
    """x >= 0 as after PReLU, dy zero-mean per channel as BatchNorm's backward leaves it; both bf16-rounded."""
    n, d, h, w = shape
    x = _randn(seed, n, cin, d, h, w).abs()
    if kind != "stem":
        x = _bf16(x)                                  # the stem reads the fp32 image
    do, ho, wo = (d * kd, 2 * h, 2 * w) if kind == "convt" else (d, h, w)
    r = _randn(seed + 1, n, cout, do, ho, wo)
    dy = _bf16(r - r.mean((0, 2, 3, 4), keepdim=True))
    return x, dy


def _wgrad_ref(kind, x, dy, wshape, kd):
    """float64 weight gradient of (x, dy) and of (|x|, |dy|), the latter bounding the accumulation error."""
    out = []
    for xx, gg in ((x.double(), dy.double()), (x.double().abs(), dy.double().abs())):
        if kind == "convt":
            n, ci, d, h, w = xx.shape
            g = gg.reshape(n, gg.shape[1], d, kd, h, 2, w, 2)
            out.append(torch.einsum("nidhw,nodahbwc->ioabc", xx, g))
        else:
            pad = (1, 0, 0) if kind == "k311" else (kd // 2, 1, 1)
            out.append(torch.nn.grad.conv3d_weight(xx, wshape, gg, padding=pad))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("kind,cin,cout,kd,shape", WGRAD_CASES)
def test_wgrad_matches_float64_within_the_accumulation_bound(kind, cin, cout, kd, shape, sm_budgets, record_property):
    """The generic, h-stacked and row-stacked kernels behind fpl_conv3d_wgrad_tc and its tap-major form plus the fold,
    fpl_conv3d_wgrad_tc_k311, fpl_stem_conv_wgrad and fpl_convt_k2s2_wgrad_tc(_tapmajor), at both SM budgets (different
    split-K), accumulating into pre-filled gradients."""
    n, d, h, w = shape
    x, dy = _wgrad_operands(kind, cin, cout, kd, shape, 901)
    wshape = {"convt": (cin, cout, kd, 2, 2), "k311": (cout, cin, 3, 1, 1)}.get(kind, (cout, cin, kd, 3, 3))
    ref, bound = _wgrad_ref(kind, x, dy, wshape, kd)
    dshape = (cout, cin, 3) if kind == "k311" else wshape
    ref, bound = ref.reshape(dshape), bound.reshape(dshape)
    pre = _randn(903, *dshape) * float(ref.abs().mean())
    xb = None if kind == "stem" else slice_buf(x, cin // 8 + 2, 1)
    dyb = slice_buf(dy, cout // 8 + 1, 1)
    xa = (_p(xb), cin // 8 + 2, 1, _p(dyb), cout // 8 + 1, 1)
    taps = 4 * kd if kind == "convt" else kd * 9

    def fold(scratch, dw):
        arr = lambda t: (ctypes.c_void_p * 1)(t.data_ptr())
        one = lambda v: (ctypes.c_int * 1)(v)
        _call("fpl_wgrad_tapmajor_to_dw_batch", 1, arr(scratch), arr(dw), one(cout), one(cin),
              one(-taps if kind == "convt" else taps), None, _st())

    def run():
        outs = []
        dw = pre.clone()
        if kind == "conv":
            _call("fpl_conv3d_wgrad_tc", *xa, _p(dw), n, d, h, w, cin, cout, kd, _st())
        elif kind == "k311":
            _call("fpl_conv3d_wgrad_tc_k311", *xa, _p(dw), n, d, h, w, cin, cout, _st())
        elif kind == "stem":
            _call("fpl_stem_conv_wgrad", _p(x), _p(dyb), cout // 8 + 1, 1, _p(dw), n, cin, d, h, w, cout, kd, _st())
        else:
            _call("fpl_convt_k2s2_wgrad_tc", *xa, _p(dw), n, d, h, w, cin, cout, kd, _st())
        outs.append(dw)
        if kind in ("conv", "convt"):
            scratch = torch.zeros(taps * cout * cin, device=DEV)
            name = "fpl_conv3d_wgrad_tc_tapmajor" if kind == "conv" else "fpl_convt_k2s2_wgrad_tc_tapmajor"
            _call(name, *xa, _p(scratch), n, d, h, w, cin, cout, kd, _st())
            dw2 = pre.clone()
            fold(scratch, dw2)
            outs.append(dw2)
        return outs

    worst = 0.0
    for outs in sm_budgets(run):
        for dw in outs:
            # fp32 accumulation in TMEM / registers and fp32 atomics over the split-K slices: 2^-16 of the sum of the
            # terms' magnitudes, plus the fp32 add into the pre-filled gradient
            err = (dw.double() - (pre.double() + ref)).abs()
            tol = 2.0 ** -16 * bound + 2.0 ** -23 * (pre.double() + ref).abs()
            worst = max(worst, float((err / tol).max()))
            record_property("wgrad_err_over_sum_abs", float((err / bound.clamp_min(1e-30)).max()))
    record_property("wgrad_err_over_bar", worst)
    assert worst <= 1.0, worst
