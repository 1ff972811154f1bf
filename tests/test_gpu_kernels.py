"""GPU: every C-ABI kernel against a plain torch fp32 CPU reference of the same op (run on the
bf16-rounded inputs the kernel sees) -- the per-kernel parity layer under the network tests."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests._util import bf16_round, dropout_keep_c8, from_c8, max_rel, randn, rel_l2, to_c8

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _ops():
    from fplplus_b200 import ops
    return ops


def _call(name, *a):
    _ops().call(name, *a)


_KEEP = []


def _p(t):
    # the C ABI borrows raw pointers: keep every tensor handed to it alive until the test ends
    # (a temporary like ``w.to(DEV)`` would otherwise go back to the caching allocator at once)
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


def _conv_ref(x, w, b, kd):
    return F.conv3d(x, w, b, padding=(kd // 2, 1, 1))


# ------------------------------------------------------------------------------------------
# convolution: direct kernel vs torch, tensor-core kernel vs direct kernel
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cin,cout,kd,shape", [(16, 16, 3, (2, 4, 20, 12)), (32, 16, 3, (1, 3, 16, 8)),
                                               (8, 24, 1, (1, 2, 9, 10)), (64, 32, 3, (1, 2, 8, 8))])
def test_conv3d_direct_fwd_and_stats(cin, cout, kd, shape):
    n, d, h, w = shape
    x = bf16_round(randn(1, n, cin, d, h, w))
    wt = randn(2, cout, cin, kd, 3, 3, scale=0.1)
    b = randn(3, cout, scale=0.1)
    ref = _conv_ref(x, wt, b, kd)
    xb = to_c8(x.to(DEV))
    y = torch.empty((n, d, cout // 8, h, w, 8), dtype=torch.bfloat16, device=DEV)
    stats = torch.zeros(2 * cout, dtype=torch.float64, device=DEV)
    _call("fpl_conv3d_direct", _p(xb), cin // 8, 0, _p(wt.to(DEV)), _p(b.to(DEV)), _p(y), cout // 8, 0, _p(stats),
          n, d, h, w, cin, cout, kd, 0, 0, _st())
    out = from_c8(y).cpu()
    assert max_rel(out, ref) < 6e-3          # bf16 output rounding only
    s = stats.cpu()
    np.testing.assert_allclose(s[:cout], ref.double().sum((0, 2, 3, 4)), rtol=1e-4, atol=1e-3)
    np.testing.assert_allclose(s[cout:], (ref.double() ** 2).sum((0, 2, 3, 4)), rtol=1e-4, atol=1e-3)


TC_CASES = [
    (16, 16, 3, (2, 4, 32, 16)), (32, 16, 3, (1, 3, 20, 12)), (16, 32, 3, (1, 2, 16, 8)),
    (32, 32, 3, (1, 5, 24, 24)), (64, 32, 3, (1, 2, 16, 16)), (64, 64, 3, (2, 3, 16, 8)),
    (128, 128, 3, (1, 2, 8, 8)), (256, 128, 3, (1, 2, 4, 4)), (256, 256, 3, (2, 1, 2, 2)),
    (16, 16, 1, (1, 3, 18, 10)), (64, 64, 1, (1, 2, 16, 16)), (48, 80, 3, (1, 2, 10, 9)),
]


@pytest.mark.parametrize("cin,cout,kd,shape", TC_CASES)
def test_conv3d_tc_matches_direct_and_torch(cin, cout, kd, shape):
    from fplplus_b200 import lib as L
    n, d, h, w = shape
    x = bf16_round(randn(11, n, cin, d, h, w))
    wt = bf16_round(randn(12, cout, cin, kd, 3, 3, scale=0.1))
    b = randn(13, cout, scale=0.1)
    ref = _conv_ref(x, wt, b, kd)
    xb = to_c8(x.to(DEV))
    nbytes = L.load().fpl_conv3d_weight_image_bytes(cin, cout, kd)
    assert nbytes == cin * cout * kd * 9 * 2
    img = torch.empty(nbytes // 2, dtype=torch.bfloat16, device=DEV)
    wd, bd = wt.to(DEV), b.to(DEV)
    _call("fpl_conv3d_prep_weight", _p(wd), cin, cout, kd, 0, _p(img), _st())
    y = torch.zeros((n, d, cout // 8, h, w, 8), dtype=torch.bfloat16, device=DEV)
    stats = torch.zeros(2 * cout, dtype=torch.float64, device=DEV)
    _call("fpl_conv3d_tc", _p(xb), cin // 8, 0, _p(img), _p(bd), _p(y), cout // 8, 0, _p(stats), n, d, h, w, cin, cout,
          kd, _st())
    torch.cuda.synchronize()
    out = from_c8(y).cpu()
    assert max_rel(out, ref) < 6e-3, (max_rel(out, ref), rel_l2(out, ref))
    y2 = torch.zeros_like(y)
    _call("fpl_conv3d_direct", _p(xb), cin // 8, 0, _p(wd), _p(bd), _p(y2), cout // 8, 0, None, n, d, h, w, cin, cout,
          kd, 0, 1, _st())
    out2 = from_c8(y2).cpu()
    # same bf16 operands, fp32 accumulation in a different order: at most 1 bf16 ulp apart
    assert max_rel(out, out2) < 5e-3
    assert (out != out2).float().mean() < 0.05
    s = stats.cpu()
    np.testing.assert_allclose(s[:cout], ref.double().sum((0, 2, 3, 4)), rtol=1e-4, atol=2e-3)
    np.testing.assert_allclose(s[cout:], (ref.double() ** 2).sum((0, 2, 3, 4)), rtol=1e-4, atol=2e-3)


def test_conv3d_tc_reads_and_writes_channel_slices():
    """x is the second half of a 2C concat buffer, y the first half of another."""
    from fplplus_b200 import lib as L
    n, d, h, w, c = 1, 2, 16, 16, 16
    full = bf16_round(randn(21, n, 2 * c, d, h, w))
    wt = bf16_round(randn(22, c, c, 3, 3, 3, scale=0.1))
    ref = _conv_ref(full[:, c:], wt, None, 3)
    xb = to_c8(full.to(DEV))
    img = torch.empty(c * c * 27, dtype=torch.bfloat16, device=DEV)
    _call("fpl_conv3d_prep_weight", _p(wt.to(DEV)), c, c, 3, 0, _p(img), _st())
    y = torch.full((n, d, 2 * c // 8, h, w, 8), 7.0, dtype=torch.bfloat16, device=DEV)
    _call("fpl_conv3d_tc", _p(xb), 2 * c // 8, c // 8, _p(img), None, _p(y), 2 * c // 8, 0, None, n, d, h, w, c, c, 3, _st())
    out = from_c8(y).cpu()
    assert max_rel(out[:, :c], ref) < 6e-3
    assert torch.all(out[:, c:] == 7.0)


@pytest.mark.parametrize("impl", ["direct", "tc"])
@pytest.mark.parametrize("cin,cout,kd,shape", [(32, 16, 3, (1, 3, 16, 8)), (16, 32, 1, (1, 2, 16, 16)),
                                               (64, 64, 3, (1, 2, 8, 8))])
def test_conv3d_dgrad(impl, cin, cout, kd, shape):
    n, d, h, w = shape
    wt = bf16_round(randn(31, cout, cin, kd, 3, 3, scale=0.1))
    dy = bf16_round(randn(32, n, cout, d, h, w))
    x = torch.zeros(n, cin, d, h, w, requires_grad=True)
    _conv_ref(x, wt, None, kd).backward(dy)
    ref = x.grad
    dyb = to_c8(dy.to(DEV))
    dx = torch.empty((n, d, cin // 8, h, w, 8), dtype=torch.bfloat16, device=DEV)
    if impl == "direct":
        _call("fpl_conv3d_direct", _p(dyb), cout // 8, 0, _p(wt.to(DEV)), None, _p(dx), cin // 8, 0, None, n, d, h, w,
              cout, cin, kd, 1, 0, _st())
    else:
        img = torch.empty(cin * cout * kd * 9, dtype=torch.bfloat16, device=DEV)
        _call("fpl_conv3d_prep_weight", _p(wt.to(DEV)), cin, cout, kd, 1, _p(img), _st())
        _call("fpl_conv3d_tc", _p(dyb), cout // 8, 0, _p(img), None, _p(dx), cin // 8, 0, None, n, d, h, w, cout, cin, kd, _st())
    assert max_rel(from_c8(dx).cpu(), ref) < 6e-3


@pytest.mark.parametrize("name", ["fpl_conv3d_wgrad", "fpl_conv3d_wgrad_tc"])
@pytest.mark.parametrize("cin,cout,kd,shape", [(16, 16, 3, (2, 3, 16, 12)), (32, 16, 3, (1, 2, 8, 8)),
                                               (16, 32, 1, (1, 2, 16, 16)), (64, 48, 3, (1, 2, 6, 10)),
                                               # Cin 16 / 32, W >= 16: the h-stacked kernel (conv_wgrad_hs.cu); ragged tiles,
                                               # odd depth / height, several output-channel chunks, batch > 1
                                               (16, 16, 3, (2, 3, 16, 32)), (32, 16, 3, (1, 5, 12, 16)), (16, 32, 3, (1, 4, 10, 48)),
                                               (32, 32, 3, (2, 2, 6, 16)), (16, 16, 3, (1, 3, 7, 20)), (32, 48, 3, (1, 3, 9, 40)),
                                               (16, 16, 3, (1, 9, 24, 80))])
def test_conv3d_wgrad(name, cin, cout, kd, shape):
    from fplplus_b200 import lib as L
    if not hasattr(L.load(), name):
        pytest.skip(name + " not built")
    n, d, h, w = shape
    x = bf16_round(randn(41, n, cin, d, h, w))
    dy = bf16_round(randn(42, n, cout, d, h, w))
    wt = torch.zeros(cout, cin, kd, 3, 3, requires_grad=True)
    _conv_ref(x, wt, None, kd).backward(dy)
    ref = wt.grad
    dw = torch.zeros_like(ref, device=DEV)
    _call(name, _p(to_c8(x.to(DEV))), cin // 8, 0, _p(to_c8(dy.to(DEV))), cout // 8, 0, _p(dw), n, d, h, w, cin, cout,
          kd, _st())
    assert max_rel(dw.cpu(), ref) < 1e-4
    # accumulates
    _call(name, _p(to_c8(x.to(DEV))), cin // 8, 0, _p(to_c8(dy.to(DEV))), cout // 8, 0, _p(dw), n, d, h, w, cin, cout,
          kd, _st())
    assert max_rel(dw.cpu(), 2 * ref) < 1e-4


@pytest.mark.parametrize("cin,kd,shape", [(1, 3, (2, 3, 12, 20)), (3, 3, (2, 3, 12, 20)), (1, 1, (2, 3, 12, 20)),
                                          # 1 channel, k3, W >= 32: the tensor-core kernels that build their operand from
                                          # the image in shared memory (stem_tc.cu); ragged tiles in H and W, depth 1 and 5
                                          (1, 3, (2, 5, 20, 70)), (1, 3, (1, 1, 33, 32)), (1, 3, (1, 4, 16, 96))])
def test_stem_conv_fwd_and_wgrad(cin, kd, shape):
    (n, d, h, w), cout = shape, 16
    x = randn(51, n, cin, d, h, w)
    wt = randn(52, cout, cin, kd, 3, 3, scale=0.2).requires_grad_(True)
    b = randn(53, cout, scale=0.1)
    ref = _conv_ref(x, wt, b, kd)
    y = torch.empty((n, d, cout // 8, h, w, 8), dtype=torch.bfloat16, device=DEV)
    stats = torch.zeros(2 * cout, dtype=torch.float64, device=DEV)
    _call("fpl_stem_conv_fwd", _p(x.to(DEV)), _p(wt.detach().to(DEV)), _p(b.to(DEV)), _p(y), cout // 8, 0, _p(stats),
          n, cin, d, h, w, cout, kd, _st())
    assert max_rel(from_c8(y).cpu(), ref.detach()) < 6e-3
    np.testing.assert_allclose(stats.cpu()[:cout], ref.detach().double().sum((0, 2, 3, 4)), rtol=1e-5, atol=1e-3)
    dy = bf16_round(randn(54, n, cout, d, h, w))
    ref.backward(dy)
    dw = torch.zeros(cout, cin, kd, 3, 3, device=DEV)
    _call("fpl_stem_conv_wgrad", _p(x.to(DEV)), _p(to_c8(dy.to(DEV))), cout // 8, 0, _p(dw), n, cin, d, h, w, cout, kd, _st())
    assert max_rel(dw.cpu(), wt.grad) < 1e-4


@pytest.mark.parametrize("classes", [2, 5])
def test_head_conv_fwd_bwd(classes):
    n, d, h, w, cin = 2, 3, 12, 16, 16
    x = bf16_round(randn(61, n, cin, d, h, w)).requires_grad_(True)
    wt = randn(62, classes, cin, 1, 3, 3, scale=0.2).requires_grad_(True)
    b = randn(63, classes, scale=0.1).requires_grad_(True)
    ref = F.conv3d(x, wt, b, padding=(0, 1, 1))
    xb = to_c8(x.detach().to(DEV))
    logits = torch.empty((n, classes, d, h, w), device=DEV)
    _call("fpl_head_conv_fwd", _p(xb), cin // 8, 0, _p(wt.detach().to(DEV)), _p(b.detach().to(DEV)), _p(logits), n, d, h,
          w, cin, classes, _st())
    assert max_rel(logits.cpu(), ref.detach()) < 1e-5
    g = randn(64, n, classes, d, h, w)
    ref.backward(g)
    dx = torch.empty((n, d, cin // 8, h, w, 8), dtype=torch.bfloat16, device=DEV)
    dw = torch.zeros(classes, cin, 1, 3, 3, device=DEV)
    db = torch.zeros(classes, device=DEV)
    _call("fpl_head_conv_bwd", _p(xb), cin // 8, 0, _p(wt.detach().to(DEV)), _p(g.to(DEV)), _p(dx), cin // 8, 0, _p(dw),
          _p(db), n, d, h, w, cin, classes, _st())
    assert max_rel(from_c8(dx).cpu(), x.grad) < 6e-3
    assert max_rel(dw.cpu(), wt.grad) < 1e-4
    assert max_rel(db.cpu(), b.grad) < 1e-4


@pytest.mark.parametrize("cin,cout,kd2", [(32, 16, 2), (64, 32, 1), (256, 128, 2)])
def test_convt_k2s2_fwd_bwd(cin, cout, kd2):
    n, d, h, w = 2, 2, 4, 6
    x = bf16_round(randn(71, n, cin, d, h, w)).requires_grad_(True)
    wt = randn(72, cin, cout, kd2, 2, 2, scale=0.2).requires_grad_(True)
    b = randn(73, cout, scale=0.1).requires_grad_(True)
    ref = F.conv_transpose3d(x, wt, b, stride=(kd2, 2, 2))
    xb = to_c8(x.detach().to(DEV))
    do, ho, wo = d * kd2, h * 2, w * 2
    # written into the second half of a concat buffer
    cat = torch.zeros((n, do, 2 * cout // 8, ho, wo, 8), dtype=torch.bfloat16, device=DEV)
    _call("fpl_convt_k2s2_fwd", _p(xb), cin // 8, 0, _p(wt.detach().to(DEV)), _p(b.detach().to(DEV)), _p(cat),
          2 * cout // 8, cout // 8, n, d, h, w, cin, cout, kd2, _st())
    out = from_c8(cat).cpu()
    assert max_rel(out[:, cout:], ref.detach()) < 6e-3
    assert torch.all(out[:, :cout] == 0)
    g = bf16_round(randn(74, n, cout, do, ho, wo))
    ref.backward(g)
    gcat = torch.cat([torch.zeros_like(g), g], 1)
    dx = torch.empty((n, d, cin // 8, h, w, 8), dtype=torch.bfloat16, device=DEV)
    dw = torch.zeros(cin, cout, kd2, 2, 2, device=DEV)
    db = torch.zeros(cout, device=DEV)
    _call("fpl_convt_k2s2_bwd", _p(xb), cin // 8, 0, _p(wt.detach().to(DEV)), _p(to_c8(gcat.to(DEV))), 2 * cout // 8,
          cout // 8, _p(dx), cin // 8, 0, _p(dw), _p(db), n, d, h, w, cin, cout, kd2, _st())
    assert max_rel(from_c8(dx).cpu(), x.grad) < 6e-3
    assert max_rel(dw.cpu(), wt.grad) < 1e-4
    assert max_rel(db.cpu(), b.grad) < 1e-4


# ------------------------------------------------------------------------------------------
# DSBN + PReLU + dropout + pool
# ------------------------------------------------------------------------------------------
def _dense_mask_c8(mask_ncdhw):
    """bool [N,C,D,H,W] -> uint8 in dense C8-planar element order."""
    n, c, d, h, w = mask_ncdhw.shape
    return mask_ncdhw.reshape(n, c // 8, 8, d, h, w).permute(0, 3, 1, 4, 5, 2).contiguous().to(torch.uint8)


@pytest.mark.parametrize("training", [1, 0])
@pytest.mark.parametrize("pool_kd,drop_p", [(0, 0.0), (2, 0.0), (1, 0.0), (0, 0.4)])
def test_dsbn_act_fwd_bwd(training, pool_kd, drop_p):
    n, c, d, h, w = 2, 16, 4, 8, 12
    y = bf16_round(randn(81, n, c, d, h, w, scale=2.0) + 0.5).requires_grad_(True)
    gamma = (randn(82, c, scale=0.3) + 1.0).requires_grad_(True)
    beta = randn(83, c, scale=0.2).requires_grad_(True)
    slope = torch.tensor([0.2], requires_grad=True)
    rm, rv = randn(84, c, scale=0.1), randn(85, c, scale=0.1).abs() + 0.8
    rm_ref, rv_ref = rm.clone(), rv.clone()
    keep = torch.from_numpy(np.random.Generator(np.random.PCG64(86)).random((n, c, d, h, w)) >= drop_p)
    z = F.batch_norm(y, rm_ref, rv_ref, gamma, beta, training=bool(training), momentum=0.1, eps=1e-5)
    a = F.prelu(z, slope)
    if drop_p > 0:
        a = a * keep.float() / (1 - drop_p)
    outs = [a]
    if pool_kd:
        outs.append(F.max_pool3d(bf16_round(a.detach()) + (a - a.detach()), (pool_kd, 2, 2), (pool_kd, 2, 2)))

    yb = to_c8(y.detach().to(DEV))
    stats = torch.stack([y.detach().double().sum((0, 2, 3, 4)), (y.detach().double() ** 2).sum((0, 2, 3, 4))]).flatten().to(DEV)
    f32 = lambda: torch.zeros(c, device=DEV)
    scale, shift, mean, invstd = f32(), f32(), f32(), f32()
    rmd, rvd = rm.to(DEV), rv.to(DEV)
    nbt = torch.zeros((), dtype=torch.int64, device=DEV)
    cnt = n * d * h * w
    _call("fpl_dsbn_finalize", _p(stats), cnt, _p(gamma.detach().to(DEV)), _p(beta.detach().to(DEV)), _p(rmd), _p(rvd),
          _p(nbt), 0.1, 1e-5, training, _p(scale), _p(shift), _p(mean), _p(invstd), c, _st())
    if training:
        np.testing.assert_allclose(rmd.cpu(), rm_ref, rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(rvd.cpu(), rv_ref, rtol=1e-5, atol=1e-6)
        assert int(nbt) == 1
    else:
        assert int(nbt) == 0
    act = torch.zeros((n, d, 2 * c // 8, h, w, 8), dtype=torch.bfloat16, device=DEV)   # first half of a concat buffer
    mask = _dense_mask_c8(keep).to(DEV) if drop_p > 0 else None
    pooled = idx = None
    if pool_kd:
        pooled = torch.empty((n, d // pool_kd, c // 8, h // 2, w // 2, 8), dtype=torch.bfloat16, device=DEV)
        idx = torch.empty((n, d // pool_kd, c // 8, h // 2, w // 2, 8), dtype=torch.uint8, device=DEV)
    sl = slope.detach().to(DEV)
    _call("fpl_dsbn_act_fwd", _p(yb), _p(scale), _p(shift), _p(sl), _p(act), 2 * c // 8, 0, _p(pooled), c // 8, 0, _p(idx),
          pool_kd, drop_p, _p(mask), 0, 0, None, n, d, h, w, c, _st())
    got = from_c8(act).cpu()
    assert max_rel(got[:, :c], a.detach()) < 6e-3
    if pool_kd:
        assert max_rel(from_c8(pooled).cpu(), outs[1].detach()) < 6e-3

    # backward: gradient arrives through the activation (g1) and, when pooled, through the pool
    g1 = bf16_round(randn(87, n, c, d, h, w))
    loss = (a * g1).sum()
    gp = None
    if pool_kd:
        gp = bf16_round(randn(88, *outs[1].shape))
        loss = loss + (outs[1] * gp).sum()
    loss.backward()
    g1b = to_c8(torch.cat([g1, torch.zeros_like(g1)], 1).to(DEV))
    gpb = to_c8(gp.to(DEV)) if pool_kd else None
    red = torch.zeros(2 * c + 1, dtype=torch.float64, device=DEV)
    common = (_p(yb), _p(g1b), 2 * c // 8, 0, _p(gpb), c // 8, 0, _p(idx), pool_kd, _p(scale), _p(shift), _p(mean),
              _p(invstd), _p(sl), drop_p, _p(mask), 0, 0, None)
    _call("fpl_dsbn_act_bwd_reduce", *common, _p(red), n, d, h, w, c, _st())
    dy = torch.empty((n, d, c // 8, h, w, 8), dtype=torch.bfloat16, device=DEV)
    _call("fpl_dsbn_act_bwd_apply", *common, _p(red), training, _p(dy), n, d, h, w, c, _st())
    dgamma, dbeta, dslope, dbias = f32(), f32(), torch.zeros(1, device=DEV), f32()
    _call("fpl_dsbn_bwd_finalize", _p(red), _p(scale), _p(invstd), training, _p(dgamma), _p(dbeta), _p(dslope), _p(dbias),
          c, _st())
    assert max_rel(from_c8(dy).cpu(), y.grad) < 1e-2
    assert max_rel(dgamma.cpu(), gamma.grad) < 2e-3
    assert max_rel(dbeta.cpu(), beta.grad) < 2e-3
    assert max_rel(dslope.cpu(), slope.grad) < 2e-3


def test_philox_dropout_statistics_and_backward_consistency():
    n, c, d, h, w = 1, 32, 4, 16, 16
    p = 0.3
    yb = to_c8(torch.ones(n, c, d, h, w, device=DEV))
    one, zero = torch.ones(c, device=DEV), torch.zeros(c, device=DEV)
    sl = torch.tensor([0.25], device=DEV)
    outs = []
    for seed in (123, 123, 124):
        act = torch.empty((n, d, c // 8, h, w, 8), dtype=torch.bfloat16, device=DEV)
        _call("fpl_dsbn_act_fwd", _p(yb), _p(one), _p(zero), _p(sl), _p(act), c // 8, 0, None, 0, 0, None, 0, p, None,
              seed, 16, None, n, d, h, w, c, _st())
        outs.append(from_c8(act).cpu())
    assert torch.equal(outs[0], outs[1]) and not torch.equal(outs[0], outs[2])
    kept = outs[0] != 0
    # the exact mask of the host Philox restatement (also pins a mistake the backward pass would repeat)
    assert torch.equal(kept, dropout_keep_c8(123, 16, n, c, d, h, w, p))
    assert abs(kept.float().mean().item() - (1 - p)) < 0.02
    assert torch.allclose(outs[0][kept], torch.tensor(1 / (1 - p)), rtol=1e-2)
    # per-channel keep rate is uniform too
    assert (kept.float().mean((0, 2, 3, 4)) - (1 - p)).abs().max() < 0.06
    # backward regenerates the same mask: dy is non-zero exactly where the forward kept the unit
    g1 = to_c8(torch.ones(n, c, d, h, w, device=DEV))
    red = torch.zeros(2 * c + 1, dtype=torch.float64, device=DEV)
    dy = torch.empty((n, d, c // 8, h, w, 8), dtype=torch.bfloat16, device=DEV)
    _call("fpl_dsbn_act_bwd_apply", _p(yb), _p(g1), c // 8, 0, None, 0, 0, None, 0, _p(one), _p(zero), _p(zero), _p(one),
          _p(sl), p, None, 123, 16, None, _p(red), 0, _p(dy), n, d, h, w, c, _st())
    assert torch.equal(from_c8(dy).cpu() != 0, kept)


# ------------------------------------------------------------------------------------------
# loss, filter, window kernels
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tag", ["c2", "c5"])
@pytest.mark.parametrize("weighted", [False, True])
def test_dice_ce_against_golden_and_closed_form(golden_dir, tag, weighted):
    import os
    from oracle import losses
    from fplplus_b200.loss import CrossEntropyLoss, DiceLoss, CombinedLoss
    from fplplus_b200.registry import loss_dict
    g = np.load(os.path.join(golden_dir, "loss.npz"))
    z, y, pw = g[f"{tag}_logits"], g[f"{tag}_onehot"], g[f"{tag}_pw"]
    wt = "w" if weighted else "u"
    for name, cls in (("dice", DiceLoss), ("ce", CrossEntropyLoss)):
        zt = torch.from_numpy(z).to(DEV).requires_grad_(True)
        d = {"prediction": zt, "ground_truth": torch.from_numpy(y).to(DEV)}
        if weighted:
            d["pixel_weight"] = torch.from_numpy(pw).to(DEV)
            d["image_weight"] = torch.ones(z.shape[0], dtype=torch.float64)
        val = cls({})(d)
        (val * 0.5).backward()
        np.testing.assert_allclose(val.item(), float(g[f"{tag}_{name}_{wt}_loss"]), rtol=1e-5)
        ref = g[f"{tag}_{name}_{wt}_grad"] * 0.5
        np.testing.assert_allclose(zt.grad.cpu().numpy(), ref, rtol=2e-3, atol=1e-5 * np.abs(ref).max())
    # combined 0.3*Dice + 0.7*CE through the CombinedLoss entry, against the float64 closed form
    zt = torch.from_numpy(z).to(DEV).requires_grad_(True)
    d = {"prediction": [zt], "ground_truth": torch.from_numpy(y).to(DEV)}
    if weighted:
        d["pixel_weight"] = torch.from_numpy(pw).to(DEV)
    comb = CombinedLoss({"loss_type": ["DiceLoss", "CrossEntropyLoss"], "loss_weight": [0.3, 0.7]}, loss_dict)
    val = comb(d)
    val.backward()
    lv, dz, _ = losses.dice_ce_closed_form(z, y, pw if weighted else None, 0.3, 0.7)
    np.testing.assert_allclose(val.item(), lv, rtol=1e-5)
    np.testing.assert_allclose(zt.grad.cpu().numpy(), dz, rtol=2e-3, atol=1e-5 * np.abs(dz).max())
    hd = comb.last_hard_dice().cpu().numpy()
    ref_hd = losses.hard_dice(torch.from_numpy(z), torch.from_numpy(y)).numpy()
    np.testing.assert_allclose(hd, ref_hd, rtol=1e-6)


def test_argmax_agreement_and_weight_folding_bit_exact():
    from oracle import fpl_filter
    from fplplus_b200 import fpl
    r = np.random.Generator(np.random.PCG64(5))
    for c in (2, 5):
        za = (r.standard_normal((1, c, 6, 12, 20)) * 2).astype(np.float32)
        zb = (za + r.standard_normal(za.shape) * 0.8).astype(np.float32)
        za[0, :, 0, 0, :4] = 1.0                      # exact ties -> first index wins
        la, lb, w, cnt = fpl.agreement_weight(torch.from_numpy(za).to(DEV), torch.from_numpy(zb).to(DEV))
        ra, rb = fpl_filter.pseudo_label(za)[0], fpl_filter.pseudo_label(zb)[0]
        np.testing.assert_array_equal(la.cpu().numpy(), ra)
        np.testing.assert_array_equal(lb.cpu().numpy(), rb)
        np.testing.assert_array_equal(fpl.pseudo_label(torch.from_numpy(za).to(DEV)).cpu().numpy()[0], ra)
        ref_w = fpl_filter.agreement_weight_multiclass(ra, rb)
        if c == 2:
            np.testing.assert_array_equal(ref_w, fpl_filter.agreement_weight(ra, rb))
        np.testing.assert_array_equal(w.cpu().numpy().astype(np.float64), ref_w)
        assert int(cnt) == int((ra != rb).sum())
        _, _, wf, _ = fpl.agreement_weight(torch.from_numpy(za).to(DEV), torch.from_numpy(zb).to(DEV), image_weight=0.37)
        np.testing.assert_array_equal(wf.cpu().numpy(), fpl_filter.set_weight_(np.float32(0.37), ref_w.astype(np.float32)))


def test_mc_uncertainty_against_reference_agent_golden(golden_dir):
    """Same prepared MC logits as oracle/gen_golden_fpl.py fed the reference agent's infer()."""
    import os
    from oracle import fpl_filter
    from oracle.gen_golden_fpl import CASES, fpl_case_logits
    from fplplus_b200 import fpl
    g = np.load(os.path.join(golden_dir, "fpl_infer.npz"))
    table = {}
    for name, seed, conf in CASES:
        passes = fpl_case_logits(seed, confident=conf)
        stats, umap = fpl.mc_uncertainty([torch.from_numpy(p).to(DEV) for p in passes], want_map=True)
        ref = fpl_filter.mc_uncertainty(passes)
        v, b = stats.tolist()
        near = int((np.abs(ref["uncertainty_map"] - 0.01) < 1e-6).sum())
        assert abs(int(b) - ref["boundary"]) <= near
        # fp32 rounding floor of a sum of per-voxel variances (identical passes give ~1e-12, not 0)
        np.testing.assert_allclose(v, float(ref["vars"]), rtol=1e-5, atol=1e-9 * passes[0][0, 0].size)
        np.testing.assert_allclose(umap.cpu().numpy(), ref["uncertainty_map"][0] if ref["uncertainty_map"].ndim == 4
                                   else ref["uncertainty_map"], rtol=1e-4, atol=1e-7)
        table[name] = [fpl.finish_uncertainty(stats)]
    srt = fpl.sort_uncertainty(table)
    assert [n for _v, n in srt] == [str(n) for n in g["names"]]                 # order incl. sentinel name ties
    np.testing.assert_allclose([float(v[0]) for v, _n in srt], g["values"], rtol=1e-5)
    assert [isinstance(v[0], int) for v, _n in srt] == list(g["is_sentinel"])


def test_window_accumulate_flips_and_normalize():
    b, c, vd, vh, vw = 1, 2, 6, 10, 12
    out = torch.zeros(b, c, vd, vh, vw, device=DEV)
    cnt = torch.zeros_like(out)
    patch = randn(91, b, c, 4, 6, 8).to(DEV)
    ref = torch.zeros(b, c, vd, vh, vw)
    rc = torch.zeros_like(ref)
    for (d0, h0, w0, fh, fw, s) in ((0, 0, 0, 0, 0, 1.0), (2, 4, 4, 1, 0, 0.5), (1, 2, 3, 1, 1, 2.0), (2, 0, 4, 0, 1, 1.0)):
        _call("fpl_window_accumulate", _p(patch), _p(out), _p(cnt), b, c, vd, vh, vw, d0, h0, w0, 4, 6, 8, fh, fw, s, _st())
        pp = patch.cpu()
        dims = [d for d, f in ((-2, fh), (-1, fw)) if f]
        if dims:
            pp = torch.flip(pp, dims)
        ref[:, :, d0:d0 + 4, h0:h0 + 6, w0:w0 + 8] += s * pp
        rc[:, :, d0:d0 + 4, h0:h0 + 6, w0:w0 + 8] += 1
    torch.testing.assert_close(out.cpu(), ref)
    torch.testing.assert_close(cnt.cpu(), rc)
    cnt.clamp_(min=1)
    _call("fpl_window_normalize", _p(out), _p(cnt), 0.25, out.numel(), _st())
    torch.testing.assert_close(out.cpu(), ref / rc.clamp(min=1) * 0.25)
    from fplplus_b200 import lib as L
    with pytest.raises(L.FplError):
        _call("fpl_window_accumulate", _p(patch), _p(out), None, b, c, vd, vh, vw, 4, 0, 0, 4, 6, 8, 0, 0, 1.0, _st())


@pytest.mark.parametrize("training", [1, 0])
@pytest.mark.parametrize("pool_kd", [0, 2])
def test_dsbn_fused_finalize_entry_points_equal_the_two_step_ones(training, pool_kd):
    """fpl_dsbn_bn_act_fwd == fpl_dsbn_finalize + fpl_dsbn_act_fwd and fpl_dsbn_act_bwd_apply_fin ==
    fpl_dsbn_act_bwd_apply + fpl_dsbn_bwd_finalize, bit for bit (same arithmetic, one launch each)."""
    n, c, d, h, w = 2, 32, 4, 8, 12
    yb = to_c8((randn(181, n, c, d, h, w, scale=2.0) + 0.5).to(DEV))
    yf = from_c8(yb).double()
    stats = torch.stack([yf.sum((0, 2, 3, 4)), (yf ** 2).sum((0, 2, 3, 4))]).flatten().contiguous()
    gamma, beta = (randn(182, c, scale=0.3) + 1.0).to(DEV), randn(183, c, scale=0.2).to(DEV)
    sl = torch.tensor([0.2], device=DEV)
    cnt = n * d * h * w
    res = []
    for fused in (0, 1):
        rm, rv = randn(184, c, scale=0.1).to(DEV), (randn(185, c, scale=0.1).abs() + 0.8).to(DEV)
        nbt = torch.zeros((), dtype=torch.int64, device=DEV)
        scale, shift, mean, invstd = (torch.zeros(c, device=DEV) for _ in range(4))
        act = torch.zeros((n, d, c // 8, h, w, 8), dtype=torch.bfloat16, device=DEV)
        pooled = idx = None
        if pool_kd:
            pooled = torch.zeros((n, d // pool_kd, c // 8, h // 2, w // 2, 8), dtype=torch.bfloat16, device=DEV)
            idx = torch.zeros((n, d // pool_kd, c // 8, h // 2, w // 2, 8), dtype=torch.uint8, device=DEV)
        tail = (_p(sl), _p(act), c // 8, 0, _p(pooled), c // 8, 0, _p(idx), pool_kd, 0.0, None, 0, 0, None, n, d, h, w, c, _st())
        if fused:
            _call("fpl_dsbn_bn_act_fwd", _p(yb), _p(stats), cnt, _p(gamma), _p(beta), _p(rm), _p(rv), _p(nbt), 0.1, 1e-5,
                  training, _p(scale), _p(shift), _p(mean), _p(invstd), *tail)
        else:
            _call("fpl_dsbn_finalize", _p(stats), cnt, _p(gamma), _p(beta), _p(rm), _p(rv), _p(nbt), 0.1, 1e-5, training,
                  _p(scale), _p(shift), _p(mean), _p(invstd), c, _st())
            _call("fpl_dsbn_act_fwd", _p(yb), _p(scale), _p(shift), *tail)
        g1 = to_c8(bf16_round(randn(187, n, c, d, h, w)).to(DEV))
        gp = to_c8(bf16_round(randn(188, n, c, d // 2, h // 2, w // 2)).to(DEV)) if pool_kd else None
        red = torch.zeros(2 * c + 1, dtype=torch.float64, device=DEV)
        common = (_p(yb), _p(g1), c // 8, 0, _p(gp), c // 8, 0, _p(idx), pool_kd, _p(scale), _p(shift), _p(mean), _p(invstd),
                  _p(sl), 0.0, None, 0, 0, None)
        _call("fpl_dsbn_act_bwd_reduce", *common, _p(red), n, d, h, w, c, _st())
        dy = torch.zeros((n, d, c // 8, h, w, 8), dtype=torch.bfloat16, device=DEV)
        dg, db, dsl, dbias = torch.zeros(c, device=DEV), torch.zeros(c, device=DEV), torch.zeros(1, device=DEV), torch.zeros(c, device=DEV)
        if fused:
            _call("fpl_dsbn_act_bwd_apply_fin", *common, _p(red), training, _p(dy), n, d, h, w, c, _st(), _p(dg), _p(db),
                  _p(dsl), _p(dbias))
        else:
            _call("fpl_dsbn_act_bwd_apply", *common, _p(red), training, _p(dy), n, d, h, w, c, _st())
            _call("fpl_dsbn_bwd_finalize", _p(red), _p(scale), _p(invstd), training, _p(dg), _p(db), _p(dsl), _p(dbias), c, _st())
        torch.cuda.synchronize()
        res.append([t.clone() for t in (act, scale, shift, mean, invstd, rm, rv, nbt, dy, dg, db, dsl, dbias)]
                   + ([pooled.clone(), idx.clone()] if pool_kd else []))
    # same arithmetic up to fp32 contraction (fma vs mul+add): fp32 vectors agree to ~1 ulp, the bf16 tensors
    # except for rare 1-ulp rounding flips, the argmax codes except on exact ties
    for a, b in zip(*res):
        if a.dtype == torch.float32:
            torch.testing.assert_close(a, b, rtol=2e-5, atol=1e-6)
        elif a.dtype == torch.bfloat16:
            assert max_rel(a.float().cpu(), b.float().cpu()) < 1e-2
            assert float((a != b).float().mean()) < 2e-3
        elif a.dtype == torch.uint8:
            assert float((a != b).float().mean()) < 2e-3
        else:
            assert torch.equal(a, b)


@pytest.mark.parametrize("cin,cout,kd2,shape", [(32, 16, 2, (2, 2, 16, 8)), (64, 32, 1, (1, 3, 20, 12)),
                                                (256, 128, 2, (1, 1, 4, 6)), (128, 64, 2, (1, 2, 8, 8)),
                                                (512, 256, 2, (1, 2, 4, 8))])      # the shipped VS widths: GEMM N = 2048
def test_convt_k2s2_tensor_core_fwd_dgrad_wgrad(cin, cout, kd2, shape):
    """ConvTranspose3d k2 s2 on tcgen05 (strided TMA sub-lattices) against torch on bf16-rounded operands."""
    from fplplus_b200 import lib as L
    n, d, h, w = shape
    x = bf16_round(randn(71, n, cin, d, h, w)).requires_grad_(True)
    wt = bf16_round(randn(72, cin, cout, kd2, 2, 2, scale=0.2)).requires_grad_(True)
    b = randn(73, cout, scale=0.1)
    ref = F.conv_transpose3d(x, wt, b, stride=(kd2, 2, 2))
    g = bf16_round(randn(74, *ref.shape))
    ref.backward(g)
    xb = to_c8(x.detach().to(DEV))
    wd, bd = wt.detach().to(DEV), b.to(DEV)
    nbytes = L.load().fpl_convt_weight_image_bytes(cin, cout, kd2)
    img = torch.empty(nbytes // 2, dtype=torch.bfloat16, device=DEV)
    img_t = torch.empty(nbytes // 2, dtype=torch.bfloat16, device=DEV)
    _call("fpl_convt_prep_weight", _p(wd), cin, cout, kd2, 0, _p(img), _st())
    _call("fpl_convt_prep_weight", _p(wd), cin, cout, kd2, 1, _p(img_t), _st())
    do, ho, wo = d * kd2, 2 * h, 2 * w
    cat = torch.zeros((n, do, 2 * cout // 8, ho, wo, 8), dtype=torch.bfloat16, device=DEV)
    _call("fpl_convt_k2s2_fwd_tc", _p(xb), cin // 8, 0, _p(img), _p(bd), _p(cat), 2 * cout // 8, cout // 8, n, d, h, w, cin,
          cout, kd2, _st())
    out = from_c8(cat).cpu()
    assert max_rel(out[:, cout:], ref.detach()) < 6e-3
    assert torch.all(out[:, :cout] == 0)                      # the skip half of the concat buffer is untouched
    gcat = to_c8(torch.cat([torch.zeros_like(g), g], 1).to(DEV))
    dx = torch.zeros((n, d, cin // 8, h, w, 8), dtype=torch.bfloat16, device=DEV)
    _call("fpl_convt_k2s2_dgrad_tc", _p(gcat), 2 * cout // 8, cout // 8, _p(img_t), _p(dx), cin // 8, 0, n, d, h, w, cin, cout,
          kd2, _st())
    dw = torch.zeros(cin, cout, kd2, 2, 2, device=DEV)
    for _ in range(2):                                         # accumulates
        _call("fpl_convt_k2s2_wgrad_tc", _p(xb), cin // 8, 0, _p(gcat), 2 * cout // 8, cout // 8, _p(dw), n, d, h, w, cin, cout,
              kd2, _st())
    assert max_rel(from_c8(dx).cpu(), x.grad) < 6e-3
    assert max_rel(dw.cpu(), 2 * wt.grad) < 1e-4
    # tap-major scratch + batched fold (negative tap count = ConvTranspose weight layout)
    ntaps = 4 * kd2
    scratch = torch.zeros(ntaps * cout * cin, device=DEV)
    _call("fpl_convt_k2s2_wgrad_tc_tapmajor", _p(xb), cin // 8, 0, _p(gcat), 2 * cout // 8, cout // 8, _p(scratch), n, d, h, w,
          cin, cout, kd2, _st())
    _call("fpl_wgrad_tapmajor_to_dw_batch", 1, (ctypes.c_void_p * 1)(scratch.data_ptr()), (ctypes.c_void_p * 1)(dw.data_ptr()),
          (ctypes.c_int * 1)(cout), (ctypes.c_int * 1)(cin), (ctypes.c_int * 1)(-ntaps), None, _st())
    assert max_rel(dw.cpu(), 3 * wt.grad) < 1e-4


@pytest.mark.parametrize("transpose", [0, 1])
@pytest.mark.parametrize("cin,cout,shape", [(16, 16, (2, 4, 32, 16)), (32, 16, (1, 3, 20, 12)), (16, 32, (1, 17, 16, 8)),
                                            (64, 32, (1, 2, 16, 16)), (32, 64, (1, 9, 10, 9)), (16, 16, (1, 20, 16, 16))])
def test_conv3d_depth_folded_tensor_core_kernel(cin, cout, shape, transpose):
    """Depth-folded tcgen05 conv (N spans the 3 output planes an input plane feeds; resident weights; TMEM
    accumulators zeroed by the epilogue) against torch on bf16-rounded operands, forward and dgrad, incl.
    ragged tiles, odd depths and a short last depth chunk; and bit-compatible with fpl_conv3d_tc up to 1 ulp."""
    from fplplus_b200 import lib as L
    n, d, h, w = shape
    wt = bf16_round(randn(12, cout, cin, 3, 3, 3, scale=0.1))
    if not transpose:
        x = bf16_round(randn(11, n, cin, d, h, w))
        b = randn(13, cout, scale=0.1)
        ref = F.conv3d(x, wt, b, padding=1)
        xin, ci, co, bias = x, cin, cout, b.to(DEV)
    else:
        dy = bf16_round(randn(14, n, cout, d, h, w))
        xx = torch.zeros(n, cin, d, h, w, requires_grad=True)
        F.conv3d(xx, wt, None, padding=1).backward(dy)
        ref, xin, ci, co, bias = xx.grad, dy, cout, cin, None
    nbytes = L.load().fpl_conv3d_dfold_image_bytes(ci, co)
    assert nbytes == 27 * ci * co * 2
    xb, wd = to_c8(xin.to(DEV)), wt.to(DEV)
    img = torch.empty(nbytes // 2, dtype=torch.bfloat16, device=DEV)
    _call("fpl_conv3d_dfold_prep_weight", _p(wd), cin, cout, transpose, _p(img), _st())
    y = torch.zeros((n, d, co // 8, h, w, 8), dtype=torch.bfloat16, device=DEV)
    stats = torch.zeros(2 * co, dtype=torch.float64, device=DEV)
    for _ in range(2):           # twice: the second launch must find nothing stale (accumulators are re-zeroed per launch)
        stats.zero_()
        _call("fpl_conv3d_tc_dfold", _p(xb), ci // 8, 0, _p(img), _p(bias), _p(y), co // 8, 0, _p(stats), n, d, h, w, ci, co, _st())
    out = from_c8(y).cpu()
    rd = ref.detach()
    assert max_rel(out, rd) < 6e-3
    s = stats.cpu()
    np.testing.assert_allclose(s[:co], rd.double().sum((0, 2, 3, 4)), rtol=1e-4, atol=2e-3)
    np.testing.assert_allclose(s[co:], (rd.double() ** 2).sum((0, 2, 3, 4)), rtol=1e-4, atol=2e-3)
    img2 = torch.empty(L.load().fpl_conv3d_weight_image_bytes(ci, co, 3) // 2, dtype=torch.bfloat16, device=DEV)
    _call("fpl_conv3d_prep_weight", _p(wd), cin, cout, 3, transpose, _p(img2), _st())
    y2 = torch.zeros_like(y)
    _call("fpl_conv3d_tc", _p(xb), ci // 8, 0, _p(img2), _p(bias), _p(y2), co // 8, 0, None, n, d, h, w, ci, co, 3, _st())
    out2 = from_c8(y2).cpu()
    assert max_rel(out, out2) < 5e-3 and float((out != out2).float().mean()) < 0.05
    assert L.load().fpl_conv3d_dfold_image_bytes(128, 128) == -1         # large layers stay on fpl_conv3d_tc


@pytest.mark.parametrize("cout,shape", [(16, (2, 5, 20, 12)), (32, (1, 16, 16, 24))])
def test_stem_on_tensor_cores_patch9_k311(cout, shape):
    """Stem conv k(3,3,3), in_chns = 1: fpl_patch9_c8 turns the 9 in-plane neighbours into channels, then the conv and
    its wgrad are k(3,1,1) tensor-core kernels with ONE in-plane tap.  Against torch on the bf16-rounded image."""
    n, d, h, w = shape
    x = bf16_round(randn(201, n, 1, d, h, w))
    wt = bf16_round(randn(202, cout, 1, 3, 3, 3, scale=0.2)).requires_grad_(True)
    b = randn(203, cout, scale=0.1)
    ref = F.conv3d(x, wt, b, padding=1)
    g = bf16_round(randn(204, *ref.shape))
    ref.backward(g)
    xs = torch.empty((n, d, 2, h, w, 8), dtype=torch.bfloat16, device=DEV)
    _call("fpl_patch9_c8", _p(x.to(DEV)), _p(xs), 0, n, d, h, w, _st())
    patch = from_c8(xs).cpu()
    assert torch.equal(patch[:, 4], x[:, 0]) and torch.all(patch[:, 9:] == 0)       # centre tap = the image itself
    assert torch.equal(patch[:, 0, :, 1:, 1:], x[:, 0, :, :-1, :-1]) and torch.all(patch[:, 0, :, 0, :] == 0)
    w16 = torch.zeros(cout, 16, 3)
    w16[:, :9, :] = wt.detach()[:, 0].reshape(cout, 3, 9).permute(0, 2, 1)
    img = torch.empty(16 * 3 * cout, dtype=torch.bfloat16, device=DEV)
    _call("fpl_conv3d_k311_prep_weight", _p(w16.to(DEV)), 16, cout, _p(img), _st())
    y = torch.zeros((n, d, cout // 8, h, w, 8), dtype=torch.bfloat16, device=DEV)
    stats = torch.zeros(2 * cout, dtype=torch.float64, device=DEV)
    _call("fpl_conv3d_tc_k311", _p(xs), 2, 0, _p(img), _p(b.to(DEV)), _p(y), cout // 8, 0, _p(stats), n, d, h, w, 16, cout, 0, _st())
    rd = ref.detach()
    assert max_rel(from_c8(y).cpu(), rd) < 6e-3
    np.testing.assert_allclose(stats.cpu()[:cout], rd.double().sum((0, 2, 3, 4)), rtol=1e-4, atol=2e-3)
    dw16 = torch.zeros(cout, 16, 3, device=DEV)
    _call("fpl_conv3d_wgrad_tc_k311", _p(xs), 2, 0, _p(to_c8(g.to(DEV))), cout // 8, 0, _p(dw16), n, d, h, w, 16, cout, _st())
    dw = dw16.cpu()[:, :9, :].permute(0, 2, 1).reshape(cout, 1, 3, 3, 3)
    assert max_rel(dw, wt.grad) < 1e-4
    assert float(dw16.cpu()[:, 9:, :].abs().max()) == 0.0
    # hi/lo split: an fp32 image and fp32 weights through bf16 operands, [x_hi | x_lo | x_hi] x [w_hi | w_hi | w_lo]
    xf = randn(205, n, 1, d, h, w)
    wf = randn(206, cout, 1, 3, 3, 3, scale=0.2)
    ref32 = F.conv3d(xf, wf, b, padding=1)
    xs4 = torch.empty((n, d, 4, h, w, 8), dtype=torch.bfloat16, device=DEV)
    _call("fpl_patch9_c8", _p(xf.to(DEV)), _p(xs4), 1, n, d, h, w, _st())
    wk = wf[:, 0].reshape(cout, 3, 9).permute(0, 2, 1)
    hi = bf16_round(wk)
    w48 = torch.zeros(cout, 48, 3)
    w48[:, 0:9], w48[:, 16:25], w48[:, 32:41] = hi, hi, wk - hi
    img48 = torch.empty(48 * 3 * cout, dtype=torch.bfloat16, device=DEV)
    _call("fpl_conv3d_k311_prep_weight", _p(w48.to(DEV)), 48, cout, _p(img48), _st())
    stats.zero_()
    _call("fpl_conv3d_tc_k311", _p(xs4), 4, 0, _p(img48), _p(b.to(DEV)), _p(y), cout // 8, 0, _p(stats), n, d, h, w, 48, cout, 32, _st())
    np.testing.assert_allclose(stats.cpu()[:cout], ref32.double().sum((0, 2, 3, 4)), rtol=2e-5, atol=2e-3)   # fp32-accurate sums
    np.testing.assert_allclose(stats.cpu()[cout:], (ref32.double() ** 2).sum((0, 2, 3, 4)), rtol=2e-5, atol=2e-3)
    assert max_rel(from_c8(y).cpu(), ref32) < 4e-3                                   # only the bf16 output rounding is left


@pytest.mark.parametrize("cin,cout,kd,shape", [(16, 16, 3, (2, 4, 16, 32)), (32, 16, 3, (1, 6, 16, 16)), (64, 32, 3, (2, 4, 8, 16)),
                                               (128, 128, 3, (2, 2, 8, 8)), (16, 16, 1, (1, 3, 16, 16)), (16, 32, 3, (1, 5, 20, 36)),
                                               (32, 32, 3, (2, 3, 10, 24)), (16, 8, 1, (2, 3, 14, 40))])
def test_wgrad_tapmajor_and_fold(cin, cout, kd, shape):
    """fpl_conv3d_wgrad_tc_tapmajor writes S[tap][cout][cin]; fpl_wgrad_tapmajor_to_dw_batch folds it into the
    PyTorch layout ACCUMULATING into dw.  Against torch's conv3d weight gradient on bf16-rounded operands."""
    n, d, h, w = shape
    x = bf16_round(randn(301, n, cin, d, h, w))
    wt = torch.zeros(cout, cin, kd, 3, 3, requires_grad=True)
    y = F.conv3d(x, wt, None, padding=(kd // 2, 1, 1))
    g = bf16_round(randn(302, *y.shape))
    y.backward(g)
    taps = kd * 9
    scratch = torch.zeros(taps * cout * cin, device=DEV)
    _call("fpl_conv3d_wgrad_tc_tapmajor", _p(to_c8(x.to(DEV))), cin // 8, 0, _p(to_c8(g.to(DEV))), cout // 8, 0, _p(scratch),
          n, d, h, w, cin, cout, kd, _st())
    s = scratch.cpu().view(taps, cout, cin).permute(1, 2, 0).reshape(cout, cin, kd, 3, 3)
    assert max_rel(s, wt.grad) < 1e-4
    # fold two layers' worth in one launch, on top of existing content
    import ctypes
    pre = randn(303, cout, cin, kd, 3, 3)
    dw_a, dw_b = pre.to(DEV).contiguous(), torch.zeros(cout, cin, kd, 3, 3, device=DEV)
    arr_s = (ctypes.c_void_p * 2)(scratch.data_ptr(), scratch.data_ptr())
    arr_d = (ctypes.c_void_p * 2)(dw_a.data_ptr(), dw_b.data_ptr())
    ci = (ctypes.c_int * 2)(cout, cout)
    cj = (ctypes.c_int * 2)(cin, cin)
    ct = (ctypes.c_int * 2)(taps, taps)
    _call("fpl_wgrad_tapmajor_to_dw_batch", 2, arr_s, arr_d, ci, cj, ct, None, _st())
    # only the first rows of a wider scratch
    half = torch.zeros(cout // 2, cin, kd, 3, 3, device=DEV)
    _call("fpl_wgrad_tapmajor_to_dw_batch", 1, (ctypes.c_void_p * 1)(scratch.data_ptr()), (ctypes.c_void_p * 1)(half.data_ptr()),
          (ctypes.c_int * 1)(cout // 2), (ctypes.c_int * 1)(cin), (ctypes.c_int * 1)(taps), (ctypes.c_int * 1)(cout), _st())
    assert max_rel(half.cpu(), wt.grad[:cout // 2]) < 1e-4
    assert max_rel(dw_b.cpu(), wt.grad) < 1e-4
    assert max_rel(dw_a.cpu(), wt.grad + pre) < 1e-4


def test_grad_scatter_add():
    """Segments of a flat gradient buffer are ADDED into the master buffer at other offsets (atomics; odd tails)."""
    rng = np.random.Generator(np.random.PCG64(311))
    counts = [1, 3, 4, 5, 16, 1023, 4096, 70001]
    src_off, dst_off, so, do = [], [], 0, 8
    for c in counts:
        src_off.append(so)
        dst_off.append(do)
        so += (c + 3) // 4 * 4
        do += (c + 3) // 4 * 4 + 4
    src = torch.from_numpy(rng.standard_normal(so).astype(np.float32)).to(DEV)
    dst0 = torch.from_numpy(rng.standard_normal(do + 8).astype(np.float32))
    dst = dst0.clone().to(DEV)
    table = torch.tensor([[a, b, c] for a, b, c in zip(src_off, dst_off, counts)], dtype=torch.int32, device=DEV)
    for _ in range(2):
        _call("fpl_grad_scatter_add", _p(dst), _p(src), _p(table), len(counts), max(counts), _st())
    want = dst0.clone()
    for a, b, c in zip(src_off, dst_off, counts):
        want[b:b + c] += 2 * src.cpu()[a:a + c]
    np.testing.assert_allclose(dst.cpu().numpy(), want.numpy(), rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("cin,cout,shape", [(16, 8, (2, 8, 16, 32)), (16, 8, (1, 5, 16, 16)), (32, 8, (1, 6, 8, 16)),
                                            (16, 16, (2, 5, 16, 16)), (64, 16, (1, 4, 8, 16)),
                                            # Cin 16, Cout 8, H >= 6, W >= 16: the row-stacked kernel (conv3d_wgrad_rs_kernel)
                                            (16, 8, (1, 3, 7, 20)), (16, 8, (2, 1, 12, 32)), (16, 8, (1, 4, 30, 70))])
def test_conv3d_wgrad_tc_k133_depth_stacked(cin, cout, shape):
    """k(1,3,3) weight gradient with depth planes stacked in M and N (the head: cout = 8 = one channel group of a wider
    dy buffer, 4 planes per MMA set; cout = 16: 2 planes); depths that are not multiples of the stack."""
    n, d, h, w = shape
    x = bf16_round(randn(321, n, cin, d, h, w))
    dy = bf16_round(randn(322, n, cout, d, h, w))
    wt = torch.zeros(cout, cin, 1, 3, 3, requires_grad=True)
    _conv_ref(x, wt, None, 1).backward(dy)
    dw = torch.zeros(cout, cin, 1, 3, 3, device=DEV)
    # dy lives in the first channel groups of a buffer with 2 more (garbage) groups
    dyb = to_c8(torch.cat([dy, randn(323, n, 16, d, h, w)], 1).to(DEV))
    _call("fpl_conv3d_wgrad_tc", _p(to_c8(x.to(DEV))), cin // 8, 0, _p(dyb), (cout + 16) // 8, 0, _p(dw), n, d, h, w, cin, cout,
          1, _st())
    assert max_rel(dw.cpu(), wt.grad) < 1e-4


@pytest.mark.parametrize("cin,classes,shape", [(16, 2, (2, 3, 12, 40)), (16, 5, (1, 2, 9, 33)), (32, 2, (1, 4, 16, 32)),
                                               (32, 8, (1, 2, 8, 70)), (16, 3, (1, 2, 5, 7)), (16, 2, (2, 3, 45, 100)),
                                               (16, 7, (1, 2, 30, 64)), (32, 4, (1, 1, 17, 35))])
def test_head_cuda_core_fwd_and_dgrad(cin, classes, shape):
    """csrc/head.cu / head_tc.cu (forward, W >= 32 and <= 7 classes: the tensor-core scatter form with three-term bf16
    weights) against torch's (1,3,3) conv on the bf16-rounded activation: fp32 logits; input gradient (bf16),
    the one-channel-group bf16 copy of the logit gradient and the ACCUMULATED bias gradient from one dgrad pass."""
    n, d, h, w = shape
    x = bf16_round(randn(401, n, cin, d, h, w)).requires_grad_(True)
    wt = randn(402, classes, cin, 1, 3, 3, scale=0.2).requires_grad_(True)
    b = randn(403, classes, scale=0.1).requires_grad_(True)
    ref = F.conv3d(x, wt, b, padding=(0, 1, 1))
    dl = randn(404, *ref.shape)
    ref.backward(dl)
    xb = to_c8(torch.cat([x.detach(), randn(405, n, 8, d, h, w)], 1).to(DEV))            # a slice of a wider buffer
    logits = torch.empty(ref.shape, device=DEV)
    _call("fpl_head_fwd", _p(xb), (cin + 8) // 8, 0, _p(wt.detach().to(DEV)), _p(b.detach().to(DEV)), _p(logits), n, d, h, w, cin,
          classes, _st())
    np.testing.assert_allclose(logits.cpu().numpy(), ref.detach().numpy(), rtol=2e-5, atol=2e-5)
    g = torch.zeros((n, d, cin // 8 + 1, h, w, 8), dtype=torch.bfloat16, device=DEV)
    dl8 = torch.zeros((n, d, 1, h, w, 8), dtype=torch.bfloat16, device=DEV)
    db = torch.ones(classes, device=DEV)
    _call("fpl_head_dgrad", _p(dl.to(DEV)), _p(wt.detach().to(DEV)), _p(g), cin // 8 + 1, 1, _p(dl8), 1, 0, _p(db), n, d, h, w, cin,
          classes, _st())
    got = from_c8(g).cpu()
    assert torch.all(got[:, :8] == 0)                                                     # the neighbouring group is untouched
    assert max_rel(got[:, 8:], x.grad) < 6e-3
    copy = from_c8(dl8).cpu()
    assert torch.equal(copy[:, :classes], bf16_round(dl)) and torch.all(copy[:, classes:] == 0)
    np.testing.assert_allclose(db.cpu().numpy() - 1.0, b.grad.numpy(), rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("kd2,shape,c", [(2, (2, 3, 5, 7), 16), (1, (1, 4, 8, 8), 8), (2, (1, 1, 1, 6), 24), (2, (1, 8, 16, 16), 32)])
def test_upsample2x_align_corners_fwd_bwd(kd2, shape, c):
    """nn.Upsample(scale_factor=2, trilinear / bilinear, align_corners=True) (UpBlock bilinear mode) against torch, into a
    channel slice of a wider buffer; the gather backward against autograd."""
    n, d, h, w = shape
    x = bf16_round(randn(501, n, c, d, h, w)).requires_grad_(True)
    if kd2 == 2:
        ref = F.interpolate(x, scale_factor=2, mode="trilinear", align_corners=True)
    else:
        ref = F.interpolate(x.transpose(1, 2).reshape(n * d, c, h, w), scale_factor=2, mode="bilinear", align_corners=True)
        ref = ref.reshape(n, d, c, 2 * h, 2 * w).transpose(1, 2)
    g = bf16_round(randn(502, *ref.shape))
    ref.backward(g)
    do = d * kd2
    cat = torch.zeros((n, do, 2 * c // 8, 2 * h, 2 * w, 8), dtype=torch.bfloat16, device=DEV)
    _call("fpl_upsample2x_c8", _p(to_c8(x.detach().to(DEV))), c // 8, 0, _p(cat), 2 * c // 8, c // 8, n, d, h, w, c, kd2, _st())
    out = from_c8(cat).cpu()
    assert torch.all(out[:, :c] == 0)
    assert max_rel(out[:, c:], ref.detach()) < 6e-3
    gcat = to_c8(torch.cat([torch.zeros_like(g), g], 1).to(DEV))
    gx = torch.zeros((n, d, c // 8, h, w, 8), dtype=torch.bfloat16, device=DEV)
    _call("fpl_upsample2x_c8_bwd", _p(gcat), 2 * c // 8, c // 8, _p(gx), c // 8, 0, n, d, h, w, c, kd2, _st())
    assert max_rel(from_c8(gx).cpu(), x.grad) < 6e-3
    s = torch.ones(c, device=DEV)
    _call("fpl_channel_sum_c8", _p(gcat), 2 * c // 8, c // 8, _p(s), n, do, 2 * h, 2 * w, c, _st())
    np.testing.assert_allclose(s.cpu().numpy() - 1.0, g.sum((0, 2, 3, 4)).numpy(), rtol=2e-4, atol=2e-3)


# ------------------------------------------------------------------------------------------------------------------
# round 2: device data path of the loss (uint8 labels / agreement codes), entropy term, loss_softmax = False
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("c", [2, 5])
def test_dice_ce_uint8_labels_and_weight_codes_equal_the_fp32_layout(c):
    """SURVEY 8 f-3: a uint8 label map + a uint8 agreement code (0/1/2) + per-sample image weights give the SAME loss and
    gradient as the PyMIC layout (fp32 one-hot + fp32 pixel weight folded by set_weight_ on the host)."""
    from oracle import fpl_filter, losses, synth
    from fplplus_b200.loss import CombinedLoss
    from fplplus_b200.registry import loss_dict
    shape = (8, 24, 32)
    lab = synth.synth_label(3, c, shape, seed=5)
    r = np.random.Generator(np.random.PCG64(8))
    code = r.integers(0, 3, (3, 1) + shape).astype(np.uint8)
    iw = r.uniform(0.01, 1.01, 3).astype(np.float32)
    pw = np.stack([fpl_filter.set_weight_(iw[i], 0.5 * code[i].astype(np.float32)) for i in range(3)], 0).astype(np.float32)
    z = randn(77, 3, c, *shape, scale=2.0)
    crit = CombinedLoss({"loss_type": ["DiceLoss", "CrossEntropyLoss"], "loss_weight": [0.4, 0.6]}, loss_dict)
    out = {}
    for mode in ("fp32", "u8"):
        zz = z.clone().to(DEV).requires_grad_(True)
        if mode == "fp32":
            d = {"prediction": zz, "ground_truth": torch.from_numpy(synth.one_hot(lab, c)).to(DEV),
                 "pixel_weight": torch.from_numpy(pw).to(DEV)}
        else:
            d = {"prediction": zz, "ground_truth": torch.from_numpy(lab).to(DEV), "pixel_weight": torch.from_numpy(code).to(DEV),
                 "image_weight": torch.from_numpy(iw), "fold_image_weight": True}
        loss = crit(d)
        loss.backward()
        out[mode] = (float(loss), zz.grad.cpu(), crit.last_hard_dice().cpu())
    assert abs(out["fp32"][0] - out["u8"][0]) <= 1e-6 * abs(out["fp32"][0])
    torch.testing.assert_close(out["u8"][1], out["fp32"][1], rtol=1e-5, atol=1e-10)
    torch.testing.assert_close(out["u8"][2], out["fp32"][2], rtol=1e-9, atol=0)
    # and against the float64 closed form of the reference losses
    lv, dz, _ = losses.dice_ce_closed_form(z.numpy(), synth.one_hot(lab, c), pw, 0.4, 0.6)
    assert abs(out["u8"][0] - lv) <= 1e-5 * abs(lv)
    assert max_rel(out["u8"][1], torch.from_numpy(dz).float()) < 1e-4
    # unfolded codes (no image weight): weight = code / 2
    zz = z.clone().to(DEV).requires_grad_(True)
    l2 = crit({"prediction": zz, "ground_truth": torch.from_numpy(lab).to(DEV), "pixel_weight": torch.from_numpy(code).to(DEV)})
    lv2, _, _ = losses.dice_ce_closed_form(z.numpy(), synth.one_hot(lab, c), 0.5 * code.astype(np.float32), 0.4, 0.6)
    assert abs(float(l2) - lv2) <= 1e-5 * abs(lv2)


def test_entropy_term_and_probability_inputs_match_the_oracle():
    """a12: entropy regulariser -sum p*log2(p+1e-10)/(N*D*H*W) (agent_seg.py:353,467) as a fused term of the loss
    kernels (value + gradient); loss_softmax = False (loss/seg/abstract.py:16-21): predictions already are probabilities."""
    from oracle import losses, synth
    from fplplus_b200.loss import CombinedLoss, DiceLoss
    from fplplus_b200.registry import loss_dict
    shape, c = (8, 16, 32), 3
    lab = synth.synth_label(2, c, shape, seed=9)
    y = torch.from_numpy(synth.one_hot(lab, c))
    z = randn(78, 2, c, *shape, scale=2.0)
    crit = CombinedLoss({"loss_type": ["DiceLoss", "CrossEntropyLoss"], "loss_weight": [0.5, 0.5], "entropy_weight": 0.3}, loss_dict)
    zz = z.clone().to(DEV).requires_grad_(True)
    loss = crit({"prediction": zz, "ground_truth": y.to(DEV)})
    loss.backward()
    zr = z.clone().requires_grad_(True)
    ref = losses.combined_loss(zr, y, None, 0.5, 0.5) + 0.3 * losses.entropy_bits(zr)
    ref.backward()
    assert abs(float(loss) - float(ref)) <= 1e-5 * abs(float(ref))
    assert max_rel(zz.grad.cpu(), zr.grad) < 1e-4
    assert abs(float(crit.last_entropy()) - float(losses.entropy_bits(z))) <= 1e-5 * float(losses.entropy_bits(z))
    # probabilities in, no softmax inside
    p = torch.softmax(z, 1)
    crit2 = DiceLoss({"loss_softmax": False})
    pp = p.clone().to(DEV).requires_grad_(True)
    l2 = crit2({"prediction": pp, "ground_truth": y.to(DEV)})
    l2.backward()
    pr = p.clone().requires_grad_(True)
    r2 = losses.dice_loss(pr, y, None, softmax=False)
    r2.backward()
    assert abs(float(l2) - float(r2)) <= 1e-5 * abs(float(r2))
    assert max_rel(pp.grad.cpu(), pr.grad) < 1e-4
    with pytest.raises(ValueError):
        CombinedLoss({"loss_type": ["DiceLoss"], "loss_weight": [1.0], "entropy_weight": 0.1, "loss_softmax": False}, loss_dict)(
            {"prediction": pp, "ground_truth": y.to(DEV)})


@pytest.mark.parametrize("weighted", [False, True])
def test_exact_data_parallel_dice_equals_the_global_batch_loss(weighted):
    """SURVEY 8e: nn.DataParallel evaluates Dice / CE over the gathered global batch.  Emulation of two ranks on one
    GPU: per-rank reduce passes, the (6C+3) sums added (what the all-reduce does), per-rank gradient passes with
    n_global = 2n and gradient scale 2 (the parameter gradients are averaged over ranks afterwards).  The loss equals the
    loss of ONE call on the concatenated batch and each rank's dlogits equal 2x its slice of that call's dlogits."""
    from oracle import synth
    shape, c, n = (8, 16, 32), 2, 2
    lab = synth.synth_label(2 * n, c, shape, seed=31)
    y = torch.from_numpy(synth.one_hot(lab, c)).to(DEV)
    z = randn(32, 2 * n, c, *shape, scale=2.0).to(DEV)
    w = torch.from_numpy(synth.synth_pixel_weight(lab, seed=31)[0]).to(DEV) if weighted else None
    sp = shape[0] * shape[1] * shape[2]
    one = torch.ones((), device=DEV)

    def reduce_(zz, yy, ww, sums, nn_):
        _call("fpl_dice_ce_reduce_ex", _p(zz), _p(yy), None, _p(ww), None, None, _p(sums), nn_, c, sp, 0, 0, _st())

    def grad_(zz, yy, ww, sums, nn_, scale, n_global):
        loss = torch.zeros((), device=DEV)
        dz = torch.empty_like(zz)
        _call("fpl_dice_ce_grad_ex", _p(zz), _p(yy), None, _p(ww), None, None, _p(sums), 0.5, 0.5, 0.0, scale, _p(one),
              _p(loss), _p(dz), nn_, c, sp, 0, n_global, _st())
        return float(loss), dz

    full = torch.zeros(6 * c + 3, dtype=torch.float64, device=DEV)
    reduce_(z, y, w, full, 2 * n)
    loss_full, dz_full = grad_(z, y, w, full, 2 * n, 1.0, 0)
    halves = [(z[:n].contiguous(), y[:n].contiguous(), None if w is None else w[:n].contiguous()),
              (z[n:].contiguous(), y[n:].contiguous(), None if w is None else w[n:].contiguous())]
    parts = []
    for zz, yy, ww in halves:
        s_ = torch.zeros(6 * c + 3, dtype=torch.float64, device=DEV)
        reduce_(zz, yy, ww, s_, n)
        parts.append(s_)
    total = parts[0] + parts[1]                                  # the all-reduce
    torch.testing.assert_close(total, full, rtol=1e-12, atol=1e-9)
    for r, (zz, yy, ww) in enumerate(halves):
        loss_r, dz_r = grad_(zz, yy, ww, total, n, 2.0, 2 * n)
        assert abs(loss_r - loss_full) <= 1e-6 * abs(loss_full)
        torch.testing.assert_close(dz_r, 2.0 * dz_full[r * n:(r + 1) * n], rtol=1e-5, atol=1e-10)
        # and it is NOT the per-rank loss (Dice is a ratio of sums)
        loss_local, _ = grad_(zz, yy, ww, parts[r], n, 1.0, 0)
        assert abs(loss_local - loss_full) > 1e-5 * abs(loss_full)
