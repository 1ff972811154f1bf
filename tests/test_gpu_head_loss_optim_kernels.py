"""Per-kernel parity of the rest of the training step at the sizes the benchmark runs: the output head forward and data
gradient (tensor-core and CUDA-core forms), the ConvTranspose k2 s2 forward, the fused Dice + CE loss (reduction, loss
value, hard Dice and gradient) and the multi-tensor Adam over the network's parameter list.  Each kernel is compared with
a float64 reference of the same operation on the operands it sees (computed on the device); each bar names the rounding
it allows and is applied per element, or per sum where the output is a sum.

The case lists are chosen with host restatements of the launch decisions (first section, no GPU needed) so that at the
full SM budget and at 16 SMs the persistent head kernels walk more tiles per CTA than their ring has stages and cross
from one sample to the next, the loss threads walk several load batches with a partial last one, and the Adam blocks walk
several chunks.  Outputs go into a channel slice of a wider buffer whose other groups hold SENTINEL, or into a buffer
with a SENTINEL guard tail; inputs come from a slice at a non-zero group offset wherever the entry point takes one."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests._util import (DEV, FULL_SMS, SENTINEL, bitwise_equal, cdiv, read_slice, run_sm_budgets, sentinel_buf,
                         slice_buf)

U24 = 2.0 ** -24                        # fp32 unit roundoff
GUARD = 4096                            # SENTINEL elements after every fp32 output


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


def _gen(seed):
    g = torch.Generator(device=DEV)
    g.manual_seed(seed)
    return g


def _randn(seed, *shape):
    return torch.randn(shape, generator=_gen(seed), device=DEV)


def _rand(seed, *shape):
    return torch.rand(shape, generator=_gen(seed), device=DEV)


def _bf16(t):
    return t.to(torch.bfloat16).float()


def _guarded(numel, fill=float("nan")):
    """(an fp32 output of numel elements filled with `fill`, the whole buffer with a SENTINEL guard tail)."""
    buf = torch.full((numel + GUARD,), SENTINEL, device=DEV)
    buf[:numel] = fill
    return buf[:numel], buf


def _tail_ok(buf, numel):
    return bool((buf[numel:] == SENTINEL).all())


# ------------------------------------------------------------------------------------------
# host restatements of launch decisions (so that the case lists provably reach them)
# ------------------------------------------------------------------------------------------
def _head_fwd_plan(sms, n, d, h, w, cin, classes):
    """fpl_head_fwd (csrc/head.cu, head_tc.cu): ("tc", grid, tiles, stages, nb) when fpl_head_fwd_tc_eligible -- tiles of
    16 rows x 30 interior columns, UMMA N = 9 * classes rounded up to 16, two CTAs per SM (100 KB) when nb <= 32 else
    one (160 KB), stages from that budget, at most 6 -- else ("cuda", blocks, 0, 0, 0): 8 rows x 64 columns per block."""
    if cin in (16, 32) and 1 <= classes <= 7 and h >= 4 and w >= 32:
        nb = cdiv(9 * classes, 16) * 16
        a_bytes = (cin // 8) * 18 * 32 * 16
        b_bytes = cdiv(3 * (cin // 8) * nb * 16, 128) * 128
        stages = min(6, ((100 if nb <= 32 else 160) * 1024 - b_bytes - 512) // a_bytes)
        tiles = cdiv(h, 16) * cdiv(w, 30) * n * d
        return "tc", min((2 if nb <= 32 else 1) * sms, tiles), tiles, stages, nb
    return "cuda", cdiv(w, 64) * cdiv(h, 8) * n * d, 0, 0, 0


def _head_dgrad_plan(sms, n, d, h, w, cin, classes):
    """fpl_head_dgrad: ("tc", grid, tiles, 3 stages) when fpl_head_dgrad_tc_eligible -- tiles of 16 rows x 32 columns,
    two CTAs per SM -- else ("cuda", blocks, voxels per thread, 0): 8 rows x 16 threads x VPT columns per block."""
    if cin in (16, 32) and 1 <= classes <= 2 and h >= 4 and w >= 32:
        tiles = cdiv(h, 16) * cdiv(w, 32) * n * d
        return "tc", min(2 * sms, tiles), tiles, 3
    vpt = 4 if cin == 16 else 2
    return "cuda", cdiv(w, 16 * vpt) * cdiv(h, 8) * n * d, vpt, 0


def _walks(grid, tiles, per_sample):
    """(most tiles a CTA walks, whether some CTA's next tile belongs to the next sample) of a grid-stride tile walk."""
    t = np.arange(max(tiles - grid, 0))
    return cdiv(tiles, grid), bool(np.any(t // per_sample != (t + grid) // per_sample))


def _convt_fwd_plan(sms, cin, cout, kd2, n, d, h, w):
    """convt_gemm_launch mode 0 (csrc/convt_tc.cu): (grid, items, stages): GEMM N = taps x cout in slices of <= 128
    columns, K chunks of <= 64 channels, 16x8 low-resolution tiles x slices, two CTAs per SM."""
    ndim = 4 * kd2 * cout
    nb = ndim
    if nb > 128:
        nb = next(s for s in (128, 64, 32, 16) if ndim % s == 0)
    kc = 64
    while kc > 16 and cin % kc:
        kc //= 2
    stages = max(2, min(8, 96 * 1024 // ((kc // 8) * 2048 + kc * nb * 2)))
    items = cdiv(h, 16) * cdiv(w, 8) * d * n * (ndim // nb)
    return min(2 * sms, items), items, stages


def _loss_plan(sms, n, c, spatial, lean, per_sm, grad):
    """dice_ce_{reduce,grad}_launch (csrc/loss.cu): (U, blocks per sample, batches thread 0 walks, whether the walk ends
    in a partial batch).  U = 8 for two classes with uint8 inputs, 2 for the other lean forms up to 5 classes, else 1;
    grid_x_for caps the blocks per sample at SMs x per_sm / n, per_sm = resident_blocks (1..4), doubled for the grad
    pass of every form but the two-class lean one."""
    s4 = spatial // 4
    u = 8 if (c == 2 and lean) else (2 if (lean and c <= 5) else 1)
    if grad and not (c == 2 and lean):
        per_sm *= 2
    bx = max(1, min(cdiv(s4, 256 * u), cdiv(sms * per_sm, n)))
    stride = bx * 256
    return u, bx, cdiv(s4, u * stride), s4 % (u * stride) != 0


def _adam_plan(sms, numels):
    """fpl_adam_multi_tensor: (grid, chunks): 4096-element chunks per tensor, at most 8 blocks per SM."""
    chunks = sum(cdiv(k, 4096) for k in numels)
    return min(chunks, 8 * sms), chunks


# (cin, classes, (n, d, h, w), coherent): coherent = x >= 0 and every weight's third bf16 term > 0, so that dropping
# that term moves the logits by ~2^-18 of the sum of the terms' magnitudes
HEAD_CASES = [
    (16, 2, (4, 32, 128, 128), True),              # the bench level: 17 tiles per CTA through 5 stages
    (32, 2, (2, 28, 128, 128), False),             # the shipped VS width: 2 stages
    (16, 3, (2, 8, 100, 94), False),               # nb 32, general epilogue, ragged H; dgrad on the CUDA cores
    (16, 5, (2, 8, 64, 96), False),                # nb 48: one CTA per SM
    (32, 7, (1, 12, 72, 128), False),              # nb 64, ragged H
    (16, 1, (2, 4, 50, 70), True),                 # nb 16; the one-class tensor-core dgrad, ragged H and W
    (16, 2, (2, 6, 37, 30), False),                # W < 32: both CUDA-core kernels
    (32, 8, (1, 4, 40, 64), False),                # 8 classes: both CUDA-core kernels
]

# (cin, cout, kd2, (n, d, h, w)) with (d, h, w) the low-resolution grid
CONVT_CASES = [
    (256, 128, 2, (4, 2, 8, 8)),                   # the bench's four up levels at n = 4
    (128, 64, 2, (4, 4, 16, 16)),
    (64, 32, 2, (4, 8, 32, 32)),
    (32, 16, 2, (4, 16, 64, 64)),
    (128, 64, 1, (4, 28, 32, 32)),                 # the kd2 = 1 levels of the shipped VS configuration
    (64, 32, 1, (4, 28, 64, 64)),
    (96, 48, 1, (1, 5, 27, 13)),                   # ragged low-resolution H / W, three N slices, K chunks of 32
    (64, 32, 2, (2, 3, 20, 12)),
]

# (name, n, classes, spatial, truth, weight, entropy, prob_input); truth "u8" / "onehot" / "soft", weight None / "code"
# (agreement codes without image weight) / "code_iw" / "map" (fp32)
LOSS_CASES = [
    ("bench_target", 4, 2, 32 * 128 * 128, "u8", "code_iw", False, False),     # lean, U = 8
    ("bench_source", 4, 2, 32 * 128 * 128, "onehot", None, False, False),      # non-lean, U = 1
    ("soft_map", 2, 3, 8 * 48 * 64, "soft", "map", False, False),              # + the plain entry points
    ("c5_lean", 2, 5, 5 * 40 * 60, "u8", "code", False, False),                # lean, U = 2, S/4 = 3000
    ("c8_entropy", 3, 8, 32 * 128 * 128, "u8", "code_iw", True, False),        # lean, U = 1, odd n
    ("prob_input", 1, 2, 36 * 128 * 128, "u8", None, False, True),             # probabilities in, n = 1
]


def _loss_lean(truth, weight):
    return truth == "u8" and weight != "map"


def test_case_lists_reach_the_launch_decisions():
    """At 148 and at 16 SMs the case lists run head-forward and head-dgrad CTAs that walk more tiles than twice their
    stage count (the ring and both TMEM accumulator sets wrap), tile walks that cross from sample n to n + 1, ragged last
    tiles in H and W, both head-forward epilogues (C == 2, the general one with nb <= 32 and > 32), the CUDA-core
    fallbacks, ConvTranspose CTAs that walk several items, loss threads that walk several U-batches with a partial last
    one in all three instantiation families, and Adam blocks that walk several chunks over more than 256 tensors."""
    from fplplus_b200.net import UNet2D5_dsbn
    import bench
    fwd0 = [_head_fwd_plan(FULL_SMS, *shape, cin, c) for cin, c, shape, _co in HEAD_CASES]
    dg0 = [_head_dgrad_plan(FULL_SMS, *shape, cin, c) for cin, c, shape, _co in HEAD_CASES]
    tc_fwd = [(c, shape, p) for (cin, c, shape, _co), p in zip(HEAD_CASES, fwd0) if p[0] == "tc"]
    assert any(c == 2 for c, _s, _p in tc_fwd)
    assert any(c != 2 and p[4] <= 32 for c, _s, p in tc_fwd) and any(p[4] > 32 for _c, _s, p in tc_fwd)
    assert any(s[2] % 16 for _c, s, _p in tc_fwd) and any(s[3] % 30 for _c, s, _p in tc_fwd)
    assert any(p[0] == "cuda" and s[3] < 32 for (_ci, _c, s, _co), p in zip(HEAD_CASES, fwd0))
    assert any(p[0] == "cuda" and c > 7 for (_ci, c, _s, _co), p in zip(HEAD_CASES, fwd0))
    tc_dg = [(c, shape) for (cin, c, shape, _co), p in zip(HEAD_CASES, dg0) if p[0] == "tc"]
    assert {c for c, _s in tc_dg} == {1, 2}
    assert any(s[2] % 16 and s[3] % 32 for _c, s in tc_dg)
    cuda_dg = [(c, shape) for (cin, c, shape, _co), p in zip(HEAD_CASES, dg0) if p[0] == "cuda"]
    assert any(c >= 3 for c, _s in cuda_dg) and any(s[3] < 32 for _c, s in cuda_dg)
    families = {(_loss_plan(FULL_SMS, n, c, s, _loss_lean(t, wt), 1, False)[0], _loss_lean(t, wt))
                for _nm, n, c, s, t, wt, _e, _pi in LOSS_CASES}
    assert {(8, True), (2, True), (1, False), (1, True)} <= families
    assert any(c >= 6 and _loss_lean(t, wt) for _nm, _n, c, _s, t, wt, _e, _pi in LOSS_CASES)
    assert any((s // 4) % (256 * _loss_plan(FULL_SMS, n, c, s, _loss_lean(t, wt), 1, False)[0])
               for _nm, n, c, s, t, wt, _e, _pi in LOSS_CASES)
    numels = [p.numel() for p in UNet2D5_dsbn(dict(bench.NET_PARAMS)).parameters()]
    assert len(numels) == 268 and any(k % 4 for k in numels)
    for sms in (FULL_SMS, 16):
        for plan_fn in (_head_fwd_plan, _head_dgrad_plan):
            walks = []
            for cin, c, (n, d, h, w), _co in HEAD_CASES:
                p = plan_fn(sms, n, d, h, w, cin, c)
                if p[0] == "tc":
                    per_sample = p[2] // n
                    walks.append((*_walks(p[1], p[2], per_sample), p[3]))
            assert any(k > 2 * stages for k, _x, stages in walks), (sms, plan_fn)
            assert any(x for _k, x, _s in walks), (sms, plan_fn)
        ct = [_convt_fwd_plan(sms, *case[:3], *case[3]) for case in CONVT_CASES]
        assert any(items > 2 * grid and cdiv(items, grid) > stages for grid, items, stages in ct), sms
        for grad in (False, True):
            for per_sm in (1, 2, 3, 4):
                plans = [_loss_plan(sms, n, c, s, _loss_lean(t, wt), per_sm, grad) + (_loss_lean(t, wt), c)
                         for _nm, n, c, s, t, wt, _e, _pi in LOSS_CASES]
                assert any(b > 1 and part for _u, _bx, b, part, _l, _c in plans), (sms, grad, per_sm)
                if sms == 16:          # and in the two-class lean and the U = 1 families
                    for fam in (lambda u, lean, c: u == 8, lambda u, lean, c: u == 1 and (not lean or c >= 6)):
                        assert any(b > 1 and part for u, _bx, b, part, lean, c in plans if fam(u, lean, c)), (grad, per_sm)
        grid, chunks = _adam_plan(sms, numels)
        assert cdiv(chunks, grid) >= 2 and grid > 1 and any(k > 4096 for k in numels), sms
    # the restatements against hand-derived values of the source
    assert _head_fwd_plan(FULL_SMS, 4, 32, 128, 128, 16, 2) == ("tc", 296, 5120, 5, 32)
    assert _head_fwd_plan(16, 2, 28, 128, 128, 32, 2) == ("tc", 32, 2240, 2, 32)
    assert _head_fwd_plan(FULL_SMS, 2, 8, 64, 96, 16, 5) == ("tc", 148, 256, 6, 48)
    assert _head_dgrad_plan(16, 4, 32, 128, 128, 16, 2) == ("tc", 32, 4096, 3)
    assert _head_dgrad_plan(FULL_SMS, 2, 8, 100, 94, 16, 3)[:3] == ("cuda", 2 * 13 * 16, 4)
    assert _convt_fwd_plan(FULL_SMS, 32, 16, 2, 4, 16, 64, 64) == (296, 2048, 6)
    assert _convt_fwd_plan(FULL_SMS, 256, 128, 2, 4, 2, 8, 8) == (64, 64, 3)
    assert _loss_plan(FULL_SMS, 4, 2, 32 * 128 * 128, True, 2, False) == (8, 64, 1, False)
    assert _loss_plan(16, 4, 2, 32 * 128 * 128, True, 2, False) == (8, 8, 8, False)
    assert _loss_plan(16, 3, 8, 32 * 128 * 128, True, 1, True) == (1, 11, 47, True)
    assert _adam_plan(FULL_SMS, numels) == (1184, 2102) and _adam_plan(16, numels) == (128, 2102)


# ------------------------------------------------------------------------------------------
# 1. head forward (fpl_head_fwd)
# ------------------------------------------------------------------------------------------
def _head_weights(seed, classes, cin, coherent):
    """fp32 weights [classes, cin, 1, 3, 3].  Coherent: w = b0 + b1 + b2 with b0 a random bf16 number of exponent e,
    b1 = +-(1 + j/128) 2^(e-9) and b2 = k 2^(e-23), k in [32, 63]: 24 significant bits, so w is exact in fp32, and the
    kernel's split bf16(w), bf16(w - b0), ... returns exactly (b0, b1, b2) with a positive third term.  b1 never has
    the sign opposite to a power-of-two b0, and |b1| is never a power of two, so no rounding meets a binade edge."""
    shape = (classes, cin, 1, 3, 3)
    if not coherent:
        return _randn(seed, *shape) * 0.2
    b0 = _bf16(_randn(seed, *shape) * 0.2)
    b0 = torch.where(b0.abs() < 1e-3, torch.full_like(b0, 0.125), b0)
    e = torch.floor(torch.log2(b0.abs()))
    g = _gen(seed + 1)
    j = torch.randint(1, 128, shape, generator=g, device=DEV).float()
    s = torch.randint(0, 2, shape, generator=g, device=DEV).float() * 2 - 1
    s = torch.where(b0.abs() == torch.exp2(e), torch.sign(b0), s)
    k = torch.randint(32, 64, shape, generator=g, device=DEV).float()
    b1 = s * (1 + j / 128) * torch.exp2(e - 9)
    b2 = k * torch.exp2(e - 23)
    w = b0.double() + b1.double() + b2.double()
    assert torch.equal(w.float().double(), w)
    return w.float()


def _ulp_bf16(r):
    a = r.abs()
    e = torch.floor(torch.log2(torch.where(a > 0, a, torch.ones_like(a))))
    return torch.where(a > 0, torch.exp2(e - 7), torch.zeros_like(a))


@pytest.mark.gpu
@pytest.mark.parametrize("cin,classes,shape,coherent", HEAD_CASES)
def test_head_fwd_matches_float64_and_is_grid_independent(cin, classes, shape, coherent, sm_budgets, record_property):
    """fp32 logits of the (1,3,3) head conv, x read from channel group 1 of a wider buffer (SENTINEL elsewhere), against
    float64 conv3d on the bf16 x with the fp32 weights and bias; bitwise identical at 148 and 16 SMs (each voxel has one
    owner and a fixed summation order)."""
    n, d, h, w = shape
    kind = _head_fwd_plan(FULL_SMS, n, d, h, w, cin, classes)[0]
    x = _bf16(_randn(1001, n, cin, d, h, w))
    if coherent:
        x = x.abs()
    wt = _head_weights(1002, classes, cin, coherent)
    b = _randn(1003, classes) * 0.1
    xb = slice_buf(x, cin // 8 + 2, 1)
    numel = n * classes * d * h * w

    def run():
        out, buf = _guarded(numel)
        _call("fpl_head_fwd", _p(xb), cin // 8 + 2, 1, _p(wt), _p(b), _p(out), n, d, h, w, cin, classes, _st())
        return buf

    b148, b16 = sm_budgets(run)
    assert bitwise_equal(b148, b16)
    assert _tail_ok(b148, numel)
    got = b148[:numel].view(n, classes, d, h, w).double()
    ref = F.conv3d(x.double(), wt.double(), b.double(), padding=(0, 1, 1))
    bound = F.conv3d(x.double().abs(), wt.double().abs(), None, padding=(0, 1, 1))
    bias = b.double().abs().view(1, -1, 1, 1, 1)
    if kind == "tc":
        # exact bf16 x bf16 products of x and the three weight terms, fp32 accumulation in the tensor pipe over 3-6
        # chained MMAs of K = 16 and the fp32 sums of the epilogue: 2^-19 of the sum of the terms' magnitudes
        tol = 2.0 ** -19 * bound + 2.0 ** -22 * bias
    else:
        # a chain of 9 cin fp32 FMAs, then the bias add: (9 cin + 1) roundings of at most the sum of the magnitudes
        tol = (9 * cin + 1) * U24 * bound + U24 * bias
    ratio = float(((got - ref).abs() / tol).max())
    record_property("head_fwd_%s_err_over_bar" % kind, ratio)
    assert ratio <= 1.0, ratio


# ------------------------------------------------------------------------------------------
# 2. head data gradient (fpl_head_dgrad)
# ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cin,classes,shape,coherent", HEAD_CASES)
def test_head_dgrad_matches_float64_and_is_grid_independent(cin, classes, shape, coherent, sm_budgets, record_property):
    """dX into channel groups 1.. of a buffer with two SENTINEL groups more, the bf16 copy of dL into group 1 of two,
    and the bias gradient accumulated onto pre-filled values.  The tensor-core kernel multiplies bf16(W) by dL carried
    as hi + lo bf16 planes; the CUDA-core kernel uses the fp32 operands.  dX and dL8 are bitwise identical at 148 and 16
    SMs; the bias gradient is not (fp32 atomics)."""
    n, d, h, w = shape
    plan = {sms: _head_dgrad_plan(sms, n, d, h, w, cin, classes) for sms in (FULL_SMS, 16)}
    kind = plan[FULL_SMS][0]
    wt = _head_weights(1102, classes, cin, False)
    dl = _randn(1104, n, classes, d, h, w)
    pre = _randn(1105, classes)
    c8 = cin // 8

    def run():
        g = sentinel_buf(n, d, c8 + 2, h, w)
        dl8 = sentinel_buf(n, d, 2, h, w)
        db = pre.clone()
        _call("fpl_head_dgrad", _p(dl), _p(wt), _p(g), c8 + 2, 1, _p(dl8), 2, 1, _p(db), n, d, h, w, cin, classes, _st())
        return g, dl8, db

    (g148, l148, db148), (g16, l16, db16) = sm_budgets(run)
    assert bitwise_equal(g148, g16) and bitwise_equal(l148, l16)
    copy = read_slice(l148, 1, 8, device=DEV)
    assert torch.equal(copy[:, :classes], _bf16(dl)) and bool((copy[:, classes:] == 0).all())
    got = read_slice(g148, 1, cin, device=DEV).double()
    if kind == "tc":
        hi = _bf16(dl)
        dl_eff, w_eff = hi.double() + _bf16(dl - hi).double(), _bf16(wt).double()
        # fp32 accumulation of exact products over 3 chained MMAs of K = 16: 2^-19 of the sum of the magnitudes
        acc = 2.0 ** -19
    else:
        dl_eff, w_eff = dl.double(), wt.double()
        acc = 9 * classes * U24                  # a chain of 9 x classes fp32 FMAs
    ref = F.conv_transpose3d(dl_eff, w_eff, padding=(0, 1, 1))
    bound = F.conv_transpose3d(dl_eff.abs(), w_eff.abs(), padding=(0, 1, 1))
    # the bf16 rounding of the fp32 result (half an ulp of its magnitude) on top of the accumulation error
    acc = 1.01 * acc * bound
    tol = 0.5 * _ulp_bf16(ref.abs() + acc) + acc
    ratio = float(((got - ref).abs() / tol).max())
    record_property("head_dgrad_%s_err_over_bar" % kind, ratio)
    assert ratio <= 1.0, ratio
    # dbias: every term is an fp32 dL value; per-lane (tc) / per-thread (cuda) fp32 sums of L terms, a warp sum (5
    # levels), (cuda: 4 warps per block,) then one fp32 atomicAdd per warp (tc) / block (cuda) onto the running value
    s_ref = dl.double().sum((0, 2, 3, 4))
    s_abs = dl.double().abs().sum((0, 2, 3, 4))
    worst = 0.0
    for sms, db in ((FULL_SMS, db148), (16, db16)):
        _k, grid, a, _b = plan[sms]
        if kind == "tc":
            terms, atomics = 2 * cdiv(a, grid) + 5, 8 * grid
        else:
            terms, atomics = a + 5 + 4, grid
        bar = U24 * (terms * s_abs + atomics * (pre.double().abs() + s_abs))
        r = float(((db.double() - (pre.double() + s_ref)).abs() / bar).max())
        worst = max(worst, r)
        assert r <= 1.0, (sms, r)
    record_property("head_dbias_err_over_bar", worst)


# ------------------------------------------------------------------------------------------
# 3. ConvTranspose k2 s2 forward (fpl_convt_k2s2_fwd_tc)
# ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cin,cout,kd2,shape", CONVT_CASES)
def test_convt_fwd_matches_float64_and_is_grid_independent(cin, cout, kd2, shape, sm_budgets, record_property):
    """y = conv_transpose3d(x, W) + bias into the upper half of a 2 cout concat buffer with one more group; the lower
    half and the extra group hold SENTINEL.  x is read from group 1 of a wider buffer.  Bitwise identical at 148 and 16
    SMs."""
    n, d, h, w = shape
    x = _bf16(_randn(1201, n, cin, d, h, w))
    wt = _bf16(_randn(1202, cin, cout, kd2, 2, 2) * 0.2)
    b = _randn(1203, cout) * 0.1
    img = torch.empty(_lib().load().fpl_convt_weight_image_bytes(cin, cout, kd2) // 2, dtype=torch.bfloat16, device=DEV)
    _call("fpl_convt_prep_weight", _p(wt), cin, cout, kd2, 0, _p(img), _st())
    xb = slice_buf(x, cin // 8 + 1, 1)
    tot = 2 * cout // 8 + 1

    def run():
        y = sentinel_buf(n, d * kd2, tot, 2 * h, 2 * w)
        _call("fpl_convt_k2s2_fwd_tc", _p(xb), cin // 8 + 1, 1, _p(img), _p(b), _p(y), tot, cout // 8, n, d, h, w, cin,
              cout, kd2, _st())
        return y

    y148, y16 = sm_budgets(run)
    assert bitwise_equal(y148, y16)
    got = read_slice(y148, cout // 8, cout, device=DEV).double()
    ref = F.conv_transpose3d(x.double(), wt.double(), b.double(), stride=(kd2, 2, 2))
    bound = F.conv_transpose3d(x.double().abs(), wt.double().abs(), None, stride=(kd2, 2, 2))
    # bf16 output rounding (half an ulp) on top of fp32 accumulation over cin / 16 chained MMAs and the bias add
    acc = 2.0 ** -16 * (bound + b.double().abs().view(1, -1, 1, 1, 1))
    tol = 0.5 * _ulp_bf16(ref.abs() + acc) + acc
    ratio = float(((got - ref).abs() / tol).max())
    record_property("convt_fwd_err_over_bar", ratio)
    assert ratio <= 1.0, ratio


# ------------------------------------------------------------------------------------------
# 4. Dice + CE loss (fpl_dice_ce_reduce_ex / _loss_ex / _grad_ex, fpl_dice_ce_reduce / _grad)
# ------------------------------------------------------------------------------------------
W_DICE, W_CE, W_ENT = 0.5, 0.5, 0.3
GRAD_SCALE, GRAD_SCALE_DEV = 2.0, 0.25


def _loss_inputs(n, c, s, truth, weight, prob, seed):
    """Device tensors as the kernels read them and the float64 truth y [n, c, s] and weight w [n, s] they decode."""
    z = _randn(seed, n, c, s) * 2.0
    if prob:
        z = torch.softmax(z, 1)
    else:
        z[:, 1, ::97] = z[:, 0, ::97]                        # exact ties: the first maximum wins the argmax
    lab = torch.randint(0, c, (n, s), generator=_gen(seed + 1), device=DEV)
    dev = {"z": z.contiguous(), "soft": None, "label": None, "wmap": None, "code": None, "iw": None}
    if truth == "u8":
        dev["label"] = lab.to(torch.uint8)
        y = F.one_hot(lab, c).permute(0, 2, 1).double()
    elif truth == "onehot":
        dev["soft"] = F.one_hot(lab, c).permute(0, 2, 1).float().contiguous()
        y = dev["soft"].double()
    else:
        dev["soft"] = torch.softmax(_randn(seed + 2, n, c, s) * 3.0, 1).contiguous()
        y = dev["soft"].double()
    wf = torch.ones(n, s, device=DEV)
    if weight == "map":
        dev["wmap"] = _rand(seed + 3, n, s)
        wf = dev["wmap"]
    elif weight in ("code", "code_iw"):
        code = torch.randint(0, 3, (n, s), generator=_gen(seed + 4), device=DEV)
        dev["code"] = code.to(torch.uint8)
        a = 0.5 * code.float()
        wf = a
        if weight == "code_iw":
            dev["iw"] = (_rand(seed + 5, n) + 0.01).float()
            wf = torch.where(a < 1, torch.zeros_like(a), a) * dev["iw"].view(n, 1)    # fp32, as set_weight_
    return dev, y, wf.double()


def _loss_sums_ref(z64, y, w, c, prob, ent):
    """The 6C+3 sums of dice_ce_reduce_kernel in float64 (the entropy sum stays 0 unless requested), and the per-sum
    magnitude and term-evaluation bounds."""
    p = z64 if prob else torch.softmax(z64, 1)
    wb = w.unsqueeze(1)
    q = p * 0.999 + 5e-4
    ce = -(y * torch.log(q)).sum(1)
    l2 = torch.log2(p + 1e-10) * float(ent)
    zd = z64.detach()
    zmax = zd.amax(1, keepdim=True)
    idx = torch.arange(c, device=DEV).view(1, c, 1)
    am = torch.where(zd == zmax, idx, c).amin(1, keepdim=True)        # first maximum
    hot = (am == idx).double()
    sums = torch.cat([(wb * y * p).sum((0, 2)), (wb * y).sum((0, 2)), (wb * p).sum((0, 2)), w.sum().view(1),
                      (w * ce).sum().view(1), (hot * y).sum((0, 2)), y.sum((0, 2)), hot.sum((0, 2)),
                      (p * l2).sum().view(1)])
    pd, ced, l2d = p.detach(), ce.detach(), l2.detach()
    wa = w.abs()
    mag = torch.cat([(wa.unsqueeze(1) * y * pd).sum((0, 2)), (wa.unsqueeze(1) * y).sum((0, 2)),
                     (wa.unsqueeze(1) * pd).sum((0, 2)), wa.sum().view(1), (wa * ced.abs()).sum().view(1),
                     (hot * y).sum((0, 2)), y.sum((0, 2)), hot.sum((0, 2)), (pd * l2d.abs()).sum().view(1)])
    # evaluation error of the terms before they are added: a few ulps of the fp32 softmax in p; log(q) and log2(p)
    # absolute errors of a few 2^-24 on top of one ulp of their value
    qd = q.detach()
    ev = torch.cat([8 * (wa.unsqueeze(1) * y * pd).sum((0, 2)), torch.zeros(c, device=DEV, dtype=torch.float64),
                    8 * (wa.unsqueeze(1) * pd).sum((0, 2)), torch.zeros(1, device=DEV, dtype=torch.float64),
                    (wa * (y * (2 * torch.log(qd).abs() + 10)).sum(1)).sum().view(1),
                    torch.zeros(3 * c, device=DEV, dtype=torch.float64),
                    (pd * (6 * l2d.abs() + 12)).sum().view(1)]) * U24
    return sums, mag, ev


def _loss_of_sums(s, c, weighted, v, ent):
    i, yy, pp = s[:c], s[c:2 * c], s[2 * c:3 * c]
    dice = ((2 * i + 1e-5) / (yy + pp + 1e-5)).mean()
    cden = s[3 * c] + 1e-5 if weighted else v
    out = W_DICE * (1 - dice) + W_CE * s[3 * c + 1] / cden
    if ent:
        out = out + W_ENT * (-s[6 * c + 2] / v)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name,n,c,s,truth,weight,ent,prob", LOSS_CASES)
def test_dice_ce_matches_float64(name, n, c, s, truth, weight, ent, prob, sm_budgets, record_property):
    """Each of the 6C+3 sums against its own bar, the hard-Dice counters exactly (one-hot truth), the loss value from
    fpl_dice_ce_loss_ex and fpl_dice_ce_grad_ex, the hard Dice, and dlogits per element against float64 autograd of the
    closed form (evaluated at the kernel's sums), at 148 and 16 SMs."""
    dev, y, w = _loss_inputs(n, c, s, truth, weight, prob, 1301 + 10 * len(name))
    weighted = weight is not None
    lean = _loss_lean(truth, weight)
    ns = 6 * c + 3
    w_ent = W_ENT if ent else 0.0
    numel = n * c * s
    srcs = lambda: (_p(dev["z"]), _p(dev["soft"]), _p(dev["label"]), _p(dev["wmap"]), _p(dev["code"]), _p(dev["iw"]))
    gsd = torch.tensor([GRAD_SCALE_DEV], device=DEV)

    def run():
        sums = torch.zeros(ns, dtype=torch.float64, device=DEV)
        _call("fpl_dice_ce_reduce_ex", *srcs(), _p(sums), n, c, s, int(ent), int(prob), _st())
        loss1, hd = torch.full((1,), SENTINEL, device=DEV), torch.full((c,), SENTINEL, dtype=torch.float64, device=DEV)
        _call("fpl_dice_ce_loss_ex", *srcs(), _p(sums), W_DICE, W_CE, w_ent, _p(loss1), _p(hd), n, c, s, int(prob), 0,
              _st())
        loss2 = torch.full((1,), SENTINEL, device=DEV)
        dz, buf = _guarded(numel)
        _call("fpl_dice_ce_grad_ex", *srcs(), _p(sums), W_DICE, W_CE, w_ent, GRAD_SCALE, _p(gsd), _p(loss2), _p(dz), n, c,
              s, int(prob), 0, _st())
        res = dict(sums=sums, loss1=loss1, hd=hd, loss2=loss2, buf=buf)
        if truth == "soft":                   # the plain entry points are the same kernels with the PyMIC layout
            sums_p = torch.zeros(ns, dtype=torch.float64, device=DEV)
            _call("fpl_dice_ce_reduce", _p(dev["z"]), _p(dev["soft"]), _p(dev["wmap"]), _p(sums_p), n, c, s, _st())
            lp = torch.full((1,), SENTINEL, device=DEV)
            dzp, bufp = _guarded(numel)
            _call("fpl_dice_ce_grad", _p(dev["z"]), _p(dev["soft"]), _p(dev["wmap"]), _p(sums_p), W_DICE, W_CE, GRAD_SCALE,
                  _p(gsd), _p(lp), _p(dzp), n, c, s, _st())
            res.update(sums_p=sums_p, lp=lp, bufp=bufp)
        return res

    outs = sm_budgets(run)
    z64 = dev["z"].double().requires_grad_(True)
    ref, mag, ev = _loss_sums_ref(z64, y, w, c, prob, ent)
    ref = ref.detach()
    v = float(n * s)
    sc = GRAD_SCALE * GRAD_SCALE_DEV
    p = (z64 if prob else torch.softmax(z64, 1)).detach()
    wb = w.unsqueeze(1)
    worst = {"sums": 0.0, "loss": 0.0, "dz": 0.0}
    for sms, r in zip((FULL_SMS, 16), outs):
        # fp32 per-thread partials over at most L terms, a 5-level warp sum, then fp64: (L + 5) 2^-24 of the sum of
        # the terms' magnitudes, plus the evaluation error of each term
        u, _bx, batches, _part = _loss_plan(sms, n, c, s, lean, 1, False)
        L = 4 * u * batches
        per = torch.full((ns,), float(L + 5), dtype=torch.float64, device=DEV)
        per[6 * c + 2] = float(c * L + 5)
        bar = per * U24 * mag + ev + 1e-300
        assert torch.equal(r["loss1"], r["loss2"]), sms
        hi_, hy_, hp_ = (r["sums"][3 * c + 2 + k * c:3 * c + 2 + (k + 1) * c] for k in range(3))
        assert torch.equal(r["hd"], (2.0 * hi_ + 1e-5) / (hy_ + hp_ + 1e-5)), sms
        sets = [(r["sums"], r["loss2"], r["buf"])]
        if truth == "soft":
            sets.append((r["sums_p"], r["lp"], r["bufp"]))
        for ks, kl, buf in sets:
            err = (ks - ref).abs()
            worst["sums"] = max(worst["sums"], float((err / bar).max()))
            assert bool((err <= bar).all()), (sms, (err / bar).tolist())
            if truth != "soft":
                hard = slice(3 * c + 2, 6 * c + 2)
                assert torch.equal(ks[hard], ref[hard]), sms            # integer counts below 2^24: exact
            # the loss: the float64 closed form of the kernel's sums rounded to fp32 (half an ulp, and the double
            # arithmetic's order); that closed form differs from the reference's by the sums' errors times its slope
            sv = ks.clone().requires_grad_(True)
            lk = _loss_of_sums(sv, c, weighted, v, ent)
            lk.backward()
            lk = float(lk.detach())
            l_ref = float(_loss_of_sums(ref, c, weighted, v, ent))
            assert abs(float(kl) - lk) <= 2 * U24 * abs(lk), sms
            lbar = float((sv.grad.abs() * bar).sum()) * 1.01 + 2 * U24 * abs(l_ref)
            worst["loss"] = max(worst["loss"], abs(float(kl) - l_ref) / lbar)
            assert abs(float(kl) - l_ref) <= lbar, sms
            # dlogits: float64 autograd of the closed form evaluated at the kernel's sums
            z64.grad = None
            s_ref, _m, _e = _loss_sums_ref(z64, y, w, c, prob, ent)
            (_loss_of_sums(s_ref + (ks - s_ref.detach()), c, weighted, v, ent) * sc).backward()
            dz_ref = z64.grad
            assert _tail_ok(buf, numel)
            dz = buf[:numel].view(n, c, s).double()
            # per voxel: dL/dp_c in fp32 from the fp32-rounded per-class constants (terms of magnitude G_c, a few ulps
            # each), then the softmax backward p (g - p.g): 32 2^-24 of the magnitudes it combines
            den = ks[c:2 * c] + ks[2 * c:3 * c] + 1e-5
            a_c = (-W_DICE * 2.0 / (c * den)).view(1, c, 1)
            b_c = (W_DICE * (2 * ks[:c] + 1e-5) / (c * den * den)).view(1, c, 1)
            cden = float(ks[3 * c]) + 1e-5 if weighted else v
            G = (wb * (a_c * y + b_c)).abs() + (W_CE * 0.999 / cden) * wb.abs() * y / (p * 0.999 + 5e-4)
            if ent:
                G = G + (W_ENT / v) * (torch.log2(p + 1e-10).abs() + 2)
            if prob:
                tol = sc * 16 * U24 * G
            else:
                tol = sc * 32 * U24 * p * (G + (p * G).sum(1, keepdim=True))
            rz = float(((dz - dz_ref).abs() / (tol + 1e-30)).max())
            worst["dz"] = max(worst["dz"], rz)
            assert rz <= 1.0, (sms, rz)
    for k, val in worst.items():
        record_property("loss_%s_err_over_bar" % k, val)


# ------------------------------------------------------------------------------------------
# 5. fused Adam at the network's parameter list
# ------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_fused_adam_over_the_network_parameters_matches_torch_adam(sm_budgets, record_property):
    """FusedAdam over the 268 parameters of UNet2D5_dsbn(bench.NET_PARAMS) (7.69 M elements, 2102 chunks: blocks walk
    2 chunks at 148 SMs and 16-17 at 16, the last block bumps 268 step counters, more than its 256 threads) for three steps with a device
    learning rate; in the second step domain 1's BatchNorm parameters have no gradient.  Against torch.optim.Adam at
    rtol 1e-6 (the kernel repeats torch's fp32 arithmetic); per-tensor step counters exactly; bitwise the same at 148
    and 16 SMs (element-wise arithmetic)."""
    from fplplus_b200.net import UNet2D5_dsbn
    from fplplus_b200.optim import FusedAdam
    import bench
    named = list(UNet2D5_dsbn(dict(bench.NET_PARAMS)).named_parameters())
    init = [p.detach().to(DEV).clone() for _n, p in named]
    skip = {i for i, (nm, _p) in enumerate(named) if ".bns.1." in nm}
    assert 0 < len(skip) and len(named) > 256
    lr = 1e-4
    grads = []
    for step in range(3):
        gs = []
        for i, t in enumerate(init):
            g = _randn(1400 + 300 * step + i, *t.shape) * (10.0 ** ((i % 3) - 3))
            gs.append(None if (step == 1 and i in skip) else g)
        grads.append(gs)

    def run(opt_cls, lr_arg):
        params = [torch.nn.Parameter(t.clone()) for t in init]
        opt = opt_cls(params, lr_arg, weight_decay=1e-5)
        for gs in grads:
            for p, g in zip(params, gs):
                p.grad = None if g is None else g.clone()
            opt.step()
        return params, opt

    ref_params, ref_opt = run(torch.optim.Adam, lr)
    outs = sm_budgets(lambda: run(FusedAdam, torch.tensor(lr, dtype=torch.float32, device=DEV)))
    for (pa, _oa), (pb, _ob) in zip(outs[:1], outs[1:]):
        for a, b in zip(pa, pb):
            assert bitwise_equal(a.detach(), b.detach())
    params, opt = outs[0]
    worst = 0.0
    for i, (p, q) in enumerate(zip(params, ref_params)):
        d = (p.detach() - q.detach()).abs()
        worst = max(worst, float((d / (1e-7 + 1e-6 * q.detach().abs())).max()))
        torch.testing.assert_close(p.detach(), q.detach(), rtol=1e-6, atol=1e-7, msg=lambda m: "tensor %d: %s" % (i, m))
        so, sr = opt.state[p], ref_opt.state[q]
        assert float(so["step"]) == float(sr["step"]) == (2.0 if i in skip else 3.0), i
        # exp_avg can cancel to near 0 over the steps: rtol 1e-6 of the magnitudes it combines, (1 - beta1) |g| per
        # step (the weight-decayed gradient may round an ulp apart in torch's kernels and here)
        gsum = sum(g[i].double().abs() for g in grads if g[i] is not None)
        m_err = (so["exp_avg"].double() - sr["exp_avg"].double()).abs()
        assert bool((m_err <= 1e-6 * (sr["exp_avg"].double().abs() + 0.1 * gsum)).all()), i
        torch.testing.assert_close(so["exp_avg_sq"], sr["exp_avg_sq"], rtol=1e-6, atol=1e-15)
    record_property("adam_err_over_bar", worst)
