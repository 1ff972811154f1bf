"""Per-kernel parity of the no-grad forward path: the conv kernels with the eval-mode BatchNorm + PReLU (+ dropout)
epilogue, the eval affine batch, the activation-only max-pool, the tensor-core head, the batched weight staging and the
NCDHW -> C8 pack.  Every kernel is compared with a plain torch / float64 reference of the same operation, the dropout
masks with the host Philox restatement of tests/_util.py.  Each bar is bit-exact where the operation is exact and
otherwise names the rounding it allows.

Outputs go into a channel slice of a wider buffer whose other channel groups hold SENTINEL, inputs come from a slice
where the entry point takes one, and the persistent kernels run under the full SM budget and under 16 SMs (several
tiles / items per CTA) with bitwise-identical results."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests._util import (DEV, FULL_SMS, SENTINEL, bf16_round, bitwise_equal, cdiv, dropout_keep_c8, max_rel,
                         philox4x32_10, randn, read_slice, run_sm_budgets, sentinel_buf, slice_buf, to_c8)


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
    _KEEP.append(t)
    return _ops().ptr(t)


def _parr(ts):
    """HOST array of DEVICE pointers (None -> NULL entry)."""
    _KEEP.extend(t for t in ts if t is not None)
    return (ctypes.c_void_p * len(ts))(*[None if t is None else t.data_ptr() for t in ts])


def _iarr(vals):
    return (ctypes.c_int * len(vals))(*vals)


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


def _bn_params(seed, c):
    """gamma, beta, running mean, running var, conv bias (CPU fp32)."""
    gamma = randn(seed, c, scale=0.3) + 1.0
    beta = randn(seed + 1, c, scale=0.2)
    mean = randn(seed + 2, c, scale=0.1)
    var = randn(seed + 3, c, scale=0.2).abs() + 0.5
    bias = randn(seed + 4, c, scale=0.1)
    return gamma, beta, mean, var, bias


def _eval_affine(gamma, beta, mean, var, bias, eps=1e-5):
    """scale / shift (device fp32) of one layer through fpl_dsbn_eval_affine_batch, as the network derives them."""
    c = gamma.numel()
    scale, shift = torch.empty(c, device=DEV), torch.empty(c, device=DEV)
    dev = lambda t: None if t is None else t.to(DEV)
    _call("fpl_dsbn_eval_affine_batch", 1, _parr([dev(gamma)]), _parr([dev(beta)]), _parr([dev(mean)]), _parr([dev(var)]),
          _parr([dev(bias)]), _parr([scale]), _parr([shift]), _iarr([c]), eps, _st())
    return scale, shift


def _bcast(v):
    return v.view(1, -1, 1, 1, 1)


def _prelu_affine(acc, scale, shift, slope):
    z = acc * _bcast(scale.cpu()) + _bcast(shift.cpu())
    return torch.where(z > 0, z, slope * z)


def _tc_image(wt, cin, cout, kd):
    img = torch.empty(_lib().load().fpl_conv3d_weight_image_bytes(cin, cout, kd) // 2, dtype=torch.bfloat16, device=DEV)
    _call("fpl_conv3d_prep_weight", _p(wt.to(DEV)), cin, cout, kd, 0, _p(img), _st())
    return img


# ------------------------------------------------------------------------------------------
# host restatements of launch decisions (so that the case lists provably reach them)
# ------------------------------------------------------------------------------------------
def _tc_nsub(cin, cout, n, d, h, w):
    """The N split of conv3d_tc_launch (csrc/conv_tc.cu): make_config's nb, then nsub doubles (up to 4) while
    nb % (2*16*nsub) == 0, nb / (2*nsub) >= 32 and tiles * slices * nsub < 96."""
    nb = cout if cout <= 128 else next(b for b in (128, 64, 32, 16) if cout % b == 0)
    mn = cdiv(h, 16) * cdiv(w, 8) * d * n * (cout // nb)
    nsub = 1
    while nsub < 4 and nb % (nsub * 2 * 16) == 0 and nb // (nsub * 2) >= 32 and mn * nsub < 96:
        nsub *= 2
    return nsub


def _dfold_tail_split(cin, cout, n, d, h, w, sms):
    """Whether dfold_launch (csrc/conv_tc_dfold.cu) cuts its last (items mod grid) depth chunks into half-depth items:
    make_df_cfg's chunk depth, shared memory and CTAs per SM, then the `rem` condition."""
    plane = 18 * 10 * 16
    nb = cout
    dc = min(16 if nb == 16 else 8, d)
    b_bytes = 9 * cin * 3 * nb * 2
    a_bytes = cin // 8 * plane
    pb = 3 if a_bytes <= 2 * plane else 2
    fixed = b_bytes + 1024 + 512 + 2 * cout * 4 + 16
    stages = next((s for s in (4, 3, 2) if fixed + s * pb * a_bytes <= 110 * 1024), None)
    if stages is None:
        stages = next(s for s in (4, 3, 2) if fixed + s * pb * a_bytes <= 220 * 1024)
    smem = fixed + stages * pb * a_bytes
    tmem = 32
    while tmem < dc * nb:
        tmem *= 2
    ctas = 2 if smem <= 110 * 1024 and tmem <= 256 else 1
    total = cdiv(h, 16) * cdiv(w, 8) * cdiv(d, dc) * n
    grid = min(sms * ctas, total)
    rem = total % grid
    return rem > 0 and 2 * rem <= grid and dc >= 8 and dc % 2 == 0 and d % dc == 0


# (cin, cout, kd, (n, d, h, w), p): ragged 16x8 tiles, odd depths, kd 1 and 3, cout 48 (nb not a power of two),
# N split 1 / 2 / 4 (also with two staged slices: 256 -> 256), and > 32 tiles for the 16-SM run
TC_ACT_CASES = [
    (16, 16, 3, (1, 3, 20, 12), 0.3),
    (32, 48, 3, (1, 3, 18, 10), 0.5),
    (64, 64, 1, (2, 3, 17, 9), 0.2),
    (64, 64, 3, (1, 3, 16, 8), 0.3),
    (128, 128, 3, (1, 2, 8, 8), 0.3),
    (128, 128, 1, (1, 3, 5, 11), 0.5),
    (256, 256, 3, (1, 2, 4, 12), 0.0),
    (16, 32, 3, (2, 5, 33, 20), 0.0),
    (32, 16, 3, (1, 5, 33, 20), 0.4),
]

# (cin, cout, (n, d, h, w)): the dfold channel pairs, depths 2 / 17 / 20 (short last depth chunks), and the tail split
DFOLD_ACT_CASES = [
    (16, 16, (1, 17, 20, 12)),
    (16, 16, (1, 20, 16, 8)),
    (16, 32, (1, 2, 16, 8)),
    (32, 16, (1, 20, 18, 10)),
    (32, 64, (2, 17, 16, 9)),
    (64, 32, (1, 20, 20, 16)),
    (64, 32, (1, 2, 17, 8)),
    (16, 16, (1, 16, 64, 80)),      # 40 items on 32 CTAs at 16 SMs: the last 8 become 16 half-depth items
]


def test_host_philox_known_answers():
    """The host Philox4x32-10 reproduces the Random123 known-answer vectors."""
    kat = [((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
           ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
           ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
            (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]
    for ctr, key, want in kat:
        assert [int(v) for v in philox4x32_10(ctr, key)] == list(want)
    # vectorised over a batch of counters: the same words as one call per counter
    ctrs = np.array([c for c, _k, _w in kat], dtype=np.uint64)
    np.testing.assert_array_equal(philox4x32_10(ctrs, (7, 9)), np.stack([philox4x32_10(c, (7, 9)) for c in ctrs]))


def test_host_mask_layout_and_launch_decisions():
    """dropout_keep_c8 indexes vectors over (n, d, c8, h, w) and draws channel i of a group from word i; the case
    lists reach the N splits 1, 2, 4 of conv3d_tc_launch and the tail split of dfold_launch."""
    n, c, d, h, w, seed, offset, p = 2, 16, 3, 2, 5, 99, 2 ** 33 + 6, 0.5
    keep = dropout_keep_c8(seed, offset, n, c, d, h, w, p)
    thr = int(np.ceil(float(np.float32(p)) * 2.0 ** 24))
    for (nn, cc, dd, hh, ww) in ((0, 0, 0, 0, 0), (1, 13, 2, 1, 4), (0, 7, 1, 1, 2), (1, 8, 0, 0, 3)):
        vec = ((nn * d + dd) * (c // 8) + cc // 8) * h * w + hh * w + ww
        ctr = 2 * vec + offset + (cc % 8) // 4
        r = int(philox4x32_10((ctr & 0xFFFFFFFF, ctr >> 32, 0, 0), (seed, 0))[(cc % 8) % 4])
        assert bool(keep[nn, cc, dd, hh, ww]) == ((r >> 8) >= thr)
    assert {_tc_nsub(ci, co, *shape) for ci, co, _kd, shape, _p in TC_ACT_CASES} == {1, 2, 4}
    assert _dfold_tail_split(16, 16, 1, 16, 64, 80, 16) and not _dfold_tail_split(16, 16, 1, 16, 64, 80, FULL_SMS)


# ------------------------------------------------------------------------------------------
# 1. eval-mode affine maps
# ------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_dsbn_eval_affine_batch_matches_float64_closed_form():
    L = _lib()
    eps = 1e-5
    eps64 = float(np.float32(eps))
    chans = [1, 7, 16, 300, 512, 8, 24, 48, 64, 128, 256, 32]
    r = np.random.Generator(np.random.PCG64(401))
    for whole_bias_null in (False, True):
        ents = []
        for e in range(48):                                      # kMaxAffine entries
            c = chans[e % len(chans)]
            gamma = torch.from_numpy((r.standard_normal(c) * 0.5 + 1.0).astype(np.float32))
            beta = torch.from_numpy(r.standard_normal(c).astype(np.float32))
            mean = torch.from_numpy((r.standard_normal(c) * 2.0).astype(np.float32))
            # variances spanning 1e-9 .. 10 and exact zeros: where var << eps the result is eps's alone
            var = torch.from_numpy((np.abs(r.standard_normal(c)) * 10.0 ** r.uniform(-9, 1, c)).astype(np.float32))
            var[::5] = 0.0
            bias = None if e % 3 == 1 else torch.from_numpy((r.standard_normal(c) * 0.5).astype(np.float32))
            ents.append([t if t is None else t.to(DEV) for t in (gamma, beta, mean, var, bias)])
        scales = [torch.full((g.numel(),), float("nan"), device=DEV) for g, *_ in ents]
        shifts = [torch.full((g.numel(),), float("nan"), device=DEV) for g, *_ in ents]
        cols = list(zip(*ents))
        _call("fpl_dsbn_eval_affine_batch", 48, _parr(cols[0]), _parr(cols[1]), _parr(cols[2]), _parr(cols[3]),
              None if whole_bias_null else _parr(cols[4]), _parr(scales), _parr(shifts), _iarr([g.numel() for g in cols[0]]),
              eps, _st())
        for (gamma, beta, mean, var, bias), sc, sh in zip(ents, scales, shifts):
            g64, be64, m64, v64 = (t.cpu().double() for t in (gamma, beta, mean, var))
            b64 = torch.zeros_like(g64) if (bias is None or whole_bias_null) else bias.cpu().double()
            scale_ref = g64 / torch.sqrt(v64 + eps64)
            shift_ref = be64 + (b64 - m64) * scale_ref
            # scale: 1 / sqrtf(var + eps) then * gamma, IEEE-rounded (no fast math): a few 2^-24 relative
            np.testing.assert_allclose(sc.cpu().double(), scale_ref, rtol=1e-6, atol=0)
            # shift: the rounding of each fp32 product / sum, relative to the magnitudes that enter it
            bound = 1e-6 * (be64.abs() + (m64 * scale_ref).abs() + (b64 * scale_ref).abs())
            assert bool(((sh.cpu().double() - shift_ref).abs() <= bound).all())
            c = gamma.numel()
            if c % 8 == 0:
                # the same scale as the eval branch of fpl_dsbn_finalize, to within 1 ulp
                fin = [torch.empty(c, device=DEV) for _ in range(4)]
                _call("fpl_dsbn_finalize", None, 0, _p(gamma), _p(beta), _p(mean), _p(var), None, 0.1, eps, 0,
                      *[_p(t) for t in fin], c, _st())
                ulps = (fin[0].cpu().view(torch.int32).long() - sc.cpu().view(torch.int32).long()).abs()
                assert int(ulps.max()) <= 1
    # count = 0 writes nothing; count = 49 is refused before any launch
    gamma, beta, mean, var, bias = (t.to(DEV) for t in _bn_params(402, 16))
    out = torch.full((16,), float("nan"), device=DEV)
    _call("fpl_dsbn_eval_affine_batch", 0, _parr([gamma]), _parr([beta]), _parr([mean]), _parr([var]), _parr([bias]),
          _parr([out]), _parr([out]), _iarr([16]), eps, _st())
    torch.cuda.synchronize()
    assert bool(torch.isnan(out).all())
    with pytest.raises(L.FplError):
        _call("fpl_dsbn_eval_affine_batch", 49, *[_parr([t] * 49) for t in (gamma, beta, mean, var, bias, out, out)],
              _iarr([16] * 49), eps, _st())
    torch.cuda.synchronize()
    assert bool(torch.isnan(out).all())


# ------------------------------------------------------------------------------------------
# 2. tensor-core conv + eval BN + PReLU + dropout epilogue
# ------------------------------------------------------------------------------------------
def _tc_act_setup(cin, cout, kd, shape, seed):
    n, d, h, w = shape
    x = bf16_round(randn(seed, n, cin, d, h, w))
    wt = bf16_round(randn(seed + 1, cout, cin, kd, 3, 3, scale=0.1))
    bn = _bn_params(seed + 2, cout)
    scale, shift = _eval_affine(*bn)
    # input: the second half of a 2*cin concat buffer (the other half holds SENTINEL)
    xb = slice_buf(x, 2 * cin // 8, cin // 8)
    return x, wt, bn, scale, shift, xb, _tc_image(wt, cin, cout, kd)


def _run_tc_act(xb, img, cin, cout, kd, shape, scale, shift, sl, p, seed, offset, seed_dev):
    n, d, h, w = shape
    a = sentinel_buf(n, d, cout // 8 + 2, h, w)                 # output: groups [1, 1 + cout/8) of a wider buffer
    _call("fpl_conv3d_tc_act", _p(xb), 2 * cin // 8, cin // 8, _p(img), _p(a), cout // 8 + 2, 1, n, d, h, w, cin, cout, kd,
          _p(scale), _p(shift), _p(sl), p, seed, offset, _p(seed_dev), _st())
    return a


def _assert_dropped_exactly(out, pre, keep):
    """The zero outputs are exactly the dropped units wherever the pre-dropout value is non-zero (with p = 0: no zero
    the reference does not have)."""
    nz = pre != 0
    assert torch.equal((out == 0)[nz], (~keep)[nz]), int(((out == 0)[nz] != (~keep)[nz]).sum())


@pytest.mark.gpu
@pytest.mark.parametrize("cin,cout,kd,shape,p", TC_ACT_CASES)
def test_conv3d_tc_act_matches_reference_with_the_exact_dropout_mask(cin, cout, kd, shape, p, sm_budgets):
    n, d, h, w = shape
    x, wt, _bn, scale, shift, xb, img = _tc_act_setup(cin, cout, kd, shape, 301)
    slope = 0.25
    sl = torch.tensor([slope], device=DEV)
    seed, offset = 0x5DEECE66D, 6 * n * d * (cout // 8) * h * w
    a148, a16 = sm_budgets(lambda: _run_tc_act(xb, img, cin, cout, kd, shape, scale, shift, sl, p, seed, offset, None))
    # an output voxel's accumulation order is fixed by its tile, not by the CTA that runs it
    assert bitwise_equal(a148, a16)
    out = read_slice(a148, 1, cout)
    pre = _prelu_affine(F.conv3d(x, wt, None, padding=(kd // 2, 1, 1)), scale, shift, slope)
    keep = dropout_keep_c8(seed, offset, n, cout, d, h, w, p) if p > 0 else torch.ones_like(pre, dtype=torch.bool)
    keep_scale = float(np.float32(1.0) / (np.float32(1.0) - np.float32(p)))
    ref = pre * keep * keep_scale
    assert max_rel(out, ref) < 6e-3                              # bf16 output rounding only
    _assert_dropped_exactly(out, pre, keep)


@pytest.mark.gpu
def test_conv3d_tc_act_seed_words_and_the_two_kernel_path():
    """The 64-bit seed (incl. the device addend and its carry into the key's high word) and the 64-bit counter offset
    reach the mask; the fused epilogue drops exactly what fpl_conv3d_tc + fpl_dsbn_finalize + fpl_dsbn_act_fwd drop."""
    cin, cout, kd, shape, p = 64, 64, 3, (1, 3, 16, 8), 0.5          # N split 2
    n, d, h, w = shape
    assert _tc_nsub(cin, cout, *shape) == 2
    x, wt, (gamma, beta, mean, var, bias), scale, shift, xb, img = _tc_act_setup(cin, cout, kd, shape, 311)
    slope = 0.25
    sl = torch.tensor([slope], device=DEV)
    pre = _prelu_affine(F.conv3d(x, wt, None, padding=1), scale, shift, slope)
    seed_dev = torch.tensor([5, 1, 9], dtype=torch.int64, device=DEV)     # forward_mc passes seed_dev[k:k+1]
    for seed, dev, offset, eff in ((0xFFFFFFFF, seed_dev[1:2], 16, 2 ** 32),
                                   (12345, None, 2 ** 32 + 16, 12345),
                                   (2 ** 63 + 7, seed_dev[2:3], 2 ** 40 + 2 ** 33, 2 ** 63 + 16)):
        keep = dropout_keep_c8(eff, offset, n, cout, d, h, w, p)
        # the masks without the high words differ, so the assertions below tell a dropped word apart
        assert not torch.equal(keep, dropout_keep_c8(eff & 0xFFFFFFFF, offset & 0xFFFFFFFF, n, cout, d, h, w, p))
        a = _run_tc_act(xb, img, cin, cout, kd, shape, scale, shift, sl, p, seed, offset, dev)
        out = read_slice(a, 1, cout)
        _assert_dropped_exactly(out, pre, keep)
        assert max_rel(out, pre * keep * 2.0) < 6e-3
        # two-kernel path: conv + bias -> bf16 y, eval-mode finalize, activation pass with the same Philox stream
        y = torch.empty((n, d, cout // 8, h, w, 8), dtype=torch.bfloat16, device=DEV)
        _call("fpl_conv3d_tc", _p(xb), 2 * cin // 8, cin // 8, _p(img), _p(bias.to(DEV)), _p(y), cout // 8, 0, None, n, d, h,
              w, cin, cout, kd, _st())
        fin = [torch.empty(cout, device=DEV) for _ in range(4)]
        _call("fpl_dsbn_finalize", None, 0, _p(gamma.to(DEV)), _p(beta.to(DEV)), _p(mean.to(DEV)), _p(var.to(DEV)), None,
              0.1, 1e-5, 0, *[_p(t) for t in fin], cout, _st())
        a2 = sentinel_buf(n, d, cout // 8 + 2, h, w)
        _call("fpl_dsbn_act_fwd", _p(y), _p(fin[0]), _p(fin[1]), _p(sl), _p(a2), cout // 8 + 2, 1, None, 0, 0, None, 0, p,
              None, seed, offset, _p(dev), n, d, h, w, cout, _st())
        out2 = read_slice(a2, 1, cout)
        assert torch.equal(out == 0, out2 == 0)
        # the two-kernel path rounds the conv output to bf16 once more before the affine map
        assert max_rel(out2, out) < 6e-3


# ------------------------------------------------------------------------------------------
# 3. depth-folded conv and the stem (k311) with the eval epilogue
# ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cin,cout,shape", DFOLD_ACT_CASES)
def test_conv3d_tc_dfold_act_matches_reference(cin, cout, shape, sm_budgets):
    n, d, h, w = shape
    L = _lib()
    x = bf16_round(randn(321, n, cin, d, h, w))
    wt = bf16_round(randn(322, cout, cin, 3, 3, 3, scale=0.1))
    scale, shift = _eval_affine(*_bn_params(323, cout))
    slope = 0.2
    sl = torch.tensor([slope], device=DEV)
    img = torch.empty(L.load().fpl_conv3d_dfold_image_bytes(cin, cout) // 2, dtype=torch.bfloat16, device=DEV)
    _call("fpl_conv3d_dfold_prep_weight", _p(wt.to(DEV)), cin, cout, 0, _p(img), _st())
    xb = slice_buf(x, 2 * cin // 8, cin // 8)                      # input: the second half of a concat buffer

    def run():
        # output: the first half of a concat buffer, as the second unit of a down level writes it
        a = sentinel_buf(n, d, 2 * cout // 8, h, w)
        _call("fpl_conv3d_tc_dfold_act", _p(xb), 2 * cin // 8, cin // 8, _p(img), _p(a), 2 * cout // 8, 0, n, d, h, w, cin,
              cout, _p(scale), _p(shift), _p(sl), _st())
        return a

    a148, a16 = sm_budgets(run)
    # an output plane sums its input planes z-1, z, z+1 in that order whichever CTA or (half) item runs it
    assert bitwise_equal(a148, a16)
    out = read_slice(a148, 0, cout)
    ref = _prelu_affine(F.conv3d(x, wt, None, padding=1), scale, shift, slope)
    assert max_rel(out, ref) < 6e-3                                 # bf16 output rounding only


@pytest.mark.gpu
@pytest.mark.parametrize("cout,shape", [(16, (2, 5, 20, 12)), (32, (1, 17, 16, 24))])
def test_stem_k311_act_hi_lo_matches_fp32_reference(cout, shape, sm_budgets):
    """The stem of the no-grad forward: fpl_patch9_c8(split) + fpl_conv3d_tc_k311_act on the 48-channel [w_hi | w_hi |
    w_lo] weights of _StemConv.sync, against the fp32 conv of the UNROUNDED image and weights."""
    n, d, h, w = shape
    xf = randn(331, n, 1, d, h, w)
    wf = randn(332, cout, 1, 3, 3, 3, scale=0.2)
    scale, shift = _eval_affine(*_bn_params(333, cout))
    slope = 0.25
    sl = torch.tensor([slope], device=DEV)
    xs4 = torch.empty((n, d, 4, h, w, 8), dtype=torch.bfloat16, device=DEV)
    _call("fpl_patch9_c8", _p(xf.to(DEV)), _p(xs4), 1, n, d, h, w, _st())
    wk = wf[:, 0].reshape(cout, 3, 9).permute(0, 2, 1)
    hi = bf16_round(wk)
    w48 = torch.zeros(cout, 48, 3)
    w48[:, 0:9], w48[:, 16:25], w48[:, 32:41] = hi, hi, wk - hi
    img = torch.empty(48 * 3 * cout, dtype=torch.bfloat16, device=DEV)
    _call("fpl_conv3d_k311_prep_weight", _p(w48.to(DEV)), 48, cout, _p(img), _st())

    def run():
        a = sentinel_buf(n, d, cout // 8 + 2, h, w)
        _call("fpl_conv3d_tc_k311_act", _p(xs4), 4, 0, _p(img), _p(a), cout // 8 + 2, 1, n, d, h, w, 48, cout, 32,
              _p(scale), _p(shift), _p(sl), _st())
        return a

    a148, a16 = sm_budgets(run)
    assert bitwise_equal(a148, a16)
    out = read_slice(a148, 1, cout)
    ref = _prelu_affine(F.conv3d(xf, wf, None, padding=1), scale, shift, slope)
    assert max_rel(out, ref) < 4e-3                  # fp32-accurate operands (hi + lo), only the bf16 output rounding


# ------------------------------------------------------------------------------------------
# 4. max-pool of an activation the epilogue already wrote
# ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("pool_kd,shape,kind", [(2, (2, 4, 6, 10), "random"), (1, (1, 3, 8, 6), "random"),
                                                (2, (1, 2, 4, 12), "negative"), (1, (2, 1, 6, 10), "ties"),
                                                (2, (1, 4, 8, 4), "ties")])
def test_maxpool_c8_is_bit_exact(pool_kd, shape, kind):
    n, d, h, w = shape
    c = 24
    x = randn(341, n, c, d, h, w)
    if kind == "negative":
        x = -(torch.round(x.abs() * 2) + 1) / 4          # every window all-negative (the -inf start), with ties
    elif kind == "ties":
        x = (torch.round(x * 2) + 0.5) / 2               # few distinct non-zero values: many tied maxima
    xb = bf16_round(x)
    a = slice_buf(xb, c // 8 + 1, 1)
    pooled = sentinel_buf(n, d // pool_kd, c // 8 + 2, h // 2, w // 2)
    _call("fpl_maxpool_c8", _p(a), c // 8 + 1, 1, _p(pooled), c // 8 + 2, 1, pool_kd, n, d, h, w, c, _st())
    got = read_slice(pooled, 1, c)
    # a max of bf16 values is one of them: exact
    assert torch.equal(got, F.max_pool3d(xb, (pool_kd, 2, 2)))


@pytest.mark.gpu
@pytest.mark.parametrize("pool_kd", [1, 2])
def test_maxpool_c8_equals_the_pooled_output_of_dsbn_act_fwd(pool_kd):
    n, c, d, h, w = 2, 16, 4, 8, 12
    y = to_c8(randn(351, n, c, d, h, w, scale=2.0).to(DEV))
    scale, shift = (randn(352, c, scale=0.3) + 1.0).to(DEV), randn(353, c, scale=0.2).to(DEV)
    sl = torch.tensor([0.2], device=DEV)
    act = sentinel_buf(n, d, c // 8 + 1, h, w)
    pooled = torch.zeros((n, d // pool_kd, c // 8, h // 2, w // 2, 8), dtype=torch.bfloat16, device=DEV)
    idx = torch.zeros(pooled.shape, dtype=torch.uint8, device=DEV)
    _call("fpl_dsbn_act_fwd", _p(y), _p(scale), _p(shift), _p(sl), _p(act), c // 8 + 1, 1, _p(pooled), c // 8, 0, _p(idx),
          pool_kd, 0.0, None, 0, 0, None, n, d, h, w, c, _st())
    pooled2 = sentinel_buf(n, d // pool_kd, c // 8, h // 2, w // 2)
    _call("fpl_maxpool_c8", _p(act), c // 8 + 1, 1, _p(pooled2), c // 8, 0, pool_kd, n, d, h, w, c, _st())
    assert bitwise_equal(pooled, pooled2)


@pytest.mark.gpu
def test_maxpool_c8_rejects_unpoolable_shapes():
    L = _lib()
    a = torch.zeros((1, 3, 2, 6, 6, 8), dtype=torch.bfloat16, device=DEV)
    pooled = torch.zeros((1, 3, 2, 3, 3, 8), dtype=torch.bfloat16, device=DEV)
    for pool_kd, d, h, w in ((1, 3, 5, 6), (1, 3, 6, 5), (2, 3, 6, 6)):      # odd H, odd W, d % pool_kd != 0
        with pytest.raises(L.FplError):
            _call("fpl_maxpool_c8", _p(a), 2, 0, _p(pooled), 2, 0, pool_kd, 1, d, h, w, 16, _st())


# ------------------------------------------------------------------------------------------
# 5. the tensor-core head
# ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("classes,cin,shape", [(1, 16, (1, 1, 20, 12)), (2, 48, (2, 3, 17, 9)), (5, 64, (1, 4, 16, 8)),
                                               (8, 16, (2, 3, 33, 10)), (8, 64, (1, 1, 18, 20)), (2, 16, (1, 4, 12, 16))])
def test_head_conv_tc_matches_reference(classes, cin, shape, sm_budgets):
    n, d, h, w = shape
    x = bf16_round(randn(361, n, cin, d, h, w))
    wt = randn(362, classes, cin, 1, 3, 3, scale=0.2)
    b = randn(363, classes, scale=0.1)
    # staged as _HeadConv does: weights and bias zero-padded to 16 output channels
    w16, b16 = torch.zeros(16, cin, 1, 3, 3), torch.zeros(16)
    w16[:classes], b16[:classes] = wt, b
    img = _tc_image(w16, cin, 16, 1)
    b16d = b16.to(DEV)
    xb = slice_buf(x, cin // 8 + 2, 1)                            # input from a slice of a wider buffer
    numel = n * classes * d * h * w

    def run():
        buf = torch.full((numel + 4096,), float("nan"), device=DEV)   # the logits, then a tail nothing may touch
        _call("fpl_head_conv_tc", _p(xb), cin // 8 + 2, 1, _p(img), _p(b16d), _p(buf), n, d, h, w, cin, classes, _st())
        return buf

    b148, b16_run = sm_budgets(run)
    assert bitwise_equal(b148[:numel], b16_run[:numel])
    assert bool(torch.isnan(b148[numel:]).all()) and bool(torch.isnan(b16_run[numel:]).all())
    got = b148[:numel].view(n, classes, d, h, w).cpu()
    ref = F.conv3d(x.double(), bf16_round(wt).double(), b.double(), padding=(0, 1, 1))
    # bf16 x bf16 products are exact in fp32: only the fp32 accumulation differs
    assert float((got.double() - ref).abs().max()) <= 2e-5 * float(ref.abs().max())


# ------------------------------------------------------------------------------------------
# 6. batched weight staging == the single-conv form, bit for bit
# ------------------------------------------------------------------------------------------
def _dev_randn(seed, *shape):
    g = torch.Generator(device=DEV)
    g.manual_seed(seed)
    return torch.randn(shape, generator=g, device=DEV) * 0.1


def _check_batch_staging(single, batch, max_count, ents, bad, wshape, image_bytes):
    """ents: the integer columns of each entry, in the order both the single and the batched form take them."""
    L = _lib()
    assert len(ents) == max_count
    ws = [_dev_randn(500 + i, *wshape(*e)) for i, e in enumerate(ents)]
    ref = []
    for wt, e in zip(ws, ents):
        img = torch.empty(image_bytes(*e) // 2, dtype=torch.bfloat16, device=DEV)
        _call(single, _p(wt), *e, _p(img), _st())
        ref.append(img)
    imgs = [torch.full_like(r, SENTINEL) for r in ref]

    def call(es, w_list, img_list, count=None):
        cols = list(zip(*es))
        _call(batch, len(es) if count is None else count, _parr(w_list), *[_iarr(c) for c in cols], _parr(img_list), _st())

    def untouched():
        torch.cuda.synchronize()
        return all(bool((i == SENTINEL).all()) for i in imgs)

    call(ents[:1], ws[:1], imgs[:1], count=0)                      # count = 0: nothing
    assert untouched()
    with pytest.raises(L.FplError):                                # one entry too many
        call(ents + ents[:1], ws + ws[:1], imgs + imgs[:1])
    with pytest.raises(L.FplError):                                # unsupported channels: refused before any launch
        call(ents[:3] + [bad], ws[:4], imgs[:4])
    assert untouched()
    call(ents, ws, imgs)
    torch.cuda.synchronize()
    for e, a, r in zip(ents, imgs, ref):
        assert bitwise_equal(a, r), e


@pytest.mark.gpu
def test_conv3d_prep_weight_batch_is_bitwise_the_single_form():
    pairs = [(16, 16), (16, 32), (32, 16), (32, 32), (16, 48), (48, 16), (48, 80), (80, 48), (32, 64), (64, 32), (64, 64),
             (64, 128), (128, 64), (128, 128), (80, 256), (256, 128), (128, 256), (256, 256), (512, 256), (256, 512)]
    ents = [(ci, co, kd, tf) for ci, co in pairs for kd in (1, 3) for tf in (0, 1)]
    L = _lib().load()
    _check_batch_staging("fpl_conv3d_prep_weight", "fpl_conv3d_prep_weight_batch", 80, ents, (24, 16, 3, 0),
                         lambda ci, co, kd, tf: (co, ci, kd, 3, 3),
                         lambda ci, co, kd, tf: L.fpl_conv3d_weight_image_bytes(co if tf else ci, ci if tf else co, kd))


@pytest.mark.gpu
def test_conv3d_dfold_prep_weight_batch_is_bitwise_the_single_form():
    pairs = [(16, 16), (16, 32), (16, 64), (32, 16), (32, 32), (32, 64), (64, 16), (64, 32)]
    ents = [(ci, co, tf) for _rep in range(4) for ci, co in pairs for tf in (0, 1)]
    L = _lib().load()
    _check_batch_staging("fpl_conv3d_dfold_prep_weight", "fpl_conv3d_dfold_prep_weight_batch", 64, ents, (16, 48, 0),
                         lambda ci, co, tf: (co, ci, 3, 3, 3),
                         lambda ci, co, tf: L.fpl_conv3d_dfold_image_bytes(co if tf else ci, ci if tf else co))


@pytest.mark.gpu
def test_convt_prep_weight_batch_is_bitwise_the_single_form():
    ents = [(ci, co, kd2, mode) for ci, co in ((32, 16), (64, 32), (256, 128), (48, 80)) for kd2 in (1, 2) for mode in (0, 1)]
    L = _lib().load()
    _check_batch_staging("fpl_convt_prep_weight", "fpl_convt_prep_weight_batch", 16, ents, (24, 16, 2, 0),
                         lambda ci, co, kd2, mode: (ci, co, kd2, 2, 2),
                         lambda ci, co, kd2, mode: L.fpl_convt_weight_image_bytes(ci, co, kd2))


# ------------------------------------------------------------------------------------------
# 7. fp32 NCDHW -> C8-planar bf16 pack (+ channel sums)
# ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("c,groups", [(1, 1), (2, 1), (5, 1), (8, 1), (1, 2), (5, 2), (8, 2), (16, 2)])
def test_pack_ncdhw_to_c8_rounds_to_nearest_even_and_accumulates_sums(c, groups):
    L = _lib()
    n, d, h, w = 2, 3, 33, 40                                      # H*W > 1024: several blocks per plane
    x = randn(371, n, c, d, h, w, scale=3.0)
    # every 7th value exactly halfway between two bf16 numbers: round-half-to-even decides
    bits = x.view(torch.int32).clone()
    mid = torch.arange(bits.numel()).view(bits.shape) % 7 == 0
    bits[mid] = (bits[mid] & ~0xFFFF) | 0x8000
    x = bits.view(torch.float32)
    tot = groups + 2
    out = sentinel_buf(n, d, tot, h, w)
    sums = torch.ones(c, device=DEV)                               # accumulated into
    _call("fpl_pack_ncdhw_to_c8", _p(x.to(DEV)), c, _p(out), tot, 1, groups, _p(sums), n, d, h, w, _st())
    got = read_slice(out, 1, groups * 8)
    assert torch.equal(got[:, :c], x.to(torch.bfloat16).float())   # torch's fp32 -> bf16 is round-to-nearest-even
    assert torch.all(got[:, c:] == 0)                              # padding channels of the groups
    xd = x.double()
    err = (sums.cpu().double() - (1.0 + xd.sum((0, 2, 3, 4)))).abs()
    assert bool((err <= 1e-5 * xd.abs().sum((0, 2, 3, 4))).all())     # fp32 partial sums
    with pytest.raises(L.FplError):                                # more channels than the groups hold
        _call("fpl_pack_ncdhw_to_c8", _p(x.to(DEV)), 9, _p(out), tot, 1, 1, None, n, d, h, w, _st())
    with pytest.raises(L.FplError):                                # channel sums are limited to 16 channels
        _call("fpl_pack_ncdhw_to_c8", _p(x.to(DEV)), 17, _p(out), 3, 0, 3, _p(sums), n, d, h, w, _st())
