"""GPU probe: what do the epilogues of the conv kernels cost?  Each variant is captured 10x into a CUDA graph and timed.
  dfold / conv_tc : plain store | + forward BatchNorm statistics; and the standalone BatchNorm-backward reduce
Usage: python tools/epi_probe.py"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from fplplus_b200 import lib, ops
from tests._util import bf16_round, randn, to_c8

DEV = "cuda:0"
L = lib.load()
P = ops.ptr


def graph_time(fn, iters=10):
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(iters):
            fn()
    g.replay()
    torch.cuda.synchronize()
    ts = []
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) / iters * 1e3)
    return sorted(ts)[1]


def probe(cin, cout, shape, kind):
    n, d, h, w = shape
    x = to_c8(bf16_round(randn(1, n, cin, d, h, w)).to(DEV))
    wt = bf16_round(randn(2, cout, cin, 3, 3, 3, scale=0.1)).to(DEV)
    y = torch.zeros((n, d, cout // 8, h, w, 8), dtype=torch.bfloat16, device=DEV)
    yprev = to_c8(bf16_round(randn(3, n, cout, d, h, w)).to(DEV))
    stats = torch.zeros(2 * cout, dtype=torch.float64, device=DEV)
    red = torch.zeros(2 * cout + 1, dtype=torch.float64, device=DEV)
    f = lambda s: randn(s, cout).to(DEV)
    sc, sh, mean, inv = f(4), f(5), f(6), f(7).abs() + 0.5
    slope = torch.tensor([0.2], device=DEV)
    st = ops.stream_ptr
    if kind == "dfold":
        img = torch.empty(L.fpl_conv3d_dfold_image_bytes(cin, cout) // 2, dtype=torch.bfloat16, device=DEV)
        ops.call("fpl_conv3d_dfold_prep_weight", P(wt), cin, cout, 0, P(img), st())
        plain = lambda: ops.call("fpl_conv3d_tc_dfold", P(x), cin // 8, 0, P(img), None, P(y), cout // 8, 0, None, n, d, h, w, cin, cout, st())
        wstat = lambda: ops.call("fpl_conv3d_tc_dfold", P(x), cin // 8, 0, P(img), None, P(y), cout // 8, 0, P(stats), n, d, h, w, cin, cout, st())
    else:
        img = torch.empty(L.fpl_conv3d_weight_image_bytes(cin, cout, 3) // 2, dtype=torch.bfloat16, device=DEV)
        ops.call("fpl_conv3d_prep_weight", P(wt), cin, cout, 3, 0, P(img), st())
        plain = lambda: ops.call("fpl_conv3d_tc", P(x), cin // 8, 0, P(img), None, P(y), cout // 8, 0, None, n, d, h, w, cin, cout, 3, st())
        wstat = lambda: ops.call("fpl_conv3d_tc", P(x), cin // 8, 0, P(img), None, P(y), cout // 8, 0, P(stats), n, d, h, w, cin, cout, 3, st())
    reduce_ = lambda: ops.call("fpl_dsbn_act_bwd_reduce", P(yprev), P(y), cout // 8, 0, None, 0, 0, None, 0, P(sc), P(sh), P(mean),
                               P(inv), P(slope), 0.0, None, 0, 0, None, P(red), n, d, h, w, cout, st())
    t = [graph_time(fn) for fn in (plain, wstat, reduce_)]
    gf = 2.0 * n * d * h * w * 27 * cin * cout / 1e9
    print("%-6s %3d->%3d %-18s plain %6.1f us (%5.0f TF/s) | +stats %6.1f | standalone reduce %6.1f" % (
        kind, cin, cout, shape, t[0], gf / t[0] / 1e-6 / 1e3, t[1], t[2]), flush=True)


for args in [(16, 16, (4, 32, 128, 128), "dfold"), (32, 16, (4, 32, 128, 128), "dfold"), (16, 32, (4, 16, 64, 64), "dfold"),
             (32, 32, (4, 16, 64, 64), "dfold"), (64, 32, (4, 16, 64, 64), "dfold"),
             (64, 64, (4, 8, 32, 32), "tc"), (128, 64, (4, 8, 32, 32), "tc"), (128, 128, (4, 4, 16, 16), "tc"),
             (256, 128, (4, 4, 16, 16), "tc"), (128, 256, (4, 2, 8, 8), "tc"), (256, 256, (4, 2, 8, 8), "tc")]:
    probe(*args)
