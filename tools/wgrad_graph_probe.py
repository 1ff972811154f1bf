"""GPU probe: every wgrad launch of the bench network (batch 4), captured 10x back to back in a CUDA graph (no host
enqueue gaps, warm L2) -- the per-launch GPU time the graph-replayed train step pays.  Development tool.
Usage: python tools/wgrad_graph_probe.py"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from fplplus_b200 import ops

DEV = "cuda:0"
SHAPES = [(16, 8, 1, (4, 32, 128, 128), 1), (16, 16, 3, (4, 32, 128, 128), 2), (32, 16, 3, (4, 32, 128, 128), 1),
          (16, 32, 3, (4, 16, 64, 64), 1), (32, 32, 3, (4, 16, 64, 64), 2), (64, 32, 3, (4, 16, 64, 64), 1),
          (32, 64, 3, (4, 8, 32, 32), 1), (64, 64, 3, (4, 8, 32, 32), 2), (128, 64, 3, (4, 8, 32, 32), 1),
          (64, 128, 3, (4, 4, 16, 16), 1), (128, 128, 3, (4, 4, 16, 16), 2), (256, 128, 3, (4, 4, 16, 16), 1),
          (128, 256, 3, (4, 2, 8, 8), 1), (256, 256, 3, (4, 2, 8, 8), 1)]
if os.environ.get("SMALLC"):
    SHAPES = SHAPES[:5]


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


def main():
    fn_name = "fpl_conv3d_wgrad_tc_tapmajor"
    total = 0.0
    print("%-30s %9s %9s %9s  (%s)" % ("layer", "us", "TFLOP/s", "x/pass", fn_name))
    for cin, cout, kd, shape, count in SHAPES:
        n, d, h, w = shape
        x = torch.randn((n, d, cin // 8, h, w, 8), device=DEV).to(torch.bfloat16)
        dy = torch.randn((n, d, max(cout // 8, 1), h, w, 8), device=DEV).to(torch.bfloat16)
        dw = torch.zeros(cout * cin * kd * 9, device=DEV)
        call = lambda: ops.call(fn_name, ops.ptr(x), cin // 8, 0, ops.ptr(dy), max(cout // 8, 1), 0, ops.ptr(dw), n, d, h, w, cin, cout, kd,
                                ops.stream_ptr())
        us = graph_time(call)
        gf = 2.0 * n * d * h * w * 9 * kd * cin * cout / 1e9
        total += us * count
        print("%-30s %9.1f %9.0f %9d" % ("%d->%d %s" % (cin, cout, "x".join(map(str, shape))), us, gf / us * 1e-3, count), flush=True)
    print("sum over one backward pass (k3 layers only): %.0f us" % total)


main()
