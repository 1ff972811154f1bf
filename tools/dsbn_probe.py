"""GPU timing of the DSBN activation kernels (fwd, pooled fwd, bwd reduce, bwd apply) on the network's layer shapes.
Prints microseconds and GB/s at the algorithmic byte counts of DESIGN.md §3.  Development tool."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from fplplus_b200 import ops

DEV = "cuda:0"
p = ops.ptr
# (channels, (n, d, h, w), pooled?)
SHAPES = [(16, (4, 32, 128, 128), 0), (16, (4, 32, 128, 128), 2), (32, (4, 16, 64, 64), 0), (32, (4, 16, 64, 64), 2),
          (64, (4, 8, 32, 32), 0), (64, (4, 8, 32, 32), 2), (128, (4, 4, 16, 16), 0), (256, (4, 2, 8, 8), 0)]
REPS = int(os.environ.get("REPS", "5"))
ONLY = os.environ.get("ONLY", "")


def timeit(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn(); fn()
    e0.record()
    for _ in range(REPS):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / REPS * 1e3


def main():
    # a buffer larger than L2, touched between measurements of different shapes
    print("%-26s %9s %9s %9s %9s   (us | GB/s)" % ("shape", "fwd", "bwd_red", "bwd_app", "sum"))
    for c, (n, d, h, w), pool in SHAPES:
        if ONLY and ONLY != "%d" % c:
            continue
        y = torch.randn((n, d, c // 8, h, w, 8), device=DEV).to(torch.bfloat16)
        g1 = torch.randn((n, d, c // 8, h, w, 8), device=DEV).to(torch.bfloat16)
        act = torch.empty_like(y)
        dy = torch.empty_like(y)
        f32 = lambda v=0.0: torch.full((c,), v, device=DEV)
        scale, shift, mean, invstd = f32(1.0), f32(), f32(), f32(1.0)
        gamma, beta, rm, rv = f32(1.0), f32(), f32(), f32(1.0)
        dgamma, dbeta, dslope, dbias = f32(), f32(), torch.zeros(1, device=DEV), f32()
        nbt = torch.zeros((), dtype=torch.int64, device=DEV)
        stats = torch.zeros(2 * c, dtype=torch.float64, device=DEV)
        stats[c:] = float(n * d * h * w)
        sl = torch.tensor([0.25], device=DEV)
        red = torch.zeros(2 * c + 1, dtype=torch.float64, device=DEV)
        pooled = idx = gp = None
        if pool:
            pooled = torch.empty((n, d // pool, c // 8, h // 2, w // 2, 8), dtype=torch.bfloat16, device=DEV)
            idx = torch.zeros((n, d // pool, c // 8, h // 2, w // 2, 8), dtype=torch.uint8, device=DEV)
            gp = torch.randn_like(pooled)
        st = ops.stream_ptr()
        cnt = n * d * h * w

        def fwd():
            ops.call("fpl_dsbn_bn_act_fwd", p(y), p(stats), cnt, p(gamma), p(beta), p(rm), p(rv), p(nbt), 0.1, 1e-5, 1,
                     p(scale), p(shift), p(mean), p(invstd), p(sl), p(act), c // 8, 0, p(pooled), c // 8, 0, p(idx), pool,
                     0.0, None, 0, 0, None, n, d, h, w, c, st)
        common = (p(y), p(g1), c // 8, 0, p(gp), c // 8, 0, p(idx), pool, p(scale), p(shift), p(mean), p(invstd), p(sl),
                  0.0, None, 0, 0, None)

        def bred():
            ops.call("fpl_dsbn_act_bwd_reduce", *common, p(red), n, d, h, w, c, st)

        def bapp():
            ops.call("fpl_dsbn_act_bwd_apply_fin", *common, p(red), 1, p(dy), n, d, h, w, c, st, p(dgamma), p(dbeta),
                     p(dslope), p(dbias))
        elems = cnt * c
        pe = elems // (4 * pool) if pool else 0          # pooled elements
        b_fwd = elems * 4 + pe * 3                        # read y, write a (+ pooled bf16 + 1-byte code)
        b_red = elems * 4 + pe * 3                        # read y, g1 (+ pooled grad + code)
        b_app = elems * 6 + pe * 3
        t = [timeit(fwd), timeit(bred), timeit(bapp)]
        gb = [b_fwd / t[0] / 1e3, b_red / t[1] / 1e3, b_app / t[2] / 1e3]
        print("%-26s " % ("c%d %s pool%d" % (c, "x".join(map(str, (n, d, h, w))), pool)) +
              " ".join("%5.1f|%4.0f" % (a, b) for a, b in zip(t, gb)) + " %8.1f" % sum(t), flush=True)


if __name__ == "__main__":
    main()
