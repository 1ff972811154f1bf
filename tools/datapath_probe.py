"""GPU timing of the training-input gather: plain `fpl_gather_patches` against per-patch NormalizeWithMeanStd
(`fpl_gather_patches_norm`: statistics kernel + normalising gather) for two domains of 4 x 1 x 32 x 128 x 128 patches cut
from resident volumes.  Kernel launches only (captured in a CUDA graph), the host's crop draws are not timed.
Development tool."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from fplplus_b200.datapath import DevicePatchSampler
from fplplus_b200.ops import call, ptr, stream_ptr
from tools.probe_util import graph_time

PATCH, BATCH = (32, 128, 128), 4


def volumes(seed):
    rng = np.random.default_rng(seed)
    out = []
    for i in range(4):
        shape = (48, 224 + 8 * i, 224)
        lab = np.zeros(shape, np.uint8)
        lab[20:28, 100:140, 90:130] = 1
        out.append({"image": 100.0 + 20.0 * rng.standard_normal((1,) + shape).astype(np.float32), "label": lab,
                    "pixel_weight": np.where(rng.random(shape) < 0.1, 0.5, 1.0).astype(np.float32), "name": "v%d" % i})
    return out


def main():
    pd, ph, pw = PATCH
    domains = []
    for d in range(2):
        vols = volumes(d)
        plain = DevicePatchSampler(vols, PATCH, BATCH, "cuda:0", seed=d)
        norm = DevicePatchSampler(vols, PATCH, BATCH, "cuda:0", seed=d, normalize={0: {}})
        plain.next_batch()
        norm.next_batch()
        torch.cuda.synchronize()
        domains.append((plain, norm))

    def run_plain():
        for plain, _ in domains:
            o = plain._out[0]
            call("fpl_gather_patches", ptr(o["rows"]), BATCH, 1, pd, ph, pw, ptr(o["image"]), ptr(o["label"]),
                 ptr(o["code"]), stream_ptr())

    def run_norm():
        for _, norm in domains:
            o, nt = norm._out[0], norm._norm
            call("fpl_gather_patches_norm", ptr(o["rows"]), BATCH, 1, pd, ph, pw, nt["mode"], nt["mean"], nt["std"],
                 ptr(nt["ws"]), nt["ws_bytes"], ptr(o["image"]), ptr(o["label"]), ptr(o["code"]), stream_ptr())

    print("device:", torch.cuda.get_device_name(0))
    for _ in range(3):                  # alternate the two forms
        t_plain, t_norm = graph_time(run_plain, 20), graph_time(run_norm, 20)
        print("2 domains x %d x 1x%dx%dx%d: plain gather %.2f us, statistics + normalising gather %.2f us (+%.2f us)"
              % (BATCH, pd, ph, pw, t_plain, t_norm, t_norm - t_plain))


if __name__ == "__main__":
    main()
