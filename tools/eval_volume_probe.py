"""GPU timing of the validation / test input path: whole-volume Pad + NormalizeWithMeanStd (fpl_pad_normalize_volume) and
the cfg-driven test pass (DeviceVolumeSet from a test CSV of NIfTI volumes) against the same volumes fed pre-transformed
through set_loaders.

Kernel times come from CUDA events around replays of a CUDA graph holding REPS launches, so the host's ctypes call cost
is not in them.  Bytes are computed from the shapes: statistics pass 4 B per voxel walked per normalised channel, pad pass
4 B read + 4 B written per output voxel per channel.  Two working sets: ONE volume (40x250x250 -> 48x256x256, 22 MB, it
stays in the 126 MB L2 between launches) and eight volumes used in turn (180 MB, more than the L2).

    python tools/eval_volume_probe.py [--out results.json] [--volumes 16]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PEAK_BPS = 7.7e12                 # HBM3e of one B200 (data sheet)
REPS = 50


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def kernel_times(src=(40, 250, 250), out=(48, 256, 256), sets=1):
    """ms per launch of fpl_pad_normalize_volume in three modes, over ``sets`` input / output pairs used in turn."""
    import ctypes
    from fplplus_b200 import lib
    from fplplus_b200.ops import call, ptr, stream_ptr
    dev = "cuda:0"
    g = torch.Generator(device=dev).manual_seed(0)
    xs = [torch.randn((1,) + src, device=dev, generator=g) * 20 + 100 for _ in range(sets)]
    ys = [torch.empty((1,) + out, device=dev) for _ in range(sets)]
    nbytes = int(lib.load().fpl_pad_normalize_volume_workspace_bytes(1, *src, *out))
    ws = torch.empty(nbytes // 8, dtype=torch.float64, device=dev)
    mean, std = (ctypes.c_float * 1)(100.0), (ctypes.c_float * 1)(20.0)
    svox, ovox = int(np.prod(src)), int(np.prod(out))
    res = {}
    for name, mode, after, nbytes_moved in (("fixed_mean_std (pad pass only)", 1, 0, 8 * ovox),
                                            ("statistics_of_source", 2, 0, 4 * svox + 8 * ovox),
                                            ("statistics_of_padded", 2, 1, 4 * ovox + 8 * ovox)):
        m = (ctypes.c_int * 1)(mode)

        def launch(i):
            call("fpl_pad_normalize_volume", ptr(xs[i % sets]), None, 1, *src, *out, m, mean, std, after, ptr(ws), nbytes,
                 ptr(ys[i % sets]), None, stream_ptr())
        s = torch.cuda.Stream()
        with torch.cuda.stream(s):
            for i in range(3):
                launch(i)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for i in range(REPS):
                launch(i)
        graph.replay()
        torch.cuda.synchronize()
        times = []
        for _ in range(10):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            graph.replay()
            b.record()
            b.synchronize()
            times.append(a.elapsed_time(b) / REPS)
        ms = float(np.median(times))
        res[name] = {"ms_per_launch": ms, "bytes": nbytes_moved, "achieved_TBps": nbytes_moved / (ms * 1e-3) / 1e12,
                     "share_of_7.7TBps": nbytes_moved / (ms * 1e-3) / PEAK_BPS, "spread_ms": [min(times), max(times)]}
    return res


def cfg_test_pass(n_vol, tmp):
    """Volumes/s of infer() from a test CSV (NIfTI rows, NormalizeWithMeanStd + Pad, tta_mode 1, one domain) and from the
    same volumes pre-transformed on the device through set_loaders, alternating; and the host share (NIfTI read + H2D)."""
    from fplplus_b200 import artefacts
    from fplplus_b200.agent import SegmentationAgent
    from oracle import synth
    from oracle.gen_golden import NET_PARAMS
    rng = np.random.default_rng(1)
    rows = []
    for i in range(n_vol):
        shape = (40, 160, 272) if i % 2 == 0 else (30, 160, 272)      # the sizes of the reference's sample volumes
        img = (100.0 + 20.0 * rng.standard_normal(shape)).astype(np.float32)
        name = "vol%02d.nii.gz" % i
        artefacts.write_nifti(img, os.path.join(tmp, name))
        rows.append([name])
    csv = os.path.join(tmp, "test.csv")
    artefacts.write_train_csv(csv, rows, fields=("image",))
    cfg = {"dataset": {"tensor_type": "float", "root_dir": tmp, "test_csv": csv,
                       "test_transform": ["NormalizeWithMeanStd", "Pad"], "normalizewithmeanstd_channels": [0],
                       "pad_output_size": [16, 32, 32], "pad_ceil_mode": True},
           "network": dict(NET_PARAMS), "training": {},
           "testing": {"fpl": False, "gpus": [0], "domian_label": 1, "evaluation_mode": True, "test_time_dropout": False,
                       "tta_mode": 1, "sliding_window_enable": False}}
    sd = {k: torch.from_numpy(np.asarray(v)) for k, v in synth.synth_state_dict().items()}

    def agent():
        ag = SegmentationAgent(cfg, "test")
        ag.create_dataset()
        ag.create_network()
        ag.net.load_state_dict(sd, strict=True)
        return ag
    cfg_agent = agent()
    pre = [cfg_agent.test_loader[i] for i in range(n_vol)]
    pre_agent = SegmentationAgent(cfg, "test")
    pre_agent.set_loaders(test=pre)
    pre_agent.create_network()
    pre_agent.net.load_state_dict(sd, strict=True)
    for ag in (cfg_agent, pre_agent):             # warm-up: modules, plans, captured graphs of every shape
        ag.infer(load_checkpoint=False)
    arms = {"cfg_test_csv": [], "pre_transformed_set_loaders": []}
    for _ in range(3):
        for key, ag in (("cfg_test_csv", cfg_agent), ("pre_transformed_set_loaders", pre_agent)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ag.infer(load_checkpoint=False)
            torch.cuda.synchronize()
            arms[key].append(n_vol / (time.perf_counter() - t0))
    host = []
    for _ in range(2):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for r in rows:
            v = np.asarray(artefacts.load_volume(os.path.join(tmp, r[0])), np.float32)
            torch.from_numpy(v).to("cuda:0")
        torch.cuda.synchronize()
        host.append((time.perf_counter() - t0) / n_vol * 1e3)
    return {"volumes": n_vol, "volumes_per_s": {k: {"median": float(np.median(v)), "runs": v} for k, v in arms.items()},
            "host_read_h2d_ms_per_volume": {"median": float(np.median(host)), "runs": host}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    ap.add_argument("--volumes", type=int, default=16)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("eval_volume_probe needs a CUDA device")
    res = {"card (name, power limit)": card(),
           "kernel_one_volume_in_L2": kernel_times(sets=1),
           "kernel_eight_volumes_180MB": kernel_times(sets=8)}
    with tempfile.TemporaryDirectory() as tmp:
        res["test_pass"] = cfg_test_pass(a.volumes, tmp)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
