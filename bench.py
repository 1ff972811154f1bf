#!/usr/bin/env python
"""bench.py -- the FPL+ hot path on B200: DSBN 3-D U-Net train step (voxels/s) + filtered-pseudo-label
pass (volumes/s), with the roofline of the dominant kernel and the reference's CPU path beside it.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

One JSON line on rank 0.  Workload of the headline metric (BASELINE.json configs[2]; configs[1] is
reported in the same line under "pl_filter"): one ``training_all`` optimiser step of the final FPL+
segmentor = zero_grad, forward of a source batch (domain 0) and a pseudo-labelled target batch
(domain 1, pixel/image-weighted), 0.5*Dice+0.5*CE, backward, Adam (weight_decay 1e-5); batch 4 per
domain per GPU of 1x32x128x128 patches, UNet2D5_dsbn ft 16-32-64-128-256, 2 classes.  Synthetic
data of that shape, synthetic weights of that architecture.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

NET_PARAMS = {"net_type": "UNet2D5_dsbn", "num_domains": 2, "class_num": 2, "in_chns": 1,
              "feature_chns": [16, 32, 64, 128, 256], "conv_dims": [3, 3, 3, 3, 3],
              "dropout": [0.0, 0.0, 0.3, 0.4, 0.5], "bilinear": False, "deep_supervise": False, "aes": False}
PATCH = (32, 128, 128)
BATCH = 4                         # per domain per GPU (BASELINE.json configs[2])
VOLUME = (48, 256, 256)           # configs[1]
TRAIN_CFG = {"train_fpl_uda": True, "dual": True, "dis": False, "val_t1": False, "val_t2": False, "gpus": [0],
             "loss_type": ["DiceLoss", "CrossEntropyLoss"], "loss_weight": [0.5, 0.5], "optimizer": "Adam",
             "learning_rate": 1e-4, "momentum": 0.9, "weight_decay": 1e-5, "lr_scheduler": "MultiStepLR",
             "lr_gamma": 0.5, "lr_milestones": [10000, 20000, 30000], "iter_start": 0, "iter_max": 40000,
             "iter_valid": 500, "ckpt_save_dir": "/tmp/fplplus_bench", "deterministic": True, "random_seed": 1}
TEST_CFG = {"fpl": True, "gpus": [0], "domian_label": 1, "ae": False, "ckpt_mode": 2, "evaluation_mode": True,
            "test_time_dropout": True, "tta_mode": 1, "sliding_window_enable": True,
            "sliding_window_size": [32, 128, 128], "sliding_window_stride": [32, 128, 128]}


def conv_gflop(params=None, patch=None):
    """Algorithmic conv GFLOP of ONE sample: (forward, train = fwd + dgrad + wgrad, forward of the dropout-free encoder
    prefix).  2 * taps * Cin * Cout per output voxel (SURVEY 8d); the stem has no dgrad; bilinear = False."""
    params, patch = params or NET_PARAMS, patch or PATCH
    ft, dims, cls = params["feature_chns"], params["conv_dims"], params["class_num"]
    vox = [float(patch[0] * patch[1] * patch[2])]
    for i in range(4):
        vox.append(vox[-1] / (8 if dims[i] == 3 else 4))
    taps = [27 if d == 3 else 9 for d in dims]
    fwd, stem = 0.0, 2.0 * taps[0] * params["in_chns"] * ft[0] * vox[0]
    chans = [params["in_chns"]] + list(ft)
    per_level = []
    for i in range(5):
        lv = 2.0 * taps[i] * (chans[i] * ft[i] + ft[i] * ft[i]) * vox[i]
        per_level.append(lv)
        fwd += lv
    for lvl in (3, 2, 1, 0):
        up_taps = 8 if dims[lvl] == 3 else 4
        fwd += 2.0 * up_taps * ft[lvl + 1] * ft[lvl] * vox[lvl + 1]                       # transposed conv k2s2
        fwd += 2.0 * taps[lvl] * (2 * ft[lvl] * ft[lvl] + ft[lvl] * ft[lvl]) * vox[lvl]
    fwd += 2.0 * 9 * ft[0] * cls * vox[0]                                                   # (1,3,3) head
    drop = params["dropout"]
    first = next((i for i in range(5) if drop[i] > 0), 5)
    return fwd / 1e9, (3 * fwd - stem) / 1e9, sum(per_level[:first]) / 1e9


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


# --------------------------------------------------------------------------------------------
# synthetic data (synthetic_data.py is the seeded generator shared with the parity tests; it is data
# generation, not the measured path, and not part of oracle/)
# --------------------------------------------------------------------------------------------
def make_batch(seed, n, shape, weighted, pinned, compact=False):
    """One batch dict.  Default: the PyMIC loader layout (io/nifty_dataset.py:171-218: 'label_prob' fp32 one-hot,
    'pixel_weight' fp32 already folded with the image weight).  ``compact``: the device data path of SURVEY 8 f-3 --
    'label' uint8 [N,D,H,W], 'pixel_weight' uint8 agreement code [N,1,D,H,W] (0/1/2 = 0/0.5/1), 'image_weight' fp32 [N];
    one-hot and NiftyDataset.set_weight_ happen inside the loss kernels.  Same voxels, same weights, bit for bit."""
    import synthetic_data as synth
    x = torch.from_numpy(synth.synth_image(n, 1, shape, seed=seed))
    lab = synth.synth_label(n, 2, shape, seed=seed)
    if compact:
        d = {"image": x, "label": torch.from_numpy(lab)}
    else:
        d = {"image": x, "label_prob": torch.from_numpy(synth.one_hot(lab, 2))}
    if weighted:
        pw, iw = synth.synth_pixel_weight(lab, seed=seed)
        if compact:
            d["pixel_weight"] = torch.from_numpy(np.where(pw > 0, 2, 1).astype(np.uint8))
            d["image_weight"] = torch.from_numpy(iw.astype(np.float32))
        else:
            d["pixel_weight"] = torch.from_numpy(pw)
            d["image_weight"] = torch.from_numpy(iw)
    if pinned:
        d = {k: (v.pin_memory() if v.dtype in (torch.float32, torch.uint8) else v) for k, v in d.items()}
    return d


def batch_bytes(b):
    return sum(v.numel() * v.element_size() for k, v in b.items() if k != "image_weight" or v.dtype == torch.float32)


# --------------------------------------------------------------------------------------------
# clocks during the timed region (B200_PROFILING.md)
# --------------------------------------------------------------------------------------------
class ClockSampler(object):
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.thr = index, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thr = threading.Thread(target=self._read, daemon=True)
        self.thr.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for t, line in self.rows:
            if t < t0 or t > t1 + 0.1:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except Exception:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------------------------
# per-kernel timing through the C-ABI call hook: CUDA events on the launching stream
# --------------------------------------------------------------------------------------------
def _conv_work(a, off):
    n, d, h, w, cin, cout, kd = a[off:off + 7]
    return 2.0 * n * d * h * w * cin * cout * kd * 9, float(n * d * h * w * (cin + cout) * 2)


def _dfold_work(a):
    n, d, h, w, cin, cout = a[9:15]
    return 2.0 * n * d * h * w * cin * cout * 27, float(n * d * h * w * (cin + cout) * 2)


def _k311_work(a, off):
    n, d, h, w, cin, cout = a[off:off + 6]
    return 2.0 * n * d * h * w * cin * cout * 3, float(n * d * h * w * (cin + cout) * 2)


def _stem_work(a, off):
    n, cin, d, h, w, cout, kd = a[off:off + 7]
    return 2.0 * n * d * h * w * cin * cout * kd * 9, float(n * d * h * w * (4 * cin + 2 * cout))


WORK = {   # entry point -> (flops, algorithmic bytes) from its argument tuple
    "fpl_conv3d_tc": lambda a: _conv_work(a, 9),
    "fpl_conv3d_tc_dfold": _dfold_work,
    "fpl_conv3d_direct": lambda a: _conv_work(a, 9),
    "fpl_conv3d_wgrad": lambda a: _conv_work(a, 7),
    "fpl_conv3d_wgrad_tc": lambda a: _conv_work(a, 7),
    "fpl_conv3d_wgrad_tc_tapmajor": lambda a: _conv_work(a, 7),
    "fpl_conv3d_wgrad_tc_k311": lambda a: _k311_work(a, 7),
    # the 1-channel stem straight from the fp32 image (csrc/stem_tc.cu): n, cin, d, h, w, cout, kd
    "fpl_stem_conv_fwd": lambda a: _stem_work(a, 7),
    "fpl_stem_conv_wgrad": lambda a: _stem_work(a, 5),
}
# entry points that launch the SAME kernel are one roofline population (the ncu capture sees kernel names):
# the wgrad entry points launch conv3d_wgrad_hs_kernel (k3, Cin 16 / 32: levels 0-1) or conv3d_wgrad_tc_kernel (the other
# k3 / k(1,3,3) wgrads, the head wgrad; the stem's k(3,1,1) wgrad when FPL_STEM_TRAIN=patch): ONE population, the weight-gradient kernels
WGRAD_KERNELS = "conv3d_wgrad_hs_kernel+conv3d_wgrad_tc_kernel"
KERNEL_OF = {"fpl_conv3d_wgrad_tc_tapmajor": WGRAD_KERNELS, "fpl_conv3d_wgrad_tc": WGRAD_KERNELS,
             "fpl_conv3d_wgrad_tc_k311": WGRAD_KERNELS, "fpl_conv3d_tc": "conv3d_tc_kernel",
             "fpl_conv3d_tc_dfold": "conv3d_tc_dfold_kernel"}


def _dsbn_work(bytes_per_elem, lo, hi):
    def f(a):
        n, d, h, w, c = a[lo:hi]
        return 0.0, float(n) * d * h * w * c * bytes_per_elem
    return f


# HBM-bound kernels: algorithmic bytes per element of DESIGN.md section 3 (bf16 activations)
WORK.update({
    "fpl_dsbn_bn_act_fwd": _dsbn_work(4, -6, -1),            # read y, write a
    "fpl_dsbn_act_bwd_reduce": _dsbn_work(4, -6, -1),        # read y, g
    "fpl_dsbn_act_bwd_apply_fin": _dsbn_work(6, -10, -5),    # read y, g, write dy
})


def _loss_work(reduce):
    """fpl_dice_ce_{reduce,grad}_ex: logits 4C B/voxel + truth (4C fp32 one-hot or 1 uint8) + weight (4, 1 or 0);
    the gradient pass also writes 4C (SURVEY 8d: 8C+4 / 12C+4 with the PyMIC layout, 4C+2 / 8C+2 with the device one)."""
    def f(a):
        soft_y, label, weight, code = a[1], a[2], a[3], a[4]
        if reduce:
            n, c, spatial = a[7], a[8], a[9]
            wr = 0
        else:
            n, c, spatial = a[14], a[15], a[16]
            if a[13] is None:                      # loss-only call (no dlogits): one thread, no streaming
                return 0.0, 0.0
            wr = 4 * c
        per = 4 * c + (4 * c if soft_y is not None else 1) + (4 if weight is not None else (1 if code is not None else 0)) + wr
        return 0.0, float(n) * spatial * per
    return f


WORK.update({"fpl_dice_ce_reduce_ex": _loss_work(True), "fpl_dice_ce_grad_ex": _loss_work(False)})
HBM_KERNELS = ("fpl_dsbn_bn_act_fwd", "fpl_dsbn_act_bwd_reduce", "fpl_dsbn_act_bwd_apply_fin", "fpl_dice_ce_reduce_ex",
               "fpl_dice_ce_grad_ex")


def measured_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel`, averaged over the launches of one train step,
    from the committed `ncu --set full` capture (profiles/roofline_traffic.json, written by tools/ncu_traffic.py)."""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if not os.path.exists(p):
        return None
    with open(p) as f:
        return json.load(f).get(kernel, {}).get("dram_bytes_per_launch")



def graph_timed_wgrad(calls, steps, dev, iters=8):
    """Launch durations of the weight-gradient population free of the host's enqueue gaps: every DISTINCT call of the eager
    steps (entry point + geometry) is re-issued on fresh buffers of the same shapes, captured `iters` times back to back in a
    CUDA graph and timed with CUDA events; the per-step total weights each shape by its launches per step."""
    from fplplus_b200.ops import call, ptr, stream_ptr
    shapes = {}
    for name, a in calls:
        k311 = name.endswith("_k311")
        n, d, h, w, cin, cout = a[7:13]
        kd = 3 if k311 else a[13]
        key = (name, a[1], a[2], a[4], a[5], n, d, h, w, cin, cout, kd)
        shapes[key] = shapes.get(key, 0) + 1
    total_us, total_fl, rows = 0.0, 0.0, []
    for key, count in shapes.items():
        name, xt, xo, dyt, dyo, n, d, h, w, cin, cout, kd = key
        k311 = name.endswith("_k311")
        x = torch.randn((n, d, xt, h, w, 8), device=dev).to(torch.bfloat16)
        dy = torch.randn((n, d, dyt, h, w, 8), device=dev).to(torch.bfloat16)
        dw = torch.zeros(max(cout, 8) * cin * 27, device=dev)
        tail = (n, d, h, w, cin, cout) if k311 else (n, d, h, w, cin, cout, kd)
        fn = lambda: call(name, ptr(x), xt, xo, ptr(dy), dyt, dyo, ptr(dw), *tail, stream_ptr())
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
        us = sorted(ts)[1]
        fl = WORK[name]((0,) * 7 + tail)[0]
        per_step = count / steps
        total_us += us * per_step
        total_fl += fl * per_step
        rows.append({"entry": name, "shape": [n, d, h, w], "cin": cin, "cout": cout, "kd": kd, "us": us, "launches_per_step": per_step,
                     "tflops": fl / us / 1e6})
        del x, dy, dw, g
    rows.sort(key=lambda r: -r["us"] * r["launches_per_step"])
    return total_us, total_fl, rows


class KernelTimer(object):
    class _Tok(object):
        __slots__ = ("rec", "e1")

        def __init__(self, rec, e1):
            self.rec, self.e1 = rec, e1

        def stop(self):
            self.e1.record()

    def __init__(self):
        self.records = []
        self.wgrad_calls = []
        self.enabled = False

    def __call__(self, name, args):
        if not self.enabled:
            return None
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        work = WORK[name](args) if name in WORK else (0.0, 0.0)
        e0.record()
        self.records.append((name, work, e0, e1))
        if KERNEL_OF.get(name) == WGRAD_KERNELS:
            self.wgrad_calls.append((name, tuple(args)))
        return KernelTimer._Tok(None, e1)

    def summary(self):
        agg = {}
        for name, (fl, by), e0, e1 in self.records:
            ms = e0.elapsed_time(e1)
            a = agg.setdefault(name, [0, 0.0, 0.0, 0.0])
            a[0] += 1
            a[1] += ms
            a[2] += fl
            a[3] += by
        return agg


# --------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------
def build_agent(stage, world):
    from fplplus_b200.agent import SegmentationAgent
    import synthetic_data as synth
    cfg = {"dataset": {"tensor_type": "float", "train_batch_size": BATCH}, "network": dict(NET_PARAMS),
           "training": dict(TRAIN_CFG), "testing": dict(TEST_CFG)}
    agent = SegmentationAgent(cfg, stage)
    agent.create_network()
    sd = synth.synth_state_dict(NET_PARAMS["in_chns"], NET_PARAMS["feature_chns"], NET_PARAMS["class_num"], NET_PARAMS["num_domains"])
    agent.net.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()}, strict=True)
    agent._pick_device("training" if stage == "train" else "testing")
    agent.net.to(agent.device)
    if stage == "train":
        agent.create_optimizer(agent.get_parameters_to_update())
        agent.create_loss_calculator()
        agent.net.train()
        if world > 1:
            agent.enable_data_parallel()
    return agent


def timed(fn, steps, warmup, barrier):
    """W warm-up calls, then exactly K calls between barrier+synchronize, CUDA events; ms total."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    timed.host_enqueue_ms = (time.time() - t0) * 1e3 / max(steps, 1)   # CPU time to enqueue one step
    torch.cuda.synchronize()
    barrier()
    t1 = time.time()
    return e0.elapsed_time(e1), t0, t1


def run_ours(args):
    import torch.distributed as dist
    from fplplus_b200 import fpl, lib
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    nccl_ctas = 0
    if world > 1:
        from fplplus_b200.agent import reserve_sms_for_nccl
        nccl_ctas = reserve_sms_for_nccl()          # before the communicator exists (NCCL_MAX_CTAS) + grid budget
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    agent = build_agent("train", world)
    dev = agent.device
    compact = not args.fp32_onehot
    host = [make_batch(11 + rank * 2, BATCH, PATCH, False, True, compact),
            make_batch(12 + rank * 2, BATCH, PATCH, True, True, compact)]
    resident = [{k: (v.to(dev) if torch.is_tensor(v) and v.dtype in (torch.float32, torch.uint8) else v) for k, v in b.items()}
                for b in host]
    vox_per_step = 2 * BATCH * PATCH[0] * PATCH[1] * PATCH[2]

    clocks = ClockSampler(local)
    clocks.start()

    # ---- kernel-side throughput: inputs resident in HBM; the step is replayed from the agent's CUDA graph ----
    last_out = [None]

    def step_resident():
        last_out[0] = agent.train_step(resident)

    for _ in range(max(args.warmup, 5)):          # includes the 3 eager steps + capture of the graph
        step_resident()
    torch.cuda.synchronize()
    ms, t0, t1 = timed(step_resident, args.steps, 0, barrier)
    host_ms = timed.host_enqueue_ms
    ms = max_over_ranks(ms)
    clk = clocks.stop(t0, t1)
    value = world * vox_per_step * args.steps / (ms / 1e3)
    if args.dump_outputs and rank == 0:
        # the legs below keep training the same network: snapshot the timed region's result before they run
        dump_outputs(args.dump_outputs, last_out[0])

    # ---- end to end through the agent with HOST buffers: H2D of the batch + D2H of the loss per step ----
    # the loss of every step is read back to the host (4 bytes into pinned memory); the read of step i is
    # completed while step i+1 is already enqueued, so the GPU never idles on the host round trip
    loss_pin = [torch.zeros((), dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_ev = [torch.cuda.Event(), torch.cuda.Event()]
    state = {"i": 0, "last": None}

    def step_e2e():
        i = state["i"]
        loss, _ = agent.train_step(host)
        loss_pin[i & 1].copy_(loss, non_blocking=True)
        loss_ev[i & 1].record()
        if i > 0:
            loss_ev[(i - 1) & 1].synchronize()
            state["last"] = float(loss_pin[(i - 1) & 1])
        state["i"] = i + 1

    ms_e2e, _, _ = timed(step_e2e, args.steps, 2, barrier)
    ms_e2e = max_over_ranks(ms_e2e)
    e2e_value = world * vox_per_step * args.steps / (ms_e2e / 1e3)
    h2d = sum(batch_bytes(b) for b in host)
    # the same step fed with the PyMIC loader layout (fp32 one-hot labels + folded fp32 pixel weights): 2.5x the H2D bytes
    e2e_alt = None
    if compact and not args.quick:
        host_alt = [make_batch(11 + rank * 2, BATCH, PATCH, False, True, False),
                    make_batch(12 + rank * 2, BATCH, PATCH, True, True, False)]
        state["i"] = 0
        host_keep, host[:] = list(host), host_alt
        for _ in range(5):
            step_e2e()                                  # this batch signature has its own captured graph
        ms_alt, _, _ = timed(step_e2e, args.steps, 0, barrier)
        ms_alt = max_over_ranks(ms_alt)
        e2e_alt = {"value": world * vox_per_step * args.steps / (ms_alt / 1e3), "unit": "voxels/s",
                   "ms_per_step": ms_alt / args.steps, "h2d_bytes_per_step": sum(batch_bytes(b) for b in host_alt),
                   "layout": "PyMIC loader layout: 'label_prob' fp32 one-hot + folded fp32 'pixel_weight'"}
        host[:] = host_keep

    # ---- roofline of the dominant kernel: a second timed region of K EAGER steps (a graph replay has no per-kernel
    #      host hook) with CUDA events on the launching stream around every C-ABI call; same kernels, same shapes ----
    timer = KernelTimer()
    lib.set_call_timer(timer)
    agent.use_cuda_graph = False
    # one stream for this pass: with the domain passes / wgrads on side streams an event bracket would also time the
    # kernels it overlaps with
    saved_streams = (agent.dual_stream, agent.net.wgrad_side_stream)
    agent.dual_stream, agent.net.wgrad_side_stream = False, False
    for _ in range(2):
        step_resident()
    torch.cuda.synchronize()
    lib.launch_count(reset=True)
    timer.enabled = True
    ms_eager, _, _ = timed(step_resident, args.steps, 0, barrier)
    timer.enabled = False
    launches = lib.launch_count()
    agent.use_cuda_graph = True
    agent.dual_stream, agent.net.wgrad_side_stream = saved_streams
    pk = peaks()
    agg = timer.summary()
    step_ms = ms / args.steps
    eager_step_ms = ms_eager / args.steps
    kern = {k: {"launches_per_step": v[0] / args.steps, "ms_per_step": v[1] / args.steps,
                "share_of_step": v[1] / args.steps / eager_step_ms} for k, v in agg.items()}
    roofline = None
    conv = {}
    for k, v in agg.items():
        if k in WORK and v[1] > 0 and v[2] > 0:
            kk = KERNEL_OF.get(k, k)
            c = conv.setdefault(kk, [0, 0.0, 0.0, 0.0, []])
            for i in range(4):
                c[i] += v[i]
            c[4].append(k)
    if conv:
        top = max(conv, key=lambda k: conv[k][1])
        n, tot_ms, fl, by, entries = conv[top]
        ach = fl / (tot_ms / 1e3) / 1e12
        tr = measured_traffic(top)
        roofline = {"kernel": top, "entry_points": sorted(entries), "bound": "tensor", "achieved": ach,
                    "peak": pk["bf16_tflops_sustained"],
                    "unit": "TFLOP/s", "frac": ach / pk["bf16_tflops_sustained"], "traffic": tr,
                    "traffic_note": "bytes per launch (dram read + write from ncu --set full), mean over ALL launches of this "
                                    "kernel in one train step -- the same population as achieved / algorithmic_mb_per_launch",
                    "peak_source": pk["source"] + " (sustained bf16, kernel timed inside a long step)",
                    "launches_per_step": n / args.steps, "avg_launch_ms": tot_ms / n,
                    "algorithmic_gflop_per_launch": fl / n / 1e9, "algorithmic_mb_per_launch": by / n / 1e6,
                    "traffic_over_algorithmic": (tr / (by / n)) if tr else None,
                    "hbm_gbs_at_algorithmic_bytes": by / (tot_ms / 1e3) / 1e9}
        if top == WGRAD_KERNELS and timer.wgrad_calls:
            # the eager brackets above include the host's enqueue gap (tensor-map encoding + launch, several us per call);
            # the same launches captured back to back in CUDA graphs give the GPU-side durations
            g_us, g_fl, g_rows = graph_timed_wgrad(timer.wgrad_calls, args.steps, dev)
            roofline["eager_brackets"] = {k: roofline[k] for k in ("achieved", "frac", "avg_launch_ms", "hbm_gbs_at_algorithmic_bytes")}
            roofline["eager_brackets"]["note"] = ("CUDA-event brackets around every launch of K eager single-stream steps: they "
                                                  "include the host's tensor-map encoding + enqueue gap of each call")
            roofline.update({"achieved": g_fl / g_us / 1e6, "frac": g_fl / g_us / 1e6 / pk["bf16_tflops_sustained"],
                             "avg_launch_ms": g_us / (n / args.steps) / 1e3, "us_per_step": g_us,
                             "hbm_gbs_at_algorithmic_bytes": (by / args.steps) / (g_us / 1e6) / 1e9,
                             "timing": "launch durations: every distinct weight-gradient launch of the step re-issued on fresh "
                                       "buffers, 8x back to back in a CUDA graph, CUDA-event timed on the launching stream "
                                       "(no host enqueue gaps); eager_brackets = the per-call brackets of the eager region",
                             "layers": g_rows[:8]})
    # per-layer roofline of every conv launch class: bound = max(tensor time at the sustained bf16 peak, HBM time at the
    # measured copy bandwidth) -- the C = 16/32 full-resolution layers are HBM-side of the ridge (SURVEY 7)
    layers = {}
    for nm, (fl, by), e0, e1 in timer.records:
        if fl > 0:
            layers.setdefault((nm, fl, by), []).append(e0.elapsed_time(e1))
    conv_layers = []
    for (nm, fl, by), ts in layers.items():
        t = sum(ts) / len(ts) / 1e3
        t_tc, t_hbm = fl / (pk["bf16_tflops_sustained"] * 1e12), by / (pk["hbm_gbs"] * 1e9)
        conv_layers.append({"entry": nm, "gflop": fl / 1e9, "mb": by / 1e6, "launches_per_step": len(ts) / args.steps,
                            "avg_us": t * 1e6, "tflops": fl / t / 1e12, "gbs": by / t / 1e9,
                            "bound": "tensor" if t_tc >= t_hbm else "hbm", "frac_of_bound": max(t_tc, t_hbm) / t})
    conv_layers.sort(key=lambda r: -r["avg_us"] * r["launches_per_step"])
    big = [r for r in conv_layers if r["gflop"] >= 1.0]
    tw = sum(r["avg_us"] * r["launches_per_step"] for r in big)
    conv_summary = {"time_weighted_frac_of_bound": (sum(r["frac_of_bound"] * r["avg_us"] * r["launches_per_step"] for r in big) / tw) if tw else None,
                    "note": "min(TC, HBM) roofline per conv launch class (>= 1 GFLOP), weighted by its time in the eager step"}
    # HBM-bound kernels: GB/s at the algorithmic bytes, over all layers of the step and for the largest layer alone
    hbm = {}
    for name in HBM_KERNELS:
        recs = [(by, e0.elapsed_time(e1)) for nm, (fl, by), e0, e1 in timer.records if nm == name and by > 0]
        if recs:
            big = max(b for b, _ in recs)
            tb = [t for b, t in recs if b == big]
            hbm[name] = {"gbs_all_layers": sum(b for b, _ in recs) / (sum(t for _, t in recs) / 1e3) / 1e9,
                         "gbs_largest_layer": big / (sum(tb) / len(tb) / 1e3) / 1e9,
                         "frac_of_hbm_peak_largest_layer": big / (sum(tb) / len(tb) / 1e3) / 1e9 / pk["hbm_gbs"],
                         "largest_layer_mb": big / 1e6}
    lib.set_call_timer(None)

    # ---- configs[1]: filtered-pseudo-label pass, volumes sharded over ranks, no communication ----
    pl = None
    if not args.skip_filter:
        pl = bench_filter(agent, rank, world, barrier, max_over_ranks, args)

    out = None
    if rank == 0:
        out = {"metric": "train_voxels_per_s", "value": value, "unit": "voxels/s", "n_gpus": world,
               "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True,
               "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
               "config": {"workload": "FPL+ final segmentor training_all step: UNet2D5_dsbn ft 16-32-64-128-256, "
                                      "2 classes, batch 4/domain/GPU x 1x32x128x128, source batch + pixel/image-"
                                      "weighted target batch, 0.5 Dice + 0.5 CE, Adam (BASELINE.json configs[2])",
                          "voxels_per_step_per_gpu": vox_per_step, "parallelism": "dp%d" % world,
                          "grad_allreduce": (type(agent.reducer).__name__ if world > 1 else None),
                          "nccl_max_ctas": nccl_ctas or None,
                          "l2": "activation working set per step >> 126 MB L2 (inputs larger than L2)",
                          "conv_gflop_per_step_per_gpu": 2 * BATCH * conv_gflop()[1], "config_name": args.config},
               "e2e": {"value": e2e_value, "unit": "voxels/s", "ms_per_step": ms_e2e / args.steps,
                       "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                       "api": "fplplus_b200.agent.SegmentationAgent.train_step(host batch dicts); every step's loss is read "
                              "back (pinned D2H), completed with a one-step lag"},
               "gpu_launches": launches, "gpu_launches_note": "kernels of this library launched by %d eager steps (the "
               "timed region replays the same kernels from a CUDA graph; torch's fused Adam adds 2 more per step)" % args.steps,
               "host_enqueue_ms_per_step": host_ms, "eager_ms_per_step": eager_step_ms,
               "clocks": clk,
               "roofline": roofline,
               "conv_layers": conv_layers[:24], "conv_layers_summary": conv_summary,
               "e2e_fp32_onehot": e2e_alt,
               "hbm_kernels": hbm,
               "kernels": kern,
               "conv_tensor_util": {"achieved_tflops_over_step": 2 * BATCH * conv_gflop()[1] * 1e9 / (step_ms / 1e3) / 1e12,
                                    "peak_tflops": pk["bf16_tflops_sustained"]},
               "pl_filter": pl}
        if not args.skip_cpu and world == 1:
            out["cpu_baseline"] = cpu_baseline(bounded_steps=12)
        elif world > 1:
            out["cpu_baseline"] = None
            out["cpu_baseline_note"] = ("timed at N=1 only: under torchrun the other ranks would spin in a barrier for the "
                                        "~15 s of CPU work and OMP_NUM_THREADS=1 starves the CPU arm; see --impl reference")
        if not args.skip_cpu and world == 1 and pl is not None and not args.quick:
            pl["cpu_baseline"] = pl_filter_cpu_baseline()
        if world == 1 and not args.quick and not args.skip_torch and args.config == "configs2":
            out["torch_cuda_baseline"] = torch_cuda_baseline(dev, args)
        if not args.skip_filter and not args.quick:
            out["filter_kernels"] = filter_kernel_rooflines(dev, pk)
    if out is not None:
        print(json.dumps(out), flush=True)
    if world > 1:
        # captured graphs hold NCCL work: drop them before the communicator, and do not let a wedged
        # communicator teardown turn a finished measurement into a hang
        dist.barrier()
        torch.cuda.synchronize()
        agent._graphs.clear()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def dump_outputs(path, step_out):
    """--dump-outputs: what train_step returned for the last timed step, as DIR/<name>.npy: ``loss`` (float32) and
    ``hard_dice_d<domain>``, the class-wise hard Dice of each domain pass (float64)."""
    loss, dices = step_out
    arrays = {"loss": loss}
    arrays.update(("hard_dice_d%d" % d, h) for d, h in enumerate(dices) if h is not None)
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        np.save(os.path.join(path, name + ".npy"), a.astype(np.float64 if a.dtype == np.float64 else np.float32))


def bench_filter(agent, rank, world, barrier, max_over_ranks, args):
    """Full FPL filter pass per volume: target pass (domain 1) + fake-source pass (domain 0) ->
    labels + agreement pixel weights; K=6 MC-dropout passes -> image uncertainty.  8 Inferer runs x
    (8 windows x 4 flips) = 256 network forwards of 1x32x128x128 per 48x256x256 volume."""
    from fplplus_b200 import fpl
    from fplplus_b200.inferer import Inferer
    import synthetic_data as synth
    import torch.nn as nn
    net = agent.net
    net.eval()
    cfg = dict(TEST_CFG)
    cfg["class_num"] = 2
    inferer = Inferer(cfg)
    nvol = max(1, args.volumes)
    vols = [torch.from_numpy(synth.synth_image(1, 1, VOLUME, seed=50 + rank * nvol + i)).pin_memory() for i in range(nvol)]
    fake = [torch.from_numpy(synth.synth_image(1, 1, VOLUME, seed=150 + rank * nvol + i)).pin_memory() for i in range(nvol)]
    results = []

    def one_volume(i):
        with torch.no_grad():
            tgt = vols[i].to(agent.device, non_blocking=True)
            src = fake[i].to(agent.device, non_blocking=True)
            one = torch.ones(1, dtype=torch.long)
            for m in net.modules():
                if type(m) == nn.Dropout:
                    m.eval()
            z_t = inferer.run(net, tgt, 1 * one)
            z_s = inferer.run(net, src, 0 * one)
            la, lb, w, cnt = fpl.agreement_weight(z_t, z_s)
            for m in net.modules():
                if type(m) == nn.Dropout:
                    m.train()
            passes = inferer.run(net, tgt, 1 * one, mc_passes=6)
            stats, _ = fpl.mc_uncertainty(passes)
            lab_host = la.cpu()                         # what leaves the GPU: u8 labels, fp32 weights, 2 scalars
            w_host = w.cpu()
            u = fpl.finish_uncertainty(stats)
            results.append((lab_host.shape, w_host.shape, u))

    one_volume(0)                                       # warm-up volume
    torch.cuda.synchronize()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(nvol):
        one_volume(i)
    e1.record()
    torch.cuda.synchronize()
    ms = max_over_ranks(e0.elapsed_time(e1))
    net.train()
    vps = world * nvol / (ms / 1e3)
    # FLOPs per volume: the reference runs 8 Inferer passes x 8 windows x 4 flips = 256 full forwards of 59.97 GFLOP
    # (15.35 TFLOP).  forward_mc computes the dropout-free encoder prefix (block0 + block1 = 13.13 GFLOP) once for the
    # 6 MC passes of a window batch, so 5 x 13.13 GFLOP per window forward set are NOT executed: 13.25 TFLOP.
    g_fwd, _g_train, g_prefix = conv_gflop(NET_PARAMS, tuple(TEST_CFG["sliding_window_size"]))
    n_win = 4 * int(np.prod([-(-VOLUME[i] // TEST_CFG["sliding_window_stride"][i]) for i in range(3)]))    # windows x 4 flips
    executed_tflop = n_win * (2 * g_fwd + 6 * g_fwd - 5 * g_prefix) / 1e3
    reference_tflop = n_win * 8 * g_fwd / 1e3
    return {"metric": "pl_filter_volumes_per_s", "value": vps, "unit": "volumes/s", "ms_per_volume": ms / nvol,
            "volumes_timed_per_gpu": nvol, "forwards_per_volume": 8 * n_win,
            "conv_tflops": executed_tflop * vps / world, "executed_tflop_per_volume": executed_tflop,
            "reference_equivalent_tflop_per_volume": reference_tflop, "reference_equivalent_tflops": reference_tflop * vps / world,
            "workload": "VS-style 1x48x256x256 volume: dual-domain sliding-window inference (window 32x128x128, "
                        "4-flip TTA) + argmax labels + agreement pixel weights + 6 MC-dropout passes -> image "
                        "uncertainty (BASELINE.json configs[1]); host volumes in, u8 labels + fp32 weights + scalar out",
            "scaling": "weak (volumes sharded round-robin, no collective)"}


# --------------------------------------------------------------------------------------------
# HBM rooflines of the filter / stitching kernels (north_star (c)): CUDA events around every launch, inputs rotated over
# enough buffers that no launch finds its data in the 126 MB L2
# --------------------------------------------------------------------------------------------
def filter_kernel_rooflines(dev, pk, iters=16):
    """GB/s at the algorithmic bytes of the filter / stitching / loss kernels at the configs[1] / configs[2] sizes.
    Each kernel is captured `iters` times back to back into a CUDA graph (inputs rotated over more buffers than fit
    the 126 MB L2) and the replay is timed with CUDA events: the figure is the average launch duration in a busy
    stream, free of the host's enqueue latency that an event bracket around a single eager launch would include."""
    from fplplus_b200 import fpl
    from fplplus_b200.loss import CombinedLoss
    from fplplus_b200.ops import call, ptr, stream_ptr
    from fplplus_b200.registry import loss_dict
    d, h, w = VOLUME
    S, C, K = d * h * w, 2, 6
    g = torch.Generator(device="cpu").manual_seed(5)
    n_sets = 8                                              # 8 x 25 MB logits volumes (+ K): far beyond L2
    vols = [torch.randn((1, C, d, h, w), generator=g).to(dev) for _ in range(n_sets + K)]
    out = {}

    def timeit(name, fn, nbytes):
        fn(0)                                               # eager warm-up (lazy module state, allocator)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for i in range(iters):
                fn(i + 1)
        graph.replay()
        torch.cuda.synchronize()
        ts = []
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            graph.replay()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        t = sorted(ts)[1] / iters / 1e3
        out[name] = {"us": t * 1e6, "algorithmic_mb": nbytes / 1e6, "gbs": nbytes / t / 1e9,
                     "frac_of_hbm_peak": nbytes / t / 1e9 / pk["hbm_gbs"]}

    timeit("fpl_mc_uncertainty_K6_C2", lambda i: fpl.mc_uncertainty([vols[(i + k) % len(vols)] for k in range(K)]),
           S * (4 * K * C))
    timeit("fpl_agree_weight_C2", lambda i: fpl.agreement_weight(vols[(2 * i) % len(vols)], vols[(2 * i + 1) % len(vols)]),
           S * (8 * C + 6))
    timeit("fpl_argmax_label_C2", lambda i: fpl.pseudo_label(vols[(i * 3) % len(vols)]), S * (4 * C + 1))
    # window accumulate: one 32x128x128 window of 2-class logits into the volume sums + visit counts (read patch, RMW out + count)
    win = (32, 128, 128)
    patches = [torch.randn((1, C) + win, generator=g).to(dev) for _ in range(4)]
    accs = [torch.zeros((1, C, d, h, w), device=dev) for _ in range(n_sets)]
    cnts = [torch.zeros((1, C, d, h, w), device=dev) for _ in range(n_sets)]
    pv = win[0] * win[1] * win[2] * C

    def wa(i):
        call("fpl_window_accumulate", ptr(patches[i % 4]), ptr(accs[i % n_sets]), ptr(cnts[i % n_sets]), 1, C, d, h, w,
             16 * (i % 2), 128 * (i % 2), 0, win[0], win[1], win[2], 0, i % 2, 1.0, stream_ptr())
    timeit("fpl_window_accumulate_32x128x128", wa, pv * 4 * 5)
    timeit("fpl_window_normalize", lambda i: call("fpl_window_normalize", ptr(accs[i % n_sets]), ptr(cnts[i % n_sets]), 1.0,
                                                  accs[0].numel(), stream_ptr()), S * C * 12)
    # loss kernels at the train-step size (batch 4 x 32x128x128, 2 classes): device layout (uint8 labels + agreement
    # codes) and PyMIC layout (fp32 one-hot + fp32 weights); reduce pass and gradient pass separately
    n, sp = BATCH, PATCH[0] * PATCH[1] * PATCH[2]
    n_rot = 12
    zs = [torch.randn((n, C) + PATCH, generator=g).to(dev) for _ in range(n_rot)]
    labs = [torch.randint(0, C, (n,) + PATCH, generator=g, dtype=torch.uint8).to(dev) for _ in range(n_rot)]
    codes = [torch.randint(1, 3, (n, 1) + PATCH, generator=g, dtype=torch.uint8).to(dev) for _ in range(n_rot)]
    onehots = [torch.nn.functional.one_hot(l.long(), C).permute(0, 4, 1, 2, 3).float().contiguous() for l in labs[:6]]
    pws = [c_.float() * 0.5 for c_ in codes[:6]]
    iw = torch.rand(n, generator=g).to(dev)
    sums = torch.zeros(6 * C + 3, dtype=torch.float64, device=dev)
    dz = torch.empty_like(zs[0])
    gs = torch.ones((), device=dev)

    def red_u8(i):
        call("fpl_dice_ce_reduce_ex", ptr(zs[i % n_rot]), None, ptr(labs[i % n_rot]), None, ptr(codes[i % n_rot]), ptr(iw),
             ptr(sums), n, C, sp, 0, 0, stream_ptr())

    def grad_u8(i):
        call("fpl_dice_ce_grad_ex", ptr(zs[i % n_rot]), None, ptr(labs[i % n_rot]), None, ptr(codes[i % n_rot]), ptr(iw),
             ptr(sums), 0.5, 0.5, 0.0, 1.0, ptr(gs), None, ptr(dz), n, C, sp, 0, 0, stream_ptr())

    def red_f32(i):
        call("fpl_dice_ce_reduce_ex", ptr(zs[i % n_rot]), ptr(onehots[i % 6]), None, ptr(pws[i % 6]), None, None,
             ptr(sums), n, C, sp, 0, 0, stream_ptr())

    def grad_f32(i):
        call("fpl_dice_ce_grad_ex", ptr(zs[i % n_rot]), ptr(onehots[i % 6]), None, ptr(pws[i % 6]), None, None,
             ptr(sums), 0.5, 0.5, 0.0, 1.0, ptr(gs), None, ptr(dz), n, C, sp, 0, 0, stream_ptr())
    red_u8(0)
    V = n * sp
    timeit("fpl_dice_ce_reduce_ex_u8_labels", red_u8, V * (4 * C + 2))
    timeit("fpl_dice_ce_grad_ex_u8_labels", grad_u8, V * (8 * C + 2))
    timeit("fpl_dice_ce_reduce_ex_fp32_onehot", red_f32, V * (8 * C + 4))
    timeit("fpl_dice_ce_grad_ex_fp32_onehot", grad_f32, V * (12 * C + 4))
    # DSBN kernels of the largest layer (16 channels x 4 x 32x128x128 = 33.5 M elements, bf16): forward (BN finalize + affine +
    # PReLU), backward reduce, backward apply -- the same entry points the eager pass brackets under "hbm_kernels", here free
    # of the host's enqueue gap
    ch = NET_PARAMS["feature_chns"][0]
    pd, ph, pw = PATCH
    rot = 6                                                 # 6 x 67 MB per tensor: beyond L2
    ys = [torch.randn((n, pd, ch // 8, ph, pw, 8), generator=g).to(torch.bfloat16).to(dev) for _ in range(rot)]
    gs1 = [torch.randn((n, pd, ch // 8, ph, pw, 8), generator=g).to(torch.bfloat16).to(dev) for _ in range(rot)]
    act = torch.empty_like(ys[0])
    dyo = torch.empty_like(ys[0])
    stats = torch.zeros(2 * ch, dtype=torch.float64, device=dev)
    stats[ch:] = float(n * sp)                              # sum of squares of a unit-variance tensor
    f32 = lambda v=0.0: torch.full((ch,), v, dtype=torch.float32, device=dev)
    gamma, beta, rm, rv = f32(1.0), f32(), f32(), f32(1.0)
    nbt = torch.zeros((), dtype=torch.int64, device=dev)
    scale, shift, mean, invstd = f32(1.0), f32(), f32(), f32(1.0)
    slope = torch.full((1,), 0.25, device=dev)
    red = torch.zeros(2 * ch + 1, dtype=torch.float64, device=dev)
    dgam, dbet, dslo, dbia = f32(), f32(), torch.zeros(1, device=dev), f32()

    def dsbn_fwd(i):
        call("fpl_dsbn_bn_act_fwd", ptr(ys[i % rot]), ptr(stats), n * sp, ptr(gamma), ptr(beta), ptr(rm), ptr(rv), ptr(nbt), 0.1, 1e-5, 1,
             ptr(scale), ptr(shift), ptr(mean), ptr(invstd), ptr(slope), ptr(act), ch // 8, 0, None, 0, 0, None, 0, 0.0, None, 0, 0,
             None, n, pd, ph, pw, ch, stream_ptr())

    def common(i):
        return (ptr(ys[i % rot]), ptr(gs1[i % rot]), ch // 8, 0, None, 0, 0, None, 0, ptr(scale), ptr(shift), ptr(mean), ptr(invstd),
                ptr(slope), 0.0, None, 0, 0, None)

    def dsbn_red(i):
        call("fpl_dsbn_act_bwd_reduce", *common(i), ptr(red), n, pd, ph, pw, ch, stream_ptr())

    def dsbn_app(i):
        call("fpl_dsbn_act_bwd_apply_fin", *common(i), ptr(red), 1, ptr(dyo), n, pd, ph, pw, ch, stream_ptr(), ptr(dgam), ptr(dbet),
             ptr(dslo), ptr(dbia))
    elems = float(n) * sp * ch
    timeit("fpl_dsbn_bn_act_fwd_16ch_full_res", dsbn_fwd, elems * 4)
    timeit("fpl_dsbn_act_bwd_reduce_16ch_full_res", dsbn_red, elems * 4)
    timeit("fpl_dsbn_act_bwd_apply_fin_16ch_full_res", dsbn_app, elems * 6)
    out["note"] = ("filter kernels at configs[1] sizes (48x256x256, 2 classes, K = 6), loss kernels at the configs[2] step "
                   "size (4 x 32x128x128); %d launches back to back in a CUDA graph, inputs rotated over > L2; peak = "
                   "MEASURED_PEAKS hbm_gbs (%s)" % (iters, pk["source"]))
    return out


# --------------------------------------------------------------------------------------------
# the same train step on stock torch modules (cuDNN / ATen) on the same GPU: the bar to beat (baseline/torch_cudnn_unet.py)
# --------------------------------------------------------------------------------------------
def torch_cuda_baseline(dev, args, steps=8):
    from baseline.torch_cudnn_unet import TorchTrainer
    out = {}
    b0, b1 = make_batch(11, BATCH, PATCH, False, False), make_batch(12, BATCH, PATCH, True, False)
    batches = [(b0["image"].to(dev), b0["label_prob"].to(dev), None),
               (b1["image"].to(dev), b1["label_prob"].to(dev), b1["pixel_weight"].to(dev))]
    vox = 2 * BATCH * PATCH[0] * PATCH[1] * PATCH[2]
    for mode in ("fp32", "bf16_channels_last"):
        try:
            torch.manual_seed(1)
            tr = TorchTrainer(dev, mode)
            for _ in range(4):
                tr.step(batches)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                tr.step(batches)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            out[mode] = {"ms_per_step": ms, "value": vox / (ms / 1e3), "unit": "voxels/s"}
            del tr
            torch.cuda.empty_cache()
        except Exception as exc:                      # a baseline must never take the product measurement down
            out[mode] = {"error": "%s: %s" % (type(exc).__name__, str(exc)[:200])}
    out["note"] = ("BASELINE, not a code path of fplplus_b200: the same DSBN 3-D U-Net + Dice/CE + Adam(fused) step as stock "
                   "torch.nn modules (cuDNN convs, ATen BatchNorm / PReLU / pooling, eager launches, cudnn.benchmark) on "
                   "this GPU, inputs resident; fp32 NCDHW is what the reference .cfg runs (tensor_type = float), bf16 "
                   "autocast + channels_last_3d is the fastest stock configuration")
    return out


# --------------------------------------------------------------------------------------------
# CPU: the oracle port of the reference path (the reference is pure Python/torch; its agent cannot
# be imported without SimpleITK/tensorboardX, see oracle/__init__.py) on the host cores
# --------------------------------------------------------------------------------------------
def _oracle_trainer(threads):
    import synthetic_data as synth
    from oracle.train_step import OracleTrainer
    torch.set_num_threads(threads)
    params = dict(NET_PARAMS)
    sd = synth.synth_state_dict(params["in_chns"], params["feature_chns"], params["class_num"], params["num_domains"])
    return OracleTrainer(sd, params, lr=1e-4, weight_decay=1e-5, w_dice=0.5, w_ce=0.5)


def cpu_baseline(bounded_steps=2, batch=1):
    threads = os.cpu_count() or 1
    tr = _oracle_trainer(threads)
    b0, b1 = make_batch(11, batch, PATCH, False, False), make_batch(12, batch, PATCH, True, False)
    batches = [(b0["image"], b0["label_prob"], None), (b1["image"], b1["label_prob"], b1["pixel_weight"])]
    tr.step(batches)
    t0 = time.time()
    for _ in range(bounded_steps):
        tr.step(batches)
    dt = (time.time() - t0) / bounded_steps
    vox = 2 * batch * PATCH[0] * PATCH[1] * PATCH[2]
    return {"value": vox / dt, "unit": "voxels/s", "cores": threads, "kind": "port",
            "sample": "%d training_all steps (1 warm-up) at batch %d/domain of 1x32x128x128 (1/%d of the GPU arm's "
                      "step), fp32 torch CPU (oneDNN), oracle.train_step.OracleTrainer" % (bounded_steps, batch, BATCH // batch),
            "s_per_step": dt}


def pl_filter_cpu_baseline():
    """BASELINE.md section 4 item 4: the oracle Inferer + NumPy filter on ONE 48x256x256 volume with tta_mode = 0 and
    K = 2 MC passes (agent_seg.py:897-931 loop), extrapolated linearly to the GPU arm's workload (4-flip TTA, K = 6)."""
    import synthetic_data as synth
    from oracle import fpl_filter, inferer as oinf, unet_dsbn
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    params = dict(NET_PARAMS)
    st = unet_dsbn.to_torch_state(synth.synth_state_dict(params["in_chns"], params["feature_chns"], params["class_num"],
                                                         params["num_domains"]), requires_grad=False)
    cfg = dict(TEST_CFG, tta_mode=0)
    vol = torch.from_numpy(synth.synth_image(1, 1, VOLUME, seed=50))
    t0 = time.time()
    with torch.no_grad():
        z_t = oinf.run(lambda x: unet_dsbn.forward(st, x, 1, params), vol, 2, cfg)
        z_s = oinf.run(lambda x: unet_dsbn.forward(st, x, 0, params), vol, 2, cfg)
        passes = [oinf.run(lambda x: unet_dsbn.forward(st, x, 1, params, drop_training=True), vol, 2, cfg).numpy()
                  for _ in range(2)]
    t_fwd = time.time() - t0                                # 4 Inferer passes x 8 windows = 32 forwards
    t0 = time.time()
    la, lb = fpl_filter.pseudo_label(z_t.numpy()), fpl_filter.pseudo_label(z_s.numpy())
    fpl_filter.agreement_weight(la, lb)
    t_lab = time.time() - t0
    t0 = time.time()
    fpl_filter.mc_uncertainty(passes)
    t_mc2 = time.time() - t0
    # full pass: (2 label passes + 6 MC passes) x 4 flips x 8 windows = 256 forwards; filter: labels once, statistics over 6
    est = t_fwd / 32 * 256 + t_lab + t_mc2 * 3
    return {"value": 1.0 / est, "unit": "volumes/s", "cores": threads, "kind": "port",
            "sample": "1 volume 48x256x256, tta_mode 0, K = 2 (32 window forwards %.1f s + labels/agreement %.2f s + MC "
                      "statistics %.2f s measured); extrapolated linearly to 256 forwards (4-flip TTA, 2 + 6 passes) and "
                      "K = 6 statistics: %.1f s per volume" % (t_fwd, t_lab, t_mc2, est),
            "s_per_volume_estimated": est}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    tr = _oracle_trainer(threads)
    batch = 1
    b0, b1 = make_batch(11, batch, PATCH, False, False), make_batch(12, batch, PATCH, True, False)
    batches = [(b0["image"], b0["label_prob"], None), (b1["image"], b1["label_prob"], b1["pixel_weight"])]
    for _ in range(max(1, min(args.warmup, 2))):
        tr.step(batches)
    t0 = time.time()
    for _ in range(args.steps):
        tr.step(batches)
    dt = time.time() - t0
    vox = 2 * batch * PATCH[0] * PATCH[1] * PATCH[2]
    v = vox * args.steps / dt
    sample = ("each step = one training_all step at batch 1/domain of 1x32x128x128 (1/4 of the GPU arm's per-GPU step), "
              "fp32 torch CPU on all host threads; warm-up capped at 2 steps")
    out = {"impl": "reference", "metric": "train_voxels_per_s", "value": v, "unit": "voxels/s",
           "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic",
           "config": {"workload": "FPL+ final segmentor training_all step (BASELINE.json configs[2]) on the host CPU, "
                                  "bounded sample", "parallelism": "cpu"},
           "cpu_baseline": {"value": v, "unit": "voxels/s", "cores": threads, "kind": "port", "sample": sample},
           "e2e": {"value": v, "unit": "voxels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out))


def apply_workload(name):
    """--config vs_shipped: the authors' own VS configuration (config_dual/data_vs/vs_t1s_S.cfg): feature_chns
    32-64-128-256-512, conv_dims [2,2,3,3,3], batch 4 x 28x128x128 patches, windows 28x128x128 -- the shape of the
    checkpoints users actually load.  The default workload stays BASELINE.json configs[2]."""
    global PATCH, VOLUME
    if name == "vs_shipped":
        NET_PARAMS.update(feature_chns=[32, 64, 128, 256, 512], conv_dims=[2, 2, 3, 3, 3])
        PATCH = (28, 128, 128)
        VOLUME = (56, 256, 256)
        TEST_CFG.update(sliding_window_size=[28, 128, 128], sliding_window_stride=[28, 128, 128])
    elif name != "configs2":
        raise SystemExit("unknown --config %s" % name)


def main():
    wd = int(os.environ.get("FPL_BENCH_WATCHDOG", "0"))
    if wd > 0:                       # debugging aid: dump every thread's stack and exit if the run wedges
        import faulthandler
        faulthandler.dump_traceback_later(wd, exit=True)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--volumes", type=int, default=2, help="volumes timed per GPU in the pl_filter leg")
    ap.add_argument("--skip-filter", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-torch", action="store_true", help="skip the stock torch/cuDNN baseline leg")
    ap.add_argument("--quick", action="store_true", help="headline numbers only (no baselines / kernel rooflines)")
    ap.add_argument("--fp32-onehot", action="store_true",
                    help="feed the PyMIC loader layout (fp32 one-hot labels, folded fp32 weights) instead of uint8 labels / codes")
    ap.add_argument("--config", default="configs2", choices=["configs2", "vs_shipped"],
                    help="configs2 = BASELINE.json configs[2] (default, the headline); vs_shipped = the authors' VS .cfg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the loss and hard Dice of the last one as DIR/<name>.npy")
    args = ap.parse_args()
    apply_workload(args.config)
    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
        run_reference(args)
        return
    if args.warmup < 3:
        args.warmup = 3
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    run_ours(args)


if __name__ == "__main__":
    main()
