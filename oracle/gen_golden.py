"""Generate tests/golden/* by running the REFERENCE's own importable modules.

Run in the build container only (needs /root/reference; the GPU box never
does):   python -m oracle.gen_golden

Inputs come from oracle/synth.py (numpy PCG64 => reproducible everywhere); the
outputs pin the oracle (tests/test_oracle_golden.py) and the CUDA path
(tests/test_gpu_*.py).
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLD = os.path.join(ROOT, "tests", "golden")
REF = "/root/reference"

sys.path.insert(0, ROOT)
from oracle import synth  # noqa: E402

NET_PARAMS = {"net_type": "UNet2D5_dsbn", "num_domains": 2, "class_num": 2, "in_chns": 1,
              "feature_chns": [16, 32, 64, 128, 256], "conv_dims": [3, 3, 3, 3, 3],
              "dropout": [0.0, 0.0, 0.3, 0.4, 0.5], "bilinear": False,
              "deep_supervise": False, "aes": False}
SHAPE = (16, 32, 32)

GRAD_KEYS = ["out_conv.weight", "out_conv.bias", "block0.conv.conv3d_1.weight", "block0.conv.conv3d_1.bias",
             "block0.conv.conv3d_2.weight", "block2.conv.conv3d_1.weight", "block4.conv.conv3d_2.weight",
             "up1.trans3d.weight", "up1.trans3d.bias", "up4.trans3d.weight", "up4.conv.conv3d_1.weight",
             "up4.conv.conv3d_2.weight", "up2.conv.conv3d_1.bias"]


def _import_reference():
    sys.path.insert(0, REF)
    sys.path.insert(0, os.path.join(REF, "PyMIC"))
    from PyMIC.pymic.net.net3d.unet2d5_dsbn import UNet2D5_dsbn
    from pymic.loss.seg.dice import DiceLoss
    from pymic.loss.seg.ce import CrossEntropyLoss
    from pymic.net_run_dsbn.infer_func import Inferer
    return UNet2D5_dsbn, DiceLoss, CrossEntropyLoss, Inferer


def _ref_net(UNet, params, seed=1):
    net = UNet(dict(params)).float()
    sd = synth.synth_state_dict(params["in_chns"], params["feature_chns"], params["class_num"],
                                params["num_domains"], seed=seed)
    net.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()}, strict=True)
    return net


def gen_net(UNet, Dice, CE):
    x = torch.from_numpy(synth.synth_image(2, 1, SHAPE, seed=1))
    lab = synth.synth_label(2, 2, SHAPE, seed=1)
    y = torch.from_numpy(synth.one_hot(lab, 2))
    pw_np, _ = synth.synth_pixel_weight(lab, seed=1)
    pw = torch.from_numpy(pw_np)
    out = {}
    # eval mode, both domains (running statistics; dropout inactive)
    net = _ref_net(UNet, NET_PARAMS)
    net.eval()
    with torch.no_grad():
        for d in (0, 1):
            out[f"eval_logits_d{d}"] = net(x, domain_label=d * torch.ones(2, dtype=torch.long)).numpy()
    # train mode, domain 1, dropout 0 so the step is deterministic; weighted 0.5*Dice+0.5*CE
    p0 = dict(NET_PARAMS, dropout=[0.0] * 5)
    net = _ref_net(UNet, p0)
    net.train()
    logits = net(x, domain_label=torch.ones(2, dtype=torch.long))
    d = {"prediction": logits, "ground_truth": y, "pixel_weight": pw}
    loss = 0.5 * Dice({})(d) + 0.5 * CE({})(d)
    loss.backward()
    out["train_logits_d1"] = logits.detach().numpy()
    out["train_loss"] = np.asarray(loss.item(), np.float64)
    named = dict(net.named_parameters())
    for k in GRAD_KEYS:
        g = named[k].grad.numpy()
        out["gradnorm::" + k] = np.asarray(np.sqrt((g.astype(np.float64) ** 2).sum()))
        # big tensors: keep the norm and a corner slice only (fixture size)
        out["grad::" + k] = g if g.size <= 20000 else np.ascontiguousarray(g[:6, :6])
    for k, p in named.items():
        if ".relu_" in k and p.grad is not None:
            out["grad::" + k] = p.grad.numpy()
        if ".bn3d" in k and ".bns.1." in k and p.grad is not None:
            out["grad::" + k] = p.grad.numpy()
    # which parameters received a gradient at all (SURVEY: 5 648 148 of 7 685 300)
    out["n_params_with_grad"] = np.asarray(sum(p.numel() for p in named.values() if p.grad is not None))
    sd = net.state_dict()
    for k in ("block0.conv.bn3d1.bns.1", "block3.conv.bn3d2.bns.1", "up4.conv.bn3d2.bns.1", "block0.conv.bn3d1.bns.0"):
        out["rm::" + k] = sd[k + ".running_mean"].numpy()
        out["rv::" + k] = sd[k + ".running_var"].numpy()
        out["nbt::" + k] = sd[k + ".num_batches_tracked"].numpy()
    np.savez_compressed(os.path.join(GOLD, "net_fwd_bwd.npz"), **out)
    print("net_fwd_bwd", {k: np.asarray(v).shape for k, v in list(out.items())[:6]}, "loss", out["train_loss"])


def gen_loss(Dice, CE):
    out = {}
    for tag, c, shape in (("c2", 2, (2, 8, 16, 16)), ("c5", 5, (1, 6, 10, 12))):
        n = shape[0]
        g = np.random.Generator(np.random.PCG64(7 + c))
        z = (g.standard_normal((n, c) + shape[1:]) * 2).astype(np.float32)
        lab = synth.synth_label(n, c, shape[1:], seed=3)
        y = synth.one_hot(lab, c)
        pw, _ = synth.synth_pixel_weight(lab, seed=3)
        out[f"{tag}_logits"], out[f"{tag}_onehot"], out[f"{tag}_pw"] = z, y, pw
        for wt in (False, True):
            for name, fn in (("dice", Dice), ("ce", CE)):
                zt = torch.from_numpy(z).requires_grad_(True)
                d = {"prediction": zt, "ground_truth": torch.from_numpy(y)}
                if wt:
                    d["pixel_weight"] = torch.from_numpy(pw)
                val = fn({})(d)
                val.backward()
                out[f"{tag}_{name}_{'w' if wt else 'u'}_loss"] = np.asarray(val.item(), np.float64)
                out[f"{tag}_{name}_{'w' if wt else 'u'}_grad"] = zt.grad.numpy()
    np.savez_compressed(os.path.join(GOLD, "loss.npz"), **out)
    print("loss", {k: float(v) for k, v in out.items() if k.endswith("_loss")})


def gen_inferer(UNet, Inferer):
    out = {}
    # (1) stitching with a cheap deterministic 'model' (depends on position inside the window)
    g = np.random.Generator(np.random.PCG64(11))
    wconv = torch.from_numpy(g.standard_normal((3, 1, 3, 3, 3)).astype(np.float32))

    class Toy(torch.nn.Module):
        def forward(self, x, domain_label=None):
            r = torch.nn.functional.conv3d(x, wconv, padding=1)
            ramp = torch.linspace(0, 1, x.shape[-1]).view(1, 1, 1, 1, -1)
            return r + ramp * (1 + domain_label[0].item())

    img = torch.from_numpy(synth.synth_image(1, 1, (20, 40, 44), seed=5))
    for tta in (0, 1):
        cfg = {"sliding_window_enable": True, "sliding_window_size": [16, 32, 32],
               "sliding_window_stride": [8, 16, 32], "tta_mode": tta, "class_num": 3}
        with torch.no_grad():
            o = Inferer(cfg).run(Toy(), img, torch.ones(1, dtype=torch.long))
        out[f"toy_tta{tta}"] = o.numpy()
    # (2) the real net through the real Inferer: 24x48x48 volume, 16x32x32 windows, flips
    net = _ref_net(UNet, NET_PARAMS)
    net.eval()
    vol = torch.from_numpy(synth.synth_image(1, 1, (24, 48, 48), seed=9))
    cfg = {"sliding_window_enable": True, "sliding_window_size": [16, 32, 32],
           "sliding_window_stride": [16, 32, 32], "tta_mode": 1, "class_num": 2}
    with torch.no_grad():
        for d in (0, 1):
            o = Inferer(cfg).run(net, vol, d * torch.ones(1, dtype=torch.long))
            out[f"net_tta1_d{d}"] = o.numpy()
    # a fixed, seeded sample of voxels (all classes of each) keeps the fixture under 1 MB: k -> [N, C, M] at the stored
    # flat voxel indices k_idx of an output of shape k_shape
    sampled = {}
    for k, a in out.items():
        vox = int(np.prod(a.shape[2:]))
        idx = np.sort(np.random.default_rng(0).choice(vox, 12000, replace=False)).astype(np.int32)
        sampled.update({k: a.reshape(a.shape[0], a.shape[1], vox)[:, :, idx], k + "_idx": idx,
                        k + "_shape": np.asarray(a.shape, np.int64)})
    np.savez_compressed(os.path.join(GOLD, "inferer.npz"), **sampled)
    print("inferer", {k: v.shape for k, v in out.items()})


def gen_image_weights():
    """The reference's only golden artefacts: the sorted-uncertainty .npy and the CSV
    built from it by the missing script."""
    import csv
    arr = np.load(os.path.join(REF, "dataset/weight/cyc121_vst1s-gan.npy"), allow_pickle=True)
    names = [os.path.basename(r[1]) for r in arr]
    values = [float(r[0][0]) for r in arr]
    sentinel = [isinstance(r[0][0], int) for r in arr]
    with open(os.path.join(REF, "config_dual/data_vs/train_vs_t1s_wi+wp.csv")) as f:
        rows = list(csv.DictReader(f))
    csv_names = [os.path.basename(r["image"]) for r in rows]
    csv_w = [float(r["image_weight"]) for r in rows]
    with open(os.path.join(GOLD, "fpl_image_weights.json"), "w") as f:
        json.dump({"source": ["dataset/weight/cyc121_vst1s-gan.npy", "config_dual/data_vs/train_vs_t1s_wi+wp.csv"],
                   "names": names, "uncertainty": values, "sentinel": sentinel,
                   "csv_names": csv_names, "csv_image_weight": csv_w}, f, indent=0)
    print("image weights", len(names), "rows;", sum(sentinel), "sentinels")


def main():
    os.makedirs(GOLD, exist_ok=True)
    torch.set_num_threads(os.cpu_count())
    UNet, Dice, CE, Inferer = _import_reference()
    gen_image_weights()
    gen_loss(Dice, CE)
    gen_net(UNet, Dice, CE)
    gen_inferer(UNet, Inferer)
    from oracle import gen_golden_fpl
    gen_golden_fpl.main()


if __name__ == "__main__":
    main()
