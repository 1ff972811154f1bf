"""GPU: per-patch NormalizeWithMeanStd of DevicePatchSampler (csrc/datapath.cu patch_stats_kernel +
gather_patches_norm_kernel) against datapath.normalize_with_mean_std of the cut, flipped patch, and a training run that
the agent builds from a cfg's CSVs alone."""
import math
import os

import numpy as np
import pytest
import torch

from oracle.gen_golden_datapath import volumes as _volumes

pytestmark = pytest.mark.gpu
PATCH = (28, 128, 128)


def _cut(vol, patch, origin, flip):
    sl = tuple(slice(o, o + p) for o, p in zip(origin, patch))
    out = vol[(slice(None),) * (vol.ndim - 3) + sl]
    axes = [a for a, bit in ((-3, 1), (-2, 2), (-1, 4)) if flip & bit]
    return np.flip(out, axes) if axes else out


def _batches(vols, normalize, seed, steps=4, bs=4):
    """(image, label, code, last_params) of ``steps`` batches of a sampler, on the host."""
    from fplplus_b200.datapath import DevicePatchSampler
    smp = DevicePatchSampler(vols, PATCH, bs, "cuda:0", seed=seed, normalize=normalize)
    out = []
    for _ in range(steps):
        b = smp.next_batch()
        torch.cuda.synchronize()
        out.append((b["image"].cpu().numpy(), b["label"].cpu().numpy(), b["pixel_weight"].cpu().numpy(),
                    list(smp.last_params)))
    return out


def _all_negative(v):
    return dict(v, image=-np.abs(v["image"]) - 0.25, name=v["name"] + "_neg")


CASES = {
    "unmasked": ({0: {}}, dict(mask_nonzero=False)),
    "masked": ({0: {"mask": True}}, dict(mask_nonzero=True)),
    "fixed": ({0: {"mean": 0.3, "std": 2.5}}, dict(mean=[0.3], std=[2.5])),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_patch_normalisation_matches_the_host_definition(case):
    from fplplus_b200.datapath import normalize_with_mean_std, pad_to
    normalize, kw = CASES[case]
    vols = _volumes(3)
    vols.append(_all_negative(vols[0]))              # masked mode: no voxel > 0, statistics of the whole patch
    padded = {v["name"]: pad_to(v["image"], PATCH) for v in vols}
    norm = _batches(vols, normalize, seed=21)
    plain = _batches(vols, None, seed=21)
    worst = 0.0
    for (img, lab, code, params), (pimg, plab, pcode, pparams) in zip(norm, plain):
        assert params == pparams                                  # same decisions, same draws
        assert np.array_equal(lab, plab) and np.array_equal(code, pcode)
        for i, (name, origin, flip) in enumerate(params):
            ref = normalize_with_mean_std(np.ascontiguousarray(_cut(padded[name], PATCH, origin, flip)), **kw)
            err = float(np.abs(img[i] - ref).max())
            worst = max(worst, err)
            assert err <= 1e-5, (case, name, origin, flip, err)
    print("%s: max |device - host| = %.3g" % (case, worst))


def test_unlisted_channel_is_the_plain_gather_bit_for_bit():
    from fplplus_b200.datapath import normalize_with_mean_std, pad_to
    vols = [dict(v, image=np.concatenate([v["image"], 40.0 * v["image"] + 3.0], 0)) for v in _volumes(4)]
    padded = {v["name"]: pad_to(v["image"], PATCH) for v in vols}
    norm = _batches(vols, {0: {"mask": True}}, seed=8)
    plain = _batches(vols, None, seed=8)
    for (img, lab, code, params), (pimg, plab, pcode, pparams) in zip(norm, plain):
        assert params == pparams and np.array_equal(lab, plab) and np.array_equal(code, pcode)
        assert np.array_equal(img[:, 1], pimg[:, 1])
        for i, (name, origin, flip) in enumerate(params):
            ref = normalize_with_mean_std(np.ascontiguousarray(_cut(padded[name], PATCH, origin, flip)), True, channels=[0])
            assert np.array_equal(ref[1], pimg[i, 1])
            assert float(np.abs(img[i, 0] - ref[0]).max()) <= 1e-5


def test_normalised_batches_are_bitwise_reproducible():
    vols = _volumes(5)
    a = _batches(vols, {0: {"mask": True}}, seed=13, steps=3)
    b = _batches(vols, {0: {"mask": True}}, seed=13, steps=3)
    for (ia, _la, _ca, pa), (ib, _lb, _cb, pb) in zip(a, b):
        assert pa == pb and np.array_equal(ia.view(np.uint32), ib.view(np.uint32))


def test_agent_trains_from_the_cfg_csvs_alone(tmp_path):
    from fplplus_b200 import artefacts
    from fplplus_b200.agent import SegmentationAgent
    from oracle.gen_golden import NET_PARAMS
    root = tmp_path / "data"
    root.mkdir()
    csvs = []
    for d, weighted in ((1, False), (2, True)):
        rows = []
        for v in _volumes(10 * d):
            img = 100.0 + 20.0 * v["image"] + 30.0 * v["label"]          # raw intensities, far from zero mean / unit std
            base = "d%d_%s" % (d, v["name"])
            np.save(root / (base + "_img.npy"), img.astype(np.float32))
            np.save(root / (base + "_lab.npy"), v["label"])
            row = [base + "_img.npy", base + "_lab.npy"]
            if weighted:
                np.save(root / (base + "_pw.npy"), v["pixel_weight"])
                row += [base + "_pw.npy", repr(v["image_weight"])]
            rows.append(row)
        path = str(tmp_path / ("train_%d.csv" % d))
        artefacts.write_train_csv(path, rows)
        csvs.append(path)
    ckpt = tmp_path / "model" / "vs_S"
    cfg = {"dataset": {"tensor_type": "float", "root_dir": str(root), "1_train_csv": csvs[0], "2_train_csv": csvs[1],
                       "train_batch_size": 2,
                       "train_transform": ["Pad", "RandomCrop", "RandomFlip", "NormalizeWithMeanStd", "LabelToProbability"],
                       "randomcrop_output_size": [16, 64, 64], "randomflip_flip_depth": False,
                       "normalizewithmeanstd_channels": [0], "labeltoprobability_class_num": 2},
           "network": dict(NET_PARAMS),
           "training": {"train_fpl_uda": True, "dual": True, "gpus": [0], "loss_type": ["DiceLoss", "CrossEntropyLoss"],
                        "loss_weight": [0.5, 0.5], "optimizer": "Adam", "learning_rate": 2e-3, "weight_decay": 1e-5,
                        "lr_scheduler": "MultiStepLR", "lr_gamma": 0.5, "lr_milestones": [8],
                        "ckpt_save_dir": str(ckpt), "iter_start": 0, "iter_max": 10, "iter_valid": 5, "iter_save": 5,
                        "early_stop_patience": None},
           "testing": {}}
    ag = SegmentationAgent(cfg, "train")
    hist = ag.run()
    assert [h[0] for h in hist] == [5, 10]
    for _it, train, _valid in hist:
        assert math.isfinite(train["loss"]) and train["loss"] > 0.0
    assert any(e["graph"] is not None for e in ag._graphs.values())
    # both domains came from the device sampler, domain 2 with its agreement codes, and the patches were normalised
    b0, b1 = ag.train_loaders[0].next_batch(), ag.train_loaders[1].next_batch()
    assert "pixel_weight" not in b0 and b1["pixel_weight"].dtype == torch.uint8
    m = b0["image"].double().mean(dim=(1, 2, 3, 4))
    assert float(m.abs().max()) < 1e-4
    for name in ("vs_S_5.pt", "vs_S_10.pt", "vs_S_latest.txt", "vs_S_best.txt"):
        assert os.path.isfile(ckpt / name), name
    assert open(ckpt / "vs_S_latest.txt").read() == "10"
