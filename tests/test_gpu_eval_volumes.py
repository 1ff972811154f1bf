"""GPU: whole-volume Pad + NormalizeWithMeanStd (csrc/datapath.cu volume_stats_kernel + pad_normalize_volume_kernel)
against np.pad composed with normalize_with_mean_std, and the validation / test stages the agent builds from a cfg's
valid / test CSVs (DeviceVolumeSet)."""
import copy
import math
import os

import numpy as np
import pytest
import torch

from oracle import fpl_filter, inferer as oracle_inferer, synth, unet_dsbn
from oracle.gen_golden import NET_PARAMS
from tests import _util

pytestmark = pytest.mark.gpu
GUARD = 512                                   # sentinel elements on each side of an output


def _modes(spec, c):
    from fplplus_b200.datapath import _norm_modes
    return _norm_modes(spec, c)


def _host(image, label, out_shape, spec, after):
    """The reference: datapath.pad_to (np.pad 'reflect' / 'edge', labels constant 0) and normalize_with_mean_std per
    listed channel, in the transform list's order."""
    from fplplus_b200.datapath import normalize_with_mean_std, pad_to

    def norm(img):
        for c, s in sorted(spec.items()):
            img = normalize_with_mean_std(img, s["mask"], [c], [s["mean"]], [s["std"]])
        return img
    img = norm(pad_to(image, out_shape)) if after else pad_to(norm(image), out_shape)
    lo = [(o - n) // 2 for n, o in zip(image.shape[1:], out_shape)]
    margins = [(l, o - n - l) for n, o, l in zip(image.shape[1:], out_shape, lo)]
    # labels pad with 0 on every axis (pad_to would switch them to 'edge' next to an axis of size 1)
    lab = None if label is None else np.pad(label, margins, "constant")
    return img, lab


def _guarded(n, dtype):
    """A flat output of n elements of ``dtype`` inside a sentinel buffer (tests/_util.sentinel_buf), and the guard."""
    per = torch.tensor([], dtype=dtype).element_size()
    total = (2 * GUARD + n) * per
    buf = _util.sentinel_buf(1, 1, 1, 1, -(-total // 16)).reshape(-1).view(torch.uint8)[:total].view(dtype)
    return buf, buf[GUARD:GUARD + n], buf.clone()


def _device(image, label, out_shape, spec, after):
    from fplplus_b200 import lib
    from fplplus_b200.ops import call, ptr, stream_ptr
    c, shape = image.shape[0], image.shape[1:]
    x = torch.from_numpy(np.ascontiguousarray(image)).to(_util.DEV)
    y = None if label is None else torch.from_numpy(np.ascontiguousarray(label)).to(_util.DEV)
    _m, tab = _modes(spec, c)
    nbytes = int(lib.load().fpl_pad_normalize_volume_workspace_bytes(c, *shape, *out_shape))
    ws = torch.full((nbytes // 8,), float("nan"), dtype=torch.float64, device=_util.DEV)
    ovox = int(np.prod(out_shape))
    ibuf, out, iref = _guarded(c * ovox, torch.float32)
    lbuf, lout, lref = _guarded(ovox, torch.uint8) if y is not None else (None, None, None)
    call("fpl_pad_normalize_volume", ptr(x), ptr(y), c, *shape, *out_shape, tab["mode"], tab["mean"], tab["std"], int(after),
         ptr(ws), nbytes, ptr(out), ptr(lout), stream_ptr())
    torch.cuda.synchronize()
    for buf, ref in ((ibuf, iref), (lbuf, lref)):
        if buf is not None:
            g = buf.view(torch.uint8).numel() // buf.numel() * GUARD
            bb, rb = buf.view(torch.uint8), ref.view(torch.uint8)
            assert torch.equal(bb[:g], rb[:g]) and torch.equal(bb[-g:], rb[-g:]), "write outside the output"
    img = out.view((c,) + tuple(out_shape)).cpu().numpy()
    return img, (None if lout is None else lout.view(tuple(out_shape)).cpu().numpy())


def _volume(c, shape, seed, negative=()):
    rng = _util.rng(seed)
    img = (3.0 + 2.0 * rng.standard_normal((c,) + shape)).astype(np.float32)
    for ch in negative:                       # masked statistics of a channel without a voxel > 0
        img[ch] = -np.abs(img[ch]) - 0.25
    lab = (rng.random(shape) < 0.3).astype(np.uint8) * rng.integers(1, 3, shape).astype(np.uint8)
    return img, lab


CASES = {
    # name: (C, source shape, padded shape, normalize spec, channels without a voxel > 0)
    "every_axis": (1, (20, 50, 70), (32, 64, 96), {0: {"mean": None, "std": None, "mask": False}}, ()),
    "multi_reflect": (1, (3, 5, 70), (16, 32, 96), {0: {"mean": None, "std": None, "mask": True}}, ()),
    "axis_of_one": (1, (1, 40, 50), (16, 64, 64), {0: {"mean": None, "std": None, "mask": False}}, ()),
    "no_pad": (2, (16, 32, 32), (16, 32, 32), {1: {"mean": None, "std": None, "mask": True}}, ()),
    "c3_raw_fixed_masked": (3, (13, 37, 45), (16, 64, 64), {1: {"mean": 2.5, "std": 1.5, "mask": False},
                                                            2: {"mean": None, "std": None, "mask": True}}, ()),
    "c3_stats_masked_empty": (3, (13, 37, 45), (16, 48, 48), {0: {"mean": None, "std": None, "mask": False},
                                                              2: {"mean": None, "std": None, "mask": True}}, (2,)),
}


@pytest.mark.parametrize("after", [False, True], ids=["stats_of_source", "stats_of_padded"])
@pytest.mark.parametrize("case", sorted(CASES))
def test_pad_normalize_volume_matches_np_pad_and_normalize(case, after):
    c, shape, out_shape, spec, negative = CASES[case]
    image, label = _volume(c, shape, seed=len(case) * 7 + int(after), negative=negative)
    ref_img, ref_lab = _host(image, label, out_shape, spec, after)
    got_img, got_lab = _device(image, label, out_shape, spec, after)
    assert got_img.shape == ref_img.shape and np.array_equal(got_lab, ref_lab)
    worst = 0.0
    for ch in range(c):
        if ch in spec:
            err = float(np.abs(got_img[ch] - ref_img[ch]).max())
            worst = max(worst, err)
            assert err <= 1e-5, (case, ch, err)
        else:
            assert np.array_equal(got_img[ch].view(np.uint32), ref_img[ch].view(np.uint32)), (case, ch)
    print("%s (%s): max |device - host| = %.3g" % (case, "padded" if after else "source", worst))


def test_no_padding_and_no_normalisation_copies_the_input_bitwise():
    image, label = _volume(2, (16, 32, 32), seed=4)
    got_img, got_lab = _device(image, label, (16, 32, 32), {}, False)
    assert np.array_equal(got_img.view(np.uint32), image.view(np.uint32)) and np.array_equal(got_lab, label)


def test_pad_normalize_volume_is_bitwise_reproducible_under_every_sm_budget():
    image, label = _volume(3, (13, 37, 45), seed=9)
    spec = {0: {"mean": None, "std": None, "mask": False}, 2: {"mean": None, "std": None, "mask": True}}

    def run():
        return _device(image, label, (16, 64, 64), spec, True)
    outs = [run(), run()] + _util.run_sm_budgets(run)
    for img, lab in outs[1:]:
        assert np.array_equal(img.view(np.uint32), outs[0][0].view(np.uint32)) and np.array_equal(lab, outs[0][1])


def test_volume_above_2_pow_30_voxels_is_refused_before_any_launch():
    from fplplus_b200 import lib
    from fplplus_b200.ops import call, ptr, stream_ptr
    buf = torch.zeros(1024, dtype=torch.float32, device=_util.DEV)
    mode = (lib.ctypes.c_int * 1)(2)
    before = lib.launch_count()
    with pytest.raises(lib.FplError, match="2\\^30"):
        call("fpl_pad_normalize_volume", ptr(buf), None, 1, 1, 1, 1, 1024, 1024, 1025, mode, None, None, 0, ptr(buf),
             4096, ptr(buf), None, stream_ptr())
    assert lib.launch_count() == before


# -- the agent's validation and test stages from a cfg ------------------------------------------------------------------
SHAPES = [(13, 37, 45), (11, 41, 30), (17, 29, 33)]
FPL_SHAPES = [(13, 37, 44), (11, 41, 32), (17, 29, 36)]
SPACING, ORIGIN = (0.41, 0.43, 1.5), (-12.0, 7.5, 3.25)


def _write_csv(tmp_path, name, seed, n, raw=True, shapes=SHAPES):
    """n NIfTI volumes of odd shapes (raw intensities, far from zero mean / unit std) and their labels; the CSV."""
    from fplplus_b200 import artefacts
    root = tmp_path / "data"
    root.mkdir(exist_ok=True)
    rows = []
    for i in range(n):
        shape = shapes[i % len(shapes)]
        lab = synth.synth_label(1, 2, shape, seed=seed + i)[0]
        img = synth.synth_image(1, 1, shape, seed=seed + i)[0, 0] * 0.5 + (lab > 0) * 2.0
        if raw:
            img = 100.0 + 20.0 * img
        base = "%s_%d" % (name, i)
        artefacts.write_nifti(img.astype(np.float32), str(root / (base + "_img.nii.gz")), SPACING, ORIGIN)
        artefacts.write_nifti(lab.astype(np.uint8), str(root / (base + "_lab.nii.gz")), SPACING, ORIGIN)
        rows.append([base + "_img.nii.gz", base + "_lab.nii.gz"])
    path = str(tmp_path / (name + ".csv"))
    artefacts.write_train_csv(path, rows, fields=("image", "label"))
    return path, str(root), rows


def _config(tmp_path, **dataset):
    tr = {"train_fpl_uda": False, "dual": True, "val_t1": False, "val_t2": False, "gpus": [0],
          "loss_type": ["DiceLoss", "CrossEntropyLoss"], "loss_weight": [0.5, 0.5], "optimizer": "Adam",
          "learning_rate": 2e-3, "weight_decay": 1e-5, "lr_scheduler": "MultiStepLR", "lr_gamma": 0.5,
          "lr_milestones": [8], "ckpt_save_dir": str(tmp_path / "model" / "vs_S"), "iter_start": 0, "iter_max": 10,
          "iter_valid": 5, "iter_save": 5, "early_stop_patience": None}
    te = {"fpl": False, "gpus": [0], "domian_label": 1, "ckpt_mode": 2, "evaluation_mode": True,
          "test_time_dropout": False, "tta_mode": 1, "sliding_window_enable": True, "sliding_window_size": [16, 32, 32],
          "sliding_window_stride": [8, 16, 32], "output_dir": str(tmp_path / "result"),
          "fpl_uncertainty_sorted": str(tmp_path / "sorted.npy")}
    ds = {"tensor_type": "float", "train_batch_size": 2, "normalizewithmeanstd_channels": [0],
          "pad_output_size": [16, 32, 32], "pad_ceil_mode": True, "labeltoprobability_class_num": 2}
    ds.update(dataset)
    return {"dataset": ds, "network": dict(NET_PARAMS), "training": tr, "testing": te}


def _agent(cfg, stage):
    from fplplus_b200.agent import SegmentationAgent
    ag = SegmentationAgent(cfg, stage)
    ag.create_dataset()
    ag.create_network()
    sd = synth.synth_state_dict()
    ag.net.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()}, strict=True)
    ag._pick_device("training" if stage == "train" else "testing")
    ag.net.to(ag.device)
    return ag, sd


def _host_transformed(root, row, spec):
    from fplplus_b200 import artefacts
    from fplplus_b200.datapath import padded_shape
    img = np.asarray(artefacts.load_volume(os.path.join(root, row[0])), np.float32)[None]
    lab = np.asarray(artefacts.load_volume(os.path.join(root, row[1]))).astype(np.uint8)
    return _host(img, lab, padded_shape(img.shape[1:], spec["pad"]), spec["normalize"], spec["stats_after_pad"])


def test_validation_from_the_cfg_matches_caller_loaders_and_the_oracle(tmp_path):
    from oracle import losses
    from fplplus_b200.agent import SegmentationAgent
    from fplplus_b200.datapath import eval_transform_from_config
    v1, root, rows1 = _write_csv(tmp_path, "valid1", 300, 2)
    v2, _root, rows2 = _write_csv(tmp_path, "valid2", 400, 3)
    cfg = _config(tmp_path, root_dir=root, **{"1_valid_csv": v1, "2_valid_csv": v2,
                                               "valid_transform": ["NormalizeWithMeanStd", "Pad", "LabelToProbability"]})
    ag, sd = _agent(cfg, "train")
    ag.create_loss_calculator()
    for d, rows in ((0, rows1), (1, rows2)):
        items = list(ag.valid_loaders[d])
        assert len(items) == len(rows) and [b["names"] for b in items] == [[r[0]] for r in rows]
        for b in items:
            assert b["image"].is_cuda and b["label"].is_cuda and b["label"].dtype == torch.uint8
            assert all(s % m == 0 for s, m in zip(b["image"].shape[2:], (16, 32, 32)))
    got = ag.validation()
    again = ag.validation()                                       # resident: the same volumes again
    assert again["loss"] == got["loss"] and np.array_equal(again["class_dice"], got["class_dice"])
    # a second agent given the same device tensors through set_loaders
    other = SegmentationAgent(copy.deepcopy(cfg), "train")
    other.set_loaders(valid=[list(ag.valid_loaders[0]), list(ag.valid_loaders[1])])
    other.create_network()
    other.net.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()}, strict=True)
    other._pick_device("training")
    other.net.to(other.device)
    other.create_loss_calculator()
    ref = other.validation()
    assert ref["loss"] == got["loss"] and ref["avg_dice"] == got["avg_dice"]
    assert np.array_equal(ref["class_dice"], got["class_dice"])
    # the oracle Inferer + losses on the host-transformed volumes
    spec = eval_transform_from_config(cfg, "valid")
    st = unet_dsbn.to_torch_state(sd, requires_grad=False)
    per_dom = []
    for d, rows in ((0, rows1), (1, rows2)):
        ls, ds = [], []
        for row in rows:
            img, lab = _host_transformed(root, row, spec)
            x, y = torch.from_numpy(img[None]), torch.from_numpy(synth.one_hot(lab[None], 2))
            with torch.no_grad():
                z = oracle_inferer.run(lambda t: unet_dsbn.forward(st, t, d, dict(NET_PARAMS)), x, 2, cfg["testing"])
            ls.append(float(losses.combined_loss(z, y, None, 0.5, 0.5)))
            ds.append(losses.hard_dice(z, y).numpy())
        per_dom.append((np.mean(ls), np.mean(np.stack(ds, 0), 0)))
    exp_loss = float(np.mean([p[0] for p in per_dom]))
    exp_dice = np.mean(np.stack([p[1] for p in per_dom], 0), 0)
    print("validation from the cfg: loss %.5f oracle %.5f; class dice %s oracle %s"
          % (got["loss"], exp_loss, got["class_dice"], exp_dice))
    assert abs(got["loss"] - exp_loss) <= 1e-2 * abs(exp_loss)
    np.testing.assert_allclose(got["class_dice"], exp_dice, atol=2e-2)


def test_cfg_only_run_validates_on_the_valid_csvs(tmp_path):
    from fplplus_b200.agent import SegmentationAgent
    t1, root, _rows = _write_csv(tmp_path, "train1", 10, 3)
    t2, _root, _rows = _write_csv(tmp_path, "train2", 20, 3)
    v1, _root, _rows = _write_csv(tmp_path, "valid1", 30, 2)
    v2, _root, _rows = _write_csv(tmp_path, "valid2", 40, 2)
    # Pad_ceil_mode is a key of the evaluation Pad only: the training list crops (and pads to) the patch size itself
    cfg = _config(tmp_path, root_dir=root, **{
        "1_train_csv": t1, "2_train_csv": t2, "1_valid_csv": v1, "2_valid_csv": v2,
        "train_transform": ["RandomCrop", "RandomFlip", "NormalizeWithMeanStd", "LabelToProbability"],
        "valid_transform": ["NormalizeWithMeanStd", "Pad", "LabelToProbability"],
        "randomcrop_output_size": [16, 32, 32], "randomflip_flip_depth": False})
    ag = SegmentationAgent(cfg, "train")
    hist = ag.run()
    assert [h[0] for h in hist] == [5, 10]
    assert all(v.__class__.__name__ == "DeviceVolumeSet" for v in ag.valid_loaders)
    for _it, train, valid in hist:
        assert math.isfinite(train["loss"]) and math.isfinite(valid["loss"]) and valid["loss"] > 0.0
        assert valid["avg_dice"] > 0.0


def _test_cfg(tmp_path, shapes=SHAPES, **testing):
    path, root, rows = _write_csv(tmp_path, "test", 500, 3, shapes=shapes)
    cfg = _config(tmp_path, root_dir=root, test_csv=path, test_transform=["NormalizeWithMeanStd", "Pad"])
    cfg["testing"].update(testing)
    return cfg, root, rows


@pytest.mark.parametrize("inverse", [True, False])
def test_test_stage_from_the_cfg_writes_cropped_label_volumes(tmp_path, inverse):
    from fplplus_b200 import artefacts, fpl
    from fplplus_b200.datapath import eval_transform_from_config
    cfg, root, rows = _test_cfg(tmp_path)
    cfg["dataset"]["pad_inverse"] = inverse
    ag, sd = _agent(cfg, "test")
    out = ag.infer(load_checkpoint=False)
    assert sorted(out) == sorted(r[0] for r in rows)
    spec = eval_transform_from_config(cfg, "test")
    st = unet_dsbn.to_torch_state(sd, requires_grad=False)
    for i, row in enumerate(rows):
        src = artefacts.read_nifti(os.path.join(root, row[0]))
        saved = artefacts.read_nifti(os.path.join(cfg["testing"]["output_dir"], row[0]))
        assert saved["data"].dtype == np.uint8 and np.array_equal(saved["data"], out[row[0]][0])
        np.testing.assert_allclose(saved["spacing"], src["spacing"], rtol=1e-6)
        np.testing.assert_allclose(saved["origin"], src["origin"], rtol=1e-6)
        b = ag.test_loader[i]
        padded = tuple(b["image"].shape[2:])
        if not inverse:
            assert saved["data"].shape == padded
            continue
        assert saved["data"].shape == src["data"].shape
        with torch.no_grad():
            lab = fpl.pseudo_label(ag.inferer.run(ag.net, b["image"], domain_label=torch.ones(1, dtype=torch.long)))
        assert np.array_equal(out[row[0]], ag._crop(lab, b["pad"]).cpu().numpy())
        img, _lab = _host_transformed(root, row, spec)
        with torch.no_grad():
            z = oracle_inferer.run(lambda t: unet_dsbn.forward(st, t, 1, dict(NET_PARAMS)), torch.from_numpy(img[None]), 2,
                                   cfg["testing"])
        (lo, hi) = b["pad"]
        ref = fpl_filter.pseudo_label(z.numpy())[0][lo[0]:padded[0] - hi[0], lo[1]:padded[1] - hi[1],
                                                     lo[2]:padded[2] - hi[2]]
        agree = float((ref == out[row[0]][0]).mean())
        print("%s: label agreement with the oracle %.5f" % (row[0], agree))
        assert agree >= 0.995


def test_fpl_branch_from_the_cfg_uses_the_uncropped_volumes(tmp_path):
    from fplplus_b200 import fpl
    # fpl_mc_uncertainty takes volumes of a multiple of 4 voxels (the reference's sample volumes are): odd axes, even counts
    cfg, root, rows = _test_cfg(tmp_path, FPL_SHAPES, fpl=True, test_time_dropout=True, tta_mode=0)
    ag, _sd = _agent(cfg, "test")
    torch.manual_seed(11)
    srt = ag.infer(load_checkpoint=False)
    assert sorted(n for _v, n in srt) == sorted(r[0] for r in rows)
    # by hand, from the same MC-dropout seeds: K passes of each volume, cropped to the source box, then the statistics
    torch.manual_seed(11)
    k = int(cfg["testing"].get("fpl_mc_passes", 6))
    expect = {}
    with torch.no_grad():
        for i, row in enumerate(rows):
            b = ag.test_loader[i]
            passes = ag.inferer.run(ag.net, b["image"], torch.ones(1, dtype=torch.long), mc_passes=k)
            passes = [ag._crop(p, b["pad"]) for p in passes]
            assert passes[0].shape[2:] == tuple(FPL_SHAPES[i])
            expect[row[0]] = fpl.finish_uncertainty(fpl.mc_uncertainty(passes)[0])
    for (v, name) in srt:
        assert v == [expect[name]], (name, v, expect[name])
