"""CPU: validation / test volumes from a .cfg -- the transform spec of valid_transform / test_transform
(datapath.eval_transform_from_config), the CSV rows of DeviceVolumeSet, and how infer() reads a cfg-built test set."""
import copy
import json
import os

import numpy as np
import pytest
import torch

from fplplus_b200 import agent as A
from fplplus_b200 import artefacts, datapath


def _parsed(golden_dir):
    with open(os.path.join(golden_dir, "cfg_parse.json")) as f:
        return json.load(f)["parsed"]


def _cfg(golden_dir, stage, transforms, **keys):
    cfg = copy.deepcopy(_parsed(golden_dir))
    cfg["dataset"][stage + "_transform"] = transforms
    cfg["dataset"].update(keys)
    return cfg


def test_normalize_before_pad_takes_the_statistics_of_the_source_volume(golden_dir):
    cfg = _cfg(golden_dir, "valid", ["NormalizeWithMeanStd", "Pad", "LabelToProbability"], pad_output_size=[16, 32, 32],
               normalizewithmeanstd_mask=True, normalizewithmeanstd_inverse=False, labeltoprobability_inverse=False)
    spec = datapath.eval_transform_from_config(cfg, "valid")
    assert spec == {"normalize": {0: {"mean": None, "std": None, "mask": True}},
                    "pad": {"output_size": [16, 32, 32], "ceil_mode": False, "inverse": True},
                    "stats_after_pad": False}


def test_pad_before_normalize_takes_the_statistics_of_the_padded_volume(golden_dir):
    cfg = _cfg(golden_dir, "test", ["Pad", "NormalizeWithMeanStd"], pad_output_size=[16, 32, 32], pad_ceil_mode=True,
               normalizewithmeanstd_channels=[0, 1], normalizewithmeanstd_mean=[1.0, 2.0], normalizewithmeanstd_std=[3.0, 4.0])
    spec = datapath.eval_transform_from_config(cfg, "test")
    assert spec["stats_after_pad"] is True and spec["pad"]["ceil_mode"] is True
    assert spec["normalize"] == {0: {"mean": 1.0, "std": 3.0, "mask": False}, 1: {"mean": 2.0, "std": 4.0, "mask": False}}
    # the other stage's list is read on its own; an absent list means no transform
    assert datapath.eval_transform_from_config(cfg, "valid") == {"normalize": None, "pad": None, "stats_after_pad": False}


def test_padded_shape_with_and_without_ceil_mode():
    ceil = {"output_size": [16, 32, 32], "ceil_mode": True, "inverse": True}
    assert datapath.padded_shape((20, 50, 70), ceil) == (32, 64, 96)
    assert datapath.padded_shape((16, 64, 1), ceil) == (16, 64, 32)
    plain = {"output_size": [24, 64, 64], "ceil_mode": False, "inverse": True}
    assert datapath.padded_shape((20, 50, 70), plain) == (24, 64, 70)
    assert datapath.padded_shape((40, 160, 272), None) == (40, 160, 272)


def test_pad_inverse_false(golden_dir):
    cfg = _cfg(golden_dir, "test", ["Pad"], pad_output_size=[16, 32, 32], pad_inverse=False)
    spec = datapath.eval_transform_from_config(cfg, "test")
    assert spec["pad"]["inverse"] is False and spec["normalize"] is None


@pytest.mark.parametrize("transforms, keys, match", [
    (["NormalizeWithMeanStd", "RandomCrop"], {}, "RandomCrop is not supported"),
    (["RandomFlip", "Pad"], {}, "RandomFlip is not supported"),
    (["Pad", "Rescale"], {}, "Rescale is not supported"),
    (["Pad", "NormalizeWithMeanStd", "Pad"], {}, "Pad is listed twice"),
    (["Pad"], {"pad_mode": "constant"}, "Pad_mode"),
    (["NormalizeWithMeanStd"], {"normalizewithmeanstd_foo": 1}, "NormalizeWithMeanStd_foo"),
    (["NormalizeWithMeanStd"], {"normalizewithmeanstd_mask": True, "normalizewithmeanstd_random_fill": True},
     "NormalizeWithMeanStd_random_fill"),
    (["NormalizeWithMeanStd"], {"normalizewithmeanstd_mean": [1.0]}, "both"),
    (["Pad"], {"pad_output_size": None}, "Pad_output_size"),
    (["Pad"], {"pad_output_size": [16, 32]}, "Pad_output_size"),
])
def test_unsupported_eval_transform_raises_naming_the_offender(golden_dir, transforms, keys, match):
    cfg = _cfg(golden_dir, "valid", transforms, pad_output_size=[16, 32, 32])
    cfg["dataset"].update(keys)
    with pytest.raises(ValueError, match=match):
        datapath.eval_transform_from_config(cfg, "valid")


def test_training_parser_still_rejects_pad_ceil_mode(golden_dir):
    cfg = copy.deepcopy(_parsed(golden_dir))
    cfg["dataset"]["train_transform"] = ["Pad", "RandomCrop"]
    cfg["dataset"].update(pad_output_size=[16, 32, 32], pad_ceil_mode=True)
    with pytest.raises(ValueError, match="Pad_ceil_mode"):
        datapath.sampler_args_from_config(cfg, 0)


def _write_volumes(root, n, with_label=True, shape=(6, 10, 12)):
    rng = np.random.default_rng(3)
    rows = []
    for i in range(n):
        img = rng.standard_normal(shape).astype(np.float32) + i
        np.save(os.path.join(root, "img%d.npy" % i), img)
        row = ["img%d.npy" % i]
        if with_label:
            np.save(os.path.join(root, "lab%d.npy" % i), (img > i).astype(np.int64))
            row.append("lab%d.npy" % i)
        rows.append(row)
    return rows


def test_volume_set_reads_the_csv_rows(tmp_path):
    root = tmp_path / "data"
    root.mkdir()
    rows = _write_volumes(str(root), 3)
    rows[1] = rows[1][:1]                                        # no label column
    rows[2] = rows[2] + ["extra.npy", "0.5"]                     # further columns are ignored
    path = str(tmp_path / "valid.csv")
    with open(path, "w") as f:
        f.write("image,label\n" + "\n".join(",".join(r) for r in rows) + "\n\n")
    vs = datapath.DeviceVolumeSet(path, "cpu", str(root))
    assert len(vs) == 3 and not vs.invert_pad
    for i, b in enumerate(vs):
        img = np.load(root / ("img%d.npy" % i))
        assert b["names"] == ["img%d.npy" % i] and b["pad"] is None
        assert b["image"].dtype == torch.float32 and np.array_equal(b["image"].numpy(), img[None, None])
        if i == 1:
            assert "label" not in b
        else:
            assert b["label"].dtype == torch.uint8 and np.array_equal(b["label"].numpy()[0], img > i)
    test = datapath.DeviceVolumeSet(path, "cpu", str(root), resident=False, labels=False)
    assert "label" not in test[0] and np.array_equal(test[2]["image"], vs[2]["image"])
    with pytest.raises(IndexError):
        test[3]


def test_infer_without_test_volumes_raises_before_touching_a_device(golden_dir):
    cfg = copy.deepcopy(_parsed(golden_dir))
    cfg["dataset"].pop("test_csv", None)
    ag = A.SegmentationAgent(cfg, "test")

    def no_device(section):
        raise AssertionError("infer() picked a device")
    ag._pick_device = no_device
    ag.create_dataset()
    with pytest.raises(ValueError, match=r"\[dataset\] test_csv"):
        ag.infer(load_checkpoint=False)


class _Net(torch.nn.Module):
    def forward(self, x):
        return x


class _Inferer(object):
    """Two-class logits of a volume: class 1 where the image is > 0."""
    def run(self, net, x, domain_label=None):
        return torch.cat([-x, x], 1)


def _host_pad(image, label, transform):
    """pad_normalize_volume on the host (datapath.pad_to): the CPU stand-in of the device transform."""
    out_shape = datapath.padded_shape(image.shape[1:], transform["pad"])
    out = torch.from_numpy(datapath.pad_to(image.numpy(), out_shape))
    lo = tuple((o - n) // 2 for n, o in zip(image.shape[1:], out_shape))
    hi = tuple(o - n - l for n, o, l in zip(image.shape[1:], out_shape, lo))
    return out, None, ((lo, hi) if any(lo) or any(hi) else None)


@pytest.mark.parametrize("inverse", [True, False])
def test_cfg_built_test_set_is_sharded_by_index_and_cropped_back(tmp_path, golden_dir, monkeypatch, inverse):
    root = tmp_path / "data"
    root.mkdir()
    rows = _write_volumes(str(root), 5)
    path = str(tmp_path / "test.csv")
    artefacts.write_train_csv(path, rows, fields=("image", "label"))
    cfg = copy.deepcopy(_parsed(golden_dir))
    cfg["dataset"].update(test_csv=path, root_dir=str(root), test_transform=["Pad"], pad_output_size=[8, 16, 16],
                          pad_inverse=inverse)
    cfg["testing"].update(fpl=False, output_dir=None, evaluation_mode=True, test_time_dropout=False)
    read = []
    real_load = artefacts.load_volume

    def counting_load(p):
        read.append(os.path.relpath(p, str(root)))
        return real_load(p)
    monkeypatch.setattr(artefacts, "load_volume", counting_load)
    monkeypatch.setattr(datapath, "pad_normalize_volume", _host_pad)
    monkeypatch.setattr(A.fpl, "pseudo_label", lambda z: z.argmax(1).to(torch.uint8))
    for rank in (0, 1):
        read.clear()
        ag = A.SegmentationAgent(cfg, "test")
        ag._pick_device = lambda section: torch.device("cpu")
        ag.rank, ag.world = rank, 2
        ag.create_dataset()
        assert isinstance(ag.test_loader, datapath.DeviceVolumeSet) and read == []     # nothing read up front
        ag.set_network(_Net())
        ag.set_inferer(_Inferer())
        out = ag.infer(load_checkpoint=False)
        mine = rows[rank::2]
        assert read == [r[0] for r in mine]                       # this rank's rows only, images only
        assert sorted(out) == sorted(r[0] for r in mine)
        for name, lab in out.items():
            img = np.load(root / name)
            if inverse:
                assert lab.shape == (1,) + img.shape and np.array_equal(lab[0], img > 0)
            else:
                assert lab.shape == (1, 8, 16, 16)
