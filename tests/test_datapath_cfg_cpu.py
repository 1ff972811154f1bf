"""CPU: the training samplers a .cfg describes (datapath.sampler_args_from_config / load_train_csv) and the decisions of a
sampler that normalises per patch."""
import copy
import json
import os

import numpy as np
import pytest

from oracle.gen_golden_datapath import volumes as _volumes


def _parsed(golden_dir):
    with open(os.path.join(golden_dir, "cfg_parse.json")) as f:
        return json.load(f)["parsed"]


def test_shipped_cfg_gives_the_sampler_of_the_fpl_configs(golden_dir):
    from fplplus_b200.datapath import sampler_args_from_config
    cfg = _parsed(golden_dir)
    for domain, csv in ((0, "config/train_t1.csv"), (1, "config/train_t2_wi+wp.csv")):
        a = sampler_args_from_config(cfg, domain, rank=1, world=2)
        s = a["sampler"]
        assert a["csv"] == csv and a["root_dir"] == "./data"
        assert s["patch"] == (32, 128, 128) and s["batch_size"] == 4
        assert s["flip"] == (False, True, True)
        assert s["rank"] == 1 and s["world"] == 2 and s["seed"] == 1 + domain
        # NormalizeWithMeanStd after RandomCrop: per-patch statistics of channel 0 on the device, nothing on the host
        assert s["normalize"] == {0: {"mean": None, "std": None, "mask": False}}
        assert a["host_transforms"] == []
        # keys the cfg does not set keep the sampler's defaults
        assert "fg_focus" not in s and "fg_ratio" not in s and "mask_label" not in s


def test_normalize_before_randomcrop_runs_per_volume_on_the_host(golden_dir):
    from fplplus_b200.datapath import sampler_args_from_config
    cfg = _parsed(golden_dir)
    ds = cfg["dataset"]
    ds["train_transform"] = ["Pad", "NormalizeWithMeanStd", "RandomCrop", "RandomFlip", "LabelToProbability"]
    ds.update(pad_output_size=[40, 130, 130], normalizewithmeanstd_mask=True, randomcrop_foreground_focus=False,
              randomcrop_mask_label=[1, 2], randomflip_flip_width=False, randomcrop_inverse=False,
              normalizewithmeanstd_inverse=False)
    a = sampler_args_from_config(cfg, 0)
    assert "normalize" not in a["sampler"]
    assert a["host_transforms"] == [("Pad", {"output_size": [40, 130, 130]}),
                                    ("NormalizeWithMeanStd", {0: {"mean": None, "std": None, "mask": True}})]
    s = a["sampler"]
    assert s["fg_focus"] is False and s["mask_label"] == [1, 2] and s["flip"] == (False, True, False)


def test_no_randomflip_means_no_flips_and_fixed_mean_std_are_passed(golden_dir):
    from fplplus_b200.datapath import sampler_args_from_config
    cfg = _parsed(golden_dir)
    ds = cfg["dataset"]
    ds["train_transform"] = ["RandomCrop", "NormalizeWithMeanStd"]
    ds.update(normalizewithmeanstd_channels=[0, 1], normalizewithmeanstd_mean=[10.0, 20.0],
              normalizewithmeanstd_std=[2.0, 4.0])
    s = sampler_args_from_config(cfg, 1)["sampler"]
    assert s["flip"] == (False, False, False)
    assert s["normalize"] == {0: {"mean": 10.0, "std": 2.0, "mask": False}, 1: {"mean": 20.0, "std": 4.0, "mask": False}}


@pytest.mark.parametrize("edit, match", [
    (lambda ds: ds.update(train_transform=["Pad", "RandomCrop", "RandomRotate"]), "RandomRotate"),
    (lambda ds: ds.update(train_transform=["RandomCrop", "Pad"]), "Pad must come before RandomCrop"),
    (lambda ds: ds.update(randomcrop_foreground_size=[1, 2, 3]), "RandomCrop_foreground_size"),
    (lambda ds: ds.update(normalizewithmeanstd_mask=True, normalizewithmeanstd_random_fill=True),
     "NormalizeWithMeanStd_random_fill"),
    (lambda ds: ds.update(train_transform=["Pad", "RandomFlip"]), "no RandomCrop"),
    (lambda ds: ds.update(normalizewithmeanstd_mean=[1.0]), "both"),
])
def test_unsupported_cfg_raises_naming_the_offender(golden_dir, edit, match):
    from fplplus_b200.datapath import sampler_args_from_config
    cfg = copy.deepcopy(_parsed(golden_dir))
    edit(cfg["dataset"])
    with pytest.raises(ValueError, match=match):
        sampler_args_from_config(cfg, 0)


def test_train_csv_of_npy_volumes(tmp_path):
    from fplplus_b200 import artefacts
    from fplplus_b200.datapath import code_from_pixel_weight, load_train_csv, normalize_with_mean_std, pad_to
    vols = _volumes(1)
    rows = []
    for v in vols:
        for k in ("image", "label", "pixel_weight"):
            np.save(tmp_path / ("%s_%s.npy" % (v["name"], k)), v[k] if k != "label" else v[k].astype(np.int64))
        rows.append(["%s_image.npy" % v["name"], "%s_label.npy" % v["name"], "%s_pixel_weight.npy" % v["name"],
                     repr(v["image_weight"])])
    rows[2] = rows[2][:2]                                       # image,label only: no code, image weight 1
    csv_path = str(tmp_path / "train.csv")
    artefacts.write_train_csv(csv_path, rows)
    got = load_train_csv(csv_path, str(tmp_path))
    assert [g["name"] for g in got] == [r[0] for r in rows]
    for i, (g, v) in enumerate(zip(got, vols)):
        assert g["image"].dtype == np.float32 and np.array_equal(g["image"], v["image"])
        assert g["label"].dtype == np.uint8 and np.array_equal(g["label"], v["label"])
        if i < 2:
            assert g["code"].dtype == np.uint8 and np.array_equal(g["code"], code_from_pixel_weight(v["pixel_weight"]))
            assert g["image_weight"] == v["image_weight"]
        else:
            assert "code" not in g and g["image_weight"] == 1.0
    # host transforms run per volume in the listed order: Pad, then NormalizeWithMeanStd of the padded volume
    spec = {0: {"mean": None, "std": None, "mask": True}}
    got = load_train_csv(csv_path, str(tmp_path), [("Pad", {"output_size": [24, 150, 210]}), ("NormalizeWithMeanStd", spec)])
    v = vols[1]
    np.testing.assert_array_equal(got[1]["image"], normalize_with_mean_std(pad_to(v["image"], (24, 150, 210)), True))
    np.testing.assert_array_equal(got[1]["label"], pad_to(v["label"], (24, 150, 210), "constant"))


def test_normalized_sampler_draws_the_same_decisions():
    from fplplus_b200.datapath import DevicePatchSampler
    vols = _volumes(2)
    plain = DevicePatchSampler(vols, (28, 128, 128), 2, "cpu", seed=5)
    norm = DevicePatchSampler(vols, (28, 128, 128), 2, "cpu", seed=5, normalize={0: {"mask": True}})
    for _ in range(30):
        i, j = plain._next_volume(), norm._next_volume()
        assert i == j
        assert plain.draw(plain.vols[i]) == norm.draw(norm.vols[j])
    assert plain.rng.getstate() == norm.rng.getstate()


@pytest.mark.parametrize("normalize, match", [
    ({1: {}}, "channel 1"),
    ({0: {"mean": 1.0}}, "both"),
    ({0: {"mean": 1.0, "std": 0.0}}, "> 0"),
    ({0: {"scale": 2.0}}, "unknown"),
])
def test_bad_normalize_argument_raises(normalize, match):
    from fplplus_b200.datapath import DevicePatchSampler
    with pytest.raises(ValueError, match=match):
        DevicePatchSampler(_volumes(2)[:1], (28, 128, 128), 2, "cpu", normalize=normalize)
