"""tests/golden/datapath_decisions.json: the RandomCrop (foreground focus) + RandomFlip decisions of 40 seeded trials over
three fixed volumes -- crop origin, flip code and a digest of the `random` state after each trial, which pins the number
of draws (tests/test_datapath.py::test_crop_and_flip_decisions_follow_the_reference_transforms).

The values are what DevicePatchSampler.draw makes (fpl-plus_b200/datapath.py).  With a PyMIC source tree given, every
trial is first replayed through the reference's own transform/crop.py RandomCrop and transform/flip.py RandomFlip from the
same `random` state, and the file is written only if crop origin, flip axes and the state after the trial all agree:
    python -m oracle.gen_golden_datapath [--reference <dir holding PyMIC/>]"""
import argparse
import hashlib
import json
import os
import random
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PATCH = (28, 128, 128)
SEED = 7
TRIALS = 40


def volumes(seed=0):
    rng = np.random.default_rng(seed)
    vols = []
    for i, shape in enumerate([(40, 160, 150), (20, 140, 200), (36, 128, 128)]):          # the second is thinner than the patch
        img = rng.standard_normal((1,) + shape).astype(np.float32)
        lab = np.zeros(shape, np.uint8)
        c = [s // 2 + int(rng.integers(-3, 4)) for s in shape]
        lab[c[0] - 3:c[0] + 4, c[1] - 10:c[1] + 12, c[2] - 9:c[2] + 10] = 1
        pw = np.where(rng.random(shape) < 0.1, 0.5, 1.0).astype(np.float32)
        vols.append({"image": img, "label": lab, "pixel_weight": pw, "image_weight": 0.2 + 0.3 * i, "name": "v%d" % i})
    return vols


def sampler(vols):
    from fplplus_b200.datapath import DevicePatchSampler
    return DevicePatchSampler(vols, PATCH, 2, "cpu", fg_focus=True, fg_ratio=0.5, flip=(False, True, True), seed=SEED)


def state_digest(rng):
    return hashlib.sha256(repr(rng.getstate()).encode()).hexdigest()[:16]


def record():
    smp = sampler(volumes())
    trials = []
    for trial in range(TRIALS):
        crop_min, flip = smp.draw(smp.vols[trial % 3])
        trials.append({"volume": trial % 3, "crop_min": [int(c) for c in crop_min], "flip": int(flip),
                       "state": state_digest(smp.rng)})
    return trials


def check_reference(ref_dir, trials):
    """Replays the trials through the reference transforms (needs the PyMIC tree and oracle.gen_golden_fpl's stubs)."""
    for p in (ref_dir, os.path.join(ref_dir, "PyMIC")):
        if p not in sys.path:
            sys.path.insert(0, p)
    from oracle.gen_golden_fpl import _install_stubs
    _install_stubs()
    from pymic.transform.crop import RandomCrop
    from pymic.transform.flip import RandomFlip
    from fplplus_b200.datapath import pad_to
    vols = volumes()
    smp = sampler(vols)
    params = {"randomcrop_output_size": list(PATCH), "randomcrop_foreground_focus": True, "randomcrop_foreground_ratio": 0.5,
              "randomcrop_mask_label": [1], "randomcrop_inverse": False, "task": "segmentation",
              "randomflip_flip_depth": False, "randomflip_flip_height": True, "randomflip_flip_width": True,
              "randomflip_inverse": False}
    crop, flip = RandomCrop(params), RandomFlip(params)
    random.setstate(smp.rng.getstate())                   # the reference draws from the global generator
    for t in trials:
        img = pad_to(vols[t["volume"]]["image"], PATCH)
        lab = pad_to(vols[t["volume"]]["label"], PATCH, "constant")[None]
        _s, cmin, cmax = crop._get_crop_param({"image": img, "label": lab})
        out = flip({"image": img[:, cmin[1]:cmax[1], cmin[2]:cmax[2], cmin[3]:cmax[3]]})
        axes = json.loads(out["RandomFlip_Param"])
        ref_flip = (4 if -1 in axes else 0) | (2 if -2 in axes else 0) | (1 if -3 in axes else 0)
        assert list(cmin[1:]) == t["crop_min"] and ref_flip == t["flip"], (t, cmin, axes)
        assert state_digest(random) == t["state"], t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", help="directory holding the PyMIC source tree of the original project")
    args = ap.parse_args()
    trials = record()
    if args.reference:
        check_reference(args.reference, trials)
    source = ("fplplus_b200.datapath.DevicePatchSampler.draw, checked trial by trial against PyMIC RandomCrop "
              "(transform/crop.py:213-234) + RandomFlip (transform/flip.py:38-47)" if args.reference else
              "fplplus_b200.datapath.DevicePatchSampler.draw as of commit 82fa7c0 (datapath.py unchanged since), whose "
              "test compared these decisions draw for draw with PyMIC RandomCrop + RandomFlip")
    path = os.path.join(ROOT, "tests", "golden", "datapath_decisions.json")
    with open(path, "w") as f:
        json.dump({"source": source, "patch": list(PATCH), "seed": SEED, "trials": trials}, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
