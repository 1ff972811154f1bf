"""Device data path (SURVEY 8 f-3): RandomCrop / RandomFlip decisions against the reference transforms' stored decisions
(CPU) and the gather kernel against numpy slicing (GPU)."""
import json
import os

import numpy as np
import pytest
import torch

from oracle.gen_golden_datapath import TRIALS, record, volumes as _volumes


def test_crop_and_flip_decisions_follow_the_reference_transforms(golden_dir):
    """Same python `random` stream -> the same crop origin, flip axes and number of draws as pymic.transform.crop.RandomCrop
    (crop.py:213-234, foreground focus) followed by pymic.transform.flip.RandomFlip (flip.py:38-47), trial by trial against
    the decisions stored in tests/golden/datapath_decisions.json (oracle/gen_golden_datapath.py)."""
    with open(os.path.join(golden_dir, "datapath_decisions.json")) as f:
        g = json.load(f)
    assert len(g["trials"]) == TRIALS
    for got, want in zip(record(), g["trials"]):
        assert got == want, (got, want)


@pytest.mark.gpu
def test_gather_kernel_cuts_and_flips_like_numpy():
    from fplplus_b200.datapath import DevicePatchSampler, code_from_pixel_weight, pad_to
    patch = (28, 128, 128)
    vols = _volumes(3)
    smp = DevicePatchSampler(vols, patch, 4, "cuda:0", seed=11)
    padded = {v["name"]: (pad_to(v["image"], patch), pad_to(v["label"], patch, "constant"),
                          pad_to(code_from_pixel_weight(v["pixel_weight"]), patch, "constant"), v["image_weight"]) for v in vols}
    seen_flips = set()
    for _ in range(6):
        b = smp.next_batch()
        torch.cuda.synchronize()
        assert b["image"].shape == (4, 1) + patch and b["label"].dtype == torch.uint8 and b["pixel_weight"].shape == (4, 1) + patch
        img, lab, code, iw = b["image"].cpu().numpy(), b["label"].cpu().numpy(), b["pixel_weight"].cpu().numpy(), b["image_weight"].cpu().numpy()
        for i, (name, (d0, h0, w0), flip) in enumerate(smp.last_params):
            pi, pl, pc, w_img = padded[name]
            sl = (slice(d0, d0 + patch[0]), slice(h0, h0 + patch[1]), slice(w0, w0 + patch[2]))
            axes = [a for a, bit in ((-3, 1), (-2, 2), (-1, 4)) if flip & bit]
            ri, rl, rc = pi[(slice(None),) + sl], pl[sl], pc[sl]
            if axes:
                ri, rl, rc = np.flip(ri, axes), np.flip(rl, axes), np.flip(rc, axes)
            np.testing.assert_array_equal(img[i], ri)
            np.testing.assert_array_equal(lab[i], rl)
            np.testing.assert_array_equal(code[i, 0], rc)
            assert iw[i] == np.float32(w_img) and b["names"][i] == name
            seen_flips.add(flip)
    assert len(seen_flips) >= 3 and all(f & 1 == 0 for f in seen_flips)      # height / width flips only (flip_depth False)


@pytest.mark.gpu
def test_agent_trains_from_the_device_sampler():
    """The batch dicts of DevicePatchSampler (uint8 label / agreement code / per-sample image weight, all on the device)
    drive SegmentationAgent.train_step through eager steps, capture and replays; same loss as the PyMIC layout built on the
    host from the very same crops."""
    import bench
    from fplplus_b200.datapath import DevicePatchSampler
    from oracle import fpl_filter, synth
    from tests.test_gpu_step_parity import _agent
    patch = (16, 64, 64)
    vols = _volumes(5)
    a_dev, a_host = _agent(), _agent()
    s0 = DevicePatchSampler([dict(v, pixel_weight=None, code=None) for v in vols], patch, 2, "cuda:0", seed=3)
    s1 = DevicePatchSampler(vols, patch, 2, "cuda:0", seed=4)
    for it in range(6):
        b0, b1 = s0.next_batch(), s1.next_batch()
        # the same batches in PyMIC's loader layout (fp32 one-hot, folded fp32 weight), on the host
        h0 = {"image": b0["image"].cpu(), "label_prob": torch.from_numpy(synth.one_hot(b0["label"].cpu().numpy(), 2))}
        code, iw = b1["pixel_weight"].cpu().numpy(), b1["image_weight"].cpu().numpy()
        pw = np.stack([fpl_filter.set_weight_(iw[i], 0.5 * code[i].astype(np.float32)) for i in range(2)], 0).astype(np.float32)
        h1 = {"image": b1["image"].cpu(), "label_prob": torch.from_numpy(synth.one_hot(b1["label"].cpu().numpy(), 2)),
              "pixel_weight": torch.from_numpy(pw), "image_weight": torch.from_numpy(iw)}
        ld, _ = a_dev.train_step([b0, b1])
        lh, _ = a_host.train_step([h0, h1])
        ld, lh = float(ld), float(lh)
        print("step %d device-path loss %.6f host-layout loss %.6f" % (it, ld, lh))
        assert abs(ld - lh) <= 2e-3 * abs(lh)
    assert any(e["graph"] is not None for e in a_dev._graphs.values())
