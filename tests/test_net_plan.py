"""The kernel plan of UNet2D5_dsbn (net._plan): the kernel every launch site of a pass runs and the weight images they
read, one entry per input geometry.  The CPU tests build the plan without a device (sm_100 passed in; the library's
image-size queries answer on the host); the GPU test checks where the training step stages those images."""
import collections.abc
import os

import numpy as np
import pytest
import torch

from fplplus_b200.net import UNet2D5_dsbn

BENCH = {"net_type": "UNet2D5_dsbn", "num_domains": 2, "class_num": 2, "in_chns": 1,
         "feature_chns": [16, 32, 64, 128, 256], "conv_dims": [3, 3, 3, 3, 3],
         "dropout": [0.0, 0.0, 0.3, 0.4, 0.5], "bilinear": False}
VS = dict(BENCH, feature_chns=[32, 64, 128, 256, 512], conv_dims=[2, 2, 3, 3, 3])


def _plan(params, shape, grad=True):
    net = UNet2D5_dsbn(dict(params))
    return net, net._plan(shape[0], net._geometry(shape), grad, True)


def _level_units(net, lvl):
    """The conv units that run at encoder / decoder level ``lvl`` (0 = full resolution)."""
    units = list(net._down_units[lvl])
    if lvl < 4:
        units += list(net._up_units[3 - lvl])
    return [u.name for u in units]


class _NoEnviron(collections.abc.Mapping):
    def __getitem__(self, key):
        raise AssertionError("environment read after construction: %s" % key)

    def __iter__(self):
        raise AssertionError("environment read after construction")

    def __len__(self):
        raise AssertionError("environment read after construction")


def test_benchmark_configuration_plan(monkeypatch):
    from fplplus_b200 import lib
    lib.load()
    net = UNet2D5_dsbn(dict(BENCH))
    shape = (4, 1, 32, 128, 128)
    with monkeypatch.context() as m:
        m.setattr(os, "environ", _NoEnviron())
        plan = net._plan(4, net._geometry(shape), True, True)
        infer = net._plan(4, net._geometry(shape), False, True)
    assert net._plan(4, net._geometry(shape), True, True) is plan          # memoised
    assert plan.fwd["block0.conv#1"] == "stem_direct" and plan.wgrad["block0.conv#1"] == "stem_direct"
    for lvl in (0, 1):
        for name in _level_units(net, lvl):
            if name != "block0.conv#1":
                assert plan.fwd[name] == "dfold" and plan.dgrad[name] == "dfold", name
    for lvl in (3, 4):
        for name in _level_units(net, lvl):
            assert plan.fwd[name] == "tc" and plan.dgrad[name] == "tc", name
    assert "block0.conv#1" not in plan.dgrad
    assert set(v for k, v in plan.wgrad.items() if k != "block0.conv#1") == {"tapmajor"}
    assert plan.head == "cc" and plan.up == ["tc"] * 4
    assert not any(kind == "stem" for kind, *_ in plan.images)           # the training stem reads the fp32 weights
    # no-grad forwards of the same geometry: the patch-tensor stem, forward images only
    assert infer.fwd["block0.conv#1"] == "stem_patch" and not infer.dgrad and not infer.wgrad
    assert infer.images[0][0] == "stem" and all(t == 0 for _, _, t, _ in infer.images)


def test_shipped_vs_configuration_plan():
    net, plan = _plan(VS, (4, 1, 28, 128, 128))
    # the stem of conv_dims[0] = 2 is a 2-D conv: fpl_stem_conv_fwd, and the tensor-core wgrad on one packed group
    assert plan.fwd["block0.conv#1"] == "stem_cc" and plan.wgrad["block0.conv#1"] == "stem_c8"
    for lvl in (0, 1):                                                      # 2.5-D levels: k(1,3,3), never depth-folded
        for name in _level_units(net, lvl):
            if name != "block0.conv#1":
                assert plan.fwd[name] == "tc" and plan.dgrad[name] == "tc", name
    assert "dfold" not in plan.fwd.values() and plan.head == "cc"
    # ft0 = 32 with a 3-D stem trains through the patch-tensor stem
    _, plan3 = _plan(dict(VS, conv_dims=[3] * 5), (4, 1, 32, 128, 128))
    assert plan3.fwd["block0.conv#1"] == "stem_patch" and plan3.wgrad["block0.conv#1"] == "stem_patch"
    assert plan3.images[0][0] == "stem"


@pytest.mark.parametrize("over,shape", [({"feature_chns": [64, 128, 256, 256, 512]}, (2, 1, 16, 64, 64)),
                                        ({"conv_dims": [2, 2, 2, 2, 2]}, (2, 1, 1, 64, 64))])
def test_zero_padded_head_serves_other_widths_and_single_planes(over, shape):
    net, plan = _plan(dict(BENCH, **over), shape)
    assert plan.head == "tc"
    assert [(kind, t) for kind, conv, t, _ in plan.images if conv is net._head] == [("tc", 0), ("tc", 1)]


def test_direct_convolutions_keep_tap_major_weight_gradients(monkeypatch):
    monkeypatch.setenv("FPL_CONV_IMPL", "direct")
    net, plan = _plan(BENCH, (4, 1, 32, 128, 128))
    assert plan.fwd["block0.conv#1"] == "stem_cc" and plan.wgrad["block0.conv#1"] == "stem_cc"
    assert set(v for k, v in plan.fwd.items() if k != "block0.conv#1") == {"direct"}
    assert set(plan.dgrad.values()) == {"direct"}
    assert set(v for k, v in plan.wgrad.items() if k != "block0.conv#1") == {"tapmajor"}
    assert plan.head == "direct" and plan.up == ["direct"] * 4 and plan.images == []


def test_bilinear_mode_projects_before_upsampling():
    net, plan = _plan(dict(BENCH, bilinear=True), (2, 1, 16, 64, 64))
    assert plan.up == ["proj"] * 4
    for pu in net._proj_units:
        assert [t for kind, conv, t, _ in plan.images if conv is pu.conv] == [0, 1]


@pytest.mark.gpu
def test_dual_stream_step_stages_every_weight_image_before_the_fork(tmp_path):
    """The two domain passes of a training step run on two streams; every weight image either pass reads is staged on
    the main stream before the side stream forks from it, also in the first step of a fresh network."""
    from oracle import synth
    from fplplus_b200 import lib
    from fplplus_b200.agent import SegmentationAgent
    shape, bs = (16, 32, 32), 2
    tr = {"train_fpl_uda": True, "dual": True, "dis": False, "val_t1": False, "val_t2": False, "gpus": [0],
          "loss_type": ["DiceLoss", "CrossEntropyLoss"], "loss_weight": [0.5, 0.5], "optimizer": "Adam",
          "learning_rate": 1e-4, "momentum": 0.9, "weight_decay": 1e-5, "lr_scheduler": "MultiStepLR", "lr_gamma": 0.5,
          "lr_milestones": [100], "iter_start": 0, "iter_max": 10, "iter_valid": 10, "ckpt_save_dir": str(tmp_path)}
    cfg = {"dataset": {"tensor_type": "float", "train_batch_size": bs}, "network": dict(BENCH, dropout=[0.0] * 5),
           "training": tr, "testing": {"gpus": [0]}}
    ag = SegmentationAgent(cfg, "train")
    ag.create_network()
    ag._pick_device("training")
    ag.net.to(ag.device)
    ag.create_optimizer(ag.get_parameters_to_update())
    ag.create_loss_calculator()
    ag.net.train()
    assert ag.dual_stream
    batches = []
    for d in (0, 1):
        lab = synth.synth_label(bs, 2, shape, seed=60 + d)
        batches.append({"image": torch.from_numpy(synth.synth_image(bs, 1, shape, seed=60 + d).astype(np.float32)),
                        "label_prob": torch.from_numpy(synth.one_hot(lab, 2))})
    events = []

    class SideStream(torch.cuda.Stream):
        def wait_stream(self, stream):
            events.append("fork")
            super().wait_stream(stream)

    ag._side_stream = SideStream()
    lib.set_call_timer(lambda name, args: events.append(name))
    try:
        ag.train_step(batches)
        torch.cuda.synchronize()
    finally:
        lib.set_call_timer(None)
    fork = events.index("fork")
    preps = [i for i, name in enumerate(events) if "prep_weight" in name]
    assert any("dfold_prep_weight" in events[i] for i in preps)
    assert preps and max(preps) < fork, [events[i] for i in preps if i > fork]
    assert any(name.startswith("fpl_conv3d_tc_dfold") for name in events[fork:])
