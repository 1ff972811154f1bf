"""CPU: the drop-in network's state_dict layout against the reference network's (stored under tests/golden/), and, where
the PyMIC source tree is present, INTEGRATION.md section 1 executed -- the
REFERENCE's own `pymic.net_run_dsbn.agent_seg.SegmentationAgent` (under the import stubs of oracle/gen_golden_fpl.py for
the packages its file-I/O side needs) takes the drop-in plugin objects through its own setters and factory methods:
set_net_dict -> create_network, set_loss_dict -> create_loss_calculator, set_inferer, state_dict round trip with the
reference's own network class, the test-time-dropout hook.  No arithmetic runs here (no GPU in this container); the
arithmetic behind these objects is what the -m gpu tests compare with the oracle."""
import os
import sys

import numpy as np
import pytest
import torch

REF = "/root/reference"
needs_reference = pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "PyMIC")),
                                     reason="runs the reference agent class: needs the PyMIC source tree")


@pytest.mark.parametrize("tag", ["vs_shipped", "configs2"])
def test_state_dict_layout_matches_the_reference_network(golden_dir, tag):
    """Checkpoints are interchangeable with the reference's: our state_dict has the reference UNet2D5_dsbn's 484 keys in
    the same order with the same shapes and dtypes (tests/golden/reference_state_dict.json), and a state_dict of that
    layout loads strictly."""
    import json
    from fplplus_b200.net import UNet2D5_dsbn
    with open(os.path.join(golden_dir, "reference_state_dict.json")) as f:
        g = json.load(f)["networks"][tag]
    net = UNet2D5_dsbn(dict(g["params"]))
    assert net.ft_chns == g["params"]["feature_chns"] and net.dims == g["params"]["conv_dims"]
    ours = [[k, list(v.shape), str(v.dtype).replace("torch.", "")] for k, v in net.state_dict().items()]
    assert len(ours) == 484 and ours == g["state_dict"]
    net.load_state_dict({k: torch.zeros(shape, dtype=getattr(torch, dt)) for k, shape, dt in g["state_dict"]}, strict=True)


@pytest.fixture(scope="module")
def ref_agent_cls():
    for p in (REF, os.path.join(REF, "PyMIC")):
        if p not in sys.path:
            sys.path.insert(0, p)
    from oracle.gen_golden_fpl import _install_stubs
    _install_stubs()
    from pymic.net_run_dsbn.agent_seg import SegmentationAgent
    return SegmentationAgent


@needs_reference
@pytest.mark.parametrize("cfg_name", ["vs_t1s_S.cfg", "vs_t1s_g.cfg", "vs_t1s_weights.cfg"])
def test_reference_agent_accepts_the_drop_in_plugins(ref_agent_cls, cfg_name):
    from pymic.util.parse_config import parse_config, synchronize_config
    import fplplus_b200
    from fplplus_b200.inferer import Inferer
    from fplplus_b200.net import UNet2D5_dsbn
    cfg = synchronize_config(parse_config(os.path.join(REF, "config_dual", "data_vs", cfg_name)))
    stage = "train" if cfg_name == "vs_t1s_S.cfg" else "test"
    agent = ref_agent_cls(cfg, stage)
    agent.set_net_dict(fplplus_b200.net_dict)            # agent_abstract.py:96-102
    agent.set_loss_dict(fplplus_b200.loss_dict)          # agent_abstract.py:104-110
    infer_cfg = dict(cfg["testing"])
    infer_cfg["class_num"] = cfg["network"]["class_num"]
    agent.set_inferer(Inferer(infer_cfg))                # agent_abstract.py:128-134
    agent.create_network()                               # agent_seg.py:82-105: looks net_type up in OUR dict
    assert isinstance(agent.net, UNet2D5_dsbn)
    assert agent.net.ft_chns == cfg["network"]["feature_chns"] and agent.net.dims == cfg["network"]["conv_dims"]
    sd = agent.net.state_dict()
    assert len(sd) == 484
    # strict state_dict exchange with the reference's own network class, both directions
    from pymic.net.net3d.unet2d5_dsbn import UNet2D5_dsbn as RefNet
    ref_net = RefNet(dict(cfg["network"]))
    ref_sd = ref_net.state_dict()
    assert list(ref_sd.keys()) == list(sd.keys())
    assert all(tuple(ref_sd[k].shape) == tuple(sd[k].shape) and ref_sd[k].dtype == sd[k].dtype for k in sd)
    agent.net.load_state_dict(ref_sd, strict=True)
    ref_net.load_state_dict(agent.net.state_dict(), strict=True)
    if stage == "train":
        agent.create_loss_calculator()                   # agent_seg.py:113-132
        assert type(agent.loss_calculator).__module__.startswith("fplplus_b200")
        agent.checkpoint = None
        agent.create_optimizer(agent.get_parameters_to_update())       # agent_abstract.py:320-337 on OUR parameters
        assert len(agent.optimizer.param_groups[0]["params"]) == len(list(agent.net.parameters()))
    else:
        # agent_seg.py:845-852: evaluation mode with test-time dropout finds real nn.Dropout children
        agent.net.eval()

        def test_time_dropout(m):
            if type(m) == torch.nn.Dropout:
                m.train()
        agent.net.apply(test_time_dropout)
        assert agent.net._first_dropout_level() == 2     # dropout = [0, 0, 0.3, 0.4, 0.5]
        assert agent.inferer.config["sliding_window_size"] == cfg["testing"]["sliding_window_size"]
    # the network refuses to run anywhere but on the GPU (no CPU fallback behind the plugin surface)
    with pytest.raises(RuntimeError):
        agent.net(torch.zeros(1, 1, 28, 32, 32), domain_label=torch.zeros(1, dtype=torch.long))
