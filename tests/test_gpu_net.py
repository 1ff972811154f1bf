"""GPU: the drop-in UNet2D5_dsbn / losses / Inferer against the golden vectors produced by the
reference's own modules (tests/golden, oracle/gen_golden.py) and against the CPU oracle.

Tolerances (BASELINE.json north_star): logits / loss within rel 1e-2 (bf16 conv path), argmax
labels >= 99.9 % voxel agreement end to end, fp32 elementwise pieces 1e-5 (see test_gpu_kernels)."""
import os

import numpy as np
import pytest
import torch

from oracle import synth
from oracle.gen_golden import NET_PARAMS, SHAPE
from tests._util import golden_voxels, max_rel, rel_l2

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _net(params=NET_PARAMS, seed=1):
    from fplplus_b200.net import UNet2D5_dsbn
    net = UNet2D5_dsbn(dict(params))
    sd = synth.synth_state_dict(params["in_chns"], params["feature_chns"], params["class_num"], params["num_domains"], seed=seed)
    net.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()}, strict=True)
    return net.to(DEV)


def _golden(golden_dir, name):
    return np.load(os.path.join(golden_dir, name))


def _label_agreement(a, b):
    return float((a.argmax(1) == b.argmax(1)).float().mean())


def _decided_agreement(out, ref, tol=1e-2):
    """Label agreement over the voxels the float tolerance can decide: a voxel whose reference
    top-2 logit margin is below ``tol`` * max|logit| (the rel-1e-2 logits tolerance of
    BASELINE.json) is a tie that an in-tolerance result may legitimately break either way.
    The synthetic-weight nets of these fixtures are untrained, so their margins crowd around 0;
    the >= 99.9 % end-to-end bar itself is checked on a trained net in
    test_trained_net_labels_and_dice_after_n_steps."""
    top2 = ref.topk(2, dim=1).values
    decided = (top2[:, 0] - top2[:, 1]) > tol * ref.abs().max()
    same = out.argmax(1) == ref.argmax(1)
    return float(same[decided].float().mean()), float(decided.float().mean())


def _check_labels(out, ref, overall=0.995):
    agree = _label_agreement(out, ref)
    dec, frac = _decided_agreement(out, ref)
    print(f"argmax agreement: all voxels {agree:.5f}, decided voxels {dec:.5f} ({frac:.3f} of the volume)")
    assert dec >= 0.999
    assert agree >= overall


@pytest.mark.parametrize("impl", ["tc", "direct"])
def test_eval_logits_match_reference(golden_dir, impl, monkeypatch):
    monkeypatch.setenv("FPL_CONV_IMPL", impl)
    g = _golden(golden_dir, "net_fwd_bwd.npz")
    net = _net().eval()
    x = torch.from_numpy(synth.synth_image(2, 1, SHAPE, seed=1)).to(DEV)
    for d in (0, 1):
        with torch.no_grad():
            out = net(x, domain_label=d * torch.ones(2, dtype=torch.long)).cpu()
        ref = torch.from_numpy(g[f"eval_logits_d{d}"])
        err = rel_l2(out, ref)
        agree = _label_agreement(out, ref)
        print(f"eval d{d} impl={impl}: rel_l2={err:.4f} max_rel={max_rel(out, ref):.4f} argmax agreement={agree:.5f}")
        assert err < 1e-2
        _check_labels(out, ref)


def test_train_step_matches_reference(golden_dir):
    """train-mode forward (batch statistics), weighted 0.5*Dice+0.5*CE, backward: logits, loss,
    running statistics and parameter gradients against the reference's autograd."""
    from fplplus_b200.loss import CombinedLoss
    from fplplus_b200.registry import loss_dict
    g = _golden(golden_dir, "net_fwd_bwd.npz")
    net = _net(dict(NET_PARAMS, dropout=[0.0] * 5)).train()
    x = torch.from_numpy(synth.synth_image(2, 1, SHAPE, seed=1)).to(DEV)
    lab = synth.synth_label(2, 2, SHAPE, seed=1)
    y = torch.from_numpy(synth.one_hot(lab, 2)).to(DEV)
    pw = torch.from_numpy(synth.synth_pixel_weight(lab, seed=1)[0]).to(DEV)
    logits = net(x, domain_label=torch.ones(2, dtype=torch.long))
    crit = CombinedLoss({"loss_type": ["DiceLoss", "CrossEntropyLoss"], "loss_weight": [0.5, 0.5]}, loss_dict)
    loss = crit({"prediction": logits, "ground_truth": y, "pixel_weight": pw})
    loss.backward()
    ref_logits = torch.from_numpy(g["train_logits_d1"])
    err = rel_l2(logits.detach().cpu(), ref_logits)
    print(f"train logits rel_l2={err:.4f}; loss {loss.item():.6f} vs {float(g['train_loss']):.6f}")
    assert err < 1e-2
    _check_labels(logits.detach().cpu(), ref_logits)
    np.testing.assert_allclose(loss.item(), float(g["train_loss"]), rtol=1e-2)
    named = dict(net.named_parameters())
    n_with_grad = sum(p.numel() for p in named.values() if p.grad is not None)
    assert n_with_grad == int(g["n_params_with_grad"])
    sd = net.state_dict()
    for k in g.files:
        if k.startswith("rm::"):
            assert max_rel(sd[k[4:] + ".running_mean"].cpu(), torch.from_numpy(g[k])) < 1e-2, k
        if k.startswith("rv::"):
            assert max_rel(sd[k[4:] + ".running_var"].cpu(), torch.from_numpy(g[k])) < 1e-2, k
        if k.startswith("nbt::"):
            assert int(sd[k[5:] + ".num_batches_tracked"]) == int(g[k]), k

    # gradients against the reference's fp32 autograd (golden): the error is the inherent effect of bf16
    # storage on this untrained net with an 8-voxel bottleneck (a 1e-2 forward perturbation flips PReLU
    # gates); bounded here, kernel parity proper is test_train_step_matches_bf16_emulation + the
    # per-kernel tests, training quality is test_trained_net_labels_and_dice_after_n_steps.
    worst = 0.0
    for k in g.files:
        if k.startswith("grad::"):
            name = k[6:]
            if name.endswith("conv3d_1.bias") or name.endswith("conv3d_2.bias"):
                # conv bias feeds BatchNorm: its true gradient is 0 (the reference holds rounding noise)
                assert float(named[name].grad.abs().max()) <= 1e-6, name
                continue
            if ".relu_" in name:
                continue
            ours, ref = named[name].grad.cpu(), torch.from_numpy(g[k])
            if ours.shape != ref.shape:
                ours = ours[:6, :6]
            e = rel_l2(ours, ref)
            cos = float((ours * ref).sum() / (ours.norm() * ref.norm()))
            worst = max(worst, e)
            print("grad vs fp32 reference %-36s rel_l2 %.4f cos %.4f" % (name, e, cos))
            assert cos > 0.95 and e < 0.3, (name, e, cos)
    print("worst gradient rel_l2 vs fp32 reference: %.4f" % worst)


@pytest.mark.parametrize("shape", [(16, 32, 32), (32, 64, 64)])
def test_train_step_matches_bf16_emulation(shape):
    """Whole-network kernel parity: the oracle run with the CUDA path's bf16 storage points made
    explicit (oracle/unet_dsbn.py, bf16=True) on the same inputs.  The first units agree to 1e-5..2e-4
    (rounding-boundary flips from fp32 summation order); the difference then grows chaotically through
    the BatchNorms of the small bottleneck, so the bounds below are per depth, not per ulp."""
    from oracle import losses, unet_dsbn
    from fplplus_b200.loss import CombinedLoss
    from fplplus_b200.registry import loss_dict
    params = dict(NET_PARAMS, dropout=[0.0] * 5)
    net = _net(params).train()
    x = torch.from_numpy(synth.synth_image(2, 1, shape, seed=21))
    lab = synth.synth_label(2, 2, shape, seed=21)
    y = torch.from_numpy(synth.one_hot(lab, 2))
    pw = torch.from_numpy(synth.synth_pixel_weight(lab, seed=21)[0])
    logits = net(x.to(DEV), domain_label=torch.zeros(2, dtype=torch.long))
    crit = CombinedLoss({"loss_type": ["DiceLoss", "CrossEntropyLoss"], "loss_weight": [0.5, 0.5]}, loss_dict)
    loss = crit({"prediction": logits, "ground_truth": y.to(DEV), "pixel_weight": pw.to(DEV)})
    loss.backward()
    def emulate(xin):
        st_ = unet_dsbn.to_torch_state(synth.synth_state_dict(), requires_grad=True)
        lg = unet_dsbn.forward(st_, xin, 0, params, bn_training=True, bf16=True)
        ls = losses.combined_loss(lg, y, pw, 0.5, 0.5)
        ls.backward()
        return st_, lg.detach(), ls.item()

    st, emu_logits, emu_loss = emulate(x)
    # the emulation's OWN sensitivity to an fp32-ulp-sized input perturbation: the yardstick for every
    # comparison below (a bf16-stored untrained net amplifies 1e-6 to ~5e-3 in the logits and to
    # 10-20 % in the gradients of the deep levels, see DESIGN.md "precision")
    noise = torch.from_numpy(np.random.Generator(np.random.PCG64(3)).standard_normal(x.shape).astype(np.float32))
    st2, emu2_logits, _ = emulate(x * (1 + 1e-6 * noise))
    e_log, s_log = rel_l2(logits.detach().cpu(), emu_logits), rel_l2(emu2_logits, emu_logits)
    print(f"shape {shape}: logits rel_l2={e_log:.5f} (emulation self-sensitivity {s_log:.5f}) "
          f"loss {loss.item():.6f} vs {emu_loss:.6f}")
    assert e_log < max(2 * s_log, 2e-3) and e_log < 1e-2
    np.testing.assert_allclose(loss.item(), emu_loss, rtol=2e-3)
    named = dict(net.named_parameters())
    slope_scale = max(float(v.grad.abs().max()) for k, v in st.items() if ".relu_" in k and v.grad is not None)
    worst = 0.0
    for name, p in named.items():
        if p.grad is None:
            assert st[name].grad is None or float(st[name].grad.abs().max()) == 0.0, name
            continue
        ours, emu, emu2 = p.grad.cpu(), st[name].grad, st2[name].grad
        if name.endswith("conv3d_1.bias") or name.endswith("conv3d_2.bias"):
            assert float(ours.abs().max()) <= 1e-6, name
            continue
        if ".relu_" in name:       # one scalar, a cancelling sum: absolute error against the slope-gradient scale
            e = float((ours - emu).abs().max()) / slope_scale
            sens = float((emu2 - emu).abs().max()) / slope_scale
        else:
            e, sens = rel_l2(ours, emu), rel_l2(emu2, emu)
        worst = max(worst, e)
        print("grad vs bf16-emulating oracle %-36s %.4f (self-sensitivity %.4f)" % (name, e, sens))
        assert e < max(2.5 * sens, 1e-2), (name, e, sens)
    print("worst gradient error vs bf16-emulating oracle: %.4f" % worst)


def test_dropout_mask_injection_matches_oracle():
    """train mode with dropout 0.3/0.4/0.5 on levels 2-4: the kernel consumes the oracle's masks."""
    from oracle import unet_dsbn
    params = dict(NET_PARAMS)
    net = _net(params).train()
    x_np = synth.synth_image(2, 1, SHAPE, seed=4)
    geo = [(16, 32, 32), (8, 16, 16), (4, 8, 8), (2, 4, 4), (1, 2, 2)]
    r = np.random.Generator(np.random.PCG64(99))
    masks_oracle, masks_dev = {}, {}
    ft = params["feature_chns"]
    for prefix, lvl in [("block%d.conv" % i, i) for i in range(5)] + [("up%d.conv" % k, 4 - k) for k in (1, 2, 3, 4)]:
        p = params["dropout"][lvl]
        if p <= 0:
            continue
        c = ft[lvl]
        m = torch.from_numpy(r.random((2, c) + geo[lvl]) >= p)
        masks_oracle[prefix] = m
        d, h, w = geo[lvl]
        masks_dev[prefix + "#1"] = m.reshape(2, c // 8, 8, d, h, w).permute(0, 3, 1, 4, 5, 2).contiguous().to(torch.uint8).to(DEV)
    net._dropout_masks = masks_dev
    with torch.no_grad():
        out = net(torch.from_numpy(x_np).to(DEV), domain_label=torch.zeros(2, dtype=torch.long)).cpu()
    st = unet_dsbn.to_torch_state(synth.synth_state_dict())
    with torch.no_grad():
        ref = unet_dsbn.forward(st, torch.from_numpy(x_np), 0, params, bn_training=True, masks=masks_oracle)
    err = rel_l2(out, ref)
    print("dropout mask-injection rel_l2", err)
    assert err < 1.5e-2
    _check_labels(out, ref, overall=0.99)


@pytest.mark.parametrize("fused", [False, True])
def test_two_domain_step_like_training_all(fused):
    """zero_grad; L=(L0+L1)/2 over two forwards; backward; Adam step -- vs the oracle trainer.
    ``fused=True``: torch's multi-tensor Adam does not bump tensor versions, the staged bf16 weight
    images must be invalidated explicitly (what the agent does) or step 2 would run on stale weights."""
    from oracle.train_step import OracleTrainer
    from fplplus_b200.loss import DiceLoss
    params = dict(NET_PARAMS, dropout=[0.0] * 5)
    net = _net(params).train()
    opt = torch.optim.Adam(net.parameters(), 1e-3, weight_decay=1e-5, fused=fused)
    oracle = OracleTrainer(synth.synth_state_dict(), params, lr=1e-3, weight_decay=1e-5)
    crit = DiceLoss({})
    batches = []
    for dmn in (0, 1):
        x = synth.synth_image(2, 1, SHAPE, seed=10 + dmn)
        lab = synth.synth_label(2, 2, SHAPE, seed=10 + dmn)
        batches.append((torch.from_numpy(x), torch.from_numpy(synth.one_hot(lab, 2)), None))
    trace = []
    for step in range(3):
        opt.zero_grad()
        total = 0.0
        for dmn, (x, y, _w) in enumerate(batches):
            out = net(x.to(DEV), domain_label=dmn * torch.ones(2, dtype=torch.long))
            total = total + crit({"prediction": out, "ground_truth": y.to(DEV)})
        loss = total / 2
        loss.backward()
        opt.step()
        if fused:
            net.invalidate_weight_images()
        ref_loss, _m, ref_logits = oracle.step(batches)
        print("step", step, "loss", loss.item(), "oracle", ref_loss)
        np.testing.assert_allclose(loss.item(), ref_loss, rtol=1e-2)
        trace.append((loss.item(), ref_loss))
    # the loss moves from step to step as the oracle's does (stale weights would freeze it)
    for (a0, r0), (a1, r1) in zip(trace[:-1], trace[1:]):
        assert abs((a1 - a0) - (r1 - r0)) <= 0.3 * abs(r1 - r0) + 1e-4, trace
    # after two Adam steps the weights still track the oracle's
    named = dict(net.named_parameters())
    for key in ("out_conv.weight", "up4.conv.conv3d_2.weight", "block0.conv.conv3d_1.weight", "up4.conv.relu_1.weight"):
        assert rel_l2(named[key].detach().cpu(), oracle.state[key].detach()) < 2e-2, key


def test_trained_net_labels_and_dice_after_n_steps():
    """BASELINE.json: 'end-to-end argmax labels agree on at least 99.9% of voxels' and 'Dice after a
    fixed number of steps is within 0.5 points'.  The oracle (training_all restatement) and the CUDA
    path both train 72 two-domain steps (Adam 2e-3, MultiStepLR [40,60] x0.2) from the same weights on
    the same synthetic ellipsoid task; then (i) each path's own trained net is scored by foreground
    hard Dice on 4 held-out batches per domain (must agree within 0.5 pt), (ii) the ORACLE-trained
    weights are loaded into the CUDA net and its eval labels are compared with the oracle's."""
    from oracle import losses, unet_dsbn
    from oracle.train_step import OracleTrainer
    from fplplus_b200.loss import CombinedLoss
    from fplplus_b200.registry import loss_dict
    steps = 72
    params = dict(NET_PARAMS, dropout=[0.0] * 5)
    net = _net(params).train()
    opt = torch.optim.Adam(net.parameters(), 2e-3, weight_decay=1e-5)
    sched = torch.optim.lr_scheduler.MultiStepLR(opt, [40, 60], 0.2)
    oracle = OracleTrainer(synth.synth_state_dict(), params, lr=2e-3, weight_decay=1e-5, lr_milestones=[40, 60],
                           lr_gamma=0.2, w_dice=0.5, w_ce=0.5)
    crit = CombinedLoss({"loss_type": ["DiceLoss", "CrossEntropyLoss"], "loss_weight": [0.5, 0.5]}, loss_dict)

    def batch(seed):
        lab = synth.synth_label(2, 2, SHAPE, seed=seed)
        # image = noise + a bright foreground, so the task is learnable in a few dozen steps
        x = synth.synth_image(2, 1, SHAPE, seed=seed) * 0.5 + (lab[:, None] > 0) * 2.0
        return torch.from_numpy(x.astype(np.float32)), torch.from_numpy(synth.one_hot(lab, 2))

    for step in range(steps):
        batches = [batch(100 + 2 * step + dmn) + (None,) for dmn in (0, 1)]
        opt.zero_grad()
        total = 0.0
        for dmn, (x, y, _w) in enumerate(batches):
            out = net(x.to(DEV), domain_label=dmn * torch.ones(2, dtype=torch.long))
            total = total + crit({"prediction": out, "ground_truth": y.to(DEV)})
        (total / 2).backward()
        opt.step()
        sched.step()
        ref_loss, _m, _l = oracle.step(batches)
    print("final train loss: cuda %.5f oracle %.5f" % (float(total.detach() / 2), ref_loss))
    held_out = [batch(s) for s in (999, 998, 997, 996)]
    st = {k: v.detach() for k, v in oracle.state.items()}

    def score(use_net):
        out = []
        for dmn in (0, 1):
            ds = []
            for xv, yv in held_out:
                with torch.no_grad():
                    if use_net:
                        z = net(xv.to(DEV), domain_label=dmn * torch.ones(2, dtype=torch.long)).cpu()
                    else:
                        z = unet_dsbn.forward(st, xv, dmn, params)
                ds.append(float(losses.hard_dice(z, yv)[1]))
            out.append(float(np.mean(ds)))
        return out

    net.eval()
    d_cuda, d_ref = score(True), score(False)
    print("foreground Dice after %d steps: cuda %s oracle %s" % (steps, d_cuda, d_ref))
    for a, b in zip(d_cuda, d_ref):
        assert abs(a - b) <= 0.005
    # (ii) identical (oracle-trained) weights -> labels
    net.load_state_dict({k: v.detach().clone() for k, v in oracle.state.items()}, strict=True)
    net.eval()
    for dmn in (0, 1):
        agree, n = 0.0, 0
        for xv, yv in held_out:
            with torch.no_grad():
                ours = net(xv.to(DEV), domain_label=dmn * torch.ones(2, dtype=torch.long)).cpu()
                ref = unet_dsbn.forward(st, xv, dmn, params)
            agree += _label_agreement(ours, ref)
            n += 1
            assert rel_l2(ours, ref) < 1e-2
            assert abs(float(losses.hard_dice(ours, yv)[1]) - float(losses.hard_dice(ref, yv)[1])) <= 0.005
        print("trained net d%d: label agreement %.5f" % (dmn, agree / n))
        assert agree / n >= 0.999


def test_25d_mode_matches_oracle():
    """conv_dims [2,2,3,3,3] (the shipped VS config): (1,3,3) convs, (1,2,2) pool / transposed conv."""
    from oracle import unet_dsbn
    params = dict(NET_PARAMS, conv_dims=[2, 2, 3, 3, 3], dropout=[0.0] * 5)
    net = _net(params).eval()
    x_np = synth.synth_image(1, 1, (8, 32, 32), seed=6)
    with torch.no_grad():
        out = net(torch.from_numpy(x_np).to(DEV), domain_label=torch.ones(1, dtype=torch.long)).cpu()
    st = unet_dsbn.to_torch_state(synth.synth_state_dict())
    with torch.no_grad():
        ref = unet_dsbn.forward(st, torch.from_numpy(x_np), 1, params)
    err = rel_l2(out, ref)
    print("2.5D rel_l2", err)
    assert err < 1e-2


def test_inferer_matches_reference_golden(golden_dir):
    from fplplus_b200.inferer import Inferer
    g = _golden(golden_dir, "inferer.npz")
    net = _net().eval()
    vol = torch.from_numpy(synth.synth_image(1, 1, (24, 48, 48), seed=9)).to(DEV)
    cfg = {"sliding_window_enable": True, "sliding_window_size": [16, 32, 32],
           "sliding_window_stride": [16, 32, 32], "tta_mode": 1, "class_num": 2}
    for d in (0, 1):
        with torch.no_grad():
            out = Inferer(dict(cfg)).run(net, vol, d * torch.ones(1, dtype=torch.long)).cpu()
        out = golden_voxels(out, g, f"net_tta1_d{d}")
        ref = torch.from_numpy(g[f"net_tta1_d{d}"])
        err = rel_l2(out, ref)
        print(f"inferer d{d}: rel_l2={err:.4f} agreement={_label_agreement(out, ref):.5f}")
        assert err < 1e-2
        _check_labels(out, ref)


def test_inferer_stitching_exact_with_toy_model(golden_dir):
    """Window enumeration / overlap counts / flips with a cheap torch 'model' (fp32 exact path)."""
    from fplplus_b200.inferer import Inferer
    g = _golden(golden_dir, "inferer.npz")
    gen = np.random.Generator(np.random.PCG64(11))
    wconv = torch.from_numpy(gen.standard_normal((3, 1, 3, 3, 3)).astype(np.float32)).to(DEV)

    class Toy(torch.nn.Module):
        def forward(self, x, domain_label=None):
            r = torch.nn.functional.conv3d(x, wconv, padding=1)
            ramp = torch.linspace(0, 1, x.shape[-1], device=x.device).view(1, 1, 1, 1, -1)
            return r + ramp * (1 + int(domain_label[0]))

    img = torch.from_numpy(synth.synth_image(1, 1, (20, 40, 44), seed=5)).to(DEV)
    torch.backends.cudnn.allow_tf32 = False
    for tta in (0, 1):
        cfg = {"sliding_window_enable": True, "sliding_window_size": [16, 32, 32],
               "sliding_window_stride": [8, 16, 32], "tta_mode": tta, "class_num": 3}
        out = Inferer(cfg).run(Toy(), img, torch.ones(1, dtype=torch.long)).cpu().numpy()
        np.testing.assert_allclose(golden_voxels(out, g, f"toy_tta{tta}"), g[f"toy_tta{tta}"], rtol=1e-4, atol=1e-5)


def test_strict_state_dict_round_trip_and_dropout_hook():
    net = _net()
    sd = net.state_dict()
    assert len(sd) == 484
    from fplplus_b200.net import UNet2D5_dsbn
    other = UNet2D5_dsbn(dict(NET_PARAMS))
    other.load_state_dict(sd, strict=True)
    # the agent's test-time-dropout hook (agent_seg.py:847-852) finds real nn.Dropout children
    net.eval()
    found = []

    def hook(m):
        if type(m) == torch.nn.Dropout:
            m.train()
            found.append(m)
    net.apply(hook)
    assert len(found) == 9
    x = torch.from_numpy(synth.synth_image(1, 1, SHAPE, seed=2)).to(DEV)
    torch.manual_seed(0)
    with torch.no_grad():
        a = net(x, domain_label=torch.ones(1, dtype=torch.long))
        b = net(x, domain_label=torch.ones(1, dtype=torch.long))
    torch.manual_seed(0)
    with torch.no_grad():
        a2 = net(x, domain_label=torch.ones(1, dtype=torch.long))
    assert not torch.equal(a, b)          # MC dropout is live in eval mode
    assert torch.equal(a, a2)             # and reproducible under torch.manual_seed
    with pytest.raises(ValueError):
        net(x[0], domain_label=torch.ones(1, dtype=torch.long))
    with pytest.raises(RuntimeError):
        net(x.cpu(), domain_label=torch.ones(1, dtype=torch.long))


def test_direct_gradient_delivery_equals_autograd_accumulation(monkeypatch):
    """Two domain passes through the same weights (training_all, agent_seg.py:459-495): p.grad as views of the master
    buffer filled by fpl_grad_scatter_add equals autograd's AccumulateGrad sum; zero_grad(set_to_none=True) starts a
    fresh step, a second backward without zero_grad accumulates."""
    from fplplus_b200.loss import CombinedLoss
    from fplplus_b200.registry import loss_dict
    params = dict(NET_PARAMS, dropout=[0.0] * 5)
    crit = CombinedLoss({"loss_type": ["DiceLoss", "CrossEntropyLoss"], "loss_weight": [0.5, 0.5]}, loss_dict)
    shape = (16, 32, 32)
    xs = [torch.from_numpy(synth.synth_image(2, 1, shape, seed=40 + d)).to(DEV) for d in (0, 1)]
    ys = [torch.from_numpy(synth.one_hot(synth.synth_label(2, 2, shape, seed=40 + d), 2)).to(DEV) for d in (0, 1)]

    def run(direct, repeats=1):
        monkeypatch.setenv("FPL_GRAD_DIRECT", direct)
        net = _net(params).train()
        for _ in range(repeats):
            total = 0
            for d in (0, 1):
                out = net(xs[d], domain_label=torch.full((2,), d, dtype=torch.long))
                total = total + crit({"prediction": out, "ground_truth": ys[d]})
            (total / 2).backward()
        torch.cuda.synchronize()
        return net, {k: (None if p.grad is None else p.grad.detach().cpu().clone()) for k, p in net.named_parameters()}

    net1, g1 = run("1")
    _, g0 = run("0")
    assert net1._master is not None
    n_views = 0
    for k in g0:
        assert (g0[k] is None) == (g1[k] is None), k
        if g0[k] is not None:
            n_views += 1
            scale = float(g0[k].abs().max()) + 1e-12
            assert float((g0[k] - g1[k]).abs().max()) <= 2e-3 * scale + 1e-7, k     # fp32 atomics: order differs
    assert n_views > 100
    # fresh step after zero_grad(set_to_none=True); BN running statistics moved, so only check the bookkeeping
    for p in net1.parameters():
        p.grad = None
    out = net1(xs[0], domain_label=torch.zeros(2, dtype=torch.long))
    crit({"prediction": out, "ground_truth": ys[0]}).backward()
    assert net1.block0.conv.bn3d1.bns[1].weight.grad is None and net1.block0.conv.bn3d1.bns[0].weight.grad is not None
    # accumulation without zero_grad: two identical steps give twice the gradient (same BN batch statistics)
    _, g2 = run("1", repeats=2)
    k = "out_conv.weight"
    assert float((g2[k] - 2 * g1[k]).abs().max()) <= 2e-2 * float(g1[k].abs().max())


@pytest.mark.parametrize("mc_dropout", [False, True])
@pytest.mark.parametrize("dims", [[3, 3, 3, 3, 3], [2, 2, 3, 3, 3]])
def test_inference_epilogue_fusion_matches_two_kernel_path(mc_dropout, dims, monkeypatch):
    """No-grad forwards with BatchNorm in eval mode run conv + BN + PReLU (+ dropout) as ONE kernel (EpiAct).  Same logits
    as conv -> fpl_dsbn_bn_act_fwd within the bf16 tolerance (the fused form skips one bf16 rounding), the SAME dropout
    mask (Philox positions), and both within rel 1e-2 of the fp32 oracle."""
    from oracle import unet_dsbn
    params = dict(NET_PARAMS, conv_dims=dims, dropout=[0.0, 0.0, 0.3, 0.4, 0.5])
    shape = (16, 32, 32)
    x = torch.from_numpy(synth.synth_image(2, 1, shape, seed=77))
    outs = {}
    for fuse in ("1", "0"):
        monkeypatch.setenv("FPL_EVAL_FUSE", fuse)
        net = _net(params).eval()
        net.cuda_graphs = False
        if mc_dropout:
            for m in net.modules():
                if type(m) == torch.nn.Dropout:
                    m.train()
        torch.manual_seed(5)
        with torch.no_grad():
            outs[fuse] = net(x.to(DEV), domain_label=torch.ones(2, dtype=torch.long)).cpu()
    err = rel_l2(outs["1"], outs["0"])
    print("fused vs two-kernel logits rel_l2 %.2e (mc_dropout=%s)" % (err, mc_dropout))
    assert err < 6e-3
    if not mc_dropout:
        sd = synth.synth_state_dict(params["in_chns"], params["feature_chns"], params["class_num"], params["num_domains"], seed=1)
        ref = unet_dsbn.forward(unet_dsbn.to_torch_state(sd), x, 1, params, bn_training=False).detach()
        assert rel_l2(outs["1"], ref) < 1e-2 and rel_l2(outs["0"], ref) < 1e-2
        assert rel_l2(outs["1"], ref) <= rel_l2(outs["0"], ref) * 1.25


@pytest.mark.parametrize("graphs", [False, True])
def test_forward_mc_equals_consecutive_mc_dropout_forwards(graphs):
    """K MC-dropout passes of one input through forward_mc (dropout-free encoder levels computed once) are bit-identical
    to K consecutive forward calls drawing the same seeds (agent_seg.py:897-911 runs K full passes)."""
    params = dict(NET_PARAMS, dropout=[0.0, 0.0, 0.3, 0.4, 0.5])
    net = _net(params).eval()
    net.cuda_graphs = graphs
    for m in net.modules():
        if type(m) == torch.nn.Dropout:
            m.train()
    assert net._first_dropout_level() == 2
    x = torch.from_numpy(synth.synth_image(2, 1, (16, 32, 32), seed=91)).to(DEV)
    dom = torch.ones(2, dtype=torch.long)
    K = 4
    with torch.no_grad():
        for _ in range(3):                      # eager first sight, capture, replay
            torch.manual_seed(11)
            sep = [net(x, domain_label=dom).clone() for _ in range(K)]
            torch.manual_seed(11)
            mc = net.forward_mc(x, dom, K)
            assert len(mc) == K
            for a, b in zip(sep, mc):
                assert torch.equal(a, b)
            assert not torch.equal(mc[0], mc[1])            # different dropout masks per pass


def test_inferer_mc_passes_without_dropout_equal_single_run():
    """Inferer.run(mc_passes=K) with every dropout in eval mode: K identical volumes equal to the plain run (window
    stitching, visit counts and TTA shared between the passes)."""
    from fplplus_b200.inferer import Inferer
    net = _net(dict(NET_PARAMS, dropout=[0.0, 0.0, 0.3, 0.4, 0.5])).eval()
    vol = torch.from_numpy(synth.synth_image(1, 1, (24, 48, 64), seed=92)).to(DEV)
    inf = Inferer({"class_num": 2, "sliding_window_enable": True, "sliding_window_size": [16, 32, 32],
                   "sliding_window_stride": [8, 32, 32], "tta_mode": 1})
    one = torch.ones(1, dtype=torch.long)
    with torch.no_grad():
        single = inf.run(net, vol, one)
        many = inf.run(net, vol, one, mc_passes=3)
    assert isinstance(many, list) and len(many) == 3
    for m in many:
        assert float((m - single).abs().max()) <= 1e-5 * float(single.abs().max())


@pytest.mark.parametrize("dims", [[3, 3, 3, 3, 3], [2, 2, 3, 3, 3]])
def test_bilinear_mode_matches_oracle(dims):
    """`bilinear = True` (SURVEY 8f-1): 1x1 projection + trilinear / bilinear x2 up-sampling (align_corners) instead of the
    transposed conv.  Eval logits against the fp32 oracle; one train-mode backward: the 1x1 convs (not the transposed
    convs) receive gradients that point the same way as the oracle's."""
    from oracle import unet_dsbn, losses
    from fplplus_b200.loss import CombinedLoss
    from fplplus_b200.registry import loss_dict
    params = dict(NET_PARAMS, conv_dims=dims, bilinear=True, dropout=[0.0] * 5)
    shape = (16, 32, 32)
    net = _net(params).eval()
    x_np = synth.synth_image(2, 1, shape, seed=61)
    dom = torch.ones(2, dtype=torch.long)
    sd = synth.synth_state_dict()
    with torch.no_grad():
        out = net(torch.from_numpy(x_np).to(DEV), domain_label=dom).cpu()
        ref = unet_dsbn.forward(unet_dsbn.to_torch_state(sd), torch.from_numpy(x_np), 1, params)
    err = rel_l2(out, ref)
    print("bilinear eval rel_l2", err)
    assert err < 1e-2
    # train-mode step
    net.train()
    lab = synth.synth_label(2, 2, shape, seed=61)
    y = torch.from_numpy(synth.one_hot(lab, 2))
    crit = CombinedLoss({"loss_type": ["DiceLoss", "CrossEntropyLoss"], "loss_weight": [0.5, 0.5]}, loss_dict)
    logits = net(torch.from_numpy(x_np).to(DEV), domain_label=dom)
    loss = crit({"prediction": logits, "ground_truth": y.to(DEV)})
    loss.backward()
    st = unet_dsbn.to_torch_state(sd, requires_grad=True)
    ref_logits = unet_dsbn.forward(st, torch.from_numpy(x_np), 1, params, bn_training=True)
    ref_loss = losses.combined_loss(ref_logits, y, None, 0.5, 0.5)
    ref_loss.backward()
    assert abs(float(loss.detach()) - float(ref_loss.detach())) <= 1e-2 * abs(float(ref_loss.detach()))
    named = dict(net.named_parameters())
    for k in range(1, 5):
        up_dim3 = dims[4 - k] == 3
        proj = "up%d.%s" % (k, "conv3d" if up_dim3 else "conv2d")
        trans = "up%d.%s" % (k, "trans3d" if up_dim3 else "trans2d")
        assert named[trans + ".weight"].grad is None
        for leaf in (".weight", ".bias"):
            ours, want = named[proj + leaf].grad.cpu().flatten(), st[proj + leaf].grad.flatten()
            cos = float(torch.nn.functional.cosine_similarity(ours, want, dim=0))
            print(proj + leaf, "cosine", cos, "norm ratio", float(ours.norm() / want.norm()))
            assert cos > 0.97 and 0.8 < float(ours.norm() / want.norm()) < 1.25
    cos = float(torch.nn.functional.cosine_similarity(named["out_conv.weight"].grad.cpu().flatten(),
                                                      st["out_conv.weight"].grad.flatten(), dim=0))
    assert cos > 0.99
