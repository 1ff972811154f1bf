"""CPU: the oracle restatement against the golden vectors produced by the
reference's own modules (oracle/gen_golden.py) and against the reference's
shipped artefacts (tests/golden/fpl_image_weights.json)."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import fpl_filter, inferer, losses, synth, unet_dsbn
from oracle.gen_golden import NET_PARAMS, SHAPE
from oracle.gen_golden_fpl import CASES, fpl_case_logits
from tests._util import golden_voxels


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name), allow_pickle=False)


@pytest.fixture(autouse=True)
def _recording_thread_count():
    """The golden vectors were recorded with 8 intra-op threads.  torch's CPU backward splits its float32 weight-gradient
    reductions by thread count, so the oracle runs with the same split here (the forward does not depend on it)."""
    saved = torch.get_num_threads()
    torch.set_num_threads(8)
    yield
    torch.set_num_threads(saved)


# conv biases that feed a training-mode BatchNorm: their gradient is exactly zero, so what backward computes for them
# (here and in the golden file) is float32 rounding noise whose size depends on the host's thread count and vector width
_BN_FED_BIASES = ("conv3d_1.bias", "conv3d_2.bias")


def _assert_rounding_level(st, name, ref):
    """Our gradient of ``name`` and the reference's both vanish next to the gradient of the same conv's weight."""
    scale = st[name[:-len("bias")] + "weight"].grad.double().norm().item()
    assert st[name].grad.double().norm().item() <= 1e-4 * scale, name
    assert float(np.linalg.norm(ref)) <= 1e-4 * scale, name


def test_state_dict_spec_matches_reference_count():
    sd = synth.synth_state_dict()
    assert len(sd) == 484                                  # SURVEY §8b (PROBE)
    n_param = sum(v.size for k, v in sd.items() if "running_" not in k and "num_batches" not in k)
    assert n_param == 7685300


def test_net_eval_logits(golden_dir):
    g = _load(golden_dir, "net_fwd_bwd.npz")
    x = torch.from_numpy(synth.synth_image(2, 1, SHAPE, seed=1))
    for d in (0, 1):
        st = unet_dsbn.to_torch_state(synth.synth_state_dict())
        with torch.no_grad():
            out = unet_dsbn.forward(st, x, d, NET_PARAMS, bn_training=False).numpy()
        np.testing.assert_allclose(out, g[f"eval_logits_d{d}"], rtol=1e-4, atol=1e-5)


def test_net_train_step_grads_and_running_stats(golden_dir):
    g = _load(golden_dir, "net_fwd_bwd.npz")
    x = torch.from_numpy(synth.synth_image(2, 1, SHAPE, seed=1))
    lab = synth.synth_label(2, 2, SHAPE, seed=1)
    y = torch.from_numpy(synth.one_hot(lab, 2))
    pw = torch.from_numpy(synth.synth_pixel_weight(lab, seed=1)[0])
    st = unet_dsbn.to_torch_state(synth.synth_state_dict(), requires_grad=True)
    p0 = dict(NET_PARAMS, dropout=[0.0] * 5)
    logits = unet_dsbn.forward(st, x, 1, p0, bn_training=True)
    loss = losses.combined_loss(logits, y, pw, 0.5, 0.5)
    loss.backward()
    np.testing.assert_allclose(logits.detach().numpy(), g["train_logits_d1"], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(loss.item(), float(g["train_loss"]), rtol=1e-6)
    n_with_grad = sum(v.numel() for v in st.values() if v.requires_grad and v.grad is not None)
    assert n_with_grad == int(g["n_params_with_grad"])
    for k in g.files:
        if k.startswith(("grad::", "gradnorm::")) and k.endswith(_BN_FED_BIASES):
            _assert_rounding_level(st, k.split("::", 1)[1], g[k])
            continue
        if k.startswith("grad::"):
            name = k[6:]
            ours = st[name].grad.numpy()
            ref = g[k]
            if ours.shape != ref.shape:
                ours = ours[:6, :6]
            np.testing.assert_allclose(ours, ref, rtol=2e-3, atol=1e-7, err_msg=name)
        if k.startswith("gradnorm::"):
            ours = st[k[10:]].grad.double().norm().item()
            np.testing.assert_allclose(ours, float(g[k]), rtol=1e-4)
        if k.startswith("rm::"):
            np.testing.assert_allclose(st[k[4:] + ".running_mean"].numpy(), g[k], rtol=1e-5, atol=1e-6)
        if k.startswith("rv::"):
            np.testing.assert_allclose(st[k[4:] + ".running_var"].numpy(), g[k], rtol=1e-5, atol=1e-6)
        if k.startswith("nbt::"):
            assert int(st[k[5:] + ".num_batches_tracked"]) == int(g[k])


def test_losses_value_and_grad(golden_dir):
    g = _load(golden_dir, "loss.npz")
    for tag in ("c2", "c5"):
        z, y, pw = g[f"{tag}_logits"], g[f"{tag}_onehot"], g[f"{tag}_pw"]
        for wt in ("u", "w"):
            w = torch.from_numpy(pw) if wt == "w" else None
            for name, fn, wd, wc in (("dice", losses.dice_loss, 1.0, 0.0), ("ce", losses.ce_loss, 0.0, 1.0)):
                zt = torch.from_numpy(z).requires_grad_(True)
                val = fn(zt, torch.from_numpy(y), w)
                val.backward()
                np.testing.assert_allclose(val.item(), float(g[f"{tag}_{name}_{wt}_loss"]), rtol=1e-6)
                np.testing.assert_allclose(zt.grad.numpy(), g[f"{tag}_{name}_{wt}_grad"], rtol=1e-4, atol=1e-9)
                # closed form (float64) agrees with the reference too
                lv, dz, _ = losses.dice_ce_closed_form(z, y, pw if wt == "w" else None, wd, wc)
                np.testing.assert_allclose(lv, float(g[f"{tag}_{name}_{wt}_loss"]), rtol=2e-6)
                np.testing.assert_allclose(dz, g[f"{tag}_{name}_{wt}_grad"], rtol=2e-3, atol=1e-9)


def test_inferer_toy_and_net(golden_dir):
    g = _load(golden_dir, "inferer.npz")
    gen = np.random.Generator(np.random.PCG64(11))
    wconv = torch.from_numpy(gen.standard_normal((3, 1, 3, 3, 3)).astype(np.float32))

    def toy(x):
        r = torch.nn.functional.conv3d(x, wconv, padding=1)
        return r + torch.linspace(0, 1, x.shape[-1]).view(1, 1, 1, 1, -1) * 2

    img = torch.from_numpy(synth.synth_image(1, 1, (20, 40, 44), seed=5))
    for tta in (0, 1):
        cfg = {"sliding_window_enable": True, "sliding_window_size": [16, 32, 32],
               "sliding_window_stride": [8, 16, 32], "tta_mode": tta}
        out = inferer.run(toy, img, 3, cfg).numpy()
        np.testing.assert_allclose(golden_voxels(out, g, f"toy_tta{tta}"), g[f"toy_tta{tta}"], rtol=1e-5, atol=1e-6)
    vol = torch.from_numpy(synth.synth_image(1, 1, (24, 48, 48), seed=9))
    cfg = {"sliding_window_enable": True, "sliding_window_size": [16, 32, 32],
           "sliding_window_stride": [16, 32, 32], "tta_mode": 1}
    st = unet_dsbn.to_torch_state(synth.synth_state_dict())
    with torch.no_grad():
        out = inferer.run(lambda im: unet_dsbn.forward(st, im, 1, NET_PARAMS), vol, 2, cfg).numpy()
    np.testing.assert_allclose(golden_voxels(out, g, "net_tta1_d1"), g["net_tta1_d1"], rtol=1e-4, atol=1e-5)


def test_window_enumeration_matches_survey_probe():
    starts, win = inferer.window_starts([48, 256, 256], [32, 128, 128], [32, 128, 128])
    assert len(starts) == 8 and win == [32, 128, 128]
    assert sorted(set(s[0] for s in starts)) == [0, 16]
    starts, _ = inferer.window_starts([40, 256, 256], [28, 128, 128], [28, 128, 128])
    assert sorted(set(s[0] for s in starts)) == [0, 12]
    assert inferer.window_starts([16, 32, 32], [32, 128, 128], [32, 128, 128])[0] is None


def test_fpl_infer_branch_against_reference_agent(golden_dir):
    """values/order produced by the reference's own SegmentationAgent.infer()."""
    g = _load(golden_dir, "fpl_infer.npz")
    table = {}
    for name, seed, conf in CASES:
        r = fpl_filter.mc_uncertainty(fpl_case_logits(seed, confident=conf))
        table[name] = [r["uncer_one"]]
    srt = fpl_filter.sort_uncertainty(table)
    assert [n for _v, n in srt] == [str(n) for n in g["names"]]
    np.testing.assert_allclose([float(v[0]) for v, _n in srt], g["values"], rtol=1e-12)
    assert [isinstance(v[0], int) for v, _n in srt] == list(g["is_sentinel"])


def test_image_weight_map_against_shipped_artefacts(golden_dir):
    with open(os.path.join(golden_dir, "fpl_image_weights.json")) as f:
        g = json.load(f)
    assert g["names"] == g["csv_names"]                      # same ascending order
    u = np.asarray(g["uncertainty"])
    assert np.all(np.diff(u) >= 0)
    assert sum(g["sentinel"]) == 6 and all(g["sentinel"][-6:])
    # sentinel ties are ordered by name string (python tuple ordering)
    tail = g["names"][-6:]
    assert tail == sorted(tail)
    w = fpl_filter.image_weights(u)
    np.testing.assert_allclose(w, np.asarray(g["csv_image_weight"]), rtol=0, atol=1e-12)
    # and re-sorting shuffled pairs reproduces the shipped order
    rng = np.random.Generator(np.random.PCG64(0))
    perm = rng.permutation(len(u))
    table = {g["names"][i]: [1 if g["sentinel"][i] else u[i]] for i in perm}
    assert [n for _v, n in fpl_filter.sort_uncertainty(table)] == g["names"]


def test_agreement_weight_and_set_weight():
    rng = np.random.Generator(np.random.PCG64(3))
    a = rng.integers(0, 2, (6, 9, 11)).astype(np.uint8)
    b = rng.integers(0, 2, (6, 9, 11)).astype(np.uint8)
    w = fpl_filter.agreement_weight(a, b)
    assert w.dtype == np.float64
    np.testing.assert_array_equal(w, np.where(a == b, 1.0, 0.5))
    np.testing.assert_array_equal(w, fpl_filter.agreement_weight_multiclass(a, b))
    folded = fpl_filter.set_weight_(0.37, w.astype(np.float32))
    np.testing.assert_allclose(folded, np.where(a == b, np.float32(0.37), 0.0), rtol=1e-7)


def test_pseudo_label_is_argmax():
    rng = np.random.Generator(np.random.PCG64(5))
    z = rng.standard_normal((1, 5, 4, 6, 7)).astype(np.float32)
    np.testing.assert_array_equal(fpl_filter.pseudo_label(z), z.argmax(1).astype(np.uint8))


def test_bf16_emulating_mode_tracks_the_fp32_oracle():
    """oracle.unet_dsbn.forward(bf16=True) makes the CUDA path's storage roundings explicit (kernel parity is
    asserted against it on the GPU); on CPU: it stays within the bf16 tolerance of the fp32 restatement, its
    gradients exist for exactly the same parameters, and conv-bias gradients (biases feeding BatchNorm) vanish."""
    from oracle import losses, synth, unet_dsbn
    from oracle.gen_golden import NET_PARAMS
    params = dict(NET_PARAMS, dropout=[0.0] * 5)
    shape = (16, 32, 32)
    x = torch.from_numpy(synth.synth_image(2, 1, shape, seed=5))
    lab = synth.synth_label(2, 2, shape, seed=5)
    y = torch.from_numpy(synth.one_hot(lab, 2))
    res = {}
    for bf in (False, True):
        st = unet_dsbn.to_torch_state(synth.synth_state_dict(), requires_grad=True)
        lg = unet_dsbn.forward(st, x, 0, params, bn_training=True, bf16=bf)
        losses.combined_loss(lg, y, None, 0.5, 0.5).backward()
        res[bf] = (lg.detach(), st)
    a, b = res[True][0], res[False][0]
    assert float((a - b).norm() / b.norm()) < 2e-2
    g_emu = {k for k, v in res[True][1].items() if v.requires_grad and v.grad is not None and float(v.grad.abs().max()) > 0}
    g_ref = {k for k, v in res[False][1].items() if v.requires_grad and v.grad is not None and float(v.grad.abs().max()) > 0}
    bias_keys = {k for k in g_ref if k.endswith("conv3d_1.bias") or k.endswith("conv3d_2.bias")}
    assert g_emu | bias_keys == g_ref | bias_keys
    for k in bias_keys & set(res[True][1]):
        gb = res[True][1][k].grad
        assert gb is None or float(gb.abs().max()) < 1e-4
    cos = torch.nn.functional.cosine_similarity(res[True][1]["up4.conv.conv3d_2.weight"].grad.flatten(),
                                                res[False][1]["up4.conv.conv3d_2.weight"].grad.flatten(), dim=0)
    assert float(cos) > 0.99


@pytest.mark.parametrize("tag", ["d25", "bil3d", "bil25"])
def test_network_modes_against_reference(golden_dir, tag):
    """The oracle's 2.5-D (`conv_dims` with 2) and `bilinear = True` branches against the REFERENCE network run in those
    modes (oracle/gen_golden_modes.py): eval logits, train-mode logits / loss, gradient prefixes and norms, and the number
    of parameters that receive gradients."""
    from oracle.gen_golden_modes import GRADS, MODES, SHAPE as MSHAPE
    g = _load(golden_dir, "net_modes.npz")
    params = dict(NET_PARAMS, dropout=[0.0] * 5, **MODES[tag])
    x = torch.from_numpy(synth.synth_image(1, 1, MSHAPE, seed=7))
    y = torch.from_numpy(synth.one_hot(synth.synth_label(1, 2, MSHAPE, seed=7), 2))
    st = unet_dsbn.to_torch_state(synth.synth_state_dict())
    with torch.no_grad():
        out = unet_dsbn.forward(st, x, 1, params, bn_training=False).numpy()
    np.testing.assert_allclose(out, g[tag + "_eval_logits"], rtol=1e-4, atol=1e-5)
    st = unet_dsbn.to_torch_state(synth.synth_state_dict(), requires_grad=True)
    logits = unet_dsbn.forward(st, x, 1, params, bn_training=True)
    loss = losses.combined_loss(logits, y, None, 0.5, 0.5)
    loss.backward()
    np.testing.assert_allclose(logits.detach().numpy(), g[tag + "_train_logits"], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(loss.item(), float(g[tag + "_train_loss"]), rtol=1e-6)
    n_with_grad = sum(v.numel() for v in st.values() if v.requires_grad and v.grad is not None)
    assert n_with_grad == int(g[tag + "_n_with_grad"])
    for k in GRADS[tag]:
        ours = st[k].grad
        np.testing.assert_allclose(ours.double().norm().item(), float(g[tag + "_gradnorm_" + k]), rtol=1e-4, err_msg=k)
        np.testing.assert_allclose(ours.numpy().reshape(-1)[:4096], g[tag + "_grad_" + k], rtol=2e-3,
                                   atol=1e-6 * float(ours.abs().max()), err_msg=k)
