"""Drop-in module: state_dict compatibility, eval-path equality with the reference (stored vectors,
tests/golden/make_golden_hosts.py) and the full training forward/backward against a fixture produced by the reference
itself."""
import json
import os
import random

import numpy as np
import pytest
import torch

from tests.common import GOLDEN, make_hrfp_params, make_draws, fill_state_dict, host_eval_case, host_state_dict_digest


def _criterion():
    return torch.nn.CrossEntropyLoss(ignore_index=255)


def test_state_dict_matches_reference_keys_and_shapes():
    from mrfp_b200.model import MRFPPlus
    with open(os.path.join(GOLDEN, "known_answers.json")) as f:
        known = json.load(f)
    m = MRFPPlus(19, criterion=_criterion())
    sd = m.state_dict()
    assert list(sd.keys()) == known["all_state_dict_keys"]
    assert {k: list(v.shape) for k, v in sd.items()} == known["state_dict_shapes"]
    frozen = sum(p.numel() for p in m.parameters() if not p.requires_grad)
    train = sum(p.numel() for p in m.parameters() if p.requires_grad)
    assert (frozen, train) == (known["frozen_params"], known["trainable_params"])


def test_reinit_rng_order_matches_reference():
    from mrfp_b200.model import MRFPPlus
    with open(os.path.join(GOLDEN, "known_answers.json")) as f:
        known = json.load(f)
    m = MRFPPlus(19, criterion=_criterion())
    log = []
    ok, on = torch.nn.init.kaiming_normal_, torch.nn.init.normal_
    torch.nn.init.kaiming_normal_ = lambda t, *a, **k: (log.append(["kaiming_normal_", list(t.shape)]), ok(t, *a, **k))[1]
    torch.nn.init.normal_ = lambda t, *a, **k: (log.append(["normal_", list(t.shape), k.get("std")]), on(t, *a, **k))[1]
    try:
        m.reinit_hrfp()
    finally:
        torch.nn.init.kaiming_normal_, torch.nn.init.normal_ = ok, on
    assert log == known["draw_log"][:16]


def test_eval_forward_needs_no_kernels_and_is_deterministic():
    from mrfp_b200.model import MRFPPlus
    m = MRFPPlus(19, criterion=_criterion()).eval()
    x = torch.rand(1, 3, 64, 64) * 255
    with torch.no_grad():
        a = m(x, training=False)
        b = m(x, training=False)
    assert a.shape == (1, 19, 64, 64) and torch.equal(a, b)


def _check_host_eval(name):
    """One tests.common.HOST_EVAL_CASES case against tests/golden/hosts_eval.npz (tests/golden/make_golden_hosts.py): the
    sampled outputs and sum |.| to the tolerance the reference's own modules were held to, the state_dict names and shapes
    exactly."""
    g = np.load(os.path.join(GOLDEN, "hosts_eval.npz"))
    m, out = host_eval_case(name)
    y = out.double().numpy()
    amax = float(g[f"{name}_absmax"])
    assert list(y.shape) == list(g[f"{name}_shape"])
    assert np.allclose(y.ravel()[g[f"{name}_idx"]], g[f"{name}_val"], rtol=1e-5, atol=1e-5 * amax)
    assert abs(np.abs(y).max() - amax) <= 1e-5 * amax
    assert abs(np.abs(y).sum() - float(g[f"{name}_abssum"])) <= 1e-5 * float(g[f"{name}_abssum"])
    assert host_state_dict_digest(m) == str(g[f"{name}_digest"])
    return m


def test_eval_forward_equals_reference_on_cpu():
    _check_host_eval("resnet50")


def _train_step(math_mode):
    from mrfp_b200 import model as M, npplus
    torch.backends.cudnn.allow_tf32 = False           # the fixture is an fp32 (CPU) run of the reference
    torch.backends.cuda.matmul.allow_tf32 = False
    g = np.load(os.path.join(GOLDEN, "full_model.npz"))
    m = M.MRFPPlus(19, criterion=_criterion(), math_mode=math_mode)
    fill_state_dict(m, 77)
    m = m.cuda().train()
    n, hh, ww = 2, 64, 64
    rng = np.random.default_rng(78)
    x = torch.from_numpy(rng.uniform(0, 255, (n, 3, hh, ww)).astype(np.float32)).cuda()
    gts = torch.from_numpy(rng.integers(0, 19, (n, hh, ww)).astype(np.int64))
    gts[torch.from_numpy(rng.uniform(size=(n, hh, ww)) < 0.05)] = 255
    gts = gts.cuda()
    ws, gs = make_hrfp_params(79)
    draws = [make_draws(80, n, 64), make_draws(81, n, 256)]

    def fake_reinit():
        convs, bns = m.hrfp_modules()
        with torch.no_grad():
            for k in range(8):
                convs[k].weight.copy_(torch.from_numpy(ws[k])); convs[k].bias.zero_()
                bns[k].weight.copy_(torch.from_numpy(gs[k])); bns[k].bias.zero_()

    def fake_draws(feat):
        a, e = draws.pop(0)
        return torch.from_numpy(a).to(feat.device), torch.from_numpy(e).to(feat.device)

    m.reinit_hrfp = fake_reinit
    orig = npplus.draw_np_plus_factors
    npplus.draw_np_plus_factors = fake_draws
    try:
        random.seed(4)
        loss = m(x, gts, training=True)
        loss.backward()
    finally:
        npplus.draw_np_plus_factors = orig
    return g, m, float(loss)


@pytest.mark.gpu
def test_training_step_matches_reference_fp32_mode():
    g, m, loss = _train_step(0)
    assert abs(loss - float(g["loss"])) <= 2e-4 * abs(float(g["loss"]))
    params = dict(m.named_parameters())
    # Gradients of the classifier (final2) are well conditioned and checked tightly.  Gradients that travelled back through the 50-layer random-weight trunk at this tiny
    # size (4x4 maps at layer4, BN over 32 values) are chaotic: the reference's own eager code run on the GPU
    # instead of the CPU moves them by 3-5 % of max (tools/debug_model.py), so they only get a coarse check.
    # Measured on B200 (tools/dbg_model_step.py): loss agrees to 6e-6; the worst sampled gradient
    # (layer2.0.conv2.weight) sits at 12.8 % with the two-step stem and 18.1 % with NP+ folded into the chain — two
    # fp32 rounding realisations of the same chaotic map (the folded form matches the two-step form to 5e-6 on the
    # stem itself: tests/test_hrfp_gpu.py::test_np_plus_folded_into_the_chain_equals_the_two_step_form).
    for key in [k[3:] for k in g.files if k.startswith("gs_")]:
        grad = params[key].grad.double().cpu()
        samp = grad.flatten()[:: max(1, grad.numel() // 64)][:64].numpy()
        ref = g["gs_" + key]
        tol = 2e-3 if key.startswith("final2") else 2.5e-1
        assert np.abs(samp - ref).max() <= tol * np.abs(ref).max(), key
        assert abs(float(grad.abs().sum()) - g["g_" + key][1]) <= tol * g["g_" + key][1], key
    for k in range(8):
        bn = m.hrfp_modules()[1][k]
        assert np.allclose(bn.running_mean.cpu().numpy(), g[f"rm{k}"], rtol=1e-3, atol=1e-4)


@pytest.mark.gpu
def test_training_step_bf16_mode_close_to_reference():
    g, m, loss = _train_step(2)
    # the bf16 HRFP branch perturbs the features by ~2 % (tests/test_hrfp_gpu.py); the loss moves accordingly
    assert abs(loss - float(g["loss"])) <= 5e-2 * abs(float(g["loss"]))
    grad = dict(m.named_parameters())["final2.0.weight"].grad
    assert torch.isfinite(grad).all()
    ref_l1 = g["g_final2.0.weight"][1]
    assert abs(float(grad.double().abs().sum()) - ref_l1) <= 0.2 * ref_l1


@pytest.mark.gpu
def test_gates_off_is_plain_deeplab_and_skips_hrfp():
    from mrfp_b200.model import MRFPPlus
    m = MRFPPlus(19, criterion=_criterion()).cuda().train()
    x = torch.rand(2, 3, 64, 64, device="cuda") * 255
    gts = torch.randint(0, 19, (2, 64, 64), device="cuda")
    random.seed(1)     # 0.134, 0.847, 0.763: p < .5 only  -> HRFP add without NP+ / HRFP+
    loss = m(x, gts, training=True)
    loss.backward()
    assert torch.isfinite(loss)
    nbt = int(m.OC1_bn.num_batches_tracked)
    state = random.getstate()
    random.seed(11)    # find a seed with all three gates >= 0.5
    for s in range(100):
        random.seed(s)
        if min(random.random(), random.random(), random.random()) >= 0.5:
            random.seed(s)
            break
    loss = m(x, gts, training=True)
    assert int(m.OC1_bn.num_batches_tracked) == nbt       # dead chain skipped (strict_buffers=False)
    random.setstate(state)


# ---- trunk="resnet-101" (SURVEY.md 8f-2, BASELINE config[3]): the reference's deep-stem ResNet-101 under the same hooks ----


def test_resnet101_host_shapes():
    from mrfp_b200.model import MRFPPlus
    m = MRFPPlus(19, trunk="resnet-101", criterion=_criterion())
    assert [len(l) for l in (m.layer1, m.layer2, m.layer3, m.layer4)] == [3, 4, 23, 3]
    assert m.OClayer1.in_channels == 128 and m.OCdeclayer4.out_channels == 128 and m.OClayer4.out_channels == 256
    assert isinstance(m.layer0[7], torch.nn.InstanceNorm2d) and m.layer0[7].num_features == 128
    assert m.layer1[-1].has_in and m.layer2[-1].has_in and not m.layer3[-1].has_in
    m.eval()
    with torch.no_grad():
        out = m(torch.rand(1, 3, 64, 64) * 255, training=False)
    assert out.shape == (1, 19, 64, 64)
    with pytest.raises(ValueError):
        MRFPPlus(19, trunk="resnet-18", criterion=_criterion())


def test_resnet101_trunk_equals_reference_resnet101_on_cpu():
    """layer0..layer2 (all three InstanceNorm sites) of the ResNet-101 host, which carries the reference's
    network/Resnet.py resnet101 (its conv1 / bn1 ... conv3 / bn3 stem as layer0.0 ... layer0.7)."""
    _check_host_eval("resnet101_trunk")


@pytest.mark.gpu
def test_resnet101_training_step_runs_all_branches():
    """One training step of the ResNet-101 host with all three MRFP branches on: the kernels run on the 128-channel stem
    (HRFP with NP+ call 1 folded in, IN+ReLU with plane sums -> pre-summed NP+ call 2, fused HRFP+ tail)."""
    from mrfp_b200.model import MRFPPlus
    torch.manual_seed(0)
    m = MRFPPlus(19, trunk="resnet-101", criterion=_criterion()).cuda().train()
    x = torch.rand(2, 3, 96, 128, device="cuda") * 255
    gts = torch.randint(0, 19, (2, 96, 128), device="cuda")
    random.seed(4)      # all three gates < 0.5 (tests/golden/known_answers.json)
    loss = m(x, gts, training=True)
    loss.backward()
    assert torch.isfinite(loss)
    assert int(m.OC1_bn.num_batches_tracked) == 1
    for name in ("layer0.0.weight", "layer0.7.weight", "layer1.2.instance_norm_layer.weight", "final2.0.weight"):
        g = dict(m.named_parameters())[name].grad
        assert g is not None and torch.isfinite(g).all() and float(g.abs().sum()) > 0, name


# ---- trunk="mobilenetv2" / "shufflenetv2" (SURVEY.md 8f-2, BASELINE config[4]) ----
@pytest.mark.parametrize("trunk", ["mobilenetv2", "shufflenetv2"])
def test_mobile_hosts_load_the_reference_state_dict_and_match_its_eval_forward_on_cpu(trunk):
    """The host is state_dict-compatible with the reference's DeepV3Plus(trunk) (network/deepv3.py:103-556; its `dsn`
    auxiliary head aside) and evaluates to the same logits — eval mode has no MRFP, so this pins the trunk wiring."""
    mine = _check_host_eval(trunk)
    stem = {"mobilenetv2": 16, "shufflenetv2": 24}[trunk]
    assert mine.OClayer1.in_channels == stem and mine.OCdeclayer4.out_channels == stem
    assert mine.hrfp_scale == {"mobilenetv2": 2, "shufflenetv2": 1}[trunk]


@pytest.mark.gpu
@pytest.mark.parametrize("math_mode", [0, 2])
@pytest.mark.parametrize("trunk", ["mobilenetv2", "shufflenetv2"])
def test_mobile_hosts_training_step_matches_the_eager_reference_ops(trunk, math_mode):
    """All three MRFP branches on a narrow-stem host (16 ch @ stride 2 / 24 ch @ stride 4; NP+ call 2 on 32 / 116 ch @
    stride 8): the loss through the kernels equals the loss through the reference's own op sequence (deepv3.py:268-277,
    :320-330, :356-357 written with torch operators, chain sized relative to xp) evaluated eagerly on the same model
    with the same random draws; gradients reach the stem and every MRFP-adjacent layer."""
    import torch.nn.functional as F
    from oracle import torch_port as TP
    from mrfp_b200.model import MRFPPlus
    h, w = 96, 128
    torch.manual_seed(0)
    m = MRFPPlus(19, trunk=trunk, criterion=_criterion(), math_mode=math_mode).cuda().train()
    x = torch.rand(2, 3, h, w, device="cuda") * 255
    gts = torch.randint(0, 19, (2, h, w), device="cuda")
    gates = (0.25, 0.25, 0.25)

    def run(eager):
        for mod in m.modules():                                  # same BN running buffers at the start of both runs
            if isinstance(mod, torch.nn.BatchNorm2d):
                mod.reset_running_stats()
        m.zero_grad(set_to_none=True)
        torch.manual_seed(5)
        if not eager:
            loss = m(x, gts, training=True, gates=gates)
        else:                                                    # the reference's expressions on the host's modules
            he, we = h * m.hrfp_scale, w * m.hrfp_scale
            m.reinit_hrfp()
            xp = m._stem(x)
            a1, e1 = torch.empty_like(xp[:, :, :1, :1]).normal_(1.0, 0.75), torch.empty_like(xp[:, :, :1, :1]).normal_(0.0, 0.75)
            convs, bns = m.hrfp_modules()
            oc, dec = TP.hrfp_chain(convs, bns, xp, he, we, exact_adjoint=True)
            f = m.layer1(oc + TP.np_plus(xp, a1, e1))
            a2, e2 = torch.empty_like(f[:, :, :1, :1]).normal_(1.0, 0.75), torch.empty_like(f[:, :, :1, :1]).normal_(0.0, 0.75)
            low = TP.np_plus(f, a2, e2)
            top = m.layer4(m.layer3(m.layer2(low)))
            d0 = torch.cat([m.bot_fine(low), F.interpolate(m.bot_aspp(m.aspp(top)), size=low.shape[2:], mode="bilinear", align_corners=True)], 1)
            d1 = F.interpolate(m.final1(d0), size=(he // 2, we // 2), mode="bilinear", align_corners=True) + dec
            loss = m.criterion(F.interpolate(m.final2(d1), size=(h, w), mode="bilinear", align_corners=True), gts)
        loss.backward()
        grads = {k: p.grad.detach().clone() for k, p in m.named_parameters() if p.grad is not None}
        return float(loss), grads

    l_k, g_k = run(False)
    l_e, g_e = run(True)
    tol = 1e-3 if math_mode == 0 else 5e-2
    assert abs(l_k - l_e) <= tol * abs(l_e), (l_k, l_e)
    assert set(g_k) == set(g_e)
    for key in ("final2.0.weight", "final2.0.bias"):             # well-conditioned gradients: checked against the eager run
        rel = float((g_k[key] - g_e[key]).norm() / g_e[key].norm())
        assert rel <= (5e-3 if math_mode == 0 else 2e-1), (key, rel)
    first = next(k for k in g_k if k.startswith("layer0") and k.endswith("weight"))
    for key in (first, "bot_fine.0.weight", "final1.0.weight"):
        assert torch.isfinite(g_k[key]).all() and float(g_k[key].abs().sum()) > 0, key
    assert int(m.OC1_bn.num_batches_tracked) >= 1
