"""Pins the numpy oracle (oracle/mrfp_oracle.py) against fixtures generated from the reference itself
(tests/golden/make_golden.py).  CPU only."""
import json
import math
import os

import numpy as np
import pytest

from oracle import mrfp_oracle as O
from tests.common import GOLDEN, hrfp_gx_both, make_hrfp_params, make_feat, make_draws


@pytest.fixture(scope="module")
def g_np():
    return np.load(os.path.join(GOLDEN, "npplus.npz"))


@pytest.fixture(scope="module")
def g_lut():
    return np.load(os.path.join(GOLDEN, "lut.npz"))


@pytest.fixture(scope="module")
def g_hrfp():
    return np.load(os.path.join(GOLDEN, "hrfp.npz"))


@pytest.fixture(scope="module")
def known():
    with open(os.path.join(GOLDEN, "known_answers.json")) as f:
        return json.load(f)


@pytest.mark.parametrize("i,name", list(enumerate("abcd")))
def test_npplus_forward_backward_vs_reference(g_np, i, name):
    shape = tuple(g_np[f"{name}_shape"])
    feat = make_feat(100 + i, shape).astype(np.float64)
    a, e = make_draws(200 + i, shape[0], shape[1])
    out, mean, beta = O.np_plus_forward(feat, a.astype(np.float64), e.astype(np.float64))
    ref = g_np[f"{name}_out"]
    tol = 2e-5 * np.abs(ref).max()                      # reference ran in fp32
    assert np.abs(out - ref).max() <= tol
    gout = np.random.default_rng(300 + i).standard_normal(shape).astype(np.float32).astype(np.float64)
    gin = O.np_plus_backward(gout, a.astype(np.float64), e.astype(np.float64), mean)
    refg = g_np[f"{name}_gin"]
    assert np.abs(gin - refg).max() <= 1e-4 * np.abs(refg).max()


def test_npplus_closed_form_backward_fp64(g_np):
    shape = tuple(g_np["a_shape"])
    feat = make_feat(100, shape).astype(np.float64)
    a, e = make_draws(200, shape[0], shape[1])
    a, e = a.astype(np.float64), e.astype(np.float64)
    out, mean, _ = O.np_plus_forward(feat, a, e)
    assert np.abs(out - g_np["a64_out"]).max() <= 1e-12 * np.abs(out).max()
    gout = np.random.default_rng(300).standard_normal(shape).astype(np.float32).astype(np.float64)
    gin = O.np_plus_backward(gout, a, e, mean)
    assert np.abs(gin - g_np["a64_gin"]).max() <= 1e-12 * np.abs(gin).max()


def test_npplus_batch_of_one_is_nan(g_np):
    assert bool(g_np["n1_all_nan"])
    feat = make_feat(1, (1, 4, 5, 5)).astype(np.float64)
    a, e = make_draws(2, 1, 4)
    out, _, _ = O.np_plus_forward(feat, a, e)
    assert np.isnan(out).all()


def test_npplus_equal_means_is_nan():
    feat = np.ones((3, 4, 5, 5))
    a, e = make_draws(3, 3, 4)
    out, _, _ = O.np_plus_forward(feat, a, e)
    assert np.isnan(out).all()          # d == 0 for all channels -> 0/0


def test_size_chain_768(g_lut):
    st = O.hrfp_geometry(768, 768, 192, 192)
    sizes = [192] + [s.out_h for s in st]
    assert sizes == [192, 231, 277, 332, 384, 384, 321, 256, 192]
    assert list(g_lut["768_h_sizes"]) == sizes


@pytest.mark.parametrize("tag,hw", [("768", (768, 768)), ("odd", (100, 140)), ("small", (48, 48)), ("rect", (40, 56))])
def test_nearest_lut_vs_aten(g_lut, tag, hw):
    h, w = hw
    xh, xw = int(g_lut[f"{tag}_h_sizes"][0]), int(g_lut[f"{tag}_w_sizes"][0])
    st = O.hrfp_geometry(h, w, xh, xw)
    for k, s in enumerate(st):
        assert np.array_equal(s.idx_h, g_lut[f"{tag}_h_{k}"]), (tag, "h", k)
        assert np.array_equal(s.idx_w, g_lut[f"{tag}_w_{k}"]), (tag, "w", k)


def test_nearest_rule_differs_from_ratio_rule(g_lut):
    # scale_factor mode uses float32(1/sf), not in/out: the two rules disagree on some indices (SURVEY §4)
    idx = g_lut["768_h_0"]
    ratio = np.minimum(np.floor(np.arange(231, dtype=np.float32) * (np.float32(192) / np.float32(231))), 191)
    assert (idx != ratio).sum() > 0
    counts = np.bincount(idx, minlength=192)
    assert counts[191] == 0 and set(np.unique(counts)) <= {0, 1, 2}


def test_bn_stats_of_resampled_equal_count_weighted_stats():
    rng = np.random.default_rng(0)
    y = rng.standard_normal((2, 3, 12, 12))
    st = O.hrfp_geometry(48, 48, 12, 12)[0]
    r = O.resample(y, st.idx_h, st.idx_w)
    ch = np.bincount(st.idx_h, minlength=12).astype(np.float64)
    cw = np.bincount(st.idx_w, minlength=12).astype(np.float64)
    wgt = ch[:, None] * cw[None, :]
    mu = (y * wgt).sum((0, 2, 3)) / (wgt.sum() * 2)
    assert np.allclose(mu, r.mean((0, 2, 3)), atol=1e-12)
    ex2 = (y * y * wgt).sum((0, 2, 3)) / (wgt.sum() * 2)
    assert np.allclose(ex2 - mu * mu, r.var((0, 2, 3)), atol=1e-12)


@pytest.mark.parametrize("tag", ["sq", "rect"])
def test_hrfp_forward_backward_vs_reference(g_hrfp, tag):
    n, h, w, seed = [int(v) for v in g_hrfp[f"{tag}_meta"]]
    xh, xw = math.ceil(h / 4), math.ceil(w / 4)
    ws, gs = make_hrfp_params(seed)
    ws64 = [x.astype(np.float64) for x in ws]
    gs64 = [x.astype(np.float64) for x in gs]
    xp = make_feat(seed + 50, (n, 64, xh, xw)).astype(np.float64)
    ocout, ocdec, saved = O.hrfp_forward(xp, ws64, gs64, h, w)
    ref = g_hrfp[f"{tag}_ocout"]
    assert ocout.shape == ref.shape
    assert np.abs(ocout - ref).max() <= 2e-4 * max(1.0, np.abs(ref).max())
    refd = g_hrfp[f"{tag}_ocout_dec"].astype(np.float64)          # stored as fp16
    assert np.abs(ocdec - refd).max() <= 2e-3 * max(1.0, np.abs(refd).max())
    assert np.allclose(ocdec.sum((0, 2, 3)), g_hrfp[f"{tag}_ocout_dec_sum"], rtol=1e-4, atol=1e-2)
    rng = np.random.default_rng(seed + 70)
    g1 = rng.standard_normal(ocout.shape).astype(np.float32).astype(np.float64)
    g2 = rng.standard_normal(ocdec.shape).astype(np.float32).astype(np.float64)
    for key, (a, b) in {"gx_both": (g1, g2), "gx_out": (g1, None), "gx_dec": (None, g2)}.items():
        gx = O.hrfp_backward(a, b, ws64, gs64, saved)
        refg = hrfp_gx_both(g_hrfp, tag) if key == "gx_both" else g_hrfp[f"{tag}_{key}"]
        assert np.abs(gx - refg).max() <= 5e-4 * np.abs(refg).max(), key
    # BN buffer side effect (SURVEY §8 a-8)
    for k in range(8):
        rm, rv = O.bn_running_update(np.zeros_like(saved[k]["mean"]), np.ones_like(saved[k]["var"]),
                                     saved[k]["mean"], saved[k]["var"], saved[k]["count"])
        assert np.allclose(rm, g_hrfp[f"{tag}_rm{k}"], rtol=1e-4, atol=1e-5)
        assert np.allclose(rv, g_hrfp[f"{tag}_rv{k}"], rtol=1e-4, atol=1e-5)
    assert int(g_hrfp[f"{tag}_nbt"]) >= 1


def test_hrfp_plus_add(g_hrfp):
    out = O.hrfp_plus_add(g_hrfp["plus_dec1"].astype(np.float64), g_hrfp["plus_ocd"].astype(np.float64))
    assert np.abs(out - g_hrfp["plus_out"]).max() <= 1e-5


def test_known_answers(known):
    assert known["frozen_params"] == 887232 and known["trainable_params"] == 40353203
    assert all(g < 0.5 for g in known["gates_seed4"])
    log = known["draw_log"]
    # 8 x (kaiming_normal_ W, normal_ gamma std .5) in module order, then NP+ draws (N,64,1,1)x2, (N,256,1,1)x2
    assert len(log) == 20
    for k, (cin, cout, _) in enumerate(O.HRFP_LAYERS):
        assert log[2 * k] == ["kaiming_normal_", [cout, cin, 3, 3]]
        assert log[2 * k + 1] == ["normal_", [cout], 0.5]
    assert [e[1] for e in log[16:]] == [[2, 64, 1, 1]] * 2 + [[2, 256, 1, 1]] * 2
    assert known["nbt_after"] == known["nbt_before"] + 1
    want = []
    for c, b in zip(O.HRFP_CONV_NAMES, O.HRFP_BN_NAMES):
        want += [f"{c}.weight", f"{c}.bias", f"{b}.weight", f"{b}.bias", f"{b}.running_mean",
                 f"{b}.running_var", f"{b}.num_batches_tracked"]
    assert known["oc_state_dict_keys"] == want
    assert abs(O.hrfp_init_std(64) - math.sqrt(2 / 576)) < 1e-12


def test_torch_port_npplus_vs_reference(g_np):
    import torch
    from oracle import torch_port as T
    shape = tuple(g_np["d_shape"])
    feat = torch.from_numpy(make_feat(103, shape)).requires_grad_(True)
    a, e = make_draws(203, shape[0], shape[1])
    y = T.np_plus(feat, torch.from_numpy(a).view(*shape[:2], 1, 1), torch.from_numpy(e).view(*shape[:2], 1, 1))
    y.backward(torch.from_numpy(np.random.default_rng(303).standard_normal(shape).astype(np.float32)))
    assert np.abs(y.detach().numpy() - g_np["d_out"]).max() <= 1e-5 * np.abs(g_np["d_out"]).max()
    assert np.abs(feat.grad.numpy() - g_np["d_gin"]).max() <= 1e-4 * np.abs(g_np["d_gin"]).max()


def test_torch_port_hrfp_vs_reference(g_hrfp):
    import torch
    from oracle import torch_port as T
    n, h, w, seed = [int(v) for v in g_hrfp["sq_meta"]]
    ws, gs = make_hrfp_params(seed)
    convs, bns = T.make_layers(ws, gs)
    xp = torch.from_numpy(make_feat(seed + 50, (n, 64, h // 4, w // 4))).requires_grad_(True)
    o, d = T.hrfp_chain(convs, bns, xp, h, w)
    rng = np.random.default_rng(seed + 70)
    g1 = torch.from_numpy(rng.standard_normal(tuple(o.shape)).astype(np.float32))
    g2 = torch.from_numpy(rng.standard_normal(tuple(d.shape)).astype(np.float32))
    torch.autograd.backward([o, d], [g1, g2])
    assert np.abs(o.detach().numpy() - g_hrfp["sq_ocout"]).max() <= 1e-4 * np.abs(g_hrfp["sq_ocout"]).max()
    gx_both = hrfp_gx_both(g_hrfp, "sq")
    assert np.abs(xp.grad.numpy() - gx_both).max() <= 1e-3 * np.abs(gx_both).max()


@pytest.mark.parametrize("name", list("abcd"))
def test_instance_norm_relu_vs_reference_fixture(name):
    """Oracle IN+ReLU (SURVEY 8f-3) against the reference's own Bottleneck(iw=4) layers (tests/golden/make_golden_instnorm.py)."""
    from tests.common import make_in_case
    g = np.load(os.path.join(GOLDEN, "instnorm.npz"))
    shape = tuple(int(v) for v in g[f"{name}_shape"])
    x, gamma, beta, gy = make_in_case(400 + "abcd".index(name), shape)
    y, mean, invstd, psum = O.instance_norm_relu_forward(x, gamma, beta)
    gx, gw, gb = O.instance_norm_relu_backward(gy, x, gamma, beta)
    np.testing.assert_allclose(y, g[f"{name}_y"], rtol=2e-5, atol=2e-5)
    # the fp32 reference and the fp64 oracle may disagree on the ReLU mask where |y| ~ 1e-7: compare away from it
    far = np.abs(O.instance_norm_relu_forward(x, gamma, beta, relu=False)[0]) > 1e-4
    scale = np.abs(g[f"{name}_gx"]).max()
    assert np.abs(gx - g[f"{name}_gx"])[far].max() <= 1e-4 * scale
    np.testing.assert_allclose(gw, g[f"{name}_gw"], rtol=1e-3, atol=1e-3)
    np.testing.assert_allclose(gb, g[f"{name}_gb"], rtol=1e-3, atol=1e-3)
    np.testing.assert_allclose(psum, y.sum(axis=(2, 3)))


@pytest.mark.parametrize("shape,relu", [((2, 3, 5, 7), True), ((1, 6, 16, 16), True), ((3, 4, 9, 1), False), ((2, 8, 32, 24), True)])
def test_instance_norm_relu_oracle_vs_torch_autograd_on_cpu(shape, relu):
    """Second pin of the InstanceNorm oracle: torch's own F.instance_norm (+ relu) and its autograd in float64 on CPU —
    the operators the reference's layers call (Resnet.py:176-178, :534-536)."""
    import torch
    import torch.nn.functional as F
    from tests.common import make_in_case
    x, gamma, beta, gy = make_in_case(500 + shape[1], shape)
    xt = torch.from_numpy(x).double().requires_grad_(True)
    wt = torch.from_numpy(gamma).double().requires_grad_(True)
    bt = torch.from_numpy(beta).double().requires_grad_(True)
    y = F.instance_norm(xt, weight=wt, bias=bt, eps=O.IN_EPS)
    if relu:
        y = F.relu(y)
    y.backward(torch.from_numpy(gy).double())
    oy, mean, invstd, psum = O.instance_norm_relu_forward(x, gamma, beta, relu=relu)
    ogx, ogw, ogb = O.instance_norm_relu_backward(gy, x, gamma, beta, relu=relu)
    np.testing.assert_allclose(oy, y.detach().numpy(), rtol=1e-10, atol=1e-10)
    np.testing.assert_allclose(ogx, xt.grad.numpy(), rtol=1e-8, atol=1e-10)
    np.testing.assert_allclose(ogw, wt.grad.numpy(), rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(ogb, bt.grad.numpy(), rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(mean, x.astype(np.float64).mean(axis=(2, 3)))
