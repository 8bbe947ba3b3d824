"""HRFP CUDA chain (through the C ABI) vs the numpy oracle and the reference-generated fixtures."""
import math
import os

import numpy as np
import pytest
import torch

from oracle import mrfp_oracle as O
from tests.common import GOLDEN, hrfp_gx_both, make_hrfp_params, make_feat

pytestmark = pytest.mark.gpu

# Tolerances (max |err| / max |ref|).
#  mode 0 (fp32 CUDA-core path): the reference's fp32 tolerance; measured 3e-6 fwd / 1.4e-6 bwd.
#  mode 2 (bf16 tcgen05 path): eight chained stages whose activations, conv outputs and gradients are STORED in
#  bf16.  The numpy oracle with the same storage rounding (oracle.round_bf16) sits 2.0e-2 (fwd) / 1.7e-1 (bwd) from the
#  fp32 reference on these fixtures — that distance is the format, not the kernels — and the kernels sit at
#  2.0e-2 / 1.7e-1 as well, and at 8e-3 / 7e-2 from the bf16-storage oracle (rounding-boundary chaos keeps the two
#  bf16 computations from agreeing better than the rounding noise itself).  The tensor-core conv alone is checked
#  to one bf16 ulp in tests/test_conv_tc_gpu.py.
#  mode 1 (tf32 tcgen05 path): fp32 storage, conv operands rounded to tf32 — the reference's own GPU arithmetic.
# The max-norm of a gradient through eight ReLU stages is set by a handful of mask flips of near-zero pre-activations;
# the L2-relative error (TOL_L2) is the bound that would catch a dropped or mis-scaled term, and every chain test
# asserts both.  Full-size (768^2) numbers: tests/test_hrfp_fullsize_gpu.py; single kernels: tests/test_hrfp_stage_gpu.py.
TOL = {0: dict(fwd=2e-4, bwd=1e-3),
       1: dict(fwd=1e-2, bwd=1e-1),
       2: dict(fwd=5e-2, bwd=5e-1)}
TOL_L2 = {0: dict(fwd=2e-5, bwd=2e-4),
          1: dict(fwd=3e-3, bwd=1e-1),
          2: dict(fwd=3e-2, bwd=3e-1)}
TOL_VS_BF16_ORACLE = dict(fwd=2.5e-2, bwd=1.5e-1)
MODES = [0, 1, 2]


def _modules(ws, gs, device):
    convs, bns = [], []
    for (cin, cout, dil), w, g in zip(O.HRFP_LAYERS, ws, gs):
        c = torch.nn.Conv2d(cin, cout, 3, padding=dil, dilation=dil).to(device).requires_grad_(False)
        b = torch.nn.BatchNorm2d(cout).to(device).requires_grad_(False)
        with torch.no_grad():
            c.weight.copy_(torch.from_numpy(w)); c.bias.zero_()
            b.weight.copy_(torch.from_numpy(g)); b.bias.zero_()
        convs.append(c); bns.append(b)
    return convs, bns


def _run(xp_np, ws, gs, h, w, mode, g1=None, g2=None, x_add=None):
    from mrfp_b200.hrfp import hrfp_chain
    dev = "cuda"
    convs, bns = _modules(ws, gs, dev)
    xp = torch.from_numpy(xp_np).to(dev).requires_grad_(True)
    xa = None if x_add is None else torch.from_numpy(x_add).to(dev).requires_grad_(True)
    out, dec = hrfp_chain(xp, convs, bns, h, w, x_add=xa, math_mode=mode)
    gx = None
    if g1 is not None or g2 is not None:
        outs, gr = [], []
        if g1 is not None:
            outs.append(out); gr.append(torch.from_numpy(g1).to(dev))
        if g2 is not None:
            outs.append(dec); gr.append(torch.from_numpy(g2).to(dev))
        torch.autograd.backward(outs, gr)
        gx = xp.grad.cpu().numpy()
    return out.detach().cpu().numpy(), dec.detach().cpu().numpy(), gx, bns, (None if xa is None else xa.grad)


def _relerr(got, ref):
    ref = np.asarray(ref, dtype=np.float64)
    return np.abs(got.astype(np.float64) - ref).max() / max(np.abs(ref).max(), 1e-30)


def _l2err(got, ref):
    ref = np.asarray(ref, dtype=np.float64)
    return np.linalg.norm((got.astype(np.float64) - ref).ravel()) / max(np.linalg.norm(ref.ravel()), 1e-30)


def _check(got, ref, mode, which, floor=0.0):
    """max-norm and L2-relative bounds of `mode` ('fwd' or 'bwd')."""
    assert _relerr(got, ref) <= max(TOL[mode][which], floor), (mode, which, "max", _relerr(got, ref))
    assert _l2err(got, ref) <= max(TOL_L2[mode][which], floor), (mode, which, "l2", _l2err(got, ref))


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("tag", ["sq", "rect"])
def test_vs_reference_fixture(tag, mode):
    g = np.load(os.path.join(GOLDEN, "hrfp.npz"))
    n, h, w, seed = [int(v) for v in g[f"{tag}_meta"]]
    xh, xw = math.ceil(h / 4), math.ceil(w / 4)
    ws, gs = make_hrfp_params(seed)
    xp = make_feat(seed + 50, (n, 64, xh, xw))
    rng = np.random.default_rng(seed + 70)
    g1 = rng.standard_normal((n, 64, xh, xw)).astype(np.float32)
    g2 = rng.standard_normal((n, 256, h // 2, w // 2)).astype(np.float32)
    out, dec, gx, bns, _ = _run(xp, ws, gs, h, w, mode, g1, g2)
    _check(out, g[f"{tag}_ocout"], mode, "fwd")
    _check(dec, g[f"{tag}_ocout_dec"].astype(np.float32), mode, "fwd", floor=2e-3)         # fixture stored as fp16
    _check(gx, hrfp_gx_both(g, tag), mode, "bwd")
    for k in range(8):
        rtol = {0: 1e-4, 1: 2e-3, 2: 2e-2}[mode]
        assert np.allclose(bns[k].running_mean.cpu().numpy(), g[f"{tag}_rm{k}"], rtol=rtol, atol=rtol)
        assert np.allclose(bns[k].running_var.cpu().numpy(), g[f"{tag}_rv{k}"], rtol=rtol, atol=rtol)
        assert int(bns[k].num_batches_tracked) == 1


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("which", ["out", "dec"])
def test_single_gradient_paths(which, mode):
    g = np.load(os.path.join(GOLDEN, "hrfp.npz"))
    n, h, w, seed = [int(v) for v in g["sq_meta"]]
    xh, xw = math.ceil(h / 4), math.ceil(w / 4)
    ws, gs = make_hrfp_params(seed)
    xp = make_feat(seed + 50, (n, 64, xh, xw))
    rng = np.random.default_rng(seed + 70)
    g1 = rng.standard_normal((n, 64, xh, xw)).astype(np.float32)
    g2 = rng.standard_normal((n, 256, h // 2, w // 2)).astype(np.float32)
    _, _, gx, _, _ = _run(xp, ws, gs, h, w, mode, g1 if which == "out" else None, g2 if which == "dec" else None)
    _check(gx, g[f"sq_gx_{which}"], mode, "bwd")


@pytest.mark.parametrize("mode", MODES)
def test_vs_oracle_odd_geometry_and_add(mode):
    n, h, w = 3, 60, 44
    xh, xw = 15, 11
    ws, gs = make_hrfp_params(5)
    xp = make_feat(6, (n, 64, xh, xw))
    x_add = np.random.default_rng(7).standard_normal((n, 64, xh, xw)).astype(np.float32)
    rng = np.random.default_rng(8)
    g1 = rng.standard_normal((n, 64, xh, xw)).astype(np.float32)
    g2 = rng.standard_normal((n, 256, h // 2, w // 2)).astype(np.float32)
    out, dec, gx, _, ga = _run(xp, ws, gs, h, w, mode, g1, g2, x_add=x_add)
    ws64 = [a.astype(np.float64) for a in ws]; gs64 = [a.astype(np.float64) for a in gs]
    ro, rd, saved = O.hrfp_forward(xp.astype(np.float64), ws64, gs64, h, w)
    rg = O.hrfp_backward(g1.astype(np.float64), g2.astype(np.float64), ws64, gs64, saved)
    _check(out, ro + x_add, mode, "fwd")
    _check(dec, rd, mode, "fwd")
    _check(gx, rg, mode, "bwd")
    assert torch.equal(ga.cpu(), torch.from_numpy(g1))        # d(OCout + x)/dx = identity
    if mode == 2:      # same computation with the same bf16 storage points
        qo, qd, qs = O.hrfp_forward(xp.astype(np.float64), ws64, gs64, h, w, quant=O.round_bf16)
        qg = O.hrfp_backward(g1.astype(np.float64), g2.astype(np.float64), ws64, gs64, qs, quant=O.round_bf16)
        assert _relerr(out, qo + x_add) <= TOL_VS_BF16_ORACLE["fwd"]
        assert _relerr(dec, qd) <= TOL_VS_BF16_ORACLE["fwd"]
        assert _relerr(gx, qg) <= TOL_VS_BF16_ORACLE["bwd"]


@pytest.mark.parametrize("mode", MODES)
def test_wide_stem_128_channels(mode):
    """R101-style stem (BASELINE config 4): xp has 128 channels, so OClayer1 is 128->64 and OCdeclayer4 is 64->128
    (`OCout + x` needs the stem width back).  The reference hard-wires 64 (deepv3.py:221-237); this is the documented
    extension of SURVEY.md 8f-2, checked against the oracle run with the same layer table."""
    n, h, w, xh, xw = 2, 64, 48, 16, 12
    layers = ((128, 64, 1), (64, 64, 1), (64, 128, 2), (128, 256, 2), (256, 128, 1), (128, 64, 1), (64, 64, 2), (64, 128, 2))
    rng = np.random.default_rng(21)
    ws = [(rng.standard_normal((co, ci, 3, 3)) * math.sqrt(2.0 / (9 * ci))).astype(np.float32) for ci, co, _ in layers]
    gs = [(0.5 * rng.standard_normal(co)).astype(np.float32) for _, co, _ in layers]
    xp = make_feat(22, (n, 128, xh, xw))
    g1 = rng.standard_normal((n, 128, xh, xw)).astype(np.float32)
    g2 = rng.standard_normal((n, 256, h // 2, w // 2)).astype(np.float32)
    from mrfp_b200.hrfp import hrfp_chain
    convs, bns = [], []
    for (ci, co, dil), wt, g in zip(layers, ws, gs):
        c = torch.nn.Conv2d(ci, co, 3, padding=dil, dilation=dil).to("cuda").requires_grad_(False)
        b = torch.nn.BatchNorm2d(co).to("cuda").requires_grad_(False)
        with torch.no_grad():
            c.weight.copy_(torch.from_numpy(wt)); c.bias.zero_()
            b.weight.copy_(torch.from_numpy(g)); b.bias.zero_()
        convs.append(c); bns.append(b)
    x = torch.from_numpy(xp).cuda().requires_grad_(True)
    out, dec = hrfp_chain(x, convs, bns, h, w, math_mode=mode)
    torch.autograd.backward([out, dec], [torch.from_numpy(g1).cuda(), torch.from_numpy(g2).cuda()])
    ws64 = [a.astype(np.float64) for a in ws]; gs64 = [a.astype(np.float64) for a in gs]
    ro, rd, saved = O.hrfp_forward(xp.astype(np.float64), ws64, gs64, h, w, layers=layers)
    rg = O.hrfp_backward(g1.astype(np.float64), g2.astype(np.float64), ws64, gs64, saved)
    assert out.shape == (n, 128, xh, xw)
    _check(out.detach().cpu().numpy(), ro, mode, "fwd")
    _check(dec.detach().cpu().numpy(), rd, mode, "fwd")
    _check(x.grad.cpu().numpy(), rg, mode, "bwd")


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("cin", [16, 24, 116])
def test_narrow_and_odd_stem_widths(cin, mode):
    """MobileNetV2 (16 channels) and ShuffleNetV2 (24 / 116 channels) stems (BASELINE config 5): OClayer1 is cin->64 and
    OCdeclayer4 64->cin.  Inside the chain the stem is stored zero-padded to the kernels' channel granule (64 on the
    tensor-core paths, the next power of two >= 16 on the CUDA-core path); at the boundary the tensors keep `cin`
    channels.  Checked against the oracle with the same layer table (extension of SURVEY.md 8f-2), in every math mode,
    with the NP+ call folded in (its (N, cin) side arrays are not padded)."""
    n, h, w, xh, xw = 2, 64, 48, 16, 12
    layers = ((cin, 64, 1), (64, 64, 1), (64, 128, 2), (128, 256, 2), (256, 128, 1), (128, 64, 1), (64, 64, 2), (64, cin, 2))
    rng = np.random.default_rng(31)
    ws = [(rng.standard_normal((co, ci, 3, 3)) * math.sqrt(2.0 / (9 * ci))).astype(np.float32) for ci, co, _ in layers]
    gs = [(0.5 * rng.standard_normal(co)).astype(np.float32) for _, co, _ in layers]
    xp = make_feat(32, (n, cin, xh, xw))
    g1 = rng.standard_normal((n, cin, xh, xw)).astype(np.float32)
    g2 = rng.standard_normal((n, 256, h // 2, w // 2)).astype(np.float32)
    alpha = (1 + 0.75 * rng.standard_normal((n, cin))).astype(np.float32)
    eps = (0.75 * rng.standard_normal((n, cin))).astype(np.float32)
    from mrfp_b200.hrfp import hrfp_chain
    convs, bns = [], []
    for (ci, co, dil), wt, g in zip(layers, ws, gs):
        c = torch.nn.Conv2d(ci, co, 3, padding=dil, dilation=dil).to("cuda").requires_grad_(False)
        b = torch.nn.BatchNorm2d(co).to("cuda").requires_grad_(False)
        with torch.no_grad():
            c.weight.copy_(torch.from_numpy(wt)); c.bias.zero_()
            b.weight.copy_(torch.from_numpy(g)); b.bias.zero_()
        convs.append(c); bns.append(b)
    x = torch.from_numpy(xp).cuda().requires_grad_(True)
    out, dec = hrfp_chain(x, convs, bns, h, w, math_mode=mode,
                          np_draws=(torch.from_numpy(alpha).cuda(), torch.from_numpy(eps).cuda()))
    torch.autograd.backward([out, dec], [torch.from_numpy(g1).cuda(), torch.from_numpy(g2).cuda()])
    ws64 = [a.astype(np.float64) for a in ws]; gs64 = [a.astype(np.float64) for a in gs]
    ro, rd, saved = O.hrfp_forward(xp.astype(np.float64), ws64, gs64, h, w, layers=layers)
    rg = O.hrfp_backward(g1.astype(np.float64), g2.astype(np.float64), ws64, gs64, saved)
    npf, npm, _ = O.np_plus_forward(xp.astype(np.float64), alpha.astype(np.float64), eps.astype(np.float64))
    npg = O.np_plus_backward(g1.astype(np.float64), alpha.astype(np.float64), eps.astype(np.float64), npm)
    assert out.shape == (n, cin, xh, xw) and x.grad.shape == (n, cin, xh, xw)
    _check(out.detach().cpu().numpy(), ro + npf, mode, "fwd")
    _check(dec.detach().cpu().numpy(), rd, mode, "fwd")
    _check(x.grad.cpu().numpy(), rg + npg, mode, "bwd")
    for k in (0, 7):
        assert bns[k].running_mean.shape == (layers[k][1],) and bool(torch.isfinite(bns[k].running_var).all())
    assert int(bns[7].num_batches_tracked) == 1


def test_stem_wider_than_the_kernels_is_refused_loudly():
    from mrfp_b200 import _lib
    from mrfp_b200.hrfp import get_plan
    with pytest.raises(_lib.MrfpError):
        get_plan(2, 320, 16, 12, 64, 48, torch.device("cuda"), 0)


@pytest.mark.parametrize("mode", MODES)
def test_np_plus_folded_into_the_chain_equals_the_two_step_form(mode):
    """x = OCout + NP+(xp) (deepv3.py:316-330) through the fused entry points vs NP+ kernel followed by the chain with
    x_add: same output, same gradient into xp, and NP+ vs the oracle on the difference OCout+NP+(xp) - OCout."""
    from mrfp_b200.hrfp import hrfp_chain
    from mrfp_b200.npplus import np_plus_with_draws
    n, h, w, xh, xw = 3, 96, 80, 24, 20
    ws, gs = make_hrfp_params(31)
    convs, bns = _modules(ws, gs, "cuda")
    xp_np = make_feat(32, (n, 64, xh, xw))
    rng = np.random.default_rng(33)
    alpha = torch.from_numpy((1 + 0.75 * rng.standard_normal((n, 64, 1, 1))).astype(np.float32)).cuda()
    eps = torch.from_numpy((0.75 * rng.standard_normal((n, 64, 1, 1))).astype(np.float32)).cuda()
    g1 = torch.from_numpy(rng.standard_normal((n, 64, xh, xw)).astype(np.float32)).cuda()
    g2 = torch.from_numpy(rng.standard_normal((n, 256, h // 2, w // 2)).astype(np.float32)).cuda()

    xa = torch.from_numpy(xp_np).cuda().requires_grad_(True)
    out_a, dec_a = hrfp_chain(xa, convs, bns, h, w, np_draws=(alpha, eps), math_mode=mode, update_running_stats=False)
    torch.autograd.backward([out_a, dec_a], [g1, g2])

    xb = torch.from_numpy(xp_np).cuda().requires_grad_(True)
    out_b, dec_b = hrfp_chain(xb, convs, bns, h, w, x_add=np_plus_with_draws(xb, alpha, eps), math_mode=mode,
                              update_running_stats=False)
    torch.autograd.backward([out_b, dec_b], [g1, g2])

    # fp32 mode: the two forms differ by fp32 rounding only.  bf16 mode: the BN statistics are accumulated with
    # atomics, so two runs of the SAME chain already differ by bf16 rounding flips (the documented bf16 tolerances).
    t_f, t_b = {0: (2e-6, 5e-6), 1: (5e-4, TOL[1]["bwd"]), 2: (TOL_VS_BF16_ORACLE["fwd"], TOL_VS_BF16_ORACLE["bwd"])}[mode]
    scale = out_b.abs().max().item()
    assert (out_a - out_b).abs().max().item() <= t_f * scale
    assert (dec_a - dec_b).abs().max().item() <= t_f * dec_b.abs().max().item()
    gscale = xb.grad.abs().max().item()
    assert (xa.grad - xb.grad).abs().max().item() <= t_b * gscale
    # and against the oracle's NP+ (fp64): (OCout + NP+(xp)) - OCout
    out_plain, _ = hrfp_chain(xb.detach(), convs, bns, h, w, want_dec=False, math_mode=mode, update_running_stats=False)
    ref, _, _ = O.np_plus_forward(xp_np.astype(np.float64), alpha.cpu().numpy().astype(np.float64).reshape(n, 64),
                                  eps.cpu().numpy().astype(np.float64).reshape(n, 64))
    got = (out_a - out_plain).detach().cpu().numpy()
    assert np.abs(got - ref).max() <= 1e-5 * np.abs(ref).max() + (2e-6 if mode == 0 else t_f) * scale


def test_plan_geometry_768():
    from mrfp_b200.hrfp import HrfpPlan
    p = HrfpPlan(8, 64, 192, 192, 768, 768, "cuda", 0)
    sizes = [192] + [s[5] for s in p.stages]
    assert sizes == [192, 231, 277, 332, 384, 384, 321, 256, 192]
    assert [s[:3] for s in p.stages] == [tuple(l) for l in O.HRFP_LAYERS]
    g = np.load(os.path.join(GOLDEN, "lut.npz"))
    lut = p.lut.cpu().numpy()
    # the blob starts with idx_h, idx_w of stage 0
    assert np.array_equal(lut[:231], g["768_h_0"]) and np.array_equal(lut[231:462], g["768_w_0"])


def test_plus_add():
    from mrfp_b200.hrfp import hrfp_plus_add
    a = torch.randn(2, 8, 12, 14, device="cuda", requires_grad=True)
    b = torch.randn(2, 8, 12, 14, device="cuda", requires_grad=True)
    o = hrfp_plus_add(a, b)
    assert torch.equal(o, a + b)
    o.sum().backward()
    assert torch.equal(a.grad, torch.ones_like(a)) and torch.equal(b.grad, torch.ones_like(b))


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("lo", [(12, 10), (24, 20), (7, 33)])
def test_plus_add_with_bilinear_upsample_matches_aten(lo, mode):
    """HRFP+ tail (deepv3.py:356-357): Upsample(dec1, bilinear, align_corners=True) + OCout_dec from the low-resolution
    dec1 in one kernel vs F.interpolate + the materialised add; gradient wrt dec1 = ATen's bilinear backward."""
    import torch.nn.functional as F
    from mrfp_b200.hrfp import hrfp_chain, hrfp_plus_add, hrfp_plus_add_upsampled
    n, h, w, xh, xw = 2, 96, 80, 24, 20
    ws, gs = make_hrfp_params(51)
    convs, bns = _modules(ws, gs, "cuda")
    xp = torch.from_numpy(make_feat(52, (n, 64, xh, xw))).cuda()
    torch.manual_seed(53)
    d_lo = torch.randn(n, 256, *lo, device="cuda")
    g = torch.randn(n, 256, h // 2, w // 2, device="cuda")
    xa = xp.clone().requires_grad_(True); da = d_lo.clone().requires_grad_(True)
    _, dec_a = hrfp_chain(xa, convs, bns, h, w, want_out=False, math_mode=mode, lazy_dec=True, update_running_stats=False)
    oa = hrfp_plus_add_upsampled(da, dec_a)
    oa.backward(g)
    xb = xp.clone().requires_grad_(True); db = d_lo.clone().requires_grad_(True)
    _, dec_b = hrfp_chain(xb, convs, bns, h, w, want_out=False, math_mode=mode, lazy_dec=True, update_running_stats=False)
    ob = hrfp_plus_add(F.interpolate(db, size=(h // 2, w // 2), mode="bilinear", align_corners=True), dec_b)
    ob.backward(g)
    # both sides take OCout_dec from the same stored conv output, so the forward agrees tightly in either mode (bf16 mode:
    # the BN statistics of the two chain runs differ in their last bits through the atomics' order)
    t_f, t_b = {0: (2e-6, 5e-6), 1: (5e-4, TOL[1]["bwd"]), 2: (2e-5, TOL_VS_BF16_ORACLE["bwd"])}[mode]
    assert (oa - ob).abs().max().item() <= t_f * ob.abs().max().item()
    assert torch.allclose(da.grad, db.grad, rtol=1e-6, atol=1e-6 * db.grad.abs().max().item())
    assert (xa.grad - xb.grad).abs().max().item() <= t_b * xb.grad.abs().max().item()
    # the interpolation alone, tight: subtract the OCout_dec-only output (fp32 mode is deterministic up to the BN atomics)
    zero = torch.zeros_like(d_lo)
    _, dec_c = hrfp_chain(xp, convs, bns, h, w, want_out=False, math_mode=0, lazy_dec=True, update_running_stats=False)
    only_dec = hrfp_plus_add_upsampled(zero, dec_c)
    _, dec_d = hrfp_chain(xp, convs, bns, h, w, want_out=False, math_mode=0, lazy_dec=True, update_running_stats=False)
    interp = hrfp_plus_add_upsampled(d_lo, dec_d) - only_dec
    ref = F.interpolate(d_lo, size=(h // 2, w // 2), mode="bilinear", align_corners=True)
    assert (interp - ref).abs().max().item() <= 2e-6 * ref.abs().max().item() + 2e-6 * only_dec.abs().max().item()


def test_plus_tail_multi_tile_bf16_matches_materialised_add():
    """The ldmatrix tail kernel (bf16 path) on a row of three 128-pixel tiles, the last one partial: fused Upsample + add
    from the low-resolution dec1 vs F.interpolate + the materialised add on the same chain state."""
    import torch.nn.functional as F
    from mrfp_b200.hrfp import hrfp_chain, hrfp_plus_add, hrfp_plus_add_upsampled
    n, h, w, xh, xw = 1, 96, 544, 24, 136
    ws, gs = make_hrfp_params(61)
    convs, bns = _modules(ws, gs, "cuda")
    xp = torch.from_numpy(make_feat(62, (n, 64, xh, xw))).cuda()
    torch.manual_seed(63)
    d_lo = torch.randn(n, 256, 24, 136, device="cuda")
    _, dec = hrfp_chain(xp, convs, bns, h, w, want_out=False, math_mode=2, lazy_dec=True, update_running_stats=False)
    fused = hrfp_plus_add_upsampled(d_lo, dec)
    ref = hrfp_plus_add(F.interpolate(d_lo, size=(h // 2, w // 2), mode="bilinear", align_corners=True), dec)
    assert fused.shape == (n, 256, 48, 272)
    assert (fused - ref).abs().max().item() <= 2e-6 * ref.abs().max().item()


def test_lazy_dec_handle_matches_materialised_path():
    """hrfp_plus_add on the HrfpDec handle (OCout_dec never materialised) == add of the materialised tensor,
    forward and both gradients."""
    from mrfp_b200.hrfp import hrfp_chain, hrfp_plus_add
    n, h, w = 2, 48, 48
    ws, gs = make_hrfp_params(3)
    xp_np = make_feat(4, (n, 64, 12, 12))
    res = []
    for lazy in (False, True):
        convs, bns = _modules(ws, gs, "cuda")
        xp = torch.from_numpy(xp_np).cuda().requires_grad_(True)
        dec1 = torch.from_numpy(np.random.default_rng(5).standard_normal((n, 256, 24, 24)).astype(np.float32)).cuda().requires_grad_(True)
        out, dec = hrfp_chain(xp, convs, bns, h, w, math_mode=0, lazy_dec=lazy)
        y = hrfp_plus_add(dec1, dec)
        g1 = torch.from_numpy(np.random.default_rng(6).standard_normal((n, 64, 12, 12)).astype(np.float32)).cuda()
        g2 = torch.from_numpy(np.random.default_rng(7).standard_normal((n, 256, 24, 24)).astype(np.float32)).cuda()
        torch.autograd.backward([out, y], [g1, g2])
        res.append((y.detach().clone(), xp.grad.clone(), dec1.grad.clone()))
    for a, b in zip(res[0], res[1]):
        assert torch.allclose(a, b, rtol=1e-5, atol=1e-5 * a.abs().max().item())
    # encoder-only chain with the handle (p >= .5, p3 < .5 in the reference's gating)
    convs, bns = _modules(ws, gs, "cuda")
    xp = torch.from_numpy(xp_np).cuda().requires_grad_(True)
    dec1 = torch.zeros(n, 256, 24, 24, device="cuda")
    out, dec = hrfp_chain(xp, convs, bns, h, w, math_mode=0, want_out=False, want_dec=True, lazy_dec=True)
    assert out is None
    y = hrfp_plus_add(dec1, dec)
    y.backward(g2)
    assert torch.isfinite(xp.grad).all() and xp.grad.abs().sum() > 0
    assert int(bns[3].num_batches_tracked) == 1 and int(bns[4].num_batches_tracked) == 0


def test_bad_plan_arguments():
    import ctypes
    from mrfp_b200 import _lib
    lib = _lib.load()
    h = ctypes.c_void_p()
    assert lib.mrfp_hrfp_plan_create(ctypes.byref(h), 0, 64, 12, 12, 48, 48, None, 0) == -2
    assert lib.mrfp_hrfp_plan_create(ctypes.byref(h), 2, 300, 12, 12, 48, 48, None, 0) == -4      # wider than the kernels
    assert lib.mrfp_hrfp_plan_create(ctypes.byref(h), 2, 64, 12, 12, 48, 48, None, 3) == -4        # unknown math mode
    bad_w = (ctypes.c_int * 4)(64, 48, 128, 256)
    assert lib.mrfp_hrfp_plan_create(ctypes.byref(h), 2, 64, 12, 12, 48, 48, bad_w, 2) == -4       # encoder width not a power of two
    # xp must have the size the chain ends at, (ceil(h/4), ceil(w/4)) — torch.add would raise in the reference (deepv3.py:330)
    assert lib.mrfp_hrfp_plan_create(ctypes.byref(h), 2, 64, 24, 24, 48, 48, None, 0) == -2
    assert lib.mrfp_hrfp_plan_create(ctypes.byref(h), 2, 64, 12, 13, 48, 48, None, 2) == -2
    for mode in (0, 1, 2):
        assert lib.mrfp_hrfp_plan_create(ctypes.byref(h), 2, 24, 12, 12, 48, 48, None, mode) == 0
        lib.mrfp_hrfp_plan_destroy(h)
    assert lib.mrfp_hrfp_plan_ws_bytes(None) == 0


# the last geometry has output rows of 46 pixels: rows of g are not 16-byte aligned, so the backward takes plain loads
# instead of the per-tile TMA box
# ... and the one before it the widest classifier the kernels take (24 classes), without a bias
@pytest.mark.parametrize("geom", [(2, 96, 80, (24, 20), 19), (1, 96, 544, (24, 136), 19), (2, 64, 48, (16, 12), 7),
                                  (1, 128, 160, (32, 40), -24), (2, 92, 92, (23, 20), 19)])
def test_tail_fused_through_the_classifier_equals_the_unfused_tail(geom):
    """deepv3.py:356-361: final2(Upsample(dec1) + OCout_dec) through mrfp_hrfp_tail_final2_* (one kernel per direction,
    nothing materialised at (N,256,h/2,w/2)) vs the Upsample+add kernel followed by the module's own 1x1 conv: output,
    gradients to dec1, W2, b2 and xp.  Both sides use the same stored conv output, so they differ by the bf16 rounding of
    the classifier operands (activations and W2) and of the rank-K gradient that joins the chain."""
    from mrfp_b200.hrfp import hrfp_chain, hrfp_plus_add_upsampled, hrfp_plus_final2, tail_final2_supported
    n, h, w, lo, k = geom
    has_bias, k = k > 0, abs(k)                      # a negative class count: no bias
    xh, xw = math.ceil(h / 4), math.ceil(w / 4)
    ws, gs = make_hrfp_params(71)
    convs, bns = _modules(ws, gs, "cuda")
    torch.manual_seed(72)
    final2 = torch.nn.Conv2d(256, k, 1, bias=has_bias).cuda()
    xp = torch.from_numpy(make_feat(73, (n, 64, xh, xw))).cuda()
    d_lo = torch.randn(n, 256, *lo, device="cuda")
    g = torch.randn(n, k, h // 2, w // 2, device="cuda")
    res = []
    for fused in (True, False):
        final2.zero_grad(set_to_none=True)
        xa = xp.clone().requires_grad_(True); da = d_lo.clone().requires_grad_(True)
        _, dec = hrfp_chain(xa, convs, bns, h, w, want_out=False, math_mode=2, lazy_dec=True, update_running_stats=False)
        if fused:
            assert tail_final2_supported(da, final2, dec)
            out = hrfp_plus_final2(da, final2, dec)
        else:
            out = final2(hrfp_plus_add_upsampled(da, dec))
        out.backward(g)
        gb = final2.bias.grad if has_bias else torch.ones(1, device="cuda")
        res.append([t.detach().clone() for t in (out, da.grad, final2.weight.grad, gb, xa.grad)])
    names = ("dec2", "g_dec1", "g_W2", "g_b2", "g_xp")
    tols = (1e-2, 1e-2, 1e-2, 1e-5, TOL_VS_BF16_ORACLE["bwd"])
    for name, a, b, tol in zip(names, res[0], res[1], tols):
        err = float((a.double() - b.double()).norm() / b.double().norm())
        assert err <= tol, (name, err)
    # the low-resolution half alone is exact arithmetic re-association: with OCout_dec's contribution removed by
    # linearity (zero classifier on the chain side is not expressible), check dec2 against fp64 directly
    _, dec = hrfp_chain(xp, convs, bns, h, w, want_out=False, math_mode=2, lazy_dec=True, update_running_stats=False)
    full = hrfp_plus_add_upsampled(d_lo, dec).double()
    ref = torch.nn.functional.conv2d(full, final2.weight.double(), final2.bias.double() if has_bias else None)
    _, dec = hrfp_chain(xp, convs, bns, h, w, want_out=False, math_mode=2, lazy_dec=True, update_running_stats=False)
    got = hrfp_plus_final2(d_lo, final2, dec)
    assert float((got.double() - ref).norm() / ref.norm()) <= 5e-3


# the last geometry has a stage-4 plane of 50 x 44: neither a multiple of the dgrad's 16 x 8 tile on either axis
@pytest.mark.parametrize("geom", [(2, 96, 80, (24, 20), 19), (1, 96, 544, (24, 136), 7), (2, 100, 88, (25, 20), 19)])
@pytest.mark.parametrize("fuse", [3, 1, 0])
@pytest.mark.parametrize("want_out", [True, False])
def test_rank_k_form_of_the_tail_gradient_in_the_full_chain(geom, fuse, want_out, monkeypatch):
    """The gradient of OCout_dec out of the fused classifier tail is W2^T g (rank K): by default it joins the chain as its two
    factors and the stage-4 dgrad accumulates their product as one more k-block (mrfp_hrfp_tail_final2_bwd_rk + MRFP_DEC_GRAD_RANK_K,
    conv_gather.cu ADD == 2) — against the materialised (N, h/2, w/2, 256) bf16 tensor added in that dgrad's epilogue
    (MRFP_TAIL_RANKK=0) and against the unfused tail.  Without the fused BN backward (fuse bit 1 off: fuse 0, 1) the stage-4
    dgrad is the tap kernel and the product is expanded into the dA buffer first; in the encoder-only backward
    (want_out=False, no stage-4 dgrad) the expansion is dA_3 itself."""
    from mrfp_b200.hrfp import hrfp_chain, hrfp_plus_add_upsampled, hrfp_plus_final2, tail_final2_supported
    n, h, w, lo, k = geom
    xh, xw = math.ceil(h / 4), math.ceil(w / 4)
    ws, gs = make_hrfp_params(81)
    convs, bns = _modules(ws, gs, "cuda")
    torch.manual_seed(82)
    final2 = torch.nn.Conv2d(256, k, 1, bias=True).cuda()
    xp = torch.from_numpy(make_feat(83, (n, 64, xh, xw))).cuda()
    d_lo = torch.randn(n, 256, *lo, device="cuda")
    g = torch.randn(n, k, h // 2, w // 2, device="cuda")
    gx = torch.randn(n, 64, xh, xw, device="cuda")
    res = {}
    for name in ("rank_k", "materialised", "unfused"):
        monkeypatch.setenv("MRFP_TAIL_RANKK", "0" if name == "materialised" else "1")
        final2.zero_grad(set_to_none=True)
        xa = xp.clone().requires_grad_(True); da = d_lo.clone().requires_grad_(True)
        x, dec = hrfp_chain(xa, convs, bns, h, w, want_out=want_out, math_mode=2, lazy_dec=True, update_running_stats=False,
                            fuse=fuse)
        assert dec.plan.fuse == fuse
        if name != "unfused":
            assert tail_final2_supported(da, final2, dec)
        out = hrfp_plus_final2(da, final2, dec) if name != "unfused" else final2(hrfp_plus_add_upsampled(da, dec))
        torch.autograd.backward([x, out] if want_out else [out], [gx, g] if want_out else [g])
        res[name] = [t.detach().clone() for t in (out, da.grad, final2.weight.grad, xa.grad)]
    rel = lambda a, b: float((a.double() - b.double()).norm() / b.double().norm())
    print({nm: rel(res["rank_k"][i], res["materialised"][i]) for i, nm in enumerate(("dec2", "g_dec1", "g_W2", "g_xp"))})
    for i, nm in enumerate(("dec2", "g_dec1", "g_W2")):
        assert rel(res["rank_k"][i], res["materialised"][i]) <= 1e-5, nm      # the same kernels up to the atomics' order
    assert rel(res["rank_k"][3], res["materialised"][3]) <= 2e-2              # one rounding instead of two on the way into dA_3
    assert rel(res["rank_k"][3], res["unfused"][3]) <= TOL_VS_BF16_ORACLE["bwd"]
    assert rel(res["materialised"][3], res["unfused"][3]) <= TOL_VS_BF16_ORACLE["bwd"]
