"""HRFP chain at the BENCHMARKED shapes (BASELINE config[0] / config[1]: 768x768 crop, batch 2 and 8) against the
reference's own operators evaluated in fp64 on the same GPU, next to the reference's own arithmetic (fp32 storage,
cuDNN convolutions under torch's TF32 default) measured against the same fp64 run.

SURVEY.md §7 criterion for a tensor-core path that claims the reference's precision (MRFP_MATH_TF32): error <= ~2x the
reference's TF32 error against fp64.  The default bf16 path (bf16 operands AND bf16 storage of every intermediate) is
held to stated L2-relative bounds and its distance is reported in units of the reference's TF32 error.  Errors are
L2-relative (||got - ref||_2 / ||ref||_2): the max-norm of a gradient through eight ReLU stages is dominated by a
handful of mask flips of near-zero pre-activations and says little about a systematic error.

The reference's operators run with `exact_adjoint=True` (oracle/torch_port.py): ATen's CUDA backward of
F.interpolate(mode='nearest', scale_factor=1.2) is not the adjoint of its own forward (tools/adjoint_nearest.py: <Lx,v> and
<x,L^T v> differ by 20-40 % on this torch; the CPU kernel is exact), so the as-is CUDA autograd gradient is 0.5-0.6 away
(L2) from the reference's CPU gradient, from the fixtures in tests/golden/ and from the fp64 chain rule.  The distance
of that as-is gradient is recorded next to the others; parity is defined against the adjoint (= the CPU reference).

Every measured number is written to gpurun_out/parity_fullsize.json (quoted in DESIGN.md §3.5).
"""
import json
import math
import os

import numpy as np
import pytest
import torch

from oracle import torch_port as TP
from tests.common import ROOT, make_feat, make_hrfp_params

pytestmark = pytest.mark.gpu

H = W = 768
XH = XW = 192
# L2-relative bounds of the bf16 path (operands and storage bf16, fp32 accumulate) against fp64
# (measured at batch 2 / 8: out 2.35e-2, dec 1.02e-2, gx 1.65e-1 = 3.2x the reference's own TF32 gradient error; the gradient
# of a chain of eight ReLU stages moves by ~sqrt(fraction of flipped masks), so its error is the square root of the
# activations' error, for the reference's TF32 run (5.1e-2) as for this path)
BF16_L2 = dict(out=3.0e-2, dec=1.5e-2, gx=2.5e-1)
FP32_L2 = dict(out=2e-5, dec=2e-5, gx=1e-4)


def _l2(got, ref):
    ref = ref.detach().double()
    return float(((got.detach().double() - ref).norm() / ref.norm().clamp_min(1e-300)).item())


def _mx(got, ref):
    ref = ref.detach().double()
    return float(((got.detach().double() - ref).abs().max() / ref.abs().max().clamp_min(1e-300)).item())


def _reference(xp, ws, gs, g1, g2, dtype, tf32, exact_adjoint=True):
    """The reference's operator sequence (deepv3.py:320-327 via oracle/torch_port.py) on the GPU."""
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = tf32
    torch.backends.cuda.matmul.allow_tf32 = tf32
    try:
        convs, bns = TP.make_layers(ws, gs)
        convs = [c.to("cuda", dtype) for c in convs]
        bns = [b.to("cuda", dtype) for b in bns]
        x = xp.detach().to(dtype).clone().requires_grad_(True)
        out, dec = TP.hrfp_chain(convs, bns, x, H, W, exact_adjoint=exact_adjoint)
        torch.autograd.backward([out, dec], [g1.to(dtype), g2.to(dtype)])
        res = dict(out=out.detach(), dec=dec.detach(), gx=x.grad.detach(),
                   rm=[b.running_mean.detach().double() for b in bns], rv=[b.running_var.detach().double() for b in bns])
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
    return res


def _ours(xp, ws, gs, g1, g2, mode):
    from mrfp_b200.hrfp import hrfp_chain
    convs, bns = TP.make_layers(ws, gs)
    convs = [c.cuda() for c in convs]; bns = [b.cuda() for b in bns]
    x = xp.detach().clone().requires_grad_(True)
    out, dec = hrfp_chain(x, convs, bns, H, W, math_mode=mode)
    torch.autograd.backward([out, dec], [g1, g2])
    return dict(out=out.detach(), dec=dec.detach(), gx=x.grad.detach(),
                rm=[b.running_mean.detach().double() for b in bns], rv=[b.running_var.detach().double() for b in bns])


def _record(tag, payload):
    path = os.path.join(ROOT, "gpurun_out", "parity_fullsize.json")
    os.makedirs(os.path.dirname(path), exist_ok=True)
    data = {}
    if os.path.exists(path):
        try:
            data = json.load(open(path))
        except Exception:
            data = {}
    data[tag] = payload
    with open(path, "w") as f:
        json.dump(data, f, indent=1, sort_keys=True)


@pytest.mark.parametrize("n", [2, 8])
def test_chain_at_benchmarked_shape_vs_fp64_and_vs_reference_tf32(n):
    ws, gs = make_hrfp_params(11)
    xp = torch.from_numpy(make_feat(12, (n, 64, XH, XW))).cuda()
    gen = torch.Generator(device="cuda").manual_seed(13)
    g1 = torch.randn(n, 64, XH, XW, device="cuda", generator=gen)
    g2 = torch.randn(n, 256, H // 2, W // 2, device="cuda", generator=gen)

    ref64 = _reference(xp, ws, gs, g1, g2, torch.float64, False)
    rows = {}
    for name, kw in (("reference_fp32", dict(dtype=torch.float32, tf32=False)), ("reference_tf32", dict(dtype=torch.float32, tf32=True))):
        r = _reference(xp, ws, gs, g1, g2, **kw)
        rows[name] = {k: dict(l2=_l2(r[k], ref64[k]), max=_mx(r[k], ref64[k])) for k in ("out", "dec", "gx")}
        del r
    if n == 2:      # the as-is CUDA autograd (ATen's inexact nearest backward at scale 1.2), for the record
        r = _reference(xp, ws, gs, g1, g2, torch.float64, False, exact_adjoint=False)
        rows["aten_cuda_autograd_fp64_as_is"] = {k: dict(l2=_l2(r[k], ref64[k]), max=_mx(r[k], ref64[k])) for k in ("out", "dec", "gx")}
        del r
    modes = [("ours_tf32", 1), ("ours_bf16", 2)] + ([("ours_fp32", 0)] if n == 2 else [])
    runs = {}
    for name, mode in modes:
        r = _ours(xp, ws, gs, g1, g2, mode)
        rows[name] = {k: dict(l2=_l2(r[k], ref64[k]), max=_mx(r[k], ref64[k])) for k in ("out", "dec", "gx")}
        # running statistics: error relative to the largest entry of each buffer (a channel mean near zero carries
        # the convolution's absolute error, not a relative one)
        rows[name]["running_stats_max_rel"] = max(
            max(float((a - b).abs().max() / b.abs().max()) for a, b in zip(r["rm"], ref64["rm"])),
            max(float((a - b).abs().max() / b.abs().max()) for a, b in zip(r["rv"], ref64["rv"])))
        runs[name] = r
    for name in rows:
        if name.startswith("ours"):
            rows[name]["l2_in_units_of_reference_tf32"] = {k: rows[name][k]["l2"] / max(rows["reference_tf32"][k]["l2"], 1e-30)
                                                           for k in ("out", "dec", "gx")}
    # no systematic bias hiding under the noise: the error is uncorrelated with the signal (a dropped or mis-scaled
    # BN-backward term would show as a projection of the error onto the reference gradient)
    for name in runs:
        e = (runs[name]["gx"].double() - ref64["gx"]).flatten()
        g = ref64["gx"].flatten()
        rows[name]["gx_error_projection_on_reference"] = float((e @ g) / (g @ g))
    _record(f"batch{n}_768x768", rows)
    print(json.dumps(rows, indent=1))

    t32 = rows["reference_tf32"]
    # (1) the TF32 tensor-core mode carries the reference's own precision: <= 2x its TF32 error (SURVEY §7), with a floor
    #     of the fp32 reference's own distance for quantities where TF32 happens to sit unusually close
    for k in ("out", "dec", "gx"):
        floor = 4 * rows["reference_fp32"][k]["l2"]
        assert rows["ours_tf32"][k]["l2"] <= 2.0 * t32[k]["l2"] + floor, (k, rows["ours_tf32"][k], t32[k])
    assert rows["ours_tf32"]["running_stats_max_rel"] <= 2e-3
    assert abs(rows["ours_tf32"]["gx_error_projection_on_reference"]) <= 5e-3
    # (2) the default bf16 mode: stated L2 bounds
    for k in ("out", "dec", "gx"):
        assert rows["ours_bf16"][k]["l2"] <= BF16_L2[k], (k, rows["ours_bf16"][k])
    assert rows["ours_bf16"]["running_stats_max_rel"] <= 3e-2
    assert abs(rows["ours_bf16"]["gx_error_projection_on_reference"]) <= 3e-2
    # (3) fp32 CUDA-core mode reproduces the fp32 reference (its own gradient error against fp64: 1.3e-3, mask flips)
    if "ours_fp32" in rows:
        for k in ("out", "dec"):
            assert rows["ours_fp32"][k]["l2"] <= FP32_L2[k], (k, rows["ours_fp32"][k])
        assert rows["ours_fp32"]["gx"]["l2"] <= 3 * rows["reference_fp32"]["gx"]["l2"] + 1e-4
        assert rows["ours_fp32"]["running_stats_max_rel"] <= 1e-4


def test_fused_np_plus_and_tail_at_benchmarked_shape():
    """The step bench.py times (np_draws folded into the chain, lazy OCout_dec, bilinear tail) at config[0] size against
    the reference's operators in fp64: x = OCout + NP+(xp), d1 = Upsample(dec1) + OCout_dec and the gradient into xp."""
    import torch.nn.functional as F
    from mrfp_b200.hrfp import hrfp_chain, hrfp_plus_add_upsampled
    n = 2
    ws, gs = make_hrfp_params(21)
    xp = torch.from_numpy(make_feat(22, (n, 64, XH, XW))).cuda()
    gen = torch.Generator(device="cuda").manual_seed(23)
    alpha = 1 + 0.75 * torch.randn(n, 64, 1, 1, device="cuda", generator=gen)
    eps = 0.75 * torch.randn(n, 64, 1, 1, device="cuda", generator=gen)
    d1 = torch.randn(n, 256, XH, XW, device="cuda", generator=gen)
    g1 = torch.randn(n, 64, XH, XW, device="cuda", generator=gen)
    g2 = torch.randn(n, 256, H // 2, W // 2, device="cuda", generator=gen)
    # fp64 reference
    convs, bns = TP.make_layers(ws, gs)
    convs = [c.to("cuda", torch.float64) for c in convs]; bns = [b.to("cuda", torch.float64) for b in bns]
    x64 = xp.double().requires_grad_(True)
    oc, dec = TP.hrfp_chain(convs, bns, x64, H, W, exact_adjoint=True)
    xr = oc + TP.np_plus(x64, alpha.double(), eps.double())
    dr = dec + F.interpolate(d1.double(), size=(H // 2, W // 2), mode="bilinear", align_corners=True)
    torch.autograd.backward([xr, dr], [g1.double(), g2.double()])
    rows = {}
    # the same step with the reference's own arithmetic (fp32 storage, TF32 cuDNN convolutions)
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = True
    try:
        c32, b32 = TP.make_layers(ws, gs)
        c32 = [c.cuda() for c in c32]; b32 = [b.cuda() for b in b32]
        x32 = xp.detach().clone().requires_grad_(True)
        oc32, dec32 = TP.hrfp_chain(c32, b32, x32, H, W, exact_adjoint=True)
        xr32 = oc32 + TP.np_plus(x32, alpha, eps)
        dr32 = dec32 + F.interpolate(d1, size=(H // 2, W // 2), mode="bilinear", align_corners=True)
        torch.autograd.backward([xr32, dr32], [g1, g2])
        rows["reference_tf32"] = dict(x=_l2(xr32, xr), d1=_l2(dr32, dr), gx=_l2(x32.grad, x64.grad))
        del oc32, dec32, xr32, dr32
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
    t32 = rows["reference_tf32"]
    bounds = {"tf32": tuple(2.0 * t32[k] + 1e-5 for k in ("x", "d1", "gx")),
              "bf16": (1e-2, 1e-2, BF16_L2["gx"])}       # x and d1 carry their fp32 operand (NP+(xp), Upsample(dec1)) unrounded
    for name, mode in (("tf32", 1), ("bf16", 2)):
        bx, bd, bg = bounds[name]
        convs2, bns2 = TP.make_layers(ws, gs)
        convs2 = [c.cuda() for c in convs2]; bns2 = [b.cuda() for b in bns2]
        xa = xp.clone().requires_grad_(True)
        xo, dh = hrfp_chain(xa, convs2, bns2, H, W, math_mode=mode, lazy_dec=True, np_draws=(alpha, eps))
        do = hrfp_plus_add_upsampled(d1, dh)
        torch.autograd.backward([xo, do], [g1, g2])
        rows[name] = dict(x=_l2(xo, xr), d1=_l2(do, dr), gx=_l2(xa.grad, x64.grad), bounds=[bx, bd, bg])
    _record("fused_step_batch2_768x768", rows)
    print(json.dumps(rows))
    for name in ("tf32", "bf16"):
        bx, bd, bg = rows[name]["bounds"]
        assert rows[name]["x"] <= bx and rows[name]["d1"] <= bd and rows[name]["gx"] <= bg, rows


def test_classifier_tail_at_benchmarked_shape():
    """deepv3.py:356-361 through the classifier (mrfp_hrfp_tail_final2_fwd / _bwd, csrc/tail_final2.cu) at config[0] size:
    dec2 and the high-resolution gradients of final2 against fp64 built from the materialised OCout_dec of the same
    chain (so the difference is the bf16 rounding of the classifier operands only), the gradient that joins the chain
    against W2^T g rounded to bf16."""
    import torch.nn.functional as F
    from mrfp_b200.hrfp import DEC_GRAD_NHWC, DEC_GRAD_RANK_K, hrfp_chain, hrfp_plus_add_upsampled, hrfp_plus_final2
    n, k = 2, 19
    ws, gs = make_hrfp_params(31)
    gen = torch.Generator(device="cuda").manual_seed(32)
    xp = torch.from_numpy(make_feat(33, (n, 64, XH, XW))).cuda()
    d1 = torch.randn(n, 256, XH, XW, device="cuda", generator=gen)
    g = torch.randn(n, k, H // 2, W // 2, device="cuda", generator=gen)
    torch.manual_seed(34)
    final2 = torch.nn.Conv2d(256, k, 1).cuda()

    def chain():
        convs, bns = TP.make_layers(ws, gs)
        convs = [c.cuda() for c in convs]; bns = [b.cuda() for b in bns]
        return hrfp_chain(xp, convs, bns, H, W, want_out=False, math_mode=2, lazy_dec=True, update_running_stats=False)[1]

    da = d1.clone().requires_grad_(True)
    dec = chain()
    out = hrfp_plus_final2(da, final2, dec)
    out.backward(g)
    slot = dec.slot
    assert slot.form in (DEC_GRAD_NHWC, DEC_GRAD_RANK_K), slot.form    # the tail's backward parked its gradient
    g_nhwc = slot.g if slot.form == DEC_GRAD_NHWC else None        # (N, h/2, w/2, 256) bf16: the gradient of OCout_dec
    if slot.form == DEC_GRAD_RANK_K:                               # ... left as its two factors (mrfp_hrfp_tail_final2_bwd_rk)
        g64, w2t = slot.g, slot.w2t
        assert float(g64[..., k:].abs().max()) == 0.0 and float(w2t[:, k:].abs().max()) == 0.0
        assert torch.equal(g64[..., :k], g.bfloat16().permute(0, 2, 3, 1)) and torch.equal(w2t[:, :k], final2.weight.detach().reshape(k, 256).bfloat16().t())
        g_nhwc = g64.double() @ w2t.double().t()
    full = hrfp_plus_add_upsampled(d1, chain()).double().requires_grad_(True)
    w64 = final2.weight.detach().double().requires_grad_(True); b64 = final2.bias.detach().double().requires_grad_(True)
    ref = F.conv2d(full, w64, b64)
    ref.backward(g.double())
    # W2^T g in fp64 with the classifier rounded to bf16 as the kernel sees it
    w2b = final2.weight.detach().reshape(k, 256).bfloat16().double()
    gd = torch.einsum("nkhw,kc->nhwc", g.bfloat16().double(), w2b)
    # the gradient to dec1 goes through the low-resolution product: W2^T . (adjoint of the bilinear Upsample)(g)
    d64 = d1.double().requires_grad_(True)
    F.interpolate(F.conv2d(d64, w64.detach()), size=(H // 2, W // 2), mode="bilinear", align_corners=True).backward(g.double())
    rows = dict(dec2=_l2(out, ref), g_w2=_l2(final2.weight.grad, w64.grad), g_b2=_l2(final2.bias.grad, b64.grad),
                g_dec1=_l2(da.grad, d64.grad))
    if g_nhwc is not None:
        rows["g_dec_nhwc"] = _l2(g_nhwc, gd)
    _record("classifier_tail_batch2_768x768", rows)
    print(json.dumps(rows))
    assert rows["dec2"] <= 5e-3 and rows["g_w2"] <= 5e-3 and rows["g_b2"] <= 1e-5 and rows["g_dec1"] <= 5e-3, rows
    assert rows.get("g_dec_nhwc", 0.0) <= 5e-3, rows
