"""The classifier-tail kernels alone (csrc/tail_final2.cu: tail_final2_fwd_kernel, tail_final2_bwd_kernel in both its
materialised and its rank-K form) against fp64, element by element, on caller buffers with guard bands.

The operand the tail's mma.sync sees is ReLU(BN_3(Y_3)) at the nearest source pixel, computed as fmaxf(fmaf(scale, y,
shift), 0) in fp32 and rounded once to bf16 (common.cuh: bn_relu_x2).  mrfp_hrfp_plus_add(0, dec) computes the same fp32
value on the same chain state, so `ocdec.bfloat16()` below is that operand bit for bit; everything the kernels add on top
of it is bounded per element from the arithmetic they do."""
import math

import pytest
import torch
import torch.nn.functional as F

from tests.common import make_feat, make_hrfp_params

pytestmark = pytest.mark.gpu

U = 2 ** -23          # one fp32 ulp relative to the value (covers round-to-nearest and truncating adders)
PX = 64               # output pixels per tile of both kernels
GUARD = 256           # elements of NaN behind every output buffer


def _chain(n, h, w, math_mode=2):
    from mrfp_b200.hrfp import hrfp_chain
    from tests.test_hrfp_gpu import _modules
    ws, gs = make_hrfp_params(91)
    convs, bns = _modules(ws, gs, "cuda")
    xp = torch.from_numpy(make_feat(92 + n + h + w, (n, 64, math.ceil(h / 4), math.ceil(w / 4)))).cuda()
    _, dec = hrfp_chain(xp, convs, bns, h, w, want_out=False, math_mode=math_mode, lazy_dec=True, update_running_stats=False)
    return dec


def _ocdec(dec):
    """OCout_dec = ReLU(BN_3(Y_3))[nearest] in fp32 from the handle's own saved state (no autograd record)."""
    from mrfp_b200.hrfp import hrfp_plus_add
    with torch.no_grad():
        return hrfp_plus_add(torch.zeros(dec.shape, device="cuda"), dec)


def _guarded(shape, dtype):
    numel = math.prod(shape)
    buf = torch.full((numel + GUARD,), float("nan"), device="cuda", dtype=dtype)
    return buf, buf[:numel].view(shape)


def _untouched(buf, numel):
    return bool(torch.isnan(buf[numel:]).all())


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _fwd(dec, t_lo, w2, b2):
    from mrfp_b200 import _lib
    plan = dec.plan
    n, _, oh, ow = plan.dec_shape
    k = w2.shape[0]
    buf, out = _guarded((n, k, oh, ow), torch.float32)
    rc = _lib.load().mrfp_hrfp_tail_final2_fwd(plan.handle, dec.saved.data_ptr(), plan.lut.data_ptr(), t_lo.data_ptr(),
                                               t_lo.shape[2], t_lo.shape[3], w2.data_ptr(), None if b2 is None else b2.data_ptr(),
                                               k, out.data_ptr(), _stream())
    assert rc == 0, rc
    torch.cuda.synchronize()
    assert _untouched(buf, out.numel())
    assert not torch.isnan(out).any()
    return out.double()


def _bwd(dec, g, w2, rank_k):
    """(g_dec_nhwc | (g64, w2t64), g_w2, g_b2) of one backward launch; g_w2 / g_b2 carry a NaN guard row K."""
    from mrfp_b200 import _lib
    plan = dec.plan
    n, c, oh, ow = plan.dec_shape
    k = w2.shape[0]
    gw_buf = torch.full((k + 1, c), float("nan"), device="cuda")
    gb_buf = torch.full((k + 1,), float("nan"), device="cuda")
    lib = _lib.load()
    common = (plan.handle, dec.saved.data_ptr(), plan.lut.data_ptr(), g.data_ptr(), w2.data_ptr(), k)
    if rank_k:
        g64_buf, g64 = _guarded((n, oh, ow, 64), torch.bfloat16)
        w2t_buf = torch.full((c + 1, 64), float("nan"), device="cuda", dtype=torch.bfloat16)
        rc = lib.mrfp_hrfp_tail_final2_bwd_rk(*common, g64.data_ptr(), w2t_buf.data_ptr(), gw_buf.data_ptr(), gb_buf.data_ptr(),
                                              _stream())
        outs = (g64, w2t_buf[:c])
        guards = [_untouched(g64_buf, g64.numel()), bool(torch.isnan(w2t_buf[c]).all())]
    else:
        gd_buf, gd = _guarded((n, oh, ow, c), torch.bfloat16)
        rc = lib.mrfp_hrfp_tail_final2_bwd(*common, gd.data_ptr(), gw_buf.data_ptr(), gb_buf.data_ptr(), _stream())
        outs = (gd,)
        guards = [_untouched(gd_buf, gd.numel())]
    assert rc == 0, rc
    torch.cuda.synchronize()
    assert all(guards) and bool(torch.isnan(gw_buf[k]).all()) and bool(torch.isnan(gb_buf[k]))
    return outs, gw_buf[:k], gb_buf[:k]


# (n, h, w): the chain's image; the tail runs at (h/2, w/2).  lo: (lh, lw) of dec1.
#   48 x 132   TMA path for g (OW % 4 == 0), last 64-pixel tile has 4 pixels, batch 1
#   36 x 75    OW % 4 != 0: g through plain loads; partial last tile (11 pixels), batch 3
#   50 x 65    a last tile of one pixel, OW % 4 != 0
#   192 x 196  2 x 192 x 4 = 1536 tiles: every CTA of the 296-CTA grid walks ~5 tiles across rows and images
#   384 x 384  the 768^2 training step, batch 2
SMALL_A, SMALL_B = (1, 96, 264, (24, 64)), (3, 72, 150, (18, 36))
KS = [1, 7, 8, 9, 16, 17, 24]           # the forward's n-blocks of 8 and the backward's k-blocks of 16, edges and interiors
CASES = ([(SMALL_A, k, k % 2 == 1) for k in KS] + [(SMALL_B, k, bias) for k in KS for bias in (True, False)] +
         [((1, 100, 130, (25, 32)), 19, True), ((2, 384, 392, (96, 96)), 19, True), ((2, 768, 768, (192, 192)), 19, True)])


@pytest.mark.parametrize("geom,k,bias", CASES)
def test_tail_kernels_match_fp64(geom, k, bias):
    """Forward (and its two terms alone) and both backward forms against fp64 per element; g64 / w2t64 bit for bit."""
    n, h, w, (lh, lw) = geom
    dec = _chain(n, h, w)
    _, c, oh, ow = dec.shape
    torch.manual_seed(1000 * k + h + w + int(bias))
    a = _ocdec(dec).bfloat16().double()                  # the mma operand A (>= 0 after the ReLU)
    w2 = (0.05 * torch.randn(k, c, device="cuda")).contiguous()
    b2 = torch.randn(k, device="cuda") if bias else None
    t_lo = torch.randn(n, k, lh, lw, device="cuda")
    wb = w2.bfloat16().double()
    mm = torch.einsum("kc,nchw->nkhw", wb, a)
    mag = torch.einsum("kc,nchw->nkhw", wb.abs(), a)     # sum_c |w||a| per output element
    up = F.interpolate(t_lo.double(), size=(oh, ow), mode="bilinear", align_corners=True)
    bb = torch.zeros(k, device="cuda", dtype=torch.float64) if b2 is None else b2.double()
    bb = bb[None, :, None, None]
    tmax = t_lo.abs().max().item()
    # bf16 x bf16 products are exact in fp32: a channel quarter is 4 m16n8k16 steps of 16 products + the accumulator, then
    # 3 quarter sums: 71 fp32 additions, one ulp each; 256 (one per channel) bounds them
    e_mma = 256 * U * mag
    # the source coordinate o * float((L-1)/(O-1)) is off by <= 2 roundings = 2^-23 (L-1) pixels on each axis, and the
    # interpolant's slope is <= 2 max|t|; the fp32 evaluation of the two lerps adds <= 4 roundings of max|t|
    e_up = (2 * (lh + lw) + 4) * U * tmax
    # out = acc + (b2 + up): two fp32 roundings
    e_add = U * (mag + bb.abs() + tmax)

    def check(got, ref, bound, what):
        ratio = ((got - ref).abs() / bound.clamp_min(1e-30)).max().item()
        print(f"{what}: error/bound {ratio:.3g}")
        assert ratio <= 1.0, (what, ratio)

    check(_fwd(dec, t_lo, w2, b2), mm + up + bb, e_mma + e_up + e_add, "out")
    check(_fwd(dec, t_lo, torch.zeros_like(w2), b2), up + bb, e_up + U * (bb.abs() + tmax) + 1e-30, "out, W2 = 0")
    check(_fwd(dec, torch.zeros_like(t_lo), w2, None), mm, e_mma + 1e-30, "out, t_lo = 0 and no bias")

    # ---- backward ----
    g = torch.randn(n, k, oh, ow, device="cuda")
    gb = g.bfloat16().double()
    ref_gw = torch.einsum("nkhw,nchw->kc", gb, a)
    mag_gw = torch.einsum("nkhw,nchw->kc", gb.abs(), a)
    ref_gb, mag_gb = g.double().sum((0, 2, 3)), g.double().abs().sum((0, 2, 3))
    # reductions over pixels: a CTA adds its tiles in registers (16 pixels per mma, 64 per tile), then one fp32 atomic per
    # CTA: at most 64 * ceil(tiles / grid) + grid additions on the way to each element
    tiles = n * oh * ((ow + PX - 1) // PX)
    grid = min(tiles, 2 * torch.cuda.get_device_properties(0).multi_processor_count)
    n_add = PX * ((tiles + grid - 1) // grid) + grid
    for rank_k in (False, True):
        outs, g_w2, g_b2 = _bwd(dec, g, w2, rank_k)
        form = "rank-K" if rank_k else "materialised"
        check(g_w2.double(), ref_gw, n_add * U * mag_gw + 1e-30, f"g_w2 ({form})")    # bf16(g) . A, the kernel's operands
        check(g_b2.double(), ref_gb, n_add * U * mag_gb, f"g_b2 ({form})")            # sum of g itself, not rounded
        if rank_k:
            g64, w2t64 = outs
            want = torch.zeros(n, oh, ow, 64, device="cuda", dtype=torch.bfloat16)
            want[..., :k] = g.permute(0, 2, 3, 1).bfloat16()
            assert torch.equal(g64, want)                                  # bf16(g) NHWC, classes K..63 zero
            want_w = torch.zeros(c, 64, device="cuda", dtype=torch.bfloat16)
            want_w[:, :k] = w2.t().bfloat16()
            assert torch.equal(w2t64, want_w)
        else:
            ref_d = torch.einsum("nkhw,kc->nhwc", gb, wb)
            mag_d = torch.einsum("nkhw,kc->nhwc", gb.abs(), wb.abs())
            # two m16n8k16 k-blocks of 16 exact products, each added to the accumulator: 34 fp32 additions, then one
            # rounding to bf16 (half an ulp, 2^-8), which also scales the accumulation error by (1 + 2^-8)
            check(outs[0].double(), ref_d, 2 ** -8 * ref_d.abs() + (1 + 2 ** -8) * 34 * U * mag_d + 1e-30, "g_dec_nhwc")


@pytest.mark.parametrize("case", [
    ("ok", 19, (24, 20)),
    ("ok", 24, (24, 20)),              # the widest classifier
    ("ok", 1, (1, 4)),                 # one low-resolution row, one aligned group of columns
    ("ok", 19, (48, 20)),              # lh == oh
    ("lw % 4", 19, (24, 18)),
    ("lw % 4", 19, (24, 2)),
    ("2(lw-1) > ow-1", 19, (24, 24)),
    ("lh > oh", 19, (49, 20)),
    ("K > 24", 25, (24, 20)),
    ("tf32", 19, (24, 20)),
])
def test_tail_supported_agrees_with_the_kernels(case):
    """model.py takes the fused tail when tail_final2_supported() says so and raises if the kernels then refuse: the
    predicate must be True exactly when the forward and both backward entry points accept the launch."""
    from mrfp_b200 import _lib
    from mrfp_b200.hrfp import tail_final2_supported
    why, k, (lh, lw) = case
    n, h, w = 2, 96, 80                                  # tail at 48 x 40
    dec = _chain(n, h, w, math_mode=1 if why == "tf32" else 2)
    _, c, oh, ow = dec.shape
    plan, lib = dec.plan, _lib.load()
    conv = torch.nn.Conv2d(c, k, 1).cuda()
    dec1 = torch.zeros(n, c, lh, lw, device="cuda")
    t_lo = torch.zeros(n, k, lh, lw, device="cuda")
    w2 = conv.weight.detach().reshape(k, c).contiguous()
    out = torch.empty(n, k, oh, ow, device="cuda")
    g = torch.zeros(n, k, oh, ow, device="cuda")
    gd = torch.empty(n, oh, ow, c, device="cuda", dtype=torch.bfloat16)
    g64 = torch.empty(n, oh, ow, 64, device="cuda", dtype=torch.bfloat16)
    w2t = torch.empty(c, 64, device="cuda", dtype=torch.bfloat16)
    gw, gbias = torch.empty(k, c, device="cuda"), torch.empty(k, device="cuda")
    base = (plan.handle, dec.saved.data_ptr(), plan.lut.data_ptr())
    rcs = (lib.mrfp_hrfp_tail_final2_fwd(*base, t_lo.data_ptr(), lh, lw, w2.data_ptr(), conv.bias.data_ptr(), k, out.data_ptr(),
                                         _stream()),
           lib.mrfp_hrfp_tail_final2_bwd(*base, g.data_ptr(), w2.data_ptr(), k, gd.data_ptr(), gw.data_ptr(), gbias.data_ptr(),
                                         _stream()),
           lib.mrfp_hrfp_tail_final2_bwd_rk(*base, g.data_ptr(), w2.data_ptr(), k, g64.data_ptr(), w2t.data_ptr(), gw.data_ptr(),
                                            gbias.data_ptr(), _stream()))
    torch.cuda.synchronize()
    supported = tail_final2_supported(dec1, conv, dec)
    assert supported == (why == "ok"), (why, supported)
    assert supported == all(rc == 0 for rc in rcs), (why, rcs)
    assert supported or rcs[0] != 0, (why, rcs)          # what the predicate refuses, the forward refuses
