"""tcgen05 implicit-GEMM conv kernel alone (debug hook of the C library) vs torch conv2d on the same bf16 inputs."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _conv_tc(x_nchw, w_oihw, dil, cnt_h=None, cnt_w=None, tf32=False):
    """One conv3x3_tc_kernel launch; bf16 (default) or tf32 operands (fp32 in HBM, fp32 output)."""
    from mrfp_b200 import _lib
    lib = _lib.load()
    fn = lib.mrfp_debug_conv3x3_tf32 if tf32 else lib.mrfp_debug_conv3x3_bf16
    fn.restype = ctypes.c_int
    fn.argtypes = [ctypes.c_void_p] * 3 + [ctypes.c_int] * 6 + [ctypes.c_void_p] * 4
    dt = torch.float32 if tf32 else torch.bfloat16
    n, cin, h, w = x_nchw.shape
    cout = w_oihw.shape[0]
    x = x_nchw.permute(0, 2, 3, 1).contiguous().to(dt)
    wp = w_oihw.permute(2, 3, 0, 1).reshape(9, cout, cin).contiguous().to(dt)   # [tap][co][ci]
    out = torch.full((n, h, w, cout), float("nan"), device="cuda", dtype=dt)
    acc = torch.zeros(2, 256, device="cuda", dtype=torch.float64)
    st = torch.cuda.current_stream().cuda_stream
    rc = fn(x.data_ptr(), wp.data_ptr(), out.data_ptr(), n, h, w, cin, cout, dil,
            None if cnt_h is None else cnt_h.data_ptr(), None if cnt_w is None else cnt_w.data_ptr(),
            acc.data_ptr() if cnt_h is not None else None, st)
    assert rc == 0, rc
    torch.cuda.synchronize()
    return out.permute(0, 3, 1, 2).float(), acc, x.permute(0, 3, 1, 2).float(), wp.reshape(3, 3, cout, cin).permute(2, 3, 0, 1).float()


def _tf32(t):
    """t with the low 13 mantissa bits cleared: a TF32-representable fp32 tensor (the kernel's conversion is the identity)."""
    return (t.contiguous().view(torch.int32) & ~0x1FFF).view(torch.float32)


def _random_counts(h, w):
    cnt_h = torch.zeros(((h + 15) // 16 + 1) * 16, dtype=torch.int32, device="cuda")
    cnt_w = torch.zeros(((w + 15) // 16 + 1) * 16, dtype=torch.int32, device="cuda")
    cnt_h[:h] = torch.randint(0, 3, (h,), device="cuda", dtype=torch.int32)
    cnt_w[:w] = torch.randint(0, 3, (w,), device="cuda", dtype=torch.int32)
    return cnt_h, cnt_w


def _check_stats(got, acc, cnt_h, cnt_w, cout):
    """The BN statistics are taken over the STORED conv output, weighted by the replication counts."""
    h, w = got.shape[2:]
    wgt = (cnt_h[:h].double()[:, None] * cnt_w[:w].double()[None, :])[None, None]
    gd = got.double()
    s1 = (gd * wgt).sum((0, 2, 3)); s2 = (gd * gd * wgt).sum((0, 2, 3))
    assert torch.allclose(acc[0, :cout], s1, rtol=1e-4, atol=1e-4 * s1.abs().max().item())
    assert torch.allclose(acc[1, :cout], s2, rtol=1e-4, atol=1e-4 * s2.abs().max().item())


CONV_CHANNELS = [(64, 64, 1), (64, 64, 2), (64, 128, 2), (128, 256, 2), (256, 128, 1), (128, 64, 1)]
# the last shape has 2 x 24 x 12 = 576 tiles (256-wide: 1152): every CTA of the persistent grid walks several tiles
CONV_SHAPES = [(2, 8, 16), (2, 20, 37), (1, 50, 61), (2, 192, 192)]


@pytest.mark.parametrize("cin,cout,dil", CONV_CHANNELS)
@pytest.mark.parametrize("shape", CONV_SHAPES)
def test_conv_matches_torch(cin, cout, dil, shape):
    n, h, w = shape
    torch.manual_seed(cin + cout + dil + h)
    x = torch.relu(torch.randn(n, cin, h, w, device="cuda"))
    wt = torch.randn(cout, cin, 3, 3, device="cuda") * (2.0 / (9 * cin)) ** 0.5
    cnt_h, cnt_w = _random_counts(h, w)
    got, acc, xb, wb = _conv_tc(x, wt, dil, cnt_h, cnt_w)
    ref = F.conv2d(xb.double(), wb.double(), padding=dil, dilation=dil)
    assert not torch.isnan(got).any()
    err = (got.double() - ref).abs().max().item()
    # bf16 output rounding: half an ulp = 2^-9 relative
    assert err <= 2 ** -8 * ref.abs().max().item() + 1e-6, err
    _check_stats(got, acc, cnt_h, cnt_w, cout)


@pytest.mark.parametrize("cin,cout,dil", CONV_CHANNELS)
@pytest.mark.parametrize("shape", CONV_SHAPES)
def test_tf32_conv_matches_fp64(cin, cout, dil, shape):
    """conv3x3_tc_kernel<float> (tcgen05 kind::tf32, the TF32 math mode of the chain) against fp64 on TF32-representable
    operands: every product is exact, so the only error left is the fp32 accumulation and it is bounded per element."""
    n, h, w = shape
    torch.manual_seed(cin + cout + dil + h + 1)
    x = _tf32(torch.relu(torch.randn(n, cin, h, w, device="cuda")))
    wt = _tf32(torch.randn(cout, cin, 3, 3, device="cuda") * (2.0 / (9 * cin)) ** 0.5)
    cnt_h, cnt_w = _random_counts(h, w)
    got, acc, xb, wb = _conv_tc(x, wt, dil, cnt_h, cnt_w, tf32=True)
    assert torch.equal(xb, x) and torch.equal(wb, wt)
    ref = F.conv2d(x.double(), wt.double(), padding=dil, dilation=dil)
    mag = F.conv2d(x.double().abs(), wt.double().abs(), padding=dil, dilation=dil)     # sum |x||w| per output element
    assert not torch.isnan(got).any()
    # 11-bit x 11-bit significands: products exact in fp32; 9 cin additions in fp32, each off by at most one ulp
    # (2^-23 relative, truncating adders included) of a partial sum bounded by sum |x||w|
    bound = 9 * cin * 2 ** -23 * mag
    ratio = ((got.double() - ref).abs() / bound.clamp_min(1e-30)).max().item()
    print(f"error/bound {ratio:.3g}")
    assert ratio <= 1.0, ratio
    _check_stats(got, acc, cnt_h, cnt_w, cout)


def test_conv_without_stats_full_size_linearity():
    """D1 shape of the reference chain (256->128 @384^2), batch 2: conv(a*x) = a*conv(x) and agreement with cuDNN."""
    torch.manual_seed(0)
    x = torch.relu(torch.randn(2, 256, 384, 384, device="cuda"))
    wt = torch.randn(128, 256, 3, 3, device="cuda") * (2.0 / (9 * 256)) ** 0.5
    got, _, xb, wb = _conv_tc(x, wt, 1)
    got2, _, _, _ = _conv_tc(2 * x, wt, 1)
    assert torch.equal(got2, 2 * got)                 # exact: power-of-two scaling commutes with bf16 rounding
    with torch.backends.cudnn.flags(allow_tf32=False):       # fp32 reference; the flag is restored afterwards
        ref = F.conv2d(xb, wb, padding=1)
    assert (got - ref).abs().max().item() <= 2 ** -8 * ref.abs().max().item() + 1e-5


def _nearest_idx(src, dst):
    scale = torch.tensor(src / dst, dtype=torch.float32)
    return torch.clamp(torch.floor(torch.arange(dst, dtype=torch.float32) * scale).to(torch.int64), max=src - 1).cuda()


@pytest.mark.parametrize("cin,cout,dil", [(64, 64, 1), (64, 64, 2), (64, 128, 2), (128, 256, 2), (256, 128, 1), (128, 64, 1)])
# the last geometry has 2 x 13 x 13 = 338 tiles (256-wide: 650) for the 148-CTA persistent grid: CTAs walk several tiles
@pytest.mark.parametrize("geom", [(2, 16, 16, 16, 16), (2, 20, 37, 17, 31), (1, 50, 61, 60, 75), (2, 33, 24, 28, 20),
                                  (2, 200, 196, 167, 164)])
def test_gathered_conv_matches_torch(cin, cout, dil, geom):
    """conv3x3_gather_kernel alone (csrc/conv_gather.cu): Conv2d(ReLU(scale * nearest(Y_prev) + shift)) with the operand
    built on chip, against torch on the same bf16 operand (rounded once, like the materialised A_k of the unfused path):
    up-sampling, down-sampling and identity resamples, ragged tiles, and the BN statistics of the stored output."""
    import ctypes as C
    from mrfp_b200 import _lib
    n, h, w, sh, sw = geom
    torch.manual_seed(cin + cout + dil + h + sh)
    fn = _lib.load().mrfp_debug_conv3x3_gather_fwd
    fn.restype = C.c_int
    fn.argtypes = [C.c_void_p, C.c_int, C.c_int] + [C.c_void_p] * 5 + [C.c_int] * 6 + [C.c_void_p] * 4
    y = torch.randn(n, sh, sw, cin, device="cuda").to(torch.bfloat16)
    wt = torch.randn(cout, cin, 3, 3, device="cuda") * (2.0 / (9 * cin)) ** 0.5
    wp = wt.permute(2, 3, 0, 1).reshape(9, cout, cin).contiguous().to(torch.bfloat16)
    stats = torch.zeros(4, 256, device="cuda")
    stats[2, :cin] = 0.5 + torch.rand(cin, device="cuda"); stats[3, :cin] = 0.3 * torch.randn(cin, device="cuda")
    ih, iw = _nearest_idx(sh, h), _nearest_idx(sw, w)
    ih32, iw32 = ih.to(torch.int32).contiguous(), iw.to(torch.int32).contiguous()
    cnt_h = torch.zeros(((h + 15) // 16 + 1) * 16, dtype=torch.int32, device="cuda")
    cnt_w = torch.zeros(((w + 15) // 16 + 1) * 16, dtype=torch.int32, device="cuda")
    cnt_h[:h] = torch.randint(0, 3, (h,), device="cuda", dtype=torch.int32)
    cnt_w[:w] = torch.randint(0, 3, (w,), device="cuda", dtype=torch.int32)
    acc = torch.zeros(2, 256, device="cuda", dtype=torch.float64)
    out = torch.full((n, h, w, cout), float("nan"), device="cuda", dtype=torch.bfloat16)
    rc = fn(y.data_ptr(), sh, sw, ih32.data_ptr(), iw32.data_ptr(), stats.data_ptr(), wp.data_ptr(), out.data_ptr(), n, h, w, cin,
            cout, dil, cnt_h.data_ptr(), cnt_w.data_ptr(), acc.data_ptr(), torch.cuda.current_stream().cuda_stream)
    assert rc == 0, rc
    torch.cuda.synchronize()
    a = torch.relu(torch.addcmul(stats[3, :cin], y.float().index_select(1, ih).index_select(2, iw), stats[2, :cin]))
    a = a.to(torch.bfloat16).permute(0, 3, 1, 2).double()                    # fmaf(scale, y, shift) -> one bf16 rounding
    wb = wp.reshape(3, 3, cout, cin).permute(2, 3, 0, 1).double()
    ref = F.conv2d(a, wb, padding=dil, dilation=dil)
    got = out.permute(0, 3, 1, 2).double()
    assert not torch.isnan(got).any()
    # bf16 output rounding (2^-9 relative) + the rare operand that rounds the other way (fma vs mul-add of the reference)
    assert (got - ref).abs().max().item() <= 2 ** -7 * ref.abs().max().item() + 1e-6
    assert float((got - ref).norm() / ref.norm()) <= 3e-3
    wgt = (cnt_h[:h].double()[:, None] * cnt_w[:w].double()[None, :])[None, None]
    s1 = (got * wgt).sum((0, 2, 3)); s2 = (got * got * wgt).sum((0, 2, 3))
    assert torch.allclose(acc[0, :cout], s1, rtol=1e-4, atol=1e-4 * s1.abs().max().item())
    assert torch.allclose(acc[1, :cout], s2, rtol=1e-4, atol=1e-4 * s2.abs().max().item())


# add: False nothing joins the output; True a bf16 tensor of the output's shape is added in the epilogue (ADD == 1); "rk" the
# stage-4 form with the classifier tail's gradient as a rank-K k-block, out += G . W2T^T (ADD == 2, identity resample)
@pytest.mark.parametrize("cin,cout,dil,geom,add", [
    (128, 256, 1, (2, 40, 56, 40, 56), True),      # stage-4 dgrad: identity resample, OCout_dec gradient added in the epilogue
    (64, 128, 1, (2, 33, 24, 28, 20), False),      # down-sampling: some source pixels have no replica
    (64, 64, 2, (2, 50, 61, 40, 49), False),
    (64, 64, 1, (2, 40, 56, 48, 67), False),       # up-sampling x1.2: up to 2 x 2 replicas per source pixel (extras stage)
    (64, 64, 1, (1, 50, 61, 60, 73), False),
    (64, 64, 1, (2, 200, 196, 240, 235), False),   # 2 x 13 x 13 = 338 tiles of 16 x 16 on the 148-CTA persistent grid
    (128, 256, 1, (1, 21, 13, 21, 13), "rk"),      # ragged on both axes (21 % 16, 13 % 8), batch 1
    (128, 256, 1, (3, 37, 30, 37, 30), "rk"),      # batch 3, ragged
    (128, 256, 1, (1, 10, 5, 10, 5), "rk"),        # smaller than one 16 x 8 tile
    (128, 256, 1, (2, 200, 196, 200, 196), "rk"),  # ragged, 650 tiles: each CTA carries its k-block ring across ~4 tiles
    (128, 256, 1, (2, 384, 384, 384, 384), "rk"),  # the stage-4 dgrad of the 768^2 training step
])
def test_gathered_dgrad_matches_torch(cin, cout, dil, geom, add):
    """conv3x3_gather_kernel<bwd | bwd-rep> alone: Conv2d(dY) with dY = BN-backward apply of (dA, Y) under the nearest
    adjoint built on chip, against torch in fp64 on the same bf16 operands (dY rounded to bf16 once, as the materialised
    dY of the unfused path).  The rank-K form is also checked with each of its two terms alone, with G carrying only the
    K = 19 classes the tail leaves and with all 32 columns of the block's two k-steps live.  Output and G have a NaN guard band after the last pixel."""
    import ctypes as C
    from mrfp_b200 import _lib
    n, h, w, oh, ow = geom                          # (h, w): conv resolution of the stage; (oh, ow): its resampled output
    torch.manual_seed(cin + cout + dil + h + oh)
    lib = _lib.load()
    fn = lib.mrfp_debug_conv3x3_gather_bwd
    fn.restype = C.c_int
    fn.argtypes = ([C.c_void_p] * 2 + [C.c_int] * 2 + [C.c_void_p] * 4 + [C.c_int] + [C.c_void_p] * 3 + [C.c_double] +
                   [C.c_void_p] * 2 + [C.c_int] * 6 + [C.c_void_p] * 2)
    rfn = lib.mrfp_debug_conv3x3_gather_bwd_rk
    rfn.restype = C.c_int
    rfn.argtypes = ([C.c_void_p] * 2 + [C.c_int] * 2 + [C.c_void_p] * 7 + [C.c_double] + [C.c_void_p] * 2 + [C.c_int] * 6 +
                    [C.c_void_p] * 3)
    y = torch.randn(n, h, w, cin, device="cuda").to(torch.bfloat16)
    dA = torch.randn(n, oh, ow, cin, device="cuda").to(torch.bfloat16)
    wt = torch.randn(cout, cin, 3, 3, device="cuda") * (2.0 / (9 * cin)) ** 0.5
    wp = wt.permute(2, 3, 0, 1).reshape(9, cout, cin).contiguous().to(torch.bfloat16)
    stats = torch.zeros(4, 256, device="cuda")
    stats[0, :cin] = 0.1 * torch.randn(cin, device="cuda"); stats[1, :cin] = 0.5 + torch.rand(cin, device="cuda")
    gamma = (0.5 * torch.randn(cin, device="cuda")).contiguous()
    stats[2, :cin] = gamma * stats[1, :cin]; stats[3, :cin] = -stats[0, :cin] * stats[2, :cin]
    count = float(n * oh * ow)
    acc = torch.zeros(2, 256, device="cuda", dtype=torch.float64)
    acc[0, :cin] = count * 0.05 * torch.randn(cin, device="cuda", dtype=torch.float64)
    acc[1, :cin] = count * 0.05 * torch.randn(cin, device="cuda", dtype=torch.float64)
    ih, iw = _nearest_idx(h, oh).cpu(), _nearest_idx(w, ow).cpu()      # dst -> src of the forward resample
    lo_h = torch.searchsorted(ih, torch.arange(h + 1)).to(torch.int32).contiguous()
    lo_w = torch.searchsorted(iw, torch.arange(w + 1)).to(torch.int32).contiguous()
    max_rep = int(max((lo_h[1:] - lo_h[:-1]).max(), (lo_w[1:] - lo_w[:-1]).max()))
    assert max_rep <= 2
    lo_hd, lo_wd = lo_h.cuda(), lo_w.cuda()
    npix, guard = n * h * w, 64                     # guard band: NaN pixels behind the last one of out and of G

    def guarded(c, fill):
        buf = torch.full(((npix + guard) * c,), fill, device="cuda", dtype=torch.bfloat16)
        return buf, buf[:npix * c].view(n, h, w, c)

    def run(wpack, addt=None, g64=None, w2t=None):
        obuf, out = guarded(cout, float("nan"))
        common = (stats.data_ptr(), gamma.data_ptr(), acc.data_ptr(), count, wpack.data_ptr(), out.data_ptr(), n, h, w, cin, cout, dil)
        if g64 is None:
            rc = fn(y.data_ptr(), dA.data_ptr(), oh, ow, lo_hd.data_ptr(), lo_wd.data_ptr(), lo_h.data_ptr(), lo_w.data_ptr(), max_rep,
                    *common, None if addt is None else addt.data_ptr(), torch.cuda.current_stream().cuda_stream)
        else:
            rc = rfn(y.data_ptr(), dA.data_ptr(), oh, ow, lo_hd.data_ptr(), lo_wd.data_ptr(), lo_h.data_ptr(), lo_w.data_ptr(),
                     *common, g64.data_ptr(), w2t.data_ptr(), torch.cuda.current_stream().cuda_stream)
        assert rc == 0, rc
        torch.cuda.synchronize()
        assert torch.isnan(obuf[npix * cout:]).all()                    # nothing written behind the last pixel
        assert not torch.isnan(out).any()
        return out.permute(0, 3, 1, 2).double()

    # reference: the adjoint of the nearest resample sums the replicas of each source pixel; BN backward with the given sums
    S = torch.zeros(n, h, ow, cin, device="cuda", dtype=torch.float64).index_add_(1, ih.cuda(), dA.double())
    S = torch.zeros(n, h, w, cin, device="cuda", dtype=torch.float64).index_add_(2, iw.cuda(), S)
    cnt = ((lo_hd[1:] - lo_hd[:-1]).double()[:, None] * (lo_wd[1:] - lo_wd[:-1]).double()[None, :])[None, :, :, None]
    mean, invstd, gm = stats[0, :cin].double(), stats[1, :cin].double(), gamma.double()
    S1, S2 = acc[0, :cin], invstd * (acc[1, :cin] - mean * acc[0, :cin])
    r = invstd * invstd * (gm * S2 / count)
    P, Q, R = (invstd * gm).float(), (invstd * (gm * S1 / count) - mean * r).float(), r.float()
    yf = y.float()
    mask = torch.addcmul(stats[3, :cin], yf, stats[2, :cin]) > 0
    dY = P.double() * torch.where(mask, S, torch.zeros_like(S)) - cnt * (R.double() * yf.double() + Q.double())
    del S, mask
    dY = dY.to(torch.bfloat16).permute(0, 3, 1, 2).double()
    wb = wp.reshape(3, 3, cout, cin).permute(2, 3, 0, 1).double()
    conv_ref = F.conv2d(dY, wb, padding=dil, dilation=dil)
    del dY

    def check(got, ref):
        r_max = (got - ref).abs().max().item() / (2 ** -7 * ref.abs().max().item() + 1e-6)
        r_l2 = float((got - ref).norm() / ref.norm()) / 3e-3
        print(f"error/bound max {r_max:.3g} l2 {r_l2:.3g}")
        assert r_max <= 1.0 and r_l2 <= 1.0, (r_max, r_l2)

    if add != "rk":
        addt = torch.randn(n, h, w, cout, device="cuda").to(torch.bfloat16) if add else None
        ref = conv_ref if addt is None else conv_ref + addt.permute(0, 3, 1, 2).double()
        check(run(wp, addt), ref)
        return

    # rank-K operands: G (pixels, 64) bf16 with a NaN guard band, W2T (cout, 64) bf16; classes >= k zero (the k-block reads
    # columns 0..31 — two UMMA k-steps of 16 — and columns 32..63 are zero padding, as mrfp_hrfp_tail_final2_bwd_rk leaves them)
    def operands(k):
        gbuf, g64 = guarded(64, float("nan"))
        g64.zero_()
        g64[..., :k] = torch.randn(n, h, w, k, device="cuda").to(torch.bfloat16)
        w2t = torch.zeros(cout, 64, device="cuda", dtype=torch.bfloat16)
        w2t[:, :k] = (0.05 * torch.randn(cout, k, device="cuda")).to(torch.bfloat16)
        rk = torch.einsum("nhwk,ck->nchw", g64.double(), w2t.double())
        rk_mag = torch.einsum("nhwk,ck->nchw", g64.double().abs(), w2t.double().abs())        # sum_k |G||W2T|
        return gbuf, g64, w2t, rk, rk_mag

    for k in (19, 32):                               # the K = 19 classes the tail leaves; every column the k-block reads
        gbuf, g64, w2t, rk, rk_mag = operands(k)
        check(run(wp, g64=g64, w2t=w2t), conv_ref + rk)
        # rank-K term alone (zero conv weights): exact bf16 products summed in fp32, two k-steps of 16 products + the
        # accumulator = 34 additions, then one rounding to bf16 — |err| <= 2^-8 |ref| (half an ulp) + 34 * 2^-23 * sum |G||W2T|
        # (one ulp per addition), x(1 + 2^-8) through the rounding
        got = run(torch.zeros_like(wp), g64=g64, w2t=w2t)
        bound = 2 ** -8 * rk.abs() + (1 + 2 ** -8) * 34 * 2 ** -23 * rk_mag
        ratio = ((got - rk).abs() / bound.clamp_min(1e-30)).max().item()
        print(f"rank-K term alone, K = {k}: error/bound {ratio:.3g}")
        assert ((got - rk).abs() <= bound).all(), ratio
        assert torch.isnan(gbuf[npix * 64:]).all()
    # conv term alone (G = 0): the extra k-block adds exact zeros to every fp32 accumulator, so the output is the
    # plain dgrad's (ADD == 0) bit for bit
    g0 = torch.zeros(n, h, w, 64, device="cuda", dtype=torch.bfloat16)
    assert torch.equal(run(wp, g64=g0, w2t=w2t), run(wp))
