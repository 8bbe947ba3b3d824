"""HRFP chain (high-resolution feature perturbation) on the sm_100a kernels.

Host-side mirror of /root/reference/deepv3.py:320-330 and :355-357: the 8 frozen conv/BN pairs are
ordinary `nn.Conv2d` / `nn.BatchNorm2d` modules owned by the caller (same names and state_dict keys
as the reference); this file only plans the geometry, owns the workspaces and exposes the chain as
one `torch.autograd.Function` (input gradient only — the weights are frozen, deepv3.py:221-237).
"""
import collections
import ctypes
import math
import os
import threading
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib

MATH_FP32 = 0      # CUDA-core fp32 convolutions (tight parity mode)
MATH_TF32 = 1      # tcgen05 kind::tf32, fp32 storage: the arithmetic of the reference's cuDNN convolutions (TF32 default)
MATH_BF16 = 2      # tcgen05 kind::f16 on bf16 operands and bf16 storage, fp32 accumulation (default: half the HBM traffic)
DEFAULT_WIDTHS = (64, 64, 128, 256)
# form of the gradient of OCout_dec given to mrfp_hrfp_bwd (include/mrfp_b200.h: MRFP_DEC_GRAD_*)
DEC_GRAD_NONE, DEC_GRAD_F32, DEC_GRAD_NHWC, DEC_GRAD_RANK_K = 0, 1, 2, 3


def _stream_ptr(dev) -> int:
    return torch.cuda.current_stream(dev).cuda_stream


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _ptr_array(tensors: Sequence[Optional[torch.Tensor]]):
    arr = (ctypes.c_void_p * len(tensors))()
    for i, t in enumerate(tensors):
        arr[i] = _ptr(t)
    return arr


class HrfpPlan:
    """Geometry + launch plan for one (N, cin, xh, xw, h, w, math_mode); owns LUTs and workspace."""

    def __init__(self, n, cin, xh, xw, h, w, device, math_mode=MATH_BF16, widths=DEFAULT_WIDTHS, fuse=None):
        lib = _lib.load()
        self.key = (n, cin, xh, xw, h, w, math_mode, tuple(widths), str(device), fuse)
        self.device = torch.device(device)
        handle = ctypes.c_void_p()
        warr = (ctypes.c_int * 4)(*widths)
        _lib.check(lib.mrfp_hrfp_plan_create(ctypes.byref(handle), n, cin, xh, xw, h, w, warr, math_mode),
                   "mrfp_hrfp_plan_create")
        self.handle = handle
        # operand fusion of the bf16 chain (include/mrfp_b200.h: mrfp_hrfp_plan_set_fusion); None = the library default (on)
        if fuse is None and os.environ.get("MRFP_FUSED_GATHER"):
            fuse = int(os.environ["MRFP_FUSED_GATHER"])
        if fuse is not None:
            self.fuse = lib.mrfp_hrfp_plan_set_fusion(handle, int(fuse))
            if self.fuse < 0:
                _lib.check(self.fuse, "mrfp_hrfp_plan_set_fusion")
        else:
            self.fuse = 3 if math_mode == MATH_BF16 else 0
        self.n, self.cin, self.xh, self.xw, self.h, self.w = n, cin, xh, xw, h, w
        self.math_mode = math_mode
        self.ws_bytes = lib.mrfp_hrfp_plan_ws_bytes(handle)
        self.saved_bytes = lib.mrfp_hrfp_plan_saved_bytes(handle)
        lut_bytes = lib.mrfp_hrfp_plan_lut_bytes(handle)
        host = np.empty(lut_bytes // 4, dtype=np.int32)
        _lib.check(lib.mrfp_hrfp_plan_write_luts(handle, host.ctypes.data, lut_bytes), "mrfp_hrfp_plan_write_luts")
        self.lut = torch.from_numpy(host).to(self.device)
        self.stages = []
        for k in range(8):
            out = (ctypes.c_int * 7)()
            _lib.check(lib.mrfp_hrfp_plan_stage(handle, k, out), "mrfp_hrfp_plan_stage")
            self.stages.append(tuple(out))

    def workspace(self) -> torch.Tensor:
        """Scratch for one forward or backward call: the grow-only per-(device, stream) buffer every plan shares."""
        return _lib.scratch(self.device, self.ws_bytes, "hrfp")

    @property
    def dec_shape(self):
        cin, cout, dil, ch, cw, oh, ow = self.stages[3]
        return (self.n, cout, oh, ow)

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                _lib.load().mrfp_hrfp_plan_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


_PLAN_CACHE = collections.OrderedDict()      # LRU: a plan is host geometry + a small LUT tensor; scratch is shared (_lib.scratch)
_PLAN_CACHE_CAP = 16
_PLAN_LOCK = threading.Lock()                 # nn.DataParallel runs replicas in host threads


def get_plan(n, cin, xh, xw, h, w, device, math_mode=MATH_BF16, widths=DEFAULT_WIDTHS, fuse=None) -> HrfpPlan:
    key = (n, cin, xh, xw, h, w, math_mode, tuple(widths), str(device), fuse)
    with _PLAN_LOCK:
        p = _PLAN_CACHE.get(key)
        if p is not None:
            _PLAN_CACHE.move_to_end(key)
            return p
    p = HrfpPlan(n, cin, xh, xw, h, w, device, math_mode, widths, fuse)
    with _PLAN_LOCK:
        _PLAN_CACHE[key] = p
        while len(_PLAN_CACHE) > _PLAN_CACHE_CAP:      # an evicted plan is destroyed when its last user (a ctx) lets go
            _PLAN_CACHE.popitem(last=False)
    return p


class DecGradSlot:
    """The gradient of a lazy OCout_dec, parked by the backward of its consumer until the chain's backward takes it:
    the fp32 NCHW gradients of hrfp_plus_add / hrfp_plus_add_upsampled (summed), or one form left by the classifier tail
    (an NHWC tensor, or the rank-K factors g and w2t)."""
    __slots__ = ("form", "g", "w2t")

    def __init__(self):
        self.form, self.g, self.w2t = DEC_GRAD_NONE, None, None

    def add_f32(self, g):
        if self.form not in (DEC_GRAD_NONE, DEC_GRAD_F32):
            raise _lib.MrfpError("OCout_dec was consumed both by the fused classifier tail and by a plain HRFP+ add")
        self.form, self.g = DEC_GRAD_F32, (g if self.g is None else self.g + g)

    def set_tail(self, form, g, w2t=None):
        if self.form != DEC_GRAD_NONE:
            raise _lib.MrfpError("OCout_dec handle consumed twice")
        self.form, self.g, self.w2t = form, g, w2t

    def take(self):
        """(form, g, w2t), leaving the slot empty."""
        out = (self.form, self.g, self.w2t)
        self.__init__()
        return out


class HrfpDec:
    """OCout_dec left in the chain's saved state instead of being materialised as a (N,256,h/2,w/2) fp32 tensor:
    `hrfp_plus_add(dec1_up, handle)` produces `dec1_up + OCout_dec` in one pass and routes the gradient back."""

    def __init__(self, plan, saved, token, slot):
        self.plan, self.saved, self.token = plan, saved, token
        self.slot = slot          # DecGradSlot shared with the chain's ctx (a reference to ctx would be a cycle)

    @property
    def shape(self):
        return self.plan.dec_shape


class _HrfpFn(torch.autograd.Function):
    """(xp, x_add) -> (OCout + x_add, OCout_dec | token).  x_add may be None (returns OCout alone).
    With `np_draws = (alpha, eps)` the first output is OCout + NP+(xp) (deepv3.py:316-318 folded into the chain)."""

    @staticmethod
    def forward(ctx, xp, x_add, plan, weights, gammas, betas, rmeans, rvars, momentum, eps, want_out, want_dec,
                holder, np_draws=None):
        lib = _lib.load()
        if not xp.is_cuda or xp.dtype != torch.float32:
            raise _lib.MrfpError("HRFP kernels need a CUDA fp32 tensor (no CPU fallback)")
        xp_c = xp.contiguous()
        dev = xp.device
        saved = torch.empty(plan.saved_bytes, dtype=torch.uint8, device=dev)
        ws = plan.workspace()
        ocout = torch.empty_like(xp_c) if want_out else None
        lazy_dec = want_dec and holder is not None
        ocdec = torch.empty(plan.dec_shape, dtype=torch.float32, device=dev) if (want_dec and not lazy_dec) else None
        xa = x_add.contiguous() if (x_add is not None and want_out) else None
        wa, ga = _ptr_array(weights), _ptr_array(gammas)
        ba = _ptr_array(betas) if betas is not None else None
        rma = _ptr_array(rmeans) if rmeans is not None else None
        rva = _ptr_array(rvars) if rvars is not None else None
        ctx.np = None
        np_ptrs = (None,) * 5          # np_alpha, np_eps, np_mean, np_beta, np_ws: NP+ not folded in
        if np_draws is not None:
            if x_add is not None or not want_out:
                raise _lib.MrfpError("np_draws folds NP+(xp) into OCout + x: it needs want_out and no x_add")
            n, c = plan.n, plan.cin
            np_alpha = np_draws[0].reshape(n, c).to(torch.float32).contiguous()
            np_eps = np_draws[1].reshape(n, c).to(torch.float32).contiguous()
            np_mean = torch.empty((n, c), dtype=torch.float32, device=dev)
            np_ws = _lib.scratch(dev, lib.mrfp_hrfp_np_ws_bytes(n, c), "hrfp_np")      # per-call scratch (both directions)
            np_ptrs = (np_alpha.data_ptr(), np_eps.data_ptr(), np_mean.data_ptr(), None, np_ws.data_ptr())
            ctx.np = (np_alpha, np_eps, np_mean)
        with torch.cuda.device(dev):
            rc = lib.mrfp_hrfp_fwd(plan.handle, xp_c.data_ptr(), wa, ga, ba, rma, rva, momentum, eps, _ptr(xa), *np_ptrs,
                                   _ptr(ocout), _ptr(ocdec), plan.lut.data_ptr(), saved.data_ptr(), ws.data_ptr(),
                                   _stream_ptr(dev))
        _lib.check(rc, "mrfp_hrfp_fwd")
        ctx.plan = plan
        ctx.saved_buf = saved
        ctx.gammas = [g for g in gammas]       # gamma is read again in backward: it must still be the forward's
        ctx.gamma_versions = [g._version for g in gammas]
        ctx.has_add = x_add is not None
        ctx.want_out, ctx.want_dec = want_out, want_dec
        ctx.slot = None
        outs = []
        if want_out:
            outs.append(ocout)
        if want_dec:
            if lazy_dec:
                token = torch.zeros(1, dtype=torch.float32, device=dev)    # carries the autograd edge only
                ctx.slot = DecGradSlot()
                holder.append(HrfpDec(plan, saved, token, ctx.slot))
                outs.append(token)
            else:
                outs.append(ocdec)
        return tuple(outs)

    @staticmethod
    def backward(ctx, *grads):
        lib = _lib.load()
        plan = ctx.plan
        if ctx.saved_buf is None:
            raise _lib.MrfpError("HRFP backward called a second time: the chain's saved state is freed after the first "
                                 "backward (retain_graph is not supported)")
        if any(g._version != v for g, v in zip(ctx.gammas, ctx.gamma_versions)):
            raise _lib.MrfpError("an HRFP BatchNorm weight was modified in place between forward and backward "
                                 "(e.g. reinit_hrfp() ran in between): the gradient would mix old and new parameters")
        gi = iter(grads)
        g_out = next(gi) if ctx.want_out else None
        g_dec = next(gi) if ctx.want_dec else None
        if ctx.slot is not None:             # lazy OCout_dec: its consumer parked the real gradient
            form, g_dec, w2t = ctx.slot.take()
        else:
            form, w2t = (DEC_GRAD_NONE if g_dec is None else DEC_GRAD_F32), None
        dev = plan.device
        g_out_c = g_out.contiguous() if g_out is not None else None
        g_dec_c = g_dec.contiguous() if g_dec is not None else None
        g_xp = None
        if ctx.needs_input_grad[0]:
            g_xp = torch.empty((plan.n, plan.cin, plan.xh, plan.xw), dtype=torch.float32, device=dev)
            ga = _ptr_array(ctx.gammas)
            ws = plan.workspace()
            np_ptrs = (None,) * 4          # np_alpha, np_eps, np_mean, np_ws
            if ctx.np is not None:         # gradient through NP+(xp) joins in the chain's last pass
                np_ws = _lib.scratch(dev, lib.mrfp_hrfp_np_ws_bytes(plan.n, plan.cin), "hrfp_np")
                np_ptrs = tuple(t.data_ptr() for t in ctx.np + (np_ws,))
            with torch.cuda.device(dev):
                rc = lib.mrfp_hrfp_bwd(plan.handle, _ptr(g_out_c), form, _ptr(g_dec_c), _ptr(w2t), ga, *np_ptrs,
                                       plan.lut.data_ptr(), ctx.saved_buf.data_ptr(), g_xp.data_ptr(), ws.data_ptr(),
                                       _stream_ptr(dev))
            _lib.check(rc, "mrfp_hrfp_bwd")
        g_add = g_out_c if (ctx.has_add and ctx.needs_input_grad[1]) else None
        ctx.saved_buf = None
        ctx.np = None
        return (g_xp, g_add) + (None,) * 12


def hrfp_chain(xp, convs, bns, h, w, x_add=None, want_out=True, want_dec=True, math_mode=MATH_BF16,
               update_running_stats=True, lazy_dec=False, np_draws=None, fuse=None):
    """Runs the chain of deepv3.py:320-327 on `xp` with the caller's 8 conv / 8 BN modules.

    `np_draws=(alpha, eps)` (the two draws of deepv3.py:274-275) makes the first output OCout + NP+(xp) — NP+ call 1
    (deepv3.py:316-318) rides on the chain's own passes and NP+(xp) is never materialised.

    Returns (OCout [+ x_add], OCout_dec) restricted to the requested outputs.  With `lazy_dec=True` the second
    value is an `HrfpDec` handle for `hrfp_plus_add` instead of a materialised tensor.
    `fuse` (bf16 mode; None = all on): bit 0 folds the forward resample + BatchNorm + ReLU between two convolutions into
    the next convolution's operand producer, bit 1 the BatchNorm backward in front of the dgrads of the non-replicating
    stages (mrfp_hrfp_plan_set_fusion); 0: separate passes."""
    n, cin, xh, xw = xp.shape
    widths = tuple(c.out_channels for c in convs[:4])
    if (xh, xw) != (math.ceil(h / 4), math.ceil(w / 4)):
        # deepv3.py:327 resamples to (ceil(h/4), ceil(w/4)) and :330 adds xp: torch.add would raise on a mismatch
        raise _lib.MrfpError(f"HRFP chain: xp is {xh}x{xw} but the chain ends at {math.ceil(h / 4)}x{math.ceil(w / 4)} "
                             f"for a {h}x{w} image (deepv3.py:327, :330)")
    plan = get_plan(n, cin, xh, xw, h, w, xp.device, math_mode, widths, fuse)
    weights = [c.weight for c in convs]
    gammas = [b.weight for b in bns]
    betas = [b.bias for b in bns]
    track = update_running_stats and all(b.track_running_stats and b.running_mean is not None for b in bns)
    rmeans = [b.running_mean for b in bns] if track else None
    rvars = [b.running_var for b in bns] if track else None
    momentum = bns[0].momentum if bns[0].momentum is not None else 0.1
    eps = bns[0].eps
    holder = [] if (lazy_dec and want_dec) else None
    outs = _HrfpFn.apply(xp, x_add, plan, weights, gammas, betas, rmeans, rvars, float(momentum), float(eps),
                         want_out, want_dec, holder, np_draws)
    if track:
        n_run = 8 if want_out else 4
        torch._foreach_add_([b.num_batches_tracked for b in bns[:n_run]], 1)     # one launch instead of eight
    outs = list(outs)
    out = outs.pop(0) if want_out else None
    dec = outs.pop(0) if want_dec else None
    if holder:
        holder[0].token = dec             # the autograd-tracked output of the Function
        dec = holder[0]
    return out, dec


def hrfp_plus_add(dec1_up: torch.Tensor, ocout_dec) -> torch.Tensor:
    """deepv3.py:357 — `torch.add(OCout_dec, dec1)` as one streaming kernel (autograd: identity to both).
    `ocout_dec` is either the materialised tensor or the `HrfpDec` handle of `hrfp_chain(lazy_dec=True)`."""
    if isinstance(ocout_dec, HrfpDec):
        return _PlusAddFusedFn.apply(dec1_up, ocout_dec.token, ocout_dec)
    return _AddFn.apply(dec1_up, ocout_dec)


class _PlusAddFusedFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, dec1_up, token, handle):
        lib = _lib.load()
        plan = handle.plan
        if tuple(dec1_up.shape) != tuple(plan.dec_shape) or dec1_up.dtype != torch.float32:
            raise _lib.MrfpError(f"hrfp_plus_add: dec1 must be fp32 of shape {plan.dec_shape}")
        a = dec1_up.contiguous()
        out = torch.empty_like(a)
        with torch.cuda.device(a.device):
            rc = lib.mrfp_hrfp_plus_add(plan.handle, handle.saved.data_ptr(), plan.lut.data_ptr(), a.data_ptr(),
                                        out.data_ptr(), _stream_ptr(a.device))
        _lib.check(rc, "mrfp_hrfp_plus_add")
        ctx.slot = handle.slot
        return out

    @staticmethod
    def backward(ctx, g):
        ctx.slot.add_f32(g)
        return g, torch.zeros(1, dtype=torch.float32, device=g.device), None


def hrfp_plus_add_upsampled(dec1: torch.Tensor, ocout_dec: "HrfpDec") -> torch.Tensor:
    """deepv3.py:356-357 in one kernel: Upsample(dec1) (bilinear, align_corners=True, mynn.py:114-119) + OCout_dec, from
    the low-resolution `dec1` and the `HrfpDec` handle of `hrfp_chain(lazy_dec=True)`.  Neither the upsampled dec1 nor
    OCout_dec is materialised.  Autograd: bilinear-transpose of the gradient to dec1 (gather kernel), identity to the chain."""
    return _PlusAddUpFn.apply(dec1, ocout_dec.token, ocout_dec)


class _PlusAddUpFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, dec1, token, handle):
        lib = _lib.load()
        plan = handle.plan
        n, c, oh, ow = plan.dec_shape
        if dec1.dim() != 4 or dec1.shape[0] != n or dec1.shape[1] != c or dec1.dtype != torch.float32 or not dec1.is_cuda:
            raise _lib.MrfpError(f"hrfp_plus_add_upsampled: dec1 must be CUDA fp32 (N={n}, C={c}, lh, lw)")
        a = dec1.contiguous()
        out = torch.empty(plan.dec_shape, dtype=torch.float32, device=a.device)
        with torch.cuda.device(a.device):
            rc = lib.mrfp_hrfp_plus_add_bilinear(plan.handle, handle.saved.data_ptr(), plan.lut.data_ptr(), a.data_ptr(),
                                                 a.shape[2], a.shape[3], out.data_ptr(), _stream_ptr(a.device))
        _lib.check(rc, "mrfp_hrfp_plus_add_bilinear")
        ctx.slot = handle.slot
        ctx.lo_shape = tuple(a.shape)
        return out

    @staticmethod
    def backward(ctx, g):
        ctx.slot.add_f32(g)
        g_lo = None
        if ctx.needs_input_grad[0]:
            from .bilinear import bilinear_up_backward          # gather form of ATen's scatter (csrc/bilinear.cu)
            g_lo = bilinear_up_backward(g, ctx.lo_shape[2:])
        return g_lo, torch.zeros(1, dtype=torch.float32, device=g.device), None


class _AddFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a, b):
        lib = _lib.load()
        a_c, b_c = a.contiguous(), b.contiguous()
        out = torch.empty_like(a_c)
        with torch.cuda.device(a.device):
            rc = lib.mrfp_add_f32(a_c.data_ptr(), b_c.data_ptr(), out.data_ptr(), a_c.numel(), _stream_ptr(a.device))
        _lib.check(rc, "mrfp_add_f32")
        return out

    @staticmethod
    def backward(ctx, g):
        return g, g


# ----------------------------------------------------------------------------------------------------------------------
# HRFP+ tail fused through the classifier (SURVEY.md 8f-4): deepv3.py:356-361 in one kernel per direction
# ----------------------------------------------------------------------------------------------------------------------
def tail_final2_supported(dec1: torch.Tensor, conv: torch.nn.Conv2d, ocout_dec) -> bool:
    """The fused tail exists for the bf16 path, 256 decoder channels, <= 24 classes, a 1x1 classifier and an Upsample by
    >= 2 whose source rows are 16-byte aligned; anything else takes hrfp_plus_add_upsampled + the module's own conv."""
    if not isinstance(ocout_dec, HrfpDec) or ocout_dec.plan.math_mode != MATH_BF16:
        return False
    n, c, oh, ow = ocout_dec.plan.dec_shape
    return (c == 256 and conv.kernel_size == (1, 1) and conv.stride == (1, 1) and conv.padding == (0, 0) and conv.groups == 1
            and conv.in_channels == 256 and conv.out_channels <= 24 and dec1.is_cuda and dec1.dtype == torch.float32
            and dec1.shape[3] % 4 == 0 and ow > 1 and 2 * (dec1.shape[3] - 1) <= ow - 1 and dec1.shape[2] <= oh)


class _TailFinal2Fn(torch.autograd.Function):
    """(t_lo, W2, b2, token) -> dec2 = b2 + Upsample(t_lo) + W2 . OCout_dec, with t_lo = W2 . dec1 at low resolution."""

    @staticmethod
    def forward(ctx, t_lo, weight, bias, token, handle):
        lib = _lib.load()
        plan = handle.plan
        n, c, oh, ow = plan.dec_shape
        k = weight.shape[0]
        t = t_lo.contiguous()
        w2 = weight.detach().reshape(k, c).contiguous()
        out = torch.empty((n, k, oh, ow), dtype=torch.float32, device=t.device)
        with torch.cuda.device(t.device):
            rc = lib.mrfp_hrfp_tail_final2_fwd(plan.handle, handle.saved.data_ptr(), plan.lut.data_ptr(), t.data_ptr(), t.shape[2],
                                               t.shape[3], w2.data_ptr(), None if bias is None else bias.data_ptr(), k,
                                               out.data_ptr(), _stream_ptr(t.device))
        _lib.check(rc, "mrfp_hrfp_tail_final2_fwd")
        ctx.handle, ctx.w2, ctx.lo, ctx.has_bias, ctx.wshape = handle, w2, (t.shape[2], t.shape[3]), bias is not None, weight.shape
        return out

    @staticmethod
    def backward(ctx, g):
        from .bilinear import bilinear_up_backward
        lib = _lib.load()
        handle, plan = ctx.handle, ctx.handle.plan
        n, c, oh, ow = plan.dec_shape
        k = ctx.w2.shape[0]
        gc = g.contiguous()
        g_t = bilinear_up_backward(gc, ctx.lo) if ctx.needs_input_grad[0] else None
        g_w2 = torch.empty((k, c), dtype=torch.float32, device=g.device)
        g_b2 = torch.empty((k,), dtype=torch.float32, device=g.device)
        if os.environ.get("MRFP_TAIL_RANKK", "1") != "0":
            # rank-K form: W2^T g joins the chain as its two factors (include/mrfp_b200.h: MRFP_DEC_GRAD_RANK_K)
            g64 = torch.empty((n, oh, ow, 64), dtype=torch.bfloat16, device=g.device)
            w2t = torch.empty((c, 64), dtype=torch.bfloat16, device=g.device)
            handle.slot.set_tail(DEC_GRAD_RANK_K, g64, w2t)
            with torch.cuda.device(g.device):
                rc = lib.mrfp_hrfp_tail_final2_bwd_rk(plan.handle, handle.saved.data_ptr(), plan.lut.data_ptr(), gc.data_ptr(),
                                                      ctx.w2.data_ptr(), k, g64.data_ptr(), w2t.data_ptr(), g_w2.data_ptr(),
                                                      g_b2.data_ptr(), _stream_ptr(g.device))
            _lib.check(rc, "mrfp_hrfp_tail_final2_bwd_rk")
        else:
            g_nhwc = torch.empty((n, oh, ow, c), dtype=torch.bfloat16, device=g.device)
            handle.slot.set_tail(DEC_GRAD_NHWC, g_nhwc)
            with torch.cuda.device(g.device):
                rc = lib.mrfp_hrfp_tail_final2_bwd(plan.handle, handle.saved.data_ptr(), plan.lut.data_ptr(), gc.data_ptr(),
                                                   ctx.w2.data_ptr(), k, g_nhwc.data_ptr(), g_w2.data_ptr(), g_b2.data_ptr(),
                                                   _stream_ptr(g.device))
            _lib.check(rc, "mrfp_hrfp_tail_final2_bwd")
        return (g_t, g_w2.reshape(ctx.wshape) if ctx.needs_input_grad[1] else None,
                g_b2 if (ctx.has_bias and ctx.needs_input_grad[2]) else None,
                torch.zeros(1, dtype=torch.float32, device=g.device), None)


def hrfp_plus_final2(dec1: torch.Tensor, conv: torch.nn.Conv2d, ocout_dec: "HrfpDec") -> torch.Tensor:
    """deepv3.py:356-361: final2(Upsample(dec1) + OCout_dec) for final2 = Conv2d(256, K, 1) without materialising anything
    at (N, 256, h/2, w/2).  The low-resolution product W2 . dec1 is a plain library GEMM (autograd gives the gradients to
    dec1 and the low-resolution half of the weight gradient); everything at high resolution is csrc/tail_final2.cu."""
    t_lo = torch.nn.functional.conv2d(dec1, conv.weight)
    return _TailFinal2Fn.apply(t_lo, conv.weight, conv.bias, ocout_dec.token, ocout_dec)
