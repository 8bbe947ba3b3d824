"""Argument validation of mrfp_hrfp_fwd / mrfp_hrfp_bwd: each rejected combination returns its MRFP_ERR_* code and
launches nothing (include/mrfp_b200.h: "< 0: nothing was launched").

Every buffer is real and sized for the plan, and the misaligned pointers point into spare bytes at the end of a real
buffer, so a call that slipped past validation would compute garbage rather than fault.  Either direction enqueues a
memset of `ws` before anything else; `ws` and the outputs are filled with a sentinel, and every buffer must come back
byte-identical."""
import pytest
import torch

from mrfp_b200.hrfp import DEC_GRAD_F32 as F32, DEC_GRAD_NHWC as NHWC, DEC_GRAD_NONE as NONE, DEC_GRAD_RANK_K as RANK_K

pytestmark = pytest.mark.gpu

NULL_POINTER, UNSUPPORTED = -1, -4
N, CIN, H, W = 2, 64, 48, 48
NP_KEYS = ("np_alpha", "np_eps", "np_mean", "np_ws")


class Case:
    """One plan and every buffer either direction of the chain may be given."""

    def __init__(self, math_mode, widths=(64, 64, 128, 256)):
        from mrfp_b200 import _lib
        from mrfp_b200.hrfp import HrfpPlan, _ptr_array
        self.lib = _lib.load()
        p = self.plan = HrfpPlan(N, CIN, H // 4, W // 4, H, W, "cuda", math_mode, widths, fuse=3)
        _, c3, _, _, _, oh, ow = p.stages[3]
        elem = torch.bfloat16 if math_mode == 2 else torch.float32
        gen = torch.Generator(device="cuda").manual_seed(7)

        def randn(*shape):
            return torch.randn(*shape, device="cuda", generator=gen)

        def sentinel(nbytes):
            return torch.full((nbytes,), 0xA5, dtype=torch.uint8, device="cuda")

        self.weights = [randn(cout, cin, 3, 3) for cin, cout, *_ in p.stages]
        self.gammas = [randn(cout) for _, cout, *_ in p.stages]
        self.W, self.gamma = _ptr_array(self.weights), _ptr_array(self.gammas)
        xshape = (N, CIN, p.xh, p.xw)
        self.buf = dict(
            xp=randn(*xshape), x_add=randn(*xshape), g_ocout=randn(*xshape), g_f32=randn(N, c3, oh, ow),
            # 16 spare bytes behind the NHWC and rank-K operands and np_ws keep the misaligned pointers below inside them
            g_nhwc=torch.zeros(N * oh * ow * c3 * elem.itemsize + 16, dtype=torch.uint8, device="cuda"),
            g64=torch.zeros(N * oh * ow * 64 * 2 + 16, dtype=torch.uint8, device="cuda"),
            w2t=torch.zeros(256 * 64 * 2 + 16, dtype=torch.uint8, device="cuda"),
            np_alpha=randn(N, CIN), np_eps=randn(N, CIN), np_mean=sentinel(N * CIN * 4),
            np_ws=sentinel(self.lib.mrfp_hrfp_np_ws_bytes(N, CIN) + 16),
            lut=p.lut, saved=torch.zeros(p.saved_bytes, dtype=torch.uint8, device="cuda"), ws=sentinel(p.ws_bytes),
            ocout=sentinel(N * CIN * p.xh * p.xw * 4), g_xp=sentinel(N * CIN * p.xh * p.xw * 4))
        torch.cuda.synchronize()
        self.before = {k: v.clone() for k, v in self.buf.items()}

    def ptr(self, name, offset=0):
        """Device address of a buffer of this case by name; None and ready-made addresses pass through."""
        return name if name is None or isinstance(name, int) else self.buf[name].data_ptr() + offset

    def _finish(self, rc):
        torch.cuda.synchronize()
        changed = [k for k, v in self.buf.items() if not torch.equal(v, self.before[k])]
        assert not changed, f"rc={rc} but {changed} were written"
        return rc

    def fwd(self, x_add=None, np=(None,) * 4, ocout="ocout"):
        a, e, m, w = np
        s = torch.cuda.current_stream().cuda_stream
        return self._finish(self.lib.mrfp_hrfp_fwd(
            self.plan.handle, self.ptr("xp"), self.W, self.gamma, None, None, None, 0.1, 1e-5, self.ptr(x_add),
            self.ptr(a), self.ptr(e), self.ptr(m), None, self.ptr(w), self.ptr(ocout), None, self.ptr("lut"),
            self.ptr("saved"), self.ptr("ws"), s))

    def bwd(self, form, g_dec=None, w2t=None, g_ocout="g_ocout", np=(None,) * 4):
        a, e, m, w = np
        s = torch.cuda.current_stream().cuda_stream
        return self._finish(self.lib.mrfp_hrfp_bwd(
            self.plan.handle, self.ptr(g_ocout), form, g_dec, w2t, self.gamma, self.ptr(a), self.ptr(e), self.ptr(m),
            self.ptr(w), self.ptr("lut"), self.ptr("saved"), self.ptr("g_xp"), self.ptr("ws"), s))


@pytest.fixture(scope="module")
def cases():
    return {"bf16": Case(2), "tf32": Case(1), "fp32": Case(0), "bf16_w128": Case(2, widths=(64, 64, 128, 128))}


# (plan, form, g_dec, w2t64, expected): g_dec / w2t64 name a buffer of the case, with a byte offset
BWD_REJECTED = [
    ("fp32", NHWC, ("g_nhwc", 0), None, UNSUPPORTED),           # the NHWC form needs a tensor-core plan
    ("bf16", NHWC, ("g_nhwc", 2), None, UNSUPPORTED),           # misaligned
    ("tf32", NHWC, ("g_nhwc", 4), None, UNSUPPORTED),
    ("tf32", RANK_K, ("g64", 0), ("w2t", 0), UNSUPPORTED),      # the rank-K form needs a bf16 plan ...
    ("fp32", RANK_K, ("g64", 0), ("w2t", 0), UNSUPPORTED),
    ("bf16_w128", RANK_K, ("g64", 0), ("w2t", 0), UNSUPPORTED),  # ... with widths[3] == 256
    ("bf16", RANK_K, ("g64", 2), ("w2t", 0), UNSUPPORTED),      # misaligned
    ("bf16", RANK_K, ("g64", 0), ("w2t", 8), UNSUPPORTED),
    ("bf16", F32, None, None, NULL_POINTER),
    ("bf16", NHWC, None, None, NULL_POINTER),
    ("bf16", RANK_K, None, ("w2t", 0), NULL_POINTER),
    ("bf16", RANK_K, ("g64", 0), None, NULL_POINTER),
    ("bf16", 4, ("g_f32", 0), None, UNSUPPORTED),               # unknown forms
    ("bf16", -1, ("g_f32", 0), None, UNSUPPORTED),
]


@pytest.mark.parametrize("plan,form,g_dec,w2t,expected", BWD_REJECTED)
def test_backward_rejects_the_gradient_form_before_any_launch(cases, plan, form, g_dec, w2t, expected):
    c = cases[plan]
    assert c.bwd(form, None if g_dec is None else c.ptr(*g_dec), None if w2t is None else c.ptr(*w2t)) == expected


def test_np_block_is_all_null_or_all_set(cases):
    """np_alpha, np_eps, np_mean and np_ws: none of them (NP+ not folded in) or all of them, np_ws 16-byte aligned.
    The backward cases pass no g_ocout, which makes it ignore NP+, and the forward cases an x_add, which a folded forward
    refuses: a call that got past this check could not run with the incomplete NP+ block."""
    c = cases["bf16"]
    partial = [tuple(k if (i >> j) & 1 else None for j, k in enumerate(NP_KEYS)) for i in range(1, 15)]
    misaligned = ("np_alpha", "np_eps", "np_mean", c.ptr("np_ws", 8))
    for np in partial + [misaligned]:
        assert c.bwd(NONE, g_ocout=None, np=np) == NULL_POINTER, np
        assert c.fwd(x_add="x_add", np=np) == NULL_POINTER, np
    # all four set is accepted: what rejects these calls is the one other fault in each
    assert c.bwd(4, np=NP_KEYS) == UNSUPPORTED
    assert c.fwd(x_add="x_add", np=NP_KEYS) == UNSUPPORTED      # NP+(xp) takes the place of x_add
    assert c.fwd(ocout=None, np=NP_KEYS) == NULL_POINTER        # the folded NP+ exists for OCout + NP+(xp) only
    assert c.bwd(4) == UNSUPPORTED
