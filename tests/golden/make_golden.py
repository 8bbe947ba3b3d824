"""Generate the golden fixtures from the REFERENCE ITSELF (build container only).

    python tests/golden/make_golden.py

Imports /root/reference through oracle/ref_shim.py, runs the reference's own code
(`MRFPPlus.Normalization_Perturbation_Plus`, the OC* modules evaluated with the literal expression
of deepv3.py:320-327, `F.interpolate`, the initialiser of mynn.py:57-74) on seeded inputs with
injected random draws, and writes small .npz / .json files next to this script.
"""
import json
import math
import os
import random
import sys

import numpy as np
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle.ref_shim import load_reference           # noqa: E402
from tests.common import make_hrfp_params, make_feat, make_draws, fill_state_dict   # noqa: E402

deepv3 = load_reference()
torch.set_num_threads(8)


class InjectNormal:
    """Replace torch.normal(mean_tensor, std_tensor) by injected draws, in call order."""

    def __init__(self, draws):
        self.draws = list(draws)
        self.orig = torch.normal

    def __enter__(self):
        def fake(mean, std, *a, **k):
            d = self.draws.pop(0)
            return d.to(mean.dtype).reshape(mean.shape)
        torch.normal = fake
        return self

    def __exit__(self, *a):
        torch.normal = self.orig


def ref_np_plus(feat, alpha, eps):
    n, c = alpha.shape
    with InjectNormal([alpha.reshape(n, c, 1, 1), eps.reshape(n, c, 1, 1)]):
        return deepv3.MRFPPlus.Normalization_Perturbation_Plus(None, feat)


def gen_npplus():
    out = {}
    cases = {"a": (2, 8, 12, 10), "b": (3, 5, 7, 9), "c": (4, 16, 6, 6), "d": (2, 64, 24, 24)}
    for i, (name, shape) in enumerate(cases.items()):
        feat = torch.from_numpy(make_feat(100 + i, shape)).requires_grad_(True)
        a, e = make_draws(200 + i, shape[0], shape[1])
        y = ref_np_plus(feat, torch.from_numpy(a), torch.from_numpy(e))
        gout = torch.from_numpy(np.random.default_rng(300 + i).standard_normal(shape).astype(np.float32))
        y.backward(gout)
        out[f"{name}_shape"] = np.array(shape)
        out[f"{name}_out"] = y.detach().numpy()
        out[f"{name}_gin"] = feat.grad.numpy()
    # float64 run of case a: tight pin for the closed-form backward
    shape = cases["a"]
    feat = torch.from_numpy(make_feat(100, shape)).double().requires_grad_(True)
    a, e = make_draws(200, shape[0], shape[1])
    y = ref_np_plus(feat, torch.from_numpy(a).double(), torch.from_numpy(e).double())
    gout = torch.from_numpy(np.random.default_rng(300).standard_normal(shape).astype(np.float32)).double()
    y.backward(gout)
    out["a64_out"] = y.detach().numpy()
    out["a64_gin"] = feat.grad.numpy()
    # N == 1 -> NaN everywhere (torch.std over a single sample)
    feat = torch.from_numpy(make_feat(1, (1, 4, 5, 5)))
    a, e = make_draws(2, 1, 4)
    y = ref_np_plus(feat, torch.from_numpy(a), torch.from_numpy(e))
    out["n1_all_nan"] = np.array(bool(torch.isnan(y).all()))
    np.savez_compressed(os.path.join(HERE, "npplus.npz"), **out)
    print("npplus.npz", {k: v.shape for k, v in out.items()})


def interp_index(in_size, **kw):
    """dst->src index actually used by F.interpolate(mode='nearest') along one axis."""
    x = torch.arange(in_size, dtype=torch.float32).reshape(1, 1, in_size, 1).expand(1, 1, in_size, 3).contiguous()
    if "scale_factor" in kw:
        y = F.interpolate(x, scale_factor=(kw["scale_factor"], 1.0))
    else:
        y = F.interpolate(x, size=(kw["size"], 3))
    return y[0, 0, :, 0].long().numpy()


def gen_lut():
    out = {}
    for tag, (h, w) in {"768": (768, 768), "odd": (100, 140), "small": (48, 48), "rect": (40, 56)}.items():
        for axis, full in (("h", h), ("w", w)):
            cur = math.ceil(full / 4) if tag != "768" else 192
            if tag == "768":
                cur = 192
            else:
                # stem of the reference: conv7x7/2 pad 3 then maxpool3x3/2 pad 1 (Resnet.py:523-551)
                c1 = (full + 6 - 7) // 2 + 1
                cur = (c1 + 2 - 3) // 2 + 1
            sizes = [cur]
            spec = [dict(scale_factor=1.205), dict(scale_factor=1.2), dict(scale_factor=1.2),
                    dict(size=int(full / 2)), dict(size=int(full / 2)), dict(scale_factor=0.838),
                    dict(scale_factor=0.798), dict(size=math.ceil(full / 4))]
            for k, kw in enumerate(spec):
                idx = interp_index(cur, **kw)
                out[f"{tag}_{axis}_{k}"] = idx.astype(np.int32)
                cur = len(idx)
                sizes.append(cur)
            out[f"{tag}_{axis}_sizes"] = np.array(sizes)
    np.savez_compressed(os.path.join(HERE, "lut.npz"), **out)
    print("lut.npz 768 sizes", out["768_h_sizes"])


def ref_hrfp_modules():
    """A bare object holding the reference's own OC* layer types (deepv3.py:221-237), built by MRFPPlus."""
    m = deepv3.MRFPPlus(19, criterion=torch.nn.CrossEntropyLoss(ignore_index=255))
    return m


def ref_hrfp_chain(m, xp, h, w):
    """The literal expression of deepv3.py:320-327 on the reference module's own layers."""
    OCout = F.relu(m.OC1_bn(F.interpolate(m.OClayer1(xp), scale_factor=(1.205, 1.205))))
    OCout = F.relu(m.OC2_bn(F.interpolate(m.OClayer2(OCout), scale_factor=(1.2, 1.2))))
    OCout = F.relu(m.OC3_bn(F.interpolate(m.OClayer3(OCout), scale_factor=(1.2, 1.2))))
    OCout_dec = F.relu(m.OC4_bn(F.interpolate(m.OClayer4(OCout), size=(int(h / 2), int(w / 2)))))
    OCout = F.relu(m.OC1_decbn(F.interpolate(m.OCdeclayer1(OCout_dec), size=(int(h / 2), int(w / 2)))))
    OCout = F.relu(m.OC2_decbn(F.interpolate(m.OCdeclayer2(OCout), scale_factor=(0.838, 0.838))))
    OCout = F.relu(m.OC3_decbn(F.interpolate(m.OCdeclayer3(OCout), scale_factor=(0.798, 0.798))))
    OCout = F.relu(m.OC4_decbn(F.interpolate(m.OCdeclayer4(OCout), size=(math.ceil(h / 4), math.ceil(w / 4)))))
    return OCout, OCout_dec


CONVS = ("OClayer1", "OClayer2", "OClayer3", "OClayer4", "OCdeclayer1", "OCdeclayer2", "OCdeclayer3", "OCdeclayer4")
BNS = ("OC1_bn", "OC2_bn", "OC3_bn", "OC4_bn", "OC1_decbn", "OC2_decbn", "OC3_decbn", "OC4_decbn")


def gen_hrfp(m):
    out = {}
    for tag, (n, h, w, seed) in {"sq": (2, 48, 48, 11), "rect": (2, 40, 56, 12)}.items():
        xh, xw = math.ceil(h / 4), math.ceil(w / 4)
        ws, gs = make_hrfp_params(seed)
        with torch.no_grad():
            for k in range(8):
                getattr(m, CONVS[k]).weight.copy_(torch.from_numpy(ws[k]))
                getattr(m, CONVS[k]).bias.zero_()
                bn = getattr(m, BNS[k])
                bn.weight.copy_(torch.from_numpy(gs[k])); bn.bias.zero_()
                bn.running_mean.zero_(); bn.running_var.fill_(1); bn.num_batches_tracked.zero_()
        m.train()
        xp = torch.from_numpy(make_feat(seed + 50, (n, 64, xh, xw))).requires_grad_(True)
        ocout, ocdec = ref_hrfp_chain(m, xp, h, w)
        rng = np.random.default_rng(seed + 70)
        g1 = torch.from_numpy(rng.standard_normal(tuple(ocout.shape)).astype(np.float32))
        g2 = torch.from_numpy(rng.standard_normal(tuple(ocdec.shape)).astype(np.float32))
        (gx_out,) = torch.autograd.grad([ocout], [xp], [g1], retain_graph=True)
        (gx_dec,) = torch.autograd.grad([ocdec], [xp], [g2])
        out[f"{tag}_meta"] = np.array([n, h, w, seed])
        out[f"{tag}_ocout"] = ocout.detach().numpy()
        out[f"{tag}_ocout_dec"] = ocdec.detach().numpy().astype(np.float16)   # large: fp16 storage, tolerance-tested
        out[f"{tag}_ocout_dec_sum"] = ocdec.detach().double().sum((0, 2, 3)).numpy()
        # the gradient of both outputs is their sum (tests.common.hrfp_gx_both): not stored, keeps the file under 1 MB
        out[f"{tag}_gx_out"] = gx_out.numpy()
        out[f"{tag}_gx_dec"] = gx_dec.numpy()
        for k in range(8):
            bn = getattr(m, BNS[k])
            out[f"{tag}_rm{k}"] = bn.running_mean.numpy().copy()
            out[f"{tag}_rv{k}"] = bn.running_var.numpy().copy()
        out[f"{tag}_nbt"] = np.array(int(m.OC1_bn.num_batches_tracked))
    # HRFP+ add (deepv3.py:356-357) on a small decoder feature
    dec1 = torch.from_numpy(np.random.default_rng(5).standard_normal((2, 8, 6, 7)).astype(np.float32))
    ocd = torch.from_numpy(np.random.default_rng(6).standard_normal((2, 8, 12, 14)).astype(np.float32))
    from network.mynn import Upsample
    out["plus_dec1"] = dec1.numpy(); out["plus_ocd"] = ocd.numpy()
    out["plus_out"] = torch.add(ocd, Upsample(dec1, (12, 14))).numpy()
    np.savez_compressed(os.path.join(HERE, "hrfp.npz"), **out)
    print("hrfp.npz", sum(v.nbytes for v in out.values()) / 1e6, "MB raw")


def gen_rng_order(m):
    """Known answers: RNG consumption order of one training forward with all branches on, param counts,
    BN buffer side effect, the three gate draws of random.seed(4)."""
    log = []
    ok, on = torch.nn.init.kaiming_normal_, torch.nn.init.normal_
    onormal = torch.normal

    def k_(t, *a, **k):
        log.append(["kaiming_normal_", list(t.shape)]); return ok(t, *a, **k)

    def n_(t, *a, **k):
        log.append(["normal_", list(t.shape), k.get("std")]); return on(t, *a, **k)

    def tn(mean, std, *a, **k):
        log.append(["torch.normal", list(mean.shape)]); return onormal(mean, std, *a, **k)

    torch.nn.init.kaiming_normal_, torch.nn.init.normal_, torch.normal = k_, n_, tn
    try:
        random.seed(4)
        gates = [random.random() for _ in range(3)]
        random.seed(4)
        m.train()
        x = torch.rand(2, 3, 64, 64) * 255
        gts = torch.randint(0, 19, (2, 64, 64))
        nbt0 = int(m.OC1_bn.num_batches_tracked)
        loss = m(x, gts, training=True)
        nbt1 = int(m.OC1_bn.num_batches_tracked)
    finally:
        torch.nn.init.kaiming_normal_, torch.nn.init.normal_, torch.normal = ok, on, onormal
    frozen = sum(p.numel() for p in m.parameters() if not p.requires_grad)
    train = sum(p.numel() for p in m.parameters() if p.requires_grad)
    oc_keys = [k for k in m.state_dict().keys() if k.startswith("OC")]
    info = dict(gates_seed4=gates, draw_log=log, frozen_params=frozen, trainable_params=train,
                nbt_before=nbt0, nbt_after=nbt1, loss_finite=bool(torch.isfinite(loss)),
                oc_state_dict_keys=oc_keys,
                all_state_dict_keys=list(m.state_dict().keys()),
                state_dict_shapes={k: list(v.shape) for k, v in m.state_dict().items()})
    with open(os.path.join(HERE, "known_answers.json"), "w") as f:
        json.dump(info, f, indent=0)
    print("known_answers.json: draws", len(log), "frozen", frozen, "trainable", train)


def gen_full_model(m):
    """One training forward+backward of the reference MRFPPlus on CPU, all three branches on, every random draw
    injected: loss and gradient fingerprints for the drop-in module test (tests/test_model.py)."""
    import deepv3 as ref
    fill_state_dict(m, 77)
    m.train()
    n, hh, ww = 2, 64, 64
    rng = np.random.default_rng(78)
    x = torch.from_numpy(rng.uniform(0, 255, (n, 3, hh, ww)).astype(np.float32))
    gts = torch.from_numpy(rng.integers(0, 19, (n, hh, ww)).astype(np.int64))
    gts[torch.from_numpy(rng.uniform(size=(n, hh, ww)) < 0.05)] = 255
    ws, gs = make_hrfp_params(79)
    a1, e1 = make_draws(80, n, 64)
    a2, e2 = make_draws(81, n, 256)
    calls = {"i": 0}
    orig_init = ref.initialize_weights_kaimingnormal_forOC

    def fake_init(mod):
        k = calls["i"] // 2
        with torch.no_grad():
            if isinstance(mod, torch.nn.Conv2d):
                mod.weight.copy_(torch.from_numpy(ws[k])); mod.bias.zero_()
            else:
                mod.weight.copy_(torch.from_numpy(gs[k])); mod.bias.zero_()
        calls["i"] += 1

    ref.initialize_weights_kaimingnormal_forOC = fake_init
    try:
        random.seed(4)                      # p, p2, p3 all < 0.5
        draws = [torch.from_numpy(t).reshape(n, -1, 1, 1) for t in (a1, e1, a2, e2)]
        with InjectNormal(draws):
            loss = m(x, gts, training=True)
        loss.backward()
    finally:
        ref.initialize_weights_kaimingnormal_forOC = orig_init
    assert calls["i"] == 16
    out = {"loss": np.array(float(loss))}
    for key in ("layer0.0.weight", "layer0.1.weight", "layer1.0.conv1.weight", "layer1.2.instance_norm_layer.weight",
                "layer2.0.conv2.weight", "final1.0.weight", "final2.0.weight", "final2.0.bias"):
        gparam = dict(m.named_parameters())[key].grad.double()
        out["g_" + key] = np.array([float(gparam.sum()), float(gparam.abs().sum()), float((gparam * gparam).sum())])
        out["gs_" + key] = gparam.flatten()[:: max(1, gparam.numel() // 64)][:64].numpy()
    for k in range(8):
        bn = getattr(m, BNS[k])
        out[f"rm{k}"] = bn.running_mean.numpy().copy()
    np.savez_compressed(os.path.join(HERE, "full_model.npz"), **out)
    print("full_model.npz loss", float(loss))


if __name__ == "__main__":
    gen_npplus()
    gen_lut()
    m = ref_hrfp_modules()
    gen_hrfp(m)
    gen_rng_order(m)
    gen_full_model(m)
