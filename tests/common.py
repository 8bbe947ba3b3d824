"""Shared helpers for tests, the golden generator and bench (seeded synthetic inputs)."""
import math
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")

HRFP_LAYERS = ((64, 64, 1), (64, 64, 1), (64, 128, 2), (128, 256, 2),
               (256, 128, 1), (128, 64, 1), (64, 64, 2), (64, 64, 2))


def make_hrfp_params(seed: int, layers=HRFP_LAYERS):
    """Frozen HRFP weights with the reference initialiser's distribution (mynn.py:57-74):
    W ~ N(0, 2/(9 cin)), gamma ~ N(0, 0.5); drawn from numpy PCG64 so every box regenerates them."""
    rng = np.random.default_rng(seed)
    ws, gs = [], []
    for cin, cout, _ in layers:
        ws.append((rng.standard_normal((cout, cin, 3, 3)) * math.sqrt(2.0 / (9 * cin))).astype(np.float32))
        gs.append((rng.standard_normal(cout) * 0.5).astype(np.float32))
    return ws, gs


def make_feat(seed: int, shape):
    """Post-ReLU-like features with channel-varying statistics (SURVEY.md §8d)."""
    rng = np.random.default_rng(seed)
    n, c, h, w = shape
    sig = rng.uniform(0.5, 1.5, size=(1, c, 1, 1))
    mu = rng.standard_normal((1, c, 1, 1))
    x = rng.standard_normal(shape) * sig + mu
    return np.maximum(x, 0).astype(np.float32)


def make_draws(seed: int, n: int, c: int):
    rng = np.random.default_rng(seed)
    alpha = (1.0 + 0.75 * rng.standard_normal((n, c))).astype(np.float32)
    eps = (0.75 * rng.standard_normal((n, c))).astype(np.float32)
    return alpha, eps


def fill_state_dict(model, seed: int):
    """Deterministic, name-keyed parameter fill (numpy PCG64) so the reference model in the build container and
    this repo's model on any box carry identical weights without shipping a 160 MB state_dict."""
    import zlib
    import torch
    sd = model.state_dict()
    with torch.no_grad():
        for key, t in sd.items():
            if not t.dtype.is_floating_point:
                continue
            rng = np.random.default_rng([seed, zlib.crc32(key.encode())])
            shape = tuple(t.shape)
            if key.endswith("running_var"):
                v = rng.uniform(0.5, 1.5, shape)
            elif key.endswith("running_mean"):
                v = 0.1 * rng.standard_normal(shape)
            elif t.dim() == 1 and key.endswith("weight"):
                v = 1.0 + 0.1 * rng.standard_normal(shape)
            elif t.dim() == 1:
                v = 0.1 * rng.standard_normal(shape)
            else:
                fan_in = int(np.prod(shape[1:]))
                v = rng.standard_normal(shape) * math.sqrt(2.0 / fan_in)
            t.copy_(torch.from_numpy(v.astype(np.float32)))


def hrfp_gx_both(g, tag: str):
    """Gradient into xp of both HRFP outputs from the hrfp.npz fixture.  The backward is linear in the upstream
    gradients, so the fixture keeps only the two single-output gradients; their sum matches the reference's joint
    backward to 6e-7 of max |.| (fp32 summation order), far inside every tolerance it is checked at."""
    return g[f"{tag}_gx_out"] + g[f"{tag}_gx_dec"]


# Eval-path cases of the host module on CPU: name -> (trunk, fill_state_dict seed, input shape).  Eval mode runs no
# MRFP branch, so these pin the trunk and head wiring (tests/test_model.py, tests/golden/make_golden_hosts.py).
HOST_EVAL_CASES = {"resnet50": ("resnet-50", 5, (2, 3, 64, 64)),
                   "resnet101_trunk": ("resnet-101", 6, (2, 3, 64, 64)),
                   "mobilenetv2": ("mobilenetv2", 9, (2, 3, 96, 160)),
                   "shufflenetv2": ("shufflenetv2", 9, (2, 3, 96, 160))}


def host_eval_case(name: str):
    """(model, output) of one HOST_EVAL_CASES entry: weights from fill_state_dict, U[0,255) pixels from a seeded torch
    generator.  The output is the logits, or for resnet101_trunk the layer2 feature (all three InstanceNorm sites).
    Evaluated in float64: an fp32 run moves by up to 1.4e-5 of max |.| with the CPU's kernels and thread count."""
    import torch
    from mrfp_b200.model import MRFPPlus
    trunk, seed, shape = HOST_EVAL_CASES[name]
    m = MRFPPlus(19, trunk=trunk, criterion=torch.nn.CrossEntropyLoss(ignore_index=255))
    fill_state_dict(m, seed)
    m.double().eval()
    x = torch.rand(shape, generator=torch.Generator().manual_seed(seed)).double() * 255
    with torch.no_grad():
        out = m.layer2(m.layer1(m._stem(x))) if name == "resnet101_trunk" else m(x, training=False)
    return m, out


def host_state_dict_digest(model) -> str:
    """sha256 over the names and shapes of the host's state_dict entries (the HRFP layers left out), in state_dict order."""
    import hashlib
    from mrfp_b200.model import HRFP_CONVS, HRFP_BNS
    lines = [f"{k} {list(v.shape)}" for k, v in model.state_dict().items() if k.split(".")[0] not in HRFP_CONVS + HRFP_BNS]
    return hashlib.sha256("\n".join(lines).encode()).hexdigest()


def make_in_case(seed: int, shape):
    """Inputs of one InstanceNorm2d(affine)+ReLU case: pre-norm features of both signs with channel-varying offsets,
    gamma ~ N(1, 0.3) (some negative via a sign flip), beta ~ N(0, 0.3), upstream gradient ~ N(0, 1)."""
    rng = np.random.default_rng(seed)
    n, c, h, w = shape
    x = (rng.standard_normal(shape) * rng.uniform(0.5, 2.0, size=(1, c, 1, 1)) + 3.0 * rng.standard_normal((1, c, 1, 1))).astype(np.float32)
    gamma = (1.0 + 0.3 * rng.standard_normal(c)).astype(np.float32)
    gamma[::5] *= -1.0
    beta = (0.3 * rng.standard_normal(c)).astype(np.float32)
    gy = rng.standard_normal(shape).astype(np.float32)
    return x, gamma, beta, gy
