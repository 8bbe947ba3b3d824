"""Generate tests/golden/hosts_eval.npz: eval-path outputs of the host module on CPU.

    python tests/golden/make_golden_hosts.py

For every case of tests.common.HOST_EVAL_CASES it stores a fixed sample of the output (seeded indices), the output's
shape, max |.| and sum |.|, and a digest of the host's state_dict names and shapes.  The vectors were recorded from
this module at a commit whose eval path matched the reference's own modules (MRFPPlus, resnet101, DeepV3Plus on
mobilenetv2 / shufflenetv2) to 1e-5 on CPU, with the same weights; tests/test_model.py holds every later commit to them.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from tests.common import HOST_EVAL_CASES, host_eval_case, host_state_dict_digest   # noqa: E402

SAMPLES = 2048

if __name__ == "__main__":
    out = {}
    for name in HOST_EVAL_CASES:
        m, y = host_eval_case(name)
        y = y.double().numpy()
        idx = np.sort(np.random.default_rng(1234).choice(y.size, SAMPLES, replace=False))
        out[f"{name}_shape"] = np.array(y.shape)
        out[f"{name}_idx"] = idx.astype(np.int32)
        out[f"{name}_val"] = y.ravel()[idx].astype(np.float32)
        out[f"{name}_absmax"] = np.array(np.abs(y).max())
        out[f"{name}_abssum"] = np.array(np.abs(y).sum())
        out[f"{name}_digest"] = np.array(host_state_dict_digest(m))
        print(name, y.shape, float(np.abs(y).max()))
    np.savez_compressed(os.path.join(HERE, "hosts_eval.npz"), **out)
