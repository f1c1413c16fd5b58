"""Shared helpers for tests: golden loading + case reconstruction (inputs are re-generated from seeds)."""
import json
import os

import numpy as np
import torch

from mvsformerplusplus_b200 import synth
from mvsformerplusplus_b200.config import default_args
from mvsformerplusplus_b200.params import build_hotpath_params

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TMP = [5.0, 5.0, 5.0, 1.0]


def load_golden(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    d = {k: torch.from_numpy(z[k]) for k in z.files if k != "meta"}
    meta = json.loads(bytes(z["meta"]).decode()) if "meta" in z.files else {}
    return d, meta


def at_golden_pixels(gold, key, t):
    """`t` [..., H, W] as the fixture stores `key`: whole, or at the fixed sample of pixels listed under `key`.pixels
    (oracle/gen_golden.py keeps large arrays at a sample of their pixels)."""
    idx = gold.get(key + ".pixels")
    return t if idx is None else t.reshape(t.shape[:-2] + (-1,))[..., idx.long()]


def build_case(meta, args=None):
    """Re-creates exactly the inputs oracle/gen_golden.py used (same seeds, same generators)."""
    args = args or default_args()
    feats = synth.make_features(meta["V"], meta["H"], meta["W"], seed=meta["fseed"])
    proj = synth.make_proj_matrices(meta["V"], meta["H"], meta["W"], theta_step=0.12)
    dv = synth.make_depth_values(meta["numdepth"], 425.0, 2.65 * 192 / meta["numdepth"])
    torch.manual_seed(0)
    params = build_hotpath_params(args).eval()
    sd = synth.randomize_state_dict(params, seed=meta["wseed"])
    return args, params, sd, feats, proj, dv


def max_abs(a, b):
    return float((a.double() - b.double()).abs().max())


def rel_linf(a, b):
    return float(((a.double() - b.double()).abs() / b.double().abs().clamp_min(1e-12)).max())


# ---- parity report shared by the GPU test modules (written to gpurun_out/parity_report.json as tests run)
REPORT = {}
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def rec(name, **kw):
    REPORT[name] = {k: (float(v) if isinstance(v, (int, float)) else v) for k, v in kw.items()}
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    with open(os.path.join(ROOT, "gpurun_out", "parity_report.json"), "w") as f:
        json.dump(REPORT, f, indent=1, sort_keys=True)
