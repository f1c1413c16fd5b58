"""ORACLE - TEST INFRASTRUCTURE ONLY.  Generates tests/golden/*.npz by executing the REFERENCE's own
modules (imported read-only from /root/reference, which exists only in the build container) on seeded
synthetic inputs.  The fixtures pin oracle/hotpath.py (tests/test_oracle_golden.py) and, on the GPU box,
the CUDA path (tests/test_gpu_parity.py).  It also records the state-dict inventory of the reference's full model
(tests/golden/reference_model_inventory.json).  Re-run:  python oracle/gen_golden.py

The reference has no tests/golden vectors of its own (SURVEY.md §4), so these reference-executed outputs
are the pin.  Reference code is imported, never copied.
"""
import json
import os
import sys

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("MVSF_REFERENCE", "/root/reference")
sys.path.insert(0, REPO)
sys.path.insert(0, REF)

from mvsformerplusplus_b200 import synth  # noqa: E402
from mvsformerplusplus_b200.config import default_args  # noqa: E402


from oracle.ref_hotpath import RefHotPath, import_reference as _import_reference, reference_hotpath  # noqa: E402


def import_reference():
    return _import_reference(REF)


CASES = {
    # name: (V, H, W, feature seed, weight seed)
    "hotpath_v3_96x128": dict(V=3, H=96, W=128, fseed=1234, wseed=7, numdepth=192),
    "hotpath_v4_64x96": dict(V=4, H=64, W=96, fseed=99, wseed=11, numdepth=48),
}

# Arrays with many values per pixel are stored at a fixed, seeded sample of 1 / PIXEL_FRACTION of their pixels (flat
# indices into H*W under "<key>.pixels") so that every fixture stays below 1 MB.  Depth, confidence, probability
# logits, entropy and visibility weights are stored whole.
SAMPLED = ("depth_values", "volume_mean", "fmt.")
PIXEL_FRACTION = 8


def sample_pixels(blob, seed=0):
    out = {}
    for k, a in blob.items():
        if k != "meta" and any(s in k for s in SAMPLED):
            H, W = a.shape[-2:]
            rng = np.random.default_rng(seed)
            idx = np.sort(rng.choice(H * W, max(1, H * W // PIXEL_FRACTION), replace=False)).astype(np.int32)
            out[k] = np.ascontiguousarray(a.reshape(a.shape[:-2] + (H * W,))[..., idx])
            out[k + ".pixels"] = idx
        else:
            out[k] = a
    return out


def reference_model_inventory():
    """The reference's DINOv2MVSNet built from its shipped config: `args` and every state-dict entry as
    [name, shape, dtype, "parameter" | "buffer"] in state-dict order (tests/test_host_cpu.py rebuilds a model of that
    shape to check that install() keeps a reference checkpoint loadable)."""
    from models.networks.DINOv2_mvsformer_model import DINOv2MVSNet
    cfg = json.load(open(os.path.join(REF, "config", "mvsformer++.json")))["arch"]["args"]
    torch.manual_seed(0)
    model = DINOv2MVSNet(cfg)
    params = {k for k, _ in model.named_parameters()}
    rows = [[k, list(v.shape), str(v.dtype).replace("torch.", ""), "parameter" if k in params else "buffer"]
            for k, v in model.state_dict().items()]
    return {"args": cfg, "state_dict": rows}


def make_case(c, args):
    feats = synth.make_features(c["V"], c["H"], c["W"], seed=c["fseed"])
    proj = synth.make_proj_matrices(c["V"], c["H"], c["W"], theta_step=0.12)
    dv = synth.make_depth_values(c["numdepth"], 425.0, 2.65 * 192 / c["numdepth"])
    return feats, proj, dv


def main():
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    R = import_reference()
    args = default_args()
    out_dir = os.path.join(REPO, "tests", "golden")
    os.makedirs(out_dir, exist_ok=True)
    tmp = [5.0, 5.0, 5.0, 1.0]

    for name, c in CASES.items():
        torch.manual_seed(0)
        model = RefHotPath(R, args).eval()
        synth.randomize_state_dict(model, seed=c["wseed"])
        feats, proj, dv = make_case(c, args)
        out = reference_hotpath(R, model, args, feats, proj, dv, tmp)
        blob = {}
        for s in range(4):
            so = out[f"stage{s + 1}"]
            for k in ("depth", "photometric_confidence", "depth_values", "prob_volume_pre"):  # prob_volume = softmax(pre)
                blob[f"stage{s + 1}.{k}"] = so[k][0].numpy()
            blob[f"stage{s + 1}.entropy"] = out["captured"][f"stage{s + 1}.entropy"][0].numpy()
            blob[f"stage{s + 1}.vis_weight"] = out["captured"][f"stage{s + 1}.vis_weight"][0].numpy()
            if s < 2:
                blob[f"stage{s + 1}.volume_mean"] = out["captured"][f"stage{s + 1}.volume_mean"][0].numpy()
        blob["refined_depth"] = out["refined_depth"][0].numpy()
        blob["photometric_confidence"] = out["photometric_confidence"][0].numpy()
        blob["fmt.stage1"] = out["features"]["stage1"][0].numpy()
        # full-resolution FMT outputs are large: keep view 1 (first source view) of stages 2-4 only
        for k in ("stage2", "stage3", "stage4"):
            blob[f"fmt.{k}.view1"] = out["features"][k][0, 1].numpy()
        blob["meta"] = np.frombuffer(json.dumps(c).encode(), dtype=np.uint8)
        np.savez_compressed(os.path.join(out_dir, name + ".npz"), **sample_pixels(blob))
        print(name, "refined_depth range", float(out["refined_depth"].min()), float(out["refined_depth"].max()),
              "stage4 conf mean", float(out["stage4"]["photometric_confidence"].mean()))

    # ---- warp seam alone, including out-of-image taps and per-pixel hypotheses (warping.py:69-109)
    g = torch.Generator().manual_seed(5)
    H, W, C, D = 12, 16, 8, 4
    src = torch.randn(1, C, H, W, generator=g)
    pm = synth.make_proj_matrices(3, H * 8, W * 8, theta_step=0.5)["stage1"]  # wide baseline -> taps leave the image
    from oracle.hotpath import compose_projection
    refp, srcp = compose_projection(pm[:, 0]), compose_projection(pm[:, 2])
    dvals = 425.0 + 500.0 * torch.rand(1, D, H, W, generator=g)
    warped, mask = R["homo_warp"](src, srcp, refp, dvals)
    np.savez_compressed(os.path.join(out_dir, "warp_seam.npz"), src=src.numpy(), src_proj=srcp.numpy(),
                        ref_proj=refp.numpy(), depth_values=dvals.numpy(), warped=warped.numpy(), mask=mask.numpy())
    print("warp_seam: fraction masked", float(mask.float().mean()))

    with open(os.path.join(out_dir, "reference_model_inventory.json"), "w") as f:
        inv = reference_model_inventory()
        f.write('{"args": ' + json.dumps(inv["args"]) + ',\n "state_dict": [\n')
        f.write(",\n".join("  " + json.dumps(r) for r in inv["state_dict"]) + "\n]}\n")
    print("reference_model_inventory:", len(inv["state_dict"]), "state-dict entries")


if __name__ == "__main__":
    main()
