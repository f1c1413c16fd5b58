"""Pins oracle/hotpath.py against the reference-executed fixtures (tests/golden, made by
oracle/gen_golden.py from the reference's own modules).  CPU only."""
import pytest
import torch
import torch.nn.functional as F

from oracle import hotpath as O
from tests.common import TMP, at_golden_pixels, build_case, load_golden, max_abs, rel_linf

CASES = ["hotpath_v3_96x128", "hotpath_v4_64x96"]


@pytest.fixture(scope="module", params=CASES)
def run(request):
    gold, meta = load_golden(request.param)
    args, params, sd, feats, proj, dv = build_case(meta)
    with torch.no_grad():
        out = O.hotpath_forward(feats, proj, dv, sd, args, tmp=TMP, keep_intermediates=True)
    return gold, out


def test_warp_seam_matches_reference():
    g, _ = load_golden("warp_seam")
    warped, mask = O.homo_warp(g["src"], g["src_proj"], g["ref_proj"], g["depth_values"])
    assert max_abs(warped, g["warped"]) < 2e-4
    assert float((mask != g["mask"]).float().mean()) < 0.01
    # and the explicit gather equals ATen's grid_sample on the same coordinates
    B, C, H, W = g["src"].shape
    px, py, _ = O.warp_coordinates(g["src_proj"], g["ref_proj"], g["depth_values"], H, W)
    grid = torch.stack((px / ((W - 1) / 2) - 1, py / ((H - 1) / 2) - 1), dim=3)
    ref = F.grid_sample(g["src"], grid.view(B, -1, W, 2), mode="bilinear", padding_mode="zeros", align_corners=True)
    assert max_abs(warped, ref.view_as(warped)) < 1e-5


def test_fmt_matches_reference(run):
    gold, out = run
    assert max_abs(at_golden_pixels(gold, "fmt.stage1", out["features"]["stage1"][0]), gold["fmt.stage1"]) < 2e-4
    for k in ("stage2", "stage3", "stage4"):
        key = f"fmt.{k}.view1"
        assert max_abs(at_golden_pixels(gold, key, out["features"][k][0, 1]), gold[key]) < 2e-4


@pytest.mark.parametrize("s", [1, 2, 3, 4])
def test_stage_outputs_match_reference(run, s):
    gold, out = run
    so = out[f"stage{s}"]
    key = f"stage{s}.depth_values"
    assert rel_linf(at_golden_pixels(gold, key, so["depth_values"][0]), gold[key]) < 1e-5
    assert max_abs(so["entropy"][0], gold[f"stage{s}.entropy"]) < 5e-4
    assert max_abs(so["vis_weight"][0], gold[f"stage{s}.vis_weight"]) < 5e-4
    if s <= 2:
        key = f"stage{s}.volume_mean"
        assert max_abs(at_golden_pixels(gold, key, so["volume_mean"][0]), gold[key]) < 1e-3
    gp = torch.softmax(gold[f"stage{s}.prob_volume_pre"], dim=0)
    assert max_abs(so["prob_volume"][0], gp) < 1e-4          # north-star probability tolerance
    assert max_abs(so["photometric_confidence"][0], gold[f"stage{s}.photometric_confidence"]) < 1e-4
    assert rel_linf(so["depth"][0], gold[f"stage{s}.depth"]) < 1e-3  # north-star depth tolerance


def test_final_outputs_match_reference(run):
    gold, out = run
    assert rel_linf(out["refined_depth"][0], gold["refined_depth"]) < 1e-3
    assert max_abs(out["photometric_confidence"][0], gold["photometric_confidence"]) < 1e-4


def test_aten_kernel_variant_agrees_with_explicit_restatement():
    """bench.py's CPU arm switches the oracle to the reference's own ATen kernels (grid_sample, SDPA); both forms
    must agree."""
    gold, meta = load_golden("hotpath_v4_64x96")
    args, params, sd, feats, proj, dv = build_case(meta)
    with torch.no_grad():
        a = O.hotpath_forward(feats, proj, dv, sd, args, tmp=TMP)
        O.USE_ATEN_KERNELS = True
        try:
            b = O.hotpath_forward(feats, proj, dv, sd, args, tmp=TMP)
        finally:
            O.USE_ATEN_KERNELS = False
    assert rel_linf(a["refined_depth"], b["refined_depth"]) < 1e-4
    assert max_abs(a["stage4"]["prob_volume"], b["stage4"]["prob_volume"]) < 1e-4
