"""GPU parity tests: every libmvsf_b200 entry point (called through the ctypes C ABI / the host seam mirrors) against
the CPU oracle on the same seeded inputs, and against the reference-executed golden fixtures.
Tolerances: north-star 1e-3 relative L-inf on depth, 1e-4 absolute on per-pixel probability; intermediates tighter.
A JSON report with every measured error is written to gpurun_out/parity_report.json."""
import ctypes
import json
import math
import os

import pytest
import torch
import torch.nn.functional as F

from tests.common import ROOT, TMP, at_golden_pixels, build_case, load_golden, max_abs, rec, rel_linf

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def hp():
    from mvsformerplusplus_b200 import hotpath
    return hotpath


@pytest.fixture(scope="module")
def L():
    from mvsformerplusplus_b200 import _lib
    return _lib.lib()


def P(t):
    return ctypes.c_void_p(t.data_ptr())


def S():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def ck(rc, what):
    from mvsformerplusplus_b200 import _lib
    _lib.check(rc, what)


# ----------------------------------------------------------------------------------------------- boundary helpers
def test_layout_roundtrip(dev, hp):
    x = torch.randn(3, 24, 13, 37, device=dev)
    n = hp.to_nhwc(x)
    assert torch.equal(n, x.permute(0, 2, 3, 1).contiguous())
    assert torch.equal(hp.to_nchw(n), x)
    assert hp.to_nhwc(n.permute(0, 3, 1, 2)).data_ptr() == n.data_ptr()  # channels-last view: zero copy


def test_compose_geometry(dev, L):
    from mvsformerplusplus_b200 import synth
    from oracle import hotpath as O
    pm = synth.make_proj_matrices(5, 1152, 1536)["stage3"][0]
    homs = torch.empty(4 * 12, device=dev)
    kinv = torch.empty(9, device=dev)
    pmd = pm.to(dev)
    ck(L.mvsf_compose_geometry(P(pmd), 5, P(homs), P(kinv), S()), "compose_geometry")
    pm64 = pm.double()
    ref = O.compose_projection(pm64[None, 0])[0]
    want = []
    for v in range(1, 5):
        M = O.compose_projection(pm64[None, v])[0] @ torch.inverse(ref)
        want.append(torch.cat([M[:3, :3].reshape(-1), M[:3, 3]]))
    want = torch.stack(want).reshape(-1)
    err = float(((homs.cpu().double() - want).abs() / want.abs().clamp_min(1e-3)).max())
    kerr = max_abs(kinv.cpu(), torch.inverse(pm64[0, 1, :3, :3]).reshape(-1))
    rec("compose_geometry", rel=err, kinv_abs=kerr)
    assert err < 1e-6 and kerr < 1e-7


def test_homo_warp_seam_vs_reference(dev, L):
    g, _ = load_golden("warp_seam")
    from oracle import hotpath as O
    src = g["src"][0]
    C, H, W = src.shape
    D = g["depth_values"].shape[1]
    M = (g["src_proj"].double() @ torch.inverse(g["ref_proj"].double()))[0]
    hom = torch.cat([M[:3, :3].reshape(-1), M[:3, 3]]).float().to(dev)
    src_nhwc = src.permute(1, 2, 0).contiguous().to(dev)
    warped = torch.empty(C, D, H, W, device=dev)
    mask = torch.empty(D, H, W, dtype=torch.uint8, device=dev)
    dvd = g["depth_values"][0].contiguous().to(dev)
    ck(L.mvsf_homo_warp(P(src_nhwc), P(hom), P(dvd), P(warped), P(mask), C, D, H, W, S()), "homo_warp")
    e = max_abs(warped.cpu(), g["warped"][0])
    mm = float((mask.cpu().bool() != g["mask"][0]).float().mean())
    rec("homo_warp_seam", abs=e, mask_mismatch=mm)
    assert e < 2e-4 and mm < 0.01


# ----------------------------------------------------------------------------------------------- scheduling
def test_init_and_schedule_inverse_range(dev, L):
    from oracle import hotpath as O
    dv = (425.0 + 2.65 * torch.arange(192)).float()
    D, H, W = 32, 12, 20
    out = torch.empty(D, H, W, device=dev)
    dvd = dv.to(dev)  # keep device inputs alive until the (asynchronous) kernels have consumed them
    ck(L.mvsf_init_inverse_range(P(dvd), 192, P(out), D, H, W, S()), "init_inverse_range")
    want = O.init_inverse_range(dv[None], D, H, W)[0]
    e0 = rel_linf(out.cpu(), want)
    g = torch.Generator().manual_seed(1)
    depth = 500.0 + 300.0 * torch.rand(1, H, W, generator=g)
    hyp = want[None] * (1.0 + 0.01 * torch.rand(1, D, H, W, generator=g))
    D2, H2, W2 = 16, 2 * H, 2 * W
    out2 = torch.empty(D2, H2, W2, device=dev)
    depth_d, hyp_d = depth[0].contiguous().to(dev), hyp[0].contiguous().to(dev)
    ck(L.mvsf_schedule_inverse_range(P(depth_d), P(hyp_d), D, 2.67, P(out2), D2, H2, W2, S()), "schedule_inverse_range")
    want2 = O.schedule_inverse_range(depth, hyp, D2, 2.67, H2, W2)[0]
    e1 = rel_linf(out2.cpu(), want2)
    rec("inverse_range", init_rel=e0, schedule_rel=e1)
    assert e0 < 1e-6 and e1 < 2e-6


def test_position3d(dev, L):
    from mvsformerplusplus_b200 import synth
    from oracle import hotpath as O
    H, W, D = 12, 16, 8
    pm = synth.make_proj_matrices(3, H * 8, W * 8)["stage1"]
    dv = synth.make_depth_values(192)
    ds = O.init_inverse_range(dv, D, H, W)
    want, hmin, hmax, wmin, wmax = O.get_position_3d(1, H, W, pm[:, 0, 1, :3, :3], ds, dv.min(), dv.max(), None, None, None, None)
    homs = torch.empty(2 * 12, device=dev)
    kinv = torch.empty(9, device=dev)
    pmd, dsd, dvd = pm[0].to(dev), ds[0].contiguous().to(dev), dv[0].to(dev)
    ck(L.mvsf_compose_geometry(P(pmd), 3, P(homs), P(kinv), S()), "compose_geometry")
    stats = torch.zeros(8, device=dev)
    pos = torch.empty(3, D, H, W, device=dev)
    ck(L.mvsf_position3d(P(kinv), P(dsd), P(dvd), 192, P(stats), 1, P(pos), D, H, W, S()), "position3d")
    e = max_abs(pos.cpu(), want[0])
    se = max_abs(stats[:4].cpu(), torch.stack([wmin, wmax, hmin, hmax]))
    rec("position3d", abs=e, stats_abs=se)
    assert e < 2e-6


# ----------------------------------------------------------------------------------------------- cost volume
def _rand_vis_sd(seed):
    from mvsformerplusplus_b200 import synth
    from mvsformerplusplus_b200.config import default_args
    from mvsformerplusplus_b200.params import build_hotpath_params
    torch.manual_seed(0)
    params = build_hotpath_params(default_args()).eval()
    return synth.randomize_state_dict(params, seed=seed)


COST_CASES = [  # C, D, H, W, V, theta_step, depth jitter
    (8, 4, 37, 53, 3, 0.1, 0.02), (16, 8, 24, 40, 3, 0.1, 0.02), (32, 16, 16, 24, 4, 0.12, 0.02), (64, 32, 12, 16, 5, 0.1, 0.02),
    (8, 4, 31, 45, 3, 0.6, 0.02),   # wide baseline: many taps leave the image (zero padding per corner)
    (8, 48, 10, 14, 3, 0.1, 0.02),  # generic-D path (D-sweep configuration)
    (64, 8, 9, 11, 2, 0.1, 0.02),
    # shapes served by the TMA-staged window kernels (C = 8 / 16, even H): several tiles, ragged right / bottom edges,
    # taps leaving the image, depth outliers that leave the staged window (global fallback), D = 4 / 8 / chunked D
    (8, 4, 64, 96, 3, 0.1, 0.02), (8, 4, 30, 44, 5, 0.6, 0.02), (8, 4, 48, 80, 3, 0.15, 0.4), (8, 8, 16, 40, 3, 0.1, 0.02),
    (8, 7, 18, 34, 2, 0.1, 0.02), (16, 8, 32, 48, 4, 0.1, 0.02), (16, 8, 28, 68, 3, 0.5, 0.3), (16, 4, 12, 20, 3, 0.1, 0.02),
    (16, 24, 10, 36, 3, 0.1, 0.02), (8, 96, 12, 20, 3, 0.1, 0.0),
]


@pytest.mark.parametrize("C,D,H,W,V,th,jit", COST_CASES)
def test_cost_volume_kernels(dev, L, C, D, H, W, V, th, jit):
    """Pass A (entropy), vis CNN, pass B (aggregation) against the oracle, through every organisation the library has:
    L1 gathers with recompute, L1 gathers with the correlation spill, and (where they apply) the window kernels."""
    from mvsformerplusplus_b200 import packing, synth
    from oracle import hotpath as O
    sd = _rand_vis_sd(5)
    g = torch.Generator().manual_seed(C * 1000 + D)
    feats = torch.randn(1, V, C, H, W, generator=g)
    sc = {8: 1, 16: 2, 32: 4, 64: 8}[C]
    pm = synth.make_proj_matrices(V, H * sc, W * sc, theta_step=th)[f"stage{ {1: 4, 2: 3, 4: 2, 8: 1}[sc] }"]
    dv = synth.make_depth_values(192)
    dvals = O.init_inverse_range(dv, D, H, W) * (1.0 + jit * torch.rand(1, D, H, W, generator=g))
    want = O.cost_volume(feats, pm, dvals, sd, "fusions.3.", 8)
    homs = torch.empty((V - 1) * 12, device=dev)
    kinv = torch.empty(9, device=dev)
    pmd = pm[0].to(dev)
    ck(L.mvsf_compose_geometry(P(pmd), V, P(homs), P(kinv), S()), "compose_geometry")
    f = feats[0].permute(0, 2, 3, 1).contiguous().to(dev)
    dd = dvals[0].contiguous().to(dev)
    wts = packing.pack_vis(sd, "fusions.3.vis.").to(dev)
    vol_scale = max(1.0, float(want["volume_mean"].abs().max()))

    def run_two_gathers():
        ent = torch.empty(V - 1, H, W, device=dev)
        ck(L.mvsf_warp_corr_entropy(P(f), P(homs), P(dd), P(ent), V, C, 8, D, H, W, S()), "warp_corr_entropy")
        vis = torch.empty(V - 1, H, W, device=dev)
        ck(L.mvsf_vis_cnn(P(ent), P(wts), P(vis), V - 1, H, W, S()), "vis_cnn")
        vol = torch.empty(D, H, W, 8, device=dev)
        ck(L.mvsf_warp_corr_aggregate(P(f), P(homs), P(dd), P(vis), P(vol), V, C, 8, D, H, W, S()), "warp_corr_aggregate")
        return ent, vis, vol

    ck(L.mvsf_warp_corr_set_tile_path(0), "set_tile_path")
    try:
        ent, vis, vol = run_two_gathers()
        # spill plan: pass A stores the per-view group correlations, the aggregation streams them
        ent_s = torch.empty(V - 1, H, W, device=dev)
        corr = torch.empty(V - 1, D, H, W, 8, device=dev)
        vol_s = torch.empty(D, H, W, 8, device=dev)
        ck(L.mvsf_warp_corr_entropy_store(P(f), P(homs), P(dd), P(ent_s), P(corr), V, C, 8, D, H, W, S()), "warp_corr_entropy_store")
        ck(L.mvsf_corr_aggregate(P(corr), P(vis), P(vol_s), V, 8, D, H, W, S()), "corr_aggregate")
    finally:
        ck(L.mvsf_warp_corr_set_tile_path(1), "set_tile_path")
    assert torch.equal(ent_s, ent)
    e_paths = max_abs(vol_s.cpu(), vol.cpu())
    assert e_paths <= 2e-6 * vol_scale, e_paths   # identical up to the pair sum of 8-channel groups
    assert L.mvsf_warp_corr_plan(C, 8, D, H, W, V, ctypes.c_size_t(1 << 40)) == 0      # room for the spill buffer: spill plan
    assert L.mvsf_warp_corr_plan(C, 8, D, H, W, V, ctypes.c_size_t(1024)) == 1         # no room: two gathers
    tiled = C in (8, 16) and H % 2 == 0    # shapes the window kernels serve
    e_tile = {}
    if tiled:   # window kernels: the two-gather plan ...
        ent_t, vis_t, vol_t = run_two_gathers()
        e_tile = dict(tile_vs_l1_entropy=max_abs(ent_t.cpu(), ent.cpu()), tile_vs_l1_volume=max_abs(vol_t.cpu(), vol_s.cpu()))
        assert e_tile["tile_vs_l1_entropy"] < 2e-5 and e_tile["tile_vs_l1_volume"] < 1e-5 * vol_scale, e_tile
        # ... and the spill plan: forced through the persistent TMA pipeline kernel where it exists (C = 8, D = 4; mode 2),
        # then as hotpath.py runs it (mode 1: at C = 8, D = 4 the device picks pipeline or L1 kernel per call)
        for mode in ((2, 1) if (C, D) == (8, 4) else (1,)):
            ck(L.mvsf_warp_corr_set_tile_path(mode), "set_tile_path")
            try:
                ent_p = torch.empty(V - 1, H, W, device=dev)
                corr_p = torch.full((V - 1, D, H, W, 8), float("nan"), device=dev)
                vol_p = torch.empty(D, H, W, 8, device=dev)
                ck(L.mvsf_warp_corr_entropy_store(P(f), P(homs), P(dd), P(ent_p), P(corr_p), V, C, 8, D, H, W, S()), "warp_corr_entropy_store")
            finally:
                ck(L.mvsf_warp_corr_set_tile_path(1), "set_tile_path")
            vis_p = torch.empty(V - 1, H, W, device=dev)
            ck(L.mvsf_vis_cnn(P(ent_p), P(wts), P(vis_p), V - 1, H, W, S()), "vis_cnn")
            ck(L.mvsf_corr_aggregate(P(corr_p), P(vis_p), P(vol_p), V, 8, D, H, W, S()), "corr_aggregate")
            tag = "pipe" if mode == 2 else "adaptive"
            e_tile.update({f"{tag}_vs_l1_entropy": max_abs(ent_p.cpu(), ent.cpu()), f"{tag}_vs_l1_corr": max_abs(corr_p.cpu(), corr.cpu()),
                           f"{tag}_vs_l1_volume": max_abs(vol_p.cpu(), vol_s.cpu())})
            assert bool(torch.isfinite(corr_p).all())
            assert e_tile[f"{tag}_vs_l1_entropy"] < 2e-5 and e_tile[f"{tag}_vs_l1_corr"] < 1e-5 * vol_scale * 8 and e_tile[f"{tag}_vs_l1_volume"] < 1e-5 * vol_scale, e_tile
            if mode == 1 and C == 8 and D == 4:
                used, miss = ctypes.c_int(-1), ctypes.c_int(-1)
                ck(L.mvsf_warp_corr_last_selection(ctypes.byref(used), ctypes.byref(miss)), "last_selection")
                e_tile.update(adaptive_used_pipeline=used.value, adaptive_window_miss_permille=miss.value)
                assert used.value in (0, 1) and 0 <= miss.value <= 1000
                assert used.value == (1 if miss.value <= 60 else 0)   # wide baseline (theta 0.6): 193 per mille -> L1 kernel
        ent, vis, vol_s = ent_p, vis_p, vol_p
    vol = vol_s
    e_ent = max_abs(ent.cpu(), want["entropy"][0])
    e_vis = max_abs(vis.cpu(), want["vis_weight"][0])
    e_vol = max_abs(vol.cpu().permute(3, 0, 1, 2), want["volume_mean"][0])
    # vis CNN in isolation on the oracle's entropy (removes the entropy noise from the comparison)
    vis2 = torch.empty(V - 1, H, W, device=dev)
    ent_o = want["entropy"][0].contiguous().to(dev)
    ck(L.mvsf_vis_cnn(P(ent_o), P(wts), P(vis2), V - 1, H, W, S()), "vis_cnn")
    e_vis2 = max_abs(vis2.cpu(), want["vis_weight"][0])
    rec(f"cost_volume_C{C}_D{D}_{H}x{W}_V{V}_th{th}_j{jit}", entropy=e_ent, vis=e_vis, vis_isolated=e_vis2, volume=e_vol,
        vol_scale=float(want["volume_mean"].abs().max()), tiled=int(tiled), **e_tile)
    assert e_ent < 5e-4 and e_vis < 5e-4 and e_vis2 < 2e-5 and e_vol < 1e-3


def test_vis_cnn_tile_borders(dev, L):
    from mvsformerplusplus_b200 import packing
    from oracle import hotpath as O
    sd = _rand_vis_sd(9)
    g = torch.Generator().manual_seed(3)
    for (N, H, W) in [(1, 30, 30), (2, 61, 95), (3, 7, 5), (1, 1, 1), (2, 64, 128)]:
        ent = 3.0 * torch.rand(1, N, H, W, generator=g)
        want = torch.cat([O.vis_cnn(ent[:, i:i + 1], sd, "fusions.1.") for i in range(N)], 1)[0]
        vis = torch.empty(N, H, W, device=dev)
        ent_d, wts = ent[0].contiguous().to(dev), packing.pack_vis(sd, "fusions.1.vis.").to(dev)
        ck(L.mvsf_vis_cnn(P(ent_d), P(wts), P(vis), N, H, W, S()), "vis_cnn")
        e = max_abs(vis.cpu(), want)
        rec(f"vis_cnn_{N}x{H}x{W}", abs=e)
        assert e < 2e-5


# ----------------------------------------------------------------------------------------------- regularisers
@pytest.mark.parametrize("mode,sd,cin,cout,ID,IH,IW", [
    (0, 1, 16, 16, 3, 16, 32), (0, 1, 32, 32, 2, 20, 44), (0, 1, 64, 64, 4, 9, 13), (0, 1, 16, 16, 5, 48, 160),
    (0, 1, 16, 16, 9, 64, 1200), (0, 2, 32, 32, 11, 40, 72), (1, 1, 8, 16, 6, 96, 1300), (0, 1, 16, 16, 1, 16, 16),
    (1, 1, 8, 16, 3, 32, 64), (1, 2, 8, 16, 8, 24, 40), (1, 1, 16, 32, 2, 18, 26), (1, 2, 32, 64, 4, 16, 16),
    (2, 1, 64, 32, 2, 9, 12), (2, 2, 32, 16, 3, 16, 24), (2, 1, 16, 8, 3, 20, 36), (2, 2, 16, 8, 2, 8, 8)])
@pytest.mark.parametrize("skip", [False, True])
def test_conv3d_tensor_core_layer(dev, L, mode, sd, cin, cout, ID, IH, IW, skip):
    """One 3x3x3 layer of the tcgen05 implicit-GEMM path against torch's fp64 convolution (conv / strided conv /
    transposed conv with output_padding = stride - 1, bias, ReLU, skip added after the ReLU)."""
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(mode * 100 + cin + ID)
    x = torch.randn(ID, IH, IW, cin, generator=g)
    w = torch.randn(27, cin, cout, generator=g) / (27 * cin) ** 0.5 * 1.7
    b = torch.randn(cout, generator=g) * 0.2
    xin = x.permute(3, 0, 1, 2)[None].double()
    if mode == 2:
        wt = w.reshape(3, 3, 3, cin, cout).permute(3, 4, 0, 1, 2).double()
        y = F.conv_transpose3d(xin, wt, stride=(sd, 2, 2), padding=1, output_padding=(sd - 1, 1, 1))
    else:
        wt = w.reshape(3, 3, 3, cin, cout).permute(4, 3, 0, 1, 2).double()
        y = F.conv3d(xin, wt, stride=(1, 1, 1) if mode == 0 else (sd, 2, 2), padding=1)
    y = torch.relu(y + b.double().view(1, -1, 1, 1, 1))[0].permute(1, 2, 3, 0).contiguous()
    sk = torch.randn(y.shape, generator=g) if skip else None
    if skip:
        y = y + sk.double()
    x_d, wb_d = x.contiguous().to(dev), torch.cat([w.reshape(-1), b]).to(dev)
    sk_d = sk.contiguous().to(dev) if skip else None
    out = torch.empty(y.shape, device=dev)
    ws = torch.empty((2 * x.numel() + 4 * y.numel()) // 2 + 27 * cin * max(cout, 16) * 4 + 1024, device=dev)
    ck(L.mvsf_conv3d_tc_layer(mode, sd, P(x_d), P(wb_d), P(sk_d) if skip else None, P(out), P(ws),
                              ctypes.c_size_t(ws.numel() * 4), cin, cout, ID, IH, IW, S()), "conv3d_tc_layer")
    e = float((out.cpu().double() - y).abs().max())
    rec(f"conv3d_tc_mode{mode}_sd{sd}_{cin}to{cout}_{ID}x{IH}x{IW}_skip{int(skip)}", abs=e, scale=float(y.abs().max()))
    assert e < 1e-5 * max(1.0, float(y.abs().max()))


@pytest.mark.parametrize("stage,D,H,W", [(1, 16, 16, 24), (1, 8, 8, 40), (2, 8, 16, 24), (3, 4, 24, 40), (3, 3, 8, 8)])
def test_costreg_unet(dev, L, stage, D, H, W):
    from mvsformerplusplus_b200 import packing
    from oracle import hotpath as O
    sd = _rand_vis_sd(13)
    g = torch.Generator().manual_seed(stage * 7 + D)
    vol = torch.randn(1, 8, D, H, W, generator=g) * 0.5
    p = f"fusions.{stage}.cost_reg."
    want = O.costreg_unet(vol, sd, p)[0, 0]
    kind, flat = packing.pack_costreg_unet(sd, p)
    need = ctypes.c_size_t(0)
    ck(L.mvsf_costreg_unet_workspace_bytes(kind, 8, D, H, W, ctypes.byref(need)), "ws")
    ws = torch.empty(need.value // 4 + 4, device=dev)
    logits = torch.empty(D, H, W, device=dev)
    v = vol[0].permute(1, 2, 3, 0).contiguous().to(dev)
    from mvsformerplusplus_b200.hotpath import pack_unet_tc
    flat_d = flat.to(dev)
    flat_tc = pack_unet_tc(kind, flat_d)
    ck(L.mvsf_costreg_unet_forward(kind, P(v), P(flat_d), P(flat_tc), P(logits), P(ws), ctypes.c_size_t(ws.numel() * 4),
                                   8, D, H, W, S()), "costreg_unet_forward")
    e = max_abs(logits.cpu(), want)
    rec(f"costreg_unet_stage{stage}_{D}x{H}x{W}", abs=e, scale=float(want.abs().max()))
    assert e < 2e-4 * max(1.0, float(want.abs().max()))


@pytest.mark.parametrize("D,H,W", [(8, 12, 16), (32, 16, 16), (4, 8, 8)])
def test_costreg_transformer(dev, L, D, H, W):
    from mvsformerplusplus_b200 import packing
    from mvsformerplusplus_b200.config import default_args
    from oracle import hotpath as O
    sd = _rand_vis_sd(17)
    cfg = default_args()["transformer_config"][0]
    g = torch.Generator().manual_seed(D)
    vol = torch.randn(1, 8, D, H, W, generator=g) * 0.5
    pos = torch.rand(1, 3, D, H, W, generator=g)
    p = "fusions.0.cost_reg."
    want = O.costreg_transformer(vol, pos, sd, p, cfg)[0, 0]
    flat = packing.pack_costreg_tr(sd, p, cfg["layer_num"]).to(dev)
    need = ctypes.c_size_t(0)
    ck(L.mvsf_costreg_tr_workspace_bytes(8, D, H, W, ctypes.byref(need)), "ws")
    ws = torch.empty(need.value // 4 + 4, device=dev)
    logits = torch.empty(D, H, W, device=dev)
    v = vol[0].permute(1, 2, 3, 0).contiguous().to(dev)
    n_tok = (D // 2) * (H // 4) * (W // 4)
    scale = 16 ** -0.5 * math.log(n_tok, cfg["train_avg_length"])
    pos_d = pos[0].contiguous().to(dev)
    from mvsformerplusplus_b200.hotpath import split_weights_f16
    flat16 = split_weights_f16(flat)
    ck(L.mvsf_costreg_tr_forward(P(v), P(pos_d), P(flat), P(flat16), ctypes.c_size_t(flat.numel()), P(logits), P(ws),
                                 ctypes.c_size_t(ws.numel() * 4), 8, D, H, W, cfg["layer_num"], float(scale), S()),
       "costreg_tr_forward")
    e = max_abs(logits.cpu(), want)
    rec(f"costreg_tr_{D}x{H}x{W}", abs=e, scale=float(want.abs().max()), tokens=n_tok)
    assert e < 2e-4 * max(1.0, float(want.abs().max()))


def test_softargmax(dev, L):
    g = torch.Generator().manual_seed(2)
    for D in (4, 8, 16, 32, 5):
        H, W = 9, 21
        z = 3.0 * torch.randn(D, H, W, generator=g)
        hyp = 425.0 + 500.0 * torch.rand(D, H, W, generator=g)
        prob = torch.empty(D, H, W, device=dev)
        depth = torch.empty(H, W, device=dev)
        conf = torch.empty(H, W, device=dev)
        zd, hd = z.to(dev), hyp.to(dev)
        ck(L.mvsf_softargmax(P(zd), P(hd), 5.0, P(prob), P(depth), P(conf), D, H, W, S()), "softargmax")
        wp = F.softmax(z, 0)
        wd = (F.softmax(z * 5.0, 0) * hyp).sum(0)
        e = (max_abs(prob.cpu(), wp), rel_linf(depth.cpu(), wd), max_abs(conf.cpu(), wp.max(0)[0]))
        rec(f"softargmax_D{D}", prob=e[0], depth_rel=e[1], conf=e[2])
        assert e[0] < 1e-6 and e[1] < 1e-6 and e[2] < 1e-6


# ----------------------------------------------------------------------------------------------- FMT
@pytest.mark.parametrize("V,H1,W1", [(3, 8, 12), (2, 16, 16), (4, 6, 10)])
def test_fmt_with_pathway(dev, hp, V, H1, W1):
    from mvsformerplusplus_b200 import synth
    from mvsformerplusplus_b200.config import default_args
    from oracle import hotpath as O
    args = default_args()
    torch.manual_seed(0)
    net = hp.HotPathNet(args).eval()
    sd = synth.randomize_state_dict(net, seed=23)
    net = net.to(dev)
    feats = synth.make_features(V, H1 * 8, W1 * 8, seed=V)
    out = net.FMT_module.forward({k: v.to(dev) for k, v in feats.items()})
    with torch.no_grad():
        want = O.fmt_with_pathway(feats, sd, args["FMT_config"])
    errs = {k: max_abs(out[k].cpu(), want[k]) for k in want}
    rec(f"fmt_V{V}_{H1}x{W1}", **errs)
    assert max(errs.values()) < 2e-4


# ----------------------------------------------------------------------------------------------- stage seam + cascade
@pytest.fixture(scope="module", params=["hotpath_v3_96x128", "hotpath_v4_64x96"])
def cascade(request, dev, hp):
    from oracle import hotpath as O
    gold, meta = load_golden(request.param)
    args, params, sd, feats, proj, dv = build_case(meta)
    net = hp.HotPathNet(args).eval()
    net.load_state_dict(sd, strict=True)
    net = net.to(dev)
    out = net.forward_features({k: v.to(dev) for k, v in feats.items()}, {k: v.to(dev) for k, v in proj.items()},
                               dv.to(dev), TMP, keep_intermediates=True)
    with torch.no_grad():
        ora = O.hotpath_forward(feats, proj, dv, sd, args, tmp=TMP, keep_intermediates=True)
    return request.param, gold, out, ora, net, args, sd, proj, dv


@pytest.mark.parametrize("s", [1, 2, 3, 4])
def test_stage_seam_teacher_forced(cascade, dev, s):
    """StageNet.forward on the ORACLE's stage inputs (features, hypotheses, 3-D positions): per-stage parity at the
    north-star tolerances without cascade error accumulation."""
    from oracle import hotpath as O
    name, gold, out, ora, net, args, sd, proj, dv = cascade
    f = ora["features"][f"stage{s}"]
    ds = ora[f"stage{s}"]["depth_values"]
    p3d = None
    if s == 1:
        B, _, _, H, W = f.shape
        p3d, *_ = O.get_position_3d(B, H, W, proj["stage1"][:, 0, 1, :3, :3], ds, dv.min(), dv.max(), None, None, None, None)
    so = net.fusions[s - 1].forward(f.to(dev), proj[f"stage{s}"].to(dev), ds.to(dev), TMP[s - 1],
                                    position3d=None if p3d is None else p3d.to(dev), keep_intermediates=True)
    want = ora[f"stage{s}"]
    e = dict(entropy=max_abs(so["entropy"].cpu(), want["entropy"]), vis=max_abs(so["vis_weight"].cpu(), want["vis_weight"]),
             volume=max_abs(so["volume_mean"].cpu().permute(0, 4, 1, 2, 3), want["volume_mean"]),
             logits=max_abs(so["prob_volume_pre"].cpu(), want["prob_volume_pre"]),
             prob=max_abs(so["prob_volume"].cpu(), want["prob_volume"]),
             conf=max_abs(so["photometric_confidence"].cpu(), want["photometric_confidence"]),
             depth_rel=rel_linf(so["depth"].cpu(), want["depth"]))
    rec(f"stage_seam_{name}_s{s}", **e)
    assert e["prob"] < 1e-4 and e["conf"] < 1e-4 and e["depth_rel"] < 1e-3


@pytest.mark.parametrize("s", [1, 2, 3, 4])
def test_cascade_vs_reference_golden(cascade, s):
    """Full FMT + cascade on the GPU against the reference-executed fixture (fp32 reference forward)."""
    name, gold, out, ora, *_ = cascade
    so = out[f"stage{s}"]
    gp = torch.softmax(gold[f"stage{s}.prob_volume_pre"], dim=0)
    key = f"stage{s}.depth_values"
    e = dict(depth_values_rel=rel_linf(at_golden_pixels(gold, key, so["depth_values"][0].cpu()), gold[key]),
             entropy=max_abs(so["entropy"][0].cpu(), gold[f"stage{s}.entropy"]),
             vis=max_abs(so["vis_weight"][0].cpu(), gold[f"stage{s}.vis_weight"]),
             prob=max_abs(so["prob_volume"][0].cpu(), gp),
             conf=max_abs(so["photometric_confidence"][0].cpu(), gold[f"stage{s}.photometric_confidence"]),
             depth_rel=rel_linf(so["depth"][0].cpu(), gold[f"stage{s}.depth"]))
    rec(f"cascade_{name}_s{s}", **e)
    assert e["prob"] < 1e-4 and e["conf"] < 1e-4 and e["depth_rel"] < 1e-3


def test_cascade_final_outputs(cascade):
    name, gold, out, ora, *_ = cascade
    e = dict(refined_depth_rel=rel_linf(out["refined_depth"][0].cpu(), gold["refined_depth"]),
             confidence=max_abs(out["photometric_confidence"][0].cpu(), gold["photometric_confidence"]),
             fmt_stage1=max_abs(at_golden_pixels(gold, "fmt.stage1", out["features"]["stage1"][0].cpu()), gold["fmt.stage1"]),
             fmt_stage4_view1=max_abs(at_golden_pixels(gold, "fmt.stage4.view1", out["features"]["stage4"][0, 1].cpu()),
                                      gold["fmt.stage4.view1"]))
    rec(f"cascade_{name}_final", **e)
    assert e["refined_depth_rel"] < 1e-3 and e["confidence"] < 1e-4 and e["fmt_stage1"] < 2e-4


# ----------------------------------------------------------------------------------------------- full-size properties
def test_full_size_properties(dev, hp):
    """BASELINE config 2 sizes (V=5, 1152x1536, ndepths 32/16/8/4): properties that do not need the CPU oracle."""
    from mvsformerplusplus_b200 import synth
    from mvsformerplusplus_b200.config import default_args
    args = default_args()
    V, H, W = 5, 1152, 1536
    torch.manual_seed(0)
    net = hp.HotPathNet(args).eval()
    synth.randomize_state_dict(net, seed=7)
    net = net.to(dev)
    feats = {k: v.to(dev) for k, v in synth.make_features(V, H, W, seed=1234, smooth=False).items()}
    proj = {k: v.to(dev) for k, v in synth.make_proj_matrices(V, H, W).items()}
    dv = synth.make_depth_values(192).to(dev)
    out = net.forward_features(feats, proj, dv, TMP)
    out2 = net.forward_features(feats, proj, dv, TMP)
    torch.cuda.synchronize()
    facts = {}
    for s in range(1, 5):
        so = out[f"stage{s}"]
        pv = so["prob_volume"]
        facts[f"s{s}_finite"] = bool(torch.isfinite(pv).all() and torch.isfinite(so["depth"]).all())
        facts[f"s{s}_prob_sum_err"] = float((pv.sum(1) - 1).abs().max())
        facts[f"s{s}_conf_is_max"] = float((so["photometric_confidence"] - pv.max(1)[0]).abs().max())
        lo, hi = so["depth_values"].min(1)[0], so["depth_values"].max(1)[0]
        facts[f"s{s}_depth_in_range"] = bool(((so["depth"] >= lo * (1 - 1e-5)) & (so["depth"] <= hi * (1 + 1e-5))).all())
        facts[f"s{s}_deterministic"] = bool(torch.equal(so["depth"], out2[f"stage{s}"]["depth"]))
    facts["refined_shape"] = list(out["refined_depth"].shape)
    rec("full_size_properties", **{k: (v if not isinstance(v, bool) else int(v)) for k, v in facts.items()})
    for s in range(1, 5):
        assert facts[f"s{s}_finite"] and facts[f"s{s}_depth_in_range"] and facts[f"s{s}_deterministic"]
        assert facts[f"s{s}_prob_sum_err"] < 1e-5 and facts[f"s{s}_conf_is_max"] == 0.0
    assert facts["refined_shape"] == [1, H, W]


def test_identity_homography_property(dev, L):
    """src camera == ref camera: the warp must return the source itself, so pass B equals the closed form
    vol[g] = mean_{c in g} ref*src (all views weighted alike) at full DTU stage-4 size."""
    from mvsformerplusplus_b200 import synth
    H, W, C, D, V = 1152, 1536, 8, 4, 2
    pm = synth.make_proj_matrices(1, H, W)["stage4"][0]
    pm = torch.cat([pm, pm], 0).to(dev)
    homs = torch.empty(12, device=dev)
    kinv = torch.empty(9, device=dev)
    ck(L.mvsf_compose_geometry(P(pm), 2, P(homs), P(kinv), S()), "compose_geometry")
    g = torch.Generator(device="cpu").manual_seed(0)
    f = torch.randn(V, H, W, C, generator=g).to(dev)
    dd = (425.0 + 100.0 * torch.arange(D, dtype=torch.float32)).view(D, 1, 1).expand(D, H, W).contiguous().to(dev)
    vis = torch.full((1, H, W), 0.7, device=dev)
    vol = torch.empty(D, H, W, C, device=dev)
    ck(L.mvsf_warp_corr_aggregate(P(f), P(homs), P(dd), P(vis), P(vol), V, C, 8, D, H, W, S()), "warp_corr_aggregate")
    want = (f[0] * f[1]) * (0.7 / (0.7 + 1e-6))
    e = float((vol - want[None]).abs().max())
    rec("identity_homography", abs=e)
    assert e < 5e-3  # coordinates round-trip through fp32 normalisation (<=1e-4 px) on white-noise features


# ----------------------------------------------------------------------------------------------- tensor-core attention
@pytest.mark.parametrize("N", [200, 1000, 4000, 27648, 32640])
def test_attention_tensor_core_vs_fp64(dev, L, N):
    """Product attention kernel (tcgen05, fp16 hi|lo split Q/K/V operands, fp16 softmax probabilities) against an fp64
    softmax(QK^T*scale)V evaluated with torch on the GPU (test-side ground truth, chunked over queries).
    Inputs are deliberately harsher than LayerNorm-ed tokens (std 1.5 -> |score| up to ~14 in log2 units).
    N = 32640 is the Tanks&Temples token count (odd number of 128-query tiles: the last CTA repeats a tile)."""
    g = torch.Generator().manual_seed(N)
    qkv = torch.randn(N, 192, generator=g) * 1.5
    scale = 16 ** -0.5 * math.log(N, 12185)
    qd = qkv.to(dev)
    ws = torch.empty((N + 128) * 224 + 16, device=dev)
    o0 = torch.empty(N, 64, device=dev)
    ck(L.mvsf_attention_forward(P(qd), P(o0), P(ws), ctypes.c_size_t(ws.numel() * 4), N, float(scale), S()), "attention")
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(3):
        ck(L.mvsf_attention_forward(P(qd), P(o0), P(ws), ctypes.c_size_t(ws.numel() * 4), N, float(scale), S()), "attention")
    ev[1].record()
    torch.cuda.synchronize()
    ms = ev[0].elapsed_time(ev[1]) / 3
    q, k, v = [qd[:, i * 64:(i + 1) * 64].double().view(N, 4, 16).transpose(0, 1) for i in range(3)]
    want = torch.empty(4, N, 16, dtype=torch.float64, device=dev)
    for s0 in range(0, N, 2048):
        a = torch.softmax(q[:, s0:s0 + 2048] @ k.transpose(1, 2) * scale, -1)
        want[:, s0:s0 + 2048] = a @ v
    want = want.transpose(0, 1).reshape(N, 64)
    e_tc, sc = max_abs(o0, want), float(want.abs().max())
    rms = float((o0.double() - want).pow(2).mean().sqrt())
    rec(f"attention_N{N}_plo0", tc_vs_f64=e_tc, rms=rms, scale=sc, ms_with_operand_tiling=ms)   # record name read by tools/
    # fp16 P: 2.5e-4 of the output scale 4.3 (DESIGN.md §2); an fp32 one-thread-per-query kernel measured 4.3e-4
    assert e_tc < 4e-4 * sc


def test_prefetching_runner_matches_direct_call(dev):
    """streaming.PrefetchingRunner (copy stream + two device slots) returns what a direct forward_features on
    device-resident inputs returns, for alternating batches, with and without prefetch."""
    import bench
    from mvsformerplusplus_b200.streaming import PrefetchingRunner
    net, _ = bench.make_net()
    net = net.to(dev)
    wl = bench.WORKLOADS["small"]
    batches = []
    for seed in (11, 12, 13):
        f, p, d = bench.make_inputs(wl, seed)
        batches.append(({k: v.pin_memory() for k, v in f.items()}, {k: v.pin_memory() for k, v in p.items()}, d.pin_memory()))
    want = []
    for f, p, d in batches:
        out = net.forward_features({k: v.to(dev) for k, v in f.items()}, {k: v.to(dev) for k, v in p.items()}, d.to(dev), bench.TMP)
        want.append((out["refined_depth"].clone(), out["photometric_confidence"].clone()))
    runner = PrefetchingRunner(net, dev)
    order = [0, 1, 2, 0, 2, 1, 1]
    for i, b in enumerate(order):
        nxt = batches[order[i + 1]] if i + 1 < len(order) and i % 3 != 2 else None   # every third call: no prefetch
        out = runner.run(batches[b], next_batch=nxt, tmp=bench.TMP)
        torch.cuda.synchronize()
        assert torch.equal(out["refined_depth"], want[b][0]), f"call {i} (batch {b})"
        assert torch.equal(out["photometric_confidence"], want[b][1])
