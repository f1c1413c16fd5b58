"""CPU-side tests: the C-ABI library builds/loads and exports every symbol include/mvsf_b200.h declares (no compute
calls without a GPU), host logic (config schema, state-dict key compatibility, weight packing) and loud failure
without a CUDA device."""
import os
import re

import pytest
import torch

from mvsformerplusplus_b200 import packing, synth
from mvsformerplusplus_b200.config import default_args, load_args, validate_args
from mvsformerplusplus_b200.params import build_hotpath_params

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from mvsformerplusplus_b200.build import build
    build()
    from mvsformerplusplus_b200 import _lib
    return _lib.lib()


def test_library_exports_every_declared_symbol(lib):
    hdr = open(os.path.join(ROOT, "include", "mvsf_b200.h")).read()
    names = sorted(set(re.findall(r"\b(mvsf_[a-z0-9_]+)\s*\(", hdr)))
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/mvsf_b200.h but not exported"
    assert lib.mvsf_abi_version() == 1


def test_bad_arguments_are_rejected_without_touching_the_gpu(lib):
    import ctypes
    from mvsformerplusplus_b200 import _lib
    need = ctypes.c_size_t(0)
    rc = lib.mvsf_costreg_tr_workspace_bytes(8, 31, 16, 16, ctypes.byref(need))  # D not a multiple of 2
    assert rc == -1 and b"down_rate" in lib.mvsf_last_error()
    assert lib.mvsf_costreg_unet_workspace_bytes(0, 8, 12, 16, 16, ctypes.byref(need)) == -1  # CostRegNet needs D % 8 == 0
    assert lib.mvsf_costreg_unet_workspace_bytes(1, 8, 4, 1152, 1536, ctypes.byref(need)) == 0
    # fp16 hi|lo buffers, 4 bytes per element: the split input (n0) + two buffers per level
    n0, n1, n2, n3 = 4 * 1152 * 1536 * 8, 4 * 576 * 768 * 16, 4 * 288 * 384 * 32, 4 * 144 * 192 * 64
    assert need.value == 4 * (n0 + 2 * (n1 + n2 + n3))
    assert lib.mvsf_costreg_unet_tc_bytes(ctypes.byref(need)) == 0 and need.value % 16 == 0 and need.value > 0
    with pytest.raises(RuntimeError, match="status -1"):
        _lib.check(lib.mvsf_warp_corr_entropy(None, None, None, None, 5, 8, 8, 4, 16, 16, None), "warp_corr_entropy")


def test_state_dict_keys_match_reference_inventory():
    m = build_hotpath_params(default_args())
    mine = {k: tuple(v.shape) for k, v in m.state_dict().items()}
    ref = {}
    for line in open(os.path.join(ROOT, "tests", "golden", "hotpath_state_dict_keys.txt")):
        k, s = line.strip().split(" ", 1)
        ref[k] = eval(s)
    assert mine == ref


def test_hotpath_modules_have_reference_keys_and_fail_loudly_on_cpu():
    from mvsformerplusplus_b200.hotpath import HotPathNet
    net = HotPathNet(default_args()).eval()
    ref = [l.split(" ", 1)[0] for l in open(os.path.join(ROOT, "tests", "golden", "hotpath_state_dict_keys.txt"))]
    assert sorted(net.state_dict().keys()) == sorted(ref)
    feats = synth.make_features(3, 64, 96)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        net.forward_features(feats, synth.make_proj_matrices(3, 64, 96), synth.make_depth_values(48), [5., 5., 5., 1.])


def test_config_schema_and_reference_errors():
    a = load_args({"arch": {"args": {"ndepths": [16, 8, 8, 4]}}})
    assert a["ndepths"] == [16, 8, 8, 4] and a["base_ch"] == [8, 8, 8, 8]
    validate_args(a)
    bad = default_args(); bad["fusion_type"] = "mean"
    with pytest.raises(NotImplementedError, match="Not implemented fusion type"):
        validate_args(bad)
    bad = default_args(); bad["FMT_config"]["attention_type"] = "FLASH2"
    with pytest.raises(NotImplementedError):
        validate_args(bad)


def test_packing_layout_sizes_and_bn_folding():
    m = build_hotpath_params(default_args()).eval()
    sd = synth.randomize_state_dict(m, seed=4)
    assert packing.pack_vis(sd, "fusions.0.vis.").numel() == 3652
    k0, f0 = packing.pack_costreg_unet(sd, "fusions.1.cost_reg.")
    k1, f1 = packing.pack_costreg_unet(sd, "fusions.3.cost_reg.")
    assert (k0, k1) == (0, 1) and f0.numel() == 290800 and f1.numel() == 290596
    assert packing.pack_costreg_tr(sd, "fusions.0.cost_reg.", 6).numel() == 332960
    assert packing.pack_fmt(sd).numel() == 214464
    # folded conv+bias reproduces conv -> BatchNorm(eval)
    x = torch.randn(1, 1, 9, 9)
    w = sd["fusions.0.vis.0.conv.weight"]
    bn = torch.nn.BatchNorm2d(16).eval()
    bn.load_state_dict({k.split("bn.")[1]: v for k, v in sd.items() if k.startswith("fusions.0.vis.0.bn.")})
    want = bn(torch.nn.functional.conv2d(x, w, padding=1))
    flat = packing.pack_vis(sd, "fusions.0.vis.")
    wf = flat[:144].view(9, 16).t().reshape(16, 1, 3, 3)
    got = torch.nn.functional.conv2d(x, wf, flat[144:160], padding=1)
    assert float((got - want).abs().max()) < 1e-5


def test_validate_args_rejects_hard_coded_transformer_options():
    for key, val in (("post_norm", False), ("qkv_bias", True), ("mid_channel", 32), ("num_heads", 8), ("down_rate", [2, 2, 2])):
        bad = default_args()
        bad["transformer_config"][0][key] = val
        with pytest.raises(NotImplementedError):
            validate_args(bad)
        from mvsformerplusplus_b200.hotpath import HotPathNet
        with pytest.raises(NotImplementedError):   # surfaces at construction, not at the first forward
            HotPathNet(bad)


def test_reference_arm_reproduces_golden_fixture():
    """bench.py --impl reference runs the reference's own modules through oracle/ref_hotpath.py (from oracle/_ref, the
    build-time copy, or /root/reference): it must reproduce the committed reference-executed fixture bit for bit."""
    from oracle import ref_hotpath as RH
    if RH.reference_root() is None:
        pytest.skip("no reference sources (oracle/_ref not built and /root/reference absent)")
    from tests.common import TMP, build_case, load_golden
    gold, meta = load_golden("hotpath_v4_64x96")
    args, params, sd, feats, proj, dv = build_case(meta)
    R = RH.import_reference()
    torch.manual_seed(0)
    model = RH.RefHotPath(R, args).eval()
    model.load_state_dict(sd, strict=True)
    out = RH.reference_hotpath(R, model, args, feats, proj, dv, TMP, capture=False)
    assert torch.equal(out["refined_depth"][0], gold["refined_depth"])
    assert torch.equal(out["photometric_confidence"][0], gold["photometric_confidence"])


def _reference_shaped_model():
    """A model with the `args` and every state-dict entry (name, shape, dtype, parameter or buffer) of the reference's
    DINOv2MVSNet built from its shipped config, as oracle/gen_golden.py recorded them from the reference itself."""
    import json
    inv = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_model_inventory.json")))
    tree = {}
    for name, shape, dtype, kind in inv["state_dict"]:
        *path, leaf = name.split(".")
        node = tree
        for p in path:
            node = node.setdefault(p, {})
        node[leaf] = (shape, getattr(torch, dtype), kind)

    def module(node):
        subs = {k: module(v) for k, v in node.items() if isinstance(v, dict)}
        if subs and all(k.isdigit() for k in subs):   # nn.ModuleList / nn.Sequential children
            m = torch.nn.ModuleList([subs[str(i)] for i in range(len(subs))])
        else:
            m = torch.nn.Module()
            for k, sub in subs.items():
                m.add_module(k, sub)
        for k, v in node.items():
            if not isinstance(v, dict):
                shape, dtype, kind = v
                t = torch.zeros(shape, dtype=dtype)
                if kind == "parameter":
                    m.register_parameter(k, torch.nn.Parameter(t))
                else:
                    m.register_buffer(k, t)
        return m

    model = module(tree)
    model.args = inv["args"]
    return model


def test_install_on_reference_constructed_model_keeps_the_checkpoint_contract():
    """test.py:209-220: init_model -> DINOv2MVSNet(arch.args), here a model with exactly its state-dict entries;
    install() swaps FMT_module / fusions for this package's modules; every state-dict key and value of the model is
    unchanged, so a reference checkpoint loads with strict=True before or after install()."""
    from mvsformerplusplus_b200 import hotpath
    model = _reference_shaped_model().eval()
    synth.randomize_state_dict(model.FMT_module, seed=3)
    synth.randomize_state_dict(model.fusions, seed=4)
    before = {k: v.clone() for k, v in model.state_dict().items()}
    hotpath.install(model)
    assert isinstance(model.FMT_module, hotpath.FMT_with_pathway)
    assert all(isinstance(f, hotpath.StageNet) for f in model.fusions)
    after = model.state_dict()
    assert sorted(after.keys()) == sorted(before.keys())
    for k in before:
        assert torch.equal(after[k], before[k]), k
    model.load_state_dict(before, strict=True)   # test.py:220
    # the installed modules refuse to run on the CPU instead of silently falling back
    feats = synth.make_features(3, 64, 96)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        model.FMT_module.forward(feats)
