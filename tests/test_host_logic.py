"""CPU-only checks of the host side: C-ABI surface, struct layout, config mirror, weight packing,
inference plan, refusal paths, benchmark byte model.  No kernel is launched here."""
import ctypes
import os
import re
import sys

import numpy as np
import pytest
import torch

from boostmvsnerfs_b200 import _lib, mlp_pack
from boostmvsnerfs_b200.config import RenderConfig
from boostmvsnerfs_b200.inference_plan import PlanCache, folded_copy
from boostmvsnerfs_b200.modules import CostRegNet, FeatureNet, MinCostRegNet, NeRF
from boostmvsnerfs_b200.synth import make_scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "bmv.h")).read()
    declared = set(re.findall(r"BMV_API\s+[\w\s\*]+?\b(bmv_\w+)\s*\(", hdr))
    assert {"bmv_cost_volume_var", "bmv_depth_regression", "bmv_raygen_sample_fetch", "bmv_composite_blend",
            "bmv_composite", "bmv_mask_viewport", "bmv_render_rays", "bmv_nerf_mlp", "bmv_version"} <= declared
    lib = _lib.load()
    for sym in declared:
        assert hasattr(lib, sym), f"{sym} declared in include/bmv.h but not exported"
    assert set(_lib.ENTRY_POINTS) | set(_lib.PLAIN_SYMBOLS) == declared
    assert lib.bmv_version() == 100


def test_struct_layouts_match_the_library():
    lib = _lib.load()
    for name, struct in _lib.ENTRY_POINTS.items():
        assert lib.bmv_sizeof_params(name.encode()) == ctypes.sizeof(struct), name
    assert lib.bmv_sizeof_params(b"nope") == -1


def test_invalid_arguments_return_status_not_crash():
    lib = _lib.load()
    p = _lib.CompositeBlendParams()
    p.K, p.S, p.R = 0, 2, 10
    assert lib.bmv_composite_blend(ctypes.byref(p), None) == -1
    assert b"K=0" in lib.bmv_last_error_string()
    q = _lib.CostVolumeParams()
    assert lib.bmv_cost_volume_var(ctypes.byref(q), None) == -1
    assert lib.bmv_cost_volume_var(None, None) == -1
    r = _lib.NerfMlpParams()
    r.P = -1
    assert lib.bmv_nerf_mlp(ctypes.byref(r), None) == -1
    assert lib.bmv_nerf_mlp_weight_count(11) == mlp_pack.layout(11)["TOTAL"]
    assert lib.bmv_nerf_mlp_weight_count(35) == mlp_pack.layout(35)["TOTAL"]
    assert lib.bmv_nerf_mlp_weight_count(7) == -1
    with pytest.raises(_lib.BmvError):
        _lib.call("bmv_composite_blend", p, 0)
    # the two multi-chain render entries share one argument check (render_multi_check.cuh): same status, own name in the text
    for entry in ("bmv_render_rays_multi", "bmv_render_rays_multi_umma"):
        m = _lib.RenderMultiParams()
        m.K, m.n_views = 0, 3
        assert getattr(lib, entry)(ctypes.byref(m), None) == -1
        assert entry.encode() + b": K must be" in lib.bmv_last_error_string()
        assert getattr(lib, entry)(None, None) == -1
        m.K = 2                                            # n_rays = 0: nothing to do, whatever the pointers are
        assert getattr(lib, entry)(ctypes.byref(m), None) == 0


def test_streamed_feats_is_a_dict_when_nothing_is_in_flight():
    from boostmvsnerfs_b200.network import StreamedFeats
    f = StreamedFeats({"level_0": 1, "level_1": 2})
    f["rgb_nhwc4"] = 3
    assert f["level_1"] == 2 and f.get("rgb_nhwc4") == 3 and f.get("missing") is None and sorted(f) == ["level_0", "level_1", "rgb_nhwc4"]
    f.join()                                               # no events recorded: nothing to wait for
    assert f.ready == {}


def test_ops_refuse_cpu_tensors():
    from boostmvsnerfs_b200 import ops
    with pytest.raises(_lib.BmvError):
        ops.depth_regression(torch.zeros(8, 4, 4), torch.zeros(8, 4, 4), False)
    with pytest.raises(_lib.BmvError):
        ops.composite(torch.zeros(4, 2, 4), torch.zeros(4, 2))


def test_render_config_presets():
    e = RenderConfig.enerf_eval()
    assert e.k_best == 4 and e.render_if == (False, True) and e.volume_planes == (64, 8) and e.num_samples == (8, 2)
    assert RenderConfig.enerf_pretrain(2).render_if == (True, True)
    m = RenderConfig.mvsnerf_eval(4, 128)
    assert m.num == 1 and m.depth_inv == (False,) and m.num_samples == (128,)


def test_synthetic_scene_contract():
    b = make_scene(H=64, W=96, n_views=5, seed=1)
    assert b["all_src_inps"].shape == (1, 5, 3, 64, 96) and b["all_src_inps"].abs().max() <= 1
    assert b["all_src_exts"].shape == (1, 5, 4, 4) and b["all_src_ixts"].shape == (1, 5, 3, 3)
    assert b["rays_1"].shape == (1, 64 * 96, 8) and b["rays_0"].shape == (1, 16 * 24, 8)
    r = b["rays_1"][0].view(64, 96, 8)
    assert torch.equal(r[..., 6], torch.arange(96.).expand(64, 96)) and torch.equal(r[..., 7], torch.arange(64.)[:, None].expand(64, 96))
    # every camera looks at (0,0,5): the point projects to the principal point
    p = torch.tensor([0., 0., 5., 1.])
    for v in range(5):
        c = b["all_src_exts"][0, v] @ p
        q = b["all_src_ixts"][0, v] @ c[:3]
        assert abs(q[0] / q[2] - 48) < 1e-3 and abs(q[1] / q[2] - 32) < 1e-3 and c[2] > 0


@pytest.mark.parametrize("F", [11, 35])
def test_mlp_weight_packing_reproduces_the_module(F):
    torch.manual_seed(F)
    net = NeRF(feat_ch=F).eval()
    for prm in net.parameters():
        if prm.dim() == 1:
            prm.data.normal_(0, 0.3)
    packed = mlp_pack.pack_nerf_weights(net)
    assert packed.numel() == mlp_pack.layout(F)["TOTAL"] and packed.numel() % 4 == 0
    vox, img = torch.randn(1, 777, 8), torch.randn(1, 777, 3, F + 4)
    with torch.no_grad():
        ref = net(vox, img)[0]
        got = mlp_pack.eval_packed(packed, vox[0], img[0])
    assert torch.allclose(ref, got, rtol=1e-5, atol=1e-5)
    with pytest.raises(ValueError):
        mlp_pack.pack_nerf_weights(NeRF(feat_ch=F, viewdir_agg=False))


@pytest.mark.parametrize("mk,shape", [(lambda: FeatureNet(), (2, 3, 32, 64)),
                                      (lambda: MinCostRegNet(32), (1, 32, 8, 16, 16)),
                                      (lambda: CostRegNet(16), (1, 16, 8, 16, 32))])
def test_bn_folding_is_exact_up_to_rounding(mk, shape):
    torch.manual_seed(1)
    net = mk().eval()
    gen = torch.Generator().manual_seed(2)
    for m in net.modules():
        if isinstance(m, (torch.nn.BatchNorm2d, torch.nn.BatchNorm3d)):
            m.running_mean.copy_(torch.randn(m.running_mean.shape, generator=gen) * 0.2)
            m.running_var.copy_(torch.rand(m.running_var.shape, generator=gen) + 0.5)
            m.weight.data.copy_(torch.rand(m.weight.shape, generator=gen) + 0.5)
            m.bias.data.copy_(torch.randn(m.bias.shape, generator=gen) * 0.1)
    x = torch.randn(*shape)
    folded = folded_copy(net)
    assert not any(isinstance(m, (torch.nn.BatchNorm2d, torch.nn.BatchNorm3d)) for m in folded.modules())
    assert sorted(net.state_dict()) == sorted(mk().state_dict())      # originals untouched
    with torch.no_grad():
        a, b = net(x), folded(x)
    for u, v in zip(a, b):
        assert torch.allclose(u, v, rtol=1e-4, atol=1e-5 * float(u.abs().max()))
    cache = PlanCache()
    f1 = cache.get("n", net, None)
    assert cache.get("n", net, None) is f1
    with torch.no_grad():
        next(net.parameters()).add_(1.0)            # in-place update (as load_state_dict does) -> rebuilt
    assert cache.get("n", net, None) is not f1


def test_network_refusals_and_contract():
    from boostmvsnerfs_b200 import network
    rc = RenderConfig.enerf_eval(2)
    net = network.BoostEnerfNetwork(preprocess=True, rc=rc)
    names = set(k.split(".")[0] for k in net.state_dict())
    assert names == {"feature_net", "cost_reg_0", "cost_reg_1", "nerf_0", "nerf_1"}   # checkpoint contract
    net.view_selection_outputs = {"synth_0": [0, 1]}
    scene = make_scene(H=64, W=96, n_views=4)
    with pytest.raises(RuntimeError, match="inference-only"):
        net.train()(scene)
    with pytest.raises(RuntimeError, match="no CPU path"):
        net.eval()(scene)
    with pytest.raises(FileNotFoundError):
        network.BoostEnerfNetwork(preprocess=False, view_selection_file="/nonexistent/view_selection.json")
    assert network._combinations(6, 3) == [tuple(r) for r in torch.combinations(torch.arange(6), 3).tolist()]


def test_missing_library_fails_loudly(tmp_path, monkeypatch):
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "libbmv.so"))
    with pytest.raises(_lib.BmvError, match="no CPU fallback"):
        _lib.load()


def test_bench_byte_model_matches_survey():
    sys.path.insert(0, ROOT)
    import bench
    alg = bench.algorithmic_bytes(bench.WORKLOADS["C2"], RenderConfig.enerf_eval(4))
    assert alg["cost_volume_l0"] == 79380480            # SURVEY.md §8(d): 79.4 MB
    assert alg["cost_volume_l1"] == 96092160            # 96.1 MB
    assert alg["raygen_fetch_l1"] == 350945280          # 351 MB
    assert alg["composite_blend_l1"] == 112803840       # 113 MB (216 B/ray)


def test_bench_dump_outputs_writes_float_arrays_and_a_fixed_sample_above_the_limit(tmp_path):
    import bench
    g = torch.Generator().manual_seed(0)
    outs = {"rgb": torch.rand(1, 1000, 3, generator=g).half(), "depth": torch.rand(1, 1000, generator=g),
            "count": torch.arange(7), "_size": (4, 5)}
    bench.dump_outputs(str(tmp_path / "whole"), outs)
    for k in ("rgb", "depth", "count"):
        a = np.load(tmp_path / "whole" / f"{k}.npy")
        assert a.dtype == (np.float64 if k == "count" else np.float32)
        assert np.array_equal(a, outs[k].double().numpy())
    assert sorted(os.listdir(tmp_path / "whole")) == ["count.npy", "depth.npy", "rgb.npy"]
    limit = 4000                                        # below the 16056 B of the three arrays as dumped
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), outs, limit=limit)
    total = 0
    for k in ("rgb", "depth", "count"):
        a, b = np.load(tmp_path / "a" / f"{k}.npy"), np.load(tmp_path / "b" / f"{k}.npy")
        assert np.array_equal(a, b) and a.ndim == 1 and 0 < a.size < outs[k].numel()
        assert np.isin(a, outs[k].double().numpy().reshape(-1)).all()
        total += a.nbytes
    assert total <= limit


class _YacsNode(dict):
    """Attribute access over a dict, like the reference's yacs CfgNode."""
    __getattr__ = dict.__getitem__


def test_plugin_loads_through_the_reference_factory(tmp_path, monkeypatch):
    """The plugin file loaded the way the reference's factory loads a network: imp.load_source(cfg.network_module,
    cfg.network_path).Network([preprocess]) (reference lib/networks/make_network.py:3-10), network_path being the module
    name as a path relative to the CWD (reference lib/config/config.py:166-168).  The reference's global config module
    `lib.config` is stood in for by the evaluate/enerf_ours values with enerf.cas_config.k_best 2; the network must load
    the reference network's own state dict under that config (the sd_* arrays of tests/golden/enerf_chain_eval.npz)
    strictly, and without pre-processing it needs <result_dir>/view_selection.json like the reference."""
    import dataclasses
    import json
    import types
    monkeypatch.syspath_prepend(os.path.join(ROOT, "oracle", "shims"))
    import imp                                                   # the shim of the stdlib module the factory uses
    from conftest import load_golden
    rc = dataclasses.asdict(RenderConfig.enerf_eval(2))
    top = ("cost_volume_input_views", "chunk_size", "white_bkgd", "viewdir_agg")
    module = "boostmvsnerfs_b200.reference_plugin.boost_enerf"
    cfg = _YacsNode(network_module=module, network_path=module.replace(".", "/") + ".py", result_dir=str(tmp_path),
                    enerf=_YacsNode({k: rc[k] for k in top}, cas_config=_YacsNode({k: v for k, v in rc.items() if k not in top})))
    monkeypatch.setitem(sys.modules, "lib", types.ModuleType("lib"))
    monkeypatch.setitem(sys.modules, "lib.config", types.SimpleNamespace(cfg=cfg))
    monkeypatch.delitem(sys.modules, module, raising=False)
    monkeypatch.chdir(ROOT)

    def make_network(cfg, *args):
        return imp.load_source(cfg.network_module, cfg.network_path).Network(*args)

    net = make_network(cfg, True)
    g = load_golden("enerf_chain_eval.npz")
    net.load_state_dict({k[3:]: g.t(k) for k in g.keys() if k.startswith("sd_")}, strict=True)
    assert net.rc.k_best == 2 and net.rc.render_if == (False, True)
    with pytest.raises(FileNotFoundError):
        make_network(cfg)
    (tmp_path / "view_selection.json").write_text(json.dumps({"synth_0": [1, 2]}))
    assert make_network(cfg).view_selection_outputs == {"synth_0": [1, 2]}


def test_sinks_oracle_arithmetic():
    """oracle/sinks_oracle.py against an independent float64 evaluation of the published PSNR definition and numpy's
    own casts (the reference's Evaluator cannot be imported here: lpips / skimage / cv2 are absent)."""
    import numpy as np
    from oracle import sinks_oracle as SO
    rs = np.random.RandomState(1)
    pred, gt = rs.rand(40, 50, 3).astype(np.float32), rs.rand(40, 50, 3).astype(np.float32)
    mask = (rs.rand(40, 50) > 0.5).astype(np.uint8)
    sel = mask[4:-4, 5:-5] >= 1
    mse = ((gt[4:-4, 5:-5][sel].astype(np.float64) - pred[4:-4, 5:-5][sel].astype(np.float64)) ** 2).sum() / (sel.sum() * 3)
    assert abs(SO.frame_psnr(pred, gt, mask, eval_center=True) - 10 * np.log10(1 / mse)) < 1e-12
    rgb8, d8 = SO.frame_to_u8(np.array([[0.0, 0.999, 1.0]], np.float32), np.array([2.0, 3.0, 4.0], np.float32))
    assert rgb8.tolist() == [[0, 254, 255]] and d8.tolist() == [0, 127, 255]


def test_bench_accounts_the_tensor_core_fpn_route():
    """bench.conv_kernel_bytes: compulsory HBM bytes of the FPN launches for the cuDNN route of conv1.x / conv2.x (fp32 c0 +
    its space-to-depth copy; pinned to the figures of DESIGN.md section 3) and for the bmv_conv2d_k3 route (fp16 tensors
    between the stem and the top layer, four extra launches)."""
    import bench
    from boostmvsnerfs_b200.config import RenderConfig
    wl = bench.WORKLOADS["C2"]
    rc = RenderConfig.enerf_eval(wl["K"])
    px = wl["n_views"] * wl["H"] * wl["W"]
    old = bench.conv_kernel_bytes(wl, rc, 2, "bmv_conv3d_k3_umma", False)
    new = bench.conv_kernel_bytes(wl, rc, 2, "bmv_conv3d_k3_umma", True)
    assert "bmv_conv2d_k3" not in old and [n for n, _ in new["bmv_conv2d_k3"]] == ["fpn_conv1_0", "fpn_conv1_1", "fpn_conv2_0", "fpn_conv2_1_top"]
    assert dict(old["bmv_fpn_stem"])["fpn_stem"] == px * 4 * (3 + 8 + 4 + 8)
    assert dict(new["bmv_fpn_stem"])["fpn_stem"] == px * (12 + 16 + 16)                    # image in, rgb4 + fp16 c0 out
    assert dict(new["bmv_conv2d_k3"])["fpn_conv1_0"] == px * 16 + px // 4 * 32             # fp16 c0 in, fp16 (N,16,H/2,W/2) out
    assert dict(new["bmv_conv2d_k3"])["fpn_conv2_1_top"] == px // 16 * 32 * 6              # fp16 in, fp32 top-layer out
    for (n0, b0), (n1, b1) in zip(old["bmv_fpn_topdown_smooth"], new["bmv_fpn_topdown_smooth"]):
        assert n0 == n1 and b1 < b0                                                         # fp16 lateral inputs
    assert old["bmv_conv3d_k3"] == new["bmv_conv3d_k3"]


def test_fpn_plan_routes_mid_layers_only_for_shapes_it_supports():
    """FusedTopDownFPN._mid_ok: conv1.x / conv2.x / top layer go to bmv_conv2d_k3 only when the folded plan has the
    regrouped 5x5 layers, biases everywhere and H, W are multiples of 4 (two space-to-depth steps); everything else keeps
    the cuDNN route.  Host logic only (no launch)."""
    import torch
    from boostmvsnerfs_b200.inference_plan import FusedTopDownFPN, folded_copy
    from boostmvsnerfs_b200.modules import FeatureNet
    torch.manual_seed(0)
    plan = FusedTopDownFPN(folded_copy(FeatureNet().eval(), torch.channels_last))
    assert plan._mid_ok(torch.empty(2, 3, 64, 96))
    assert not plan._mid_ok(torch.empty(2, 3, 66, 96)) and not plan._mid_ok(torch.empty(2, 3, 64, 98))
    plan.tensor_core_mid = False
    assert not plan._mid_ok(torch.empty(2, 3, 64, 96))
    plan.tensor_core_mid = True
    unfolded = FusedTopDownFPN(FeatureNet().eval())                     # BN not folded, 5x5 layers not regrouped
    assert not unfolded._mid_ok(torch.empty(2, 3, 64, 96))


def test_volume_scale_requests_follow_the_fp16_volume_gating():
    """Network._volume_scale_requests: a range scale is requested from the FPN plan only for levels >= 1 whose cost volume is
    stored in fp16 (CUDA, channels-last, TF32-class convolutions allowed, range scaling on) — never on the CPU."""
    import torch
    from boostmvsnerfs_b200 import network
    from boostmvsnerfs_b200.config import RenderConfig
    net = network.BoostEnerfNetwork(preprocess=True, rc=RenderConfig.enerf_eval(2)).eval()
    assert net._volume_scale_requests(torch.device("cpu")) is None
    assert not net._fp16_volume(1, 16, torch.device("cpu"))
    net.volume_range_scale = False
    assert net._volume_scale_requests(torch.device("cpu")) is None
