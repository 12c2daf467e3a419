"""The oracle (oracle/enerf_oracle.py) against the golden vectors produced by the UNMODIFIED
reference (oracle/gen_golden.py).  CPU only; bit-exact — the oracle restates the reference's
own ATen operation sequence, so on the same torch build nothing may differ."""
import numpy as np
import pytest
import torch

from boostmvsnerfs_b200.config import RenderConfig
from boostmvsnerfs_b200.modules import EnerfModules
from conftest import load_golden
from oracle import enerf_oracle as O

pytestmark = pytest.mark.usefixtures("golden_threads")
RC = RenderConfig.enerf_eval(k_best=2)
H, W = 64, 96


def same(a, b, what):
    a = a.detach().cpu().numpy() if torch.is_tensor(a) else a
    assert a.shape == b.shape, f"{what}: shape {a.shape} vs {b.shape}"
    bad = int((a != b).sum() - (np.isnan(a) & np.isnan(b)).sum())
    assert bad == 0, f"{what}: {bad}/{a.size} entries differ, max abs {np.nanmax(np.abs(a - b))}"


def _cams(g):
    return g.t("in_src_exts"), g.t("in_src_ixts"), g.t("in_tar_ext"), g.t("in_tar_ixt")


def test_proj_mats(ops_golden):
    g = ops_golden
    se, si, te, ti = _cams(g)
    same(O.proj_mats(se, si, te, ti, RC.im_feat_scale[0], RC.volume_scale[0]), g.np("proj_mats_l0"), "proj l0")
    same(O.proj_mats(se, si, te, ti, RC.im_feat_scale[1], RC.volume_scale[1]), g.np("proj_mats_l1"), "proj l1")


def test_depth_planes(ops_golden):
    g = ops_golden
    p0, nf0 = O.depth_planes_first(g.t("in_near_far"), 64, H // 8, W // 8, True)
    same(p0, g.np("planes_l0"), "planes l0")
    same(nf0, g.np("near_far_l0"), "near_far l0")
    p1, nf1 = O.depth_planes_next(g.t("depth_l0"), g.t("std_l0"), g.t("near_far_l0"), 8, 4.0, True, False)
    same(p1, g.np("planes_l1"), "planes l1")
    same(nf1, g.np("near_far_l1"), "near_far l1")


def test_cost_volume(ops_golden):
    g = ops_golden
    same(O.homography_warp(g.t("in_feat0")[:, 1], g.t("proj_mats_l0")[:, 1], g.t("planes_l0")),
         g.np("warped_l0_view1"), "warp")
    same(O.cost_volume_var(g.t("in_feat0"), g.t("proj_mats_l0"), g.t("planes_l0")), g.np("volume_l0"), "vol l0")
    same(O.cost_volume_var(g.t("in_feat1"), g.t("proj_mats_l1"), g.t("planes_l1")), g.np("volume_l1"), "vol l1")


def test_depth_regression(ops_golden):
    g = ops_golden
    d, s = O.depth_regression(g.t("in_logits0"), g.t("planes_l0"), True)
    same(d, g.np("depth_l0"), "depth l0"); same(s, g.np("std_l0"), "std l0")
    d, s = O.depth_regression(g.t("in_logits1"), g.t("planes_l1"), False)
    same(d, g.np("depth_l1"), "depth l1"); same(s, g.np("std_l1"), "std l1")


def test_rays_and_samples(ops_golden):
    g = ops_golden
    r1 = O.build_rays(g.t("depth_l1"), g.t("std_l1"), g.t("near_far_l1"), g.t("in_rays_1"), 2.0, False)
    same(r1, g.np("rays12_l1"), "rays12 l1")
    for S, sfx in ((2, ""), (1, "_s1")):
        xyz, uvd, z = O.sample_along_depth(r1, S, False)
        same(xyz, g.np(f"xyz_l1{sfx}"), "xyz"); same(uvd, g.np(f"uvd_l1{sfx}"), "uvd"); same(z, g.np(f"z_l1{sfx}"), "z")
    r0 = O.build_rays(g.t("depth_l0"), g.t("std_l0"), g.t("near_far_l0"), g.t("in_rays_0"), 2.0, True)
    same(r0, g.np("rays12_l0"), "rays12 l0")
    xyz, uvd, z = O.sample_along_depth(r0, 8, True)
    same(xyz, g.np("xyz_l0"), "xyz l0"); same(uvd, g.np("uvd_l0"), "uvd l0"); same(z, g.np("z_l0"), "z l0")


def test_fetches(ops_golden):
    g = ops_golden
    se, si, te, _ = _cams(g)
    uvd = O.normalise_uv(g.t("uvd_l1"), H, W)
    same(O.vox_feat(uvd.reshape(1, -1, 3), g.t("in_regvol1")), g.np("vox_feat_l1"), "vox l1")
    rgbs = O.unpreprocess(g.t("in_src_inps"), 1.0)
    same(rgbs, g.np("unpreprocess_l1"), "unpreprocess l1")
    same(O.img_feat(g.t("xyz_l1"), torch.cat((g.t("in_imfeat2"), rgbs), 2), se, si, te, 1.0),
         g.np("img_feat_l1"), "img_feat l1")
    uvd0 = O.normalise_uv(g.t("uvd_l0"), H // 4, W // 4)
    same(O.vox_feat(uvd0.reshape(1, -1, 3), g.t("in_regvol0")), g.np("vox_feat_l0"), "vox l0")
    rgbs0 = O.unpreprocess(g.t("in_src_inps"), 0.25)
    same(rgbs0, g.np("unpreprocess_l0"), "unpreprocess l0")
    same(O.img_feat(g.t("xyz_l0"), torch.cat((g.t("in_feat0"), rgbs0), 2), se, si, te, 0.25),
         g.np("img_feat_l0"), "img_feat l0")


def test_visibility(ops_golden):
    g = ops_golden
    se, si, _, _ = _cams(g)
    inv = torch.tensor([[W - 1, H - 1]], dtype=torch.float32)
    same(O.mask_viewport(g.t("xyz_l1"), se, si, inv), g.np("mask_l1"), "mask l1")
    wide = g.t("in_xyz_wide")
    m = O.mask_viewport(wide, se, si, inv)
    same(m, g.np("mask_wide"), "mask wide")
    same(O.ndc_coords(wide, se[:, 0], si[:, 0], inv), g.np("ndc_wide_view0"), "ndc")
    cnt = O.visibility_count(wide, se, si, inv)
    assert set(np.unique(cnt.numpy()).tolist()) == {0, 1, 2, 3}, "fixture must exercise every count"
    same((cnt.float() / 3).view(1, -1, 1), g.np("mask_wide"), "count/3 == mask")


def test_compositing(ops_golden):
    g = ops_golden
    raws, masks, zs = g.t("in_blend_raws"), g.t("in_blend_masks"), g.t("in_blend_z")
    out = O.composite_blend(raws, O.merge_masks(masks, raws.shape[1]), zs)
    for k in ("rgb", "depth", "weights"):
        same(out[k], g.np(f"blend_{k}"), f"blend {k}")
    out = O.composite(g.t("in_comp_raw"), g.t("in_comp_z"))
    for k in ("rgb", "depth", "weights"):
        same(out[k], g.np(f"comp_{k}"), f"composite {k}")
    with pytest.raises(NotImplementedError):
        O.composite_blend(raws, masks, zs, white_bkgd=True)


def _load_modules(g, rc):
    net = EnerfModules(rc).eval()
    sd = {k[3:]: g.t(k) for k in g.keys() if k.startswith("sd_")}
    net.load_state_dict(sd, strict=True)          # reference checkpoint names must load unchanged
    return net


def _batch(g):
    b = {k[3:]: g.t(k) for k in g.keys() if k.startswith("in_")}
    b["meta"] = {"scene": ["synth"], "tar_view": torch.tensor([0])}
    return b


@pytest.mark.parametrize("case,rc", [("chain_eval", RenderConfig.enerf_eval(2)),
                                     ("chain_pretrain", RenderConfig.enerf_pretrain(2))])
def test_boost_forward_chain(case, rc):
    g = load_golden(f"enerf_{case}.npz")
    net, batch = _load_modules(g, rc), _batch(g)
    with torch.no_grad():
        out = O.boost_enerf_forward(net, batch, rc, g.t("k_best")[None])
    expect = [k[4:] for k in g.keys() if k.startswith("out_")]
    assert sorted(out.keys()) == sorted(expect)
    for k in expect:
        same(out[k], g.np(f"out_{k}"), f"{case} {k}")
    for k in ("src_inps", "src_exts", "src_ixts"):    # reference leaves the LAST triple in batch
        same(batch[k], g.np(f"after_{k}"), f"batch[{k}] after forward")


@pytest.mark.parametrize("case,rc", [("chain_eval", RenderConfig.enerf_eval(2)),
                                     ("chain_pretrain", RenderConfig.enerf_pretrain(2))])
def test_view_selection_preprocess(case, rc):
    g = load_golden(f"enerf_{case}.npz")
    net, batch = _load_modules(g, rc), _batch(g)
    with torch.no_grad():
        cm = O.calc_mask(net, torch.tensor([0, 1, 3]), batch, rc)
        for k, v in cm.items():
            same(v, g.np(f"calc_mask_013_{k}"), f"{case} calc_mask {k}")
        sel = O.forward_view_selection(net, batch, rc)
    assert sel == {"synth_0": g.np("view_selection").tolist()}


def test_single_volume_chain():
    g = load_golden("enerf_single.npz")
    rc = RenderConfig.enerf_eval(1)
    net, batch = _load_modules(g, rc), _batch(g)
    batch["src_inps"], batch["src_exts"], batch["src_ixts"] = (
        batch["all_src_inps"], batch["all_src_exts"], batch["all_src_ixts"])
    with torch.no_grad():
        out = O.enerf_forward(net, batch, rc)
    for k in [k[4:] for k in g.keys() if k.startswith("out_")]:
        same(out[k], g.np(f"out_{k}"), f"single {k}")
