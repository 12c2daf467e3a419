"""oracle/mvsnerf_oracle.py against the golden vectors of the UNMODIFIED reference (CPU, bit-exact)."""
import numpy as np
import pytest
import torch

from boostmvsnerfs_b200.config import RenderConfig
from boostmvsnerfs_b200.modules_mvs import MvsnerfModules, MvsNerfMlp
from conftest import load_golden
from oracle import mvsnerf_oracle as M

pytestmark = pytest.mark.usefixtures("golden_threads")
H, W = 64, 96


def same(a, b, what):
    a = a.detach().cpu().numpy() if torch.is_tensor(a) else a
    assert a.shape == b.shape, f"{what}: shape {a.shape} vs {b.shape}"
    bad = int((a != b).sum() - (np.isnan(a) & np.isnan(b)).sum())
    assert bad == 0, f"{what}: {bad}/{a.size} entries differ, max abs {np.nanmax(np.abs(a - b))}"


@pytest.fixture(scope="module")
def g():
    return load_golden("mvsnerf_ops.npz")


def test_proj_mats_and_planes(g):
    same(M.proj_mats(g.t("in_src_exts"), g.t("in_src_ixts")), g.np("proj_mats"), "proj mats")
    near, far, planes = M.depth_planes(g.t("in_depth_ranges")[:, [1, 0, 3]], 8)
    same(planes, g.np("planes"), "planes")
    same(torch.stack([near, far]), g.np("near_far"), "near/far")


def test_cost_volume_41(g):
    vol = M.cost_volume_var_img(g.t("in_src_inps"), g.t("in_feats"), g.t("proj_mats"), g.t("planes"))
    same(vol, g.np("volume41"), "41-channel volume")


def test_march_ndc_and_mlp_input(g):
    rays = g.t("in_rays_sub")
    xyz, z = M.ray_marcher(rays, 8)
    same(xyz, g.np("march_xyz"), "xyz"); same(z, g.np("march_z"), "z")
    nf = g.t("near_far")
    inv = torch.tensor([W - 1, H - 1], dtype=torch.float32)
    ndc = M.ndc_coordinate(g.t("in_src_exts")[0][0], g.t("in_src_ixts")[0][0], xyz[0], inv, near=nf.min(),
                           far=nf.max(), pad=24)[None]
    same(ndc, g.np("ndc"), "ndc")
    x = M.mlp_input(xyz[0], ndc, rays[..., 3:6], g.t("in_regvol"), g.t("in_src_inps"), g.t("in_src_exts"),
                    g.t("in_src_ixts"))
    same(x, g.np("mlp_input"), "86-wide MLP input")
    from oracle import enerf_oracle as E
    same(E.mask_viewport(xyz, g.t("in_src_exts"), g.t("in_src_ixts"), inv), g.np("mask"), "visibility")


def test_mlp_module_matches_reference(g):
    mlp = MvsNerfMlp().eval()
    mlp.load_state_dict({k[len("sd_nerf."):]: g.t(k) for k in g.keys() if k.startswith("sd_nerf.")}, strict=True)
    with torch.no_grad():
        same(mlp(g.t("mlp_input")), g.np("mlp_output"), "Renderer_ours output")


def test_view_selection_mask(g):
    m = M.visibility_mask_2d(g.t("in_rays_0"), g.t("in_src_exts"), g.t("in_src_ixts"), H, W, S=128)
    same(m, g.np("calc_mask"), "2-D coverage mask")


def test_boost_mvsnerf_forward_chain():
    g = load_golden("mvsnerf_chain.npz")
    rc = RenderConfig.mvsnerf_eval(2, 8)
    net = MvsnerfModules().eval()
    net.load_state_dict({k[3:]: g.t(k) for k in g.keys() if k.startswith("sd_")}, strict=True)
    batch = {k[3:]: g.t(k) for k in g.keys() if k.startswith("in_")}
    batch["meta"] = {"scene": ["synth"], "tar_view": torch.tensor([0])}
    with torch.no_grad():
        out = M.boost_mvsnerf_forward(net, batch, rc, g.t("k_best")[None])
    for k in [k[4:] for k in g.keys() if k.startswith("out_")]:
        same(out[k], g.np(f"out_{k}"), f"chain {k}")
    for k in ("src_inps", "src_exts", "src_ixts", "near_far"):
        same(batch[k], g.np(f"after_{k}"), f"batch[{k}] after forward")
    # greedy view selection over all C(4,3) triples (reference forward_view_selection)
    from oracle import enerf_oracle as E
    masks = []
    for t in E.view_triples(4, 3):
        masks.append(M.visibility_mask_2d(batch["rays_0"], batch["all_src_exts"][:, t], batch["all_src_ixts"][:, t], H, W))
    assert M.search_k_best_views(masks, 2) == g.np("view_selection").tolist()


def test_boost_mvsnerf_forward_chain_32_planes():
    """The oracle at the shipped 32 planes / samples against the reference's outputs (mvsnerf_chain_d32.npz: same
    network, scene and selection as mvsnerf_chain.npz)."""
    g = load_golden("mvsnerf_chain.npz")
    gd = load_golden("mvsnerf_chain_d32.npz")
    rc = RenderConfig.mvsnerf_eval(2, 32)
    net = MvsnerfModules().eval()
    net.load_state_dict({k[3:]: g.t(k) for k in g.keys() if k.startswith("sd_")}, strict=True)
    batch = {k[3:]: g.t(k) for k in g.keys() if k.startswith("in_")}
    batch["meta"] = {"scene": ["synth"], "tar_view": torch.tensor([0])}
    with torch.no_grad():
        out = M.boost_mvsnerf_forward(net, batch, rc, g.t("k_best")[None])
    same(out["rgb_level0"], gd.np("out_rgb_level0"), "rgb, 32 planes")
    same(out["depth_level0"], gd.np("out_depth_level0"), "depth, 32 planes")
    same(out["weights_level0"][:, ::8], gd.np("out_weights_level0_every8"), "weights, 32 planes")
