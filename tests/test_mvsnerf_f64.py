"""oracle/mvsnerf_f64.py (the float64 restatement of K1b, the K3b row and the MLP) against the golden vectors of the
UNMODIFIED reference (tests/golden/mvsnerf_ops.npz), on the CPU.

The golden outputs are float32, so the bar is float32 accuracy: |f64 - golden| <= 1e-5 * (max |golden| + |golden|)
per element.  In-mask bits must be equal except where the float64 decision margin is below 1e-6."""
import numpy as np
import torch

from boostmvsnerfs_b200.modules_mvs import MvsNerfMlp
from conftest import load_golden
from oracle import mvsnerf_f64 as F64
from oracle import mvsnerf_oracle as M

H, W = 64, 96
RTOL = 1e-5


def close(a, b, what, rtol=RTOL, keep=None):
    a = a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
    b = np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape, f"{what}: shape {a.shape} vs {b.shape}"
    err = np.abs(a - b)
    bad = err > rtol * (np.abs(b).max() + np.abs(b))
    if keep is not None:
        bad &= keep
    assert not bad.any(), f"{what}: {int(bad.sum())}/{a.size} outside {rtol:g}; max abs err {err.max():.3e}"


def test_cost_volume_restates_the_reference():
    g = load_golden("mvsnerf_ops.npz")
    feats = g.t("in_feats")[0]
    small = torch.nn.functional.interpolate(g.t("in_src_inps")[0], (H // 4, W // 4), mode="bilinear", align_corners=False)
    r = F64.cost_volume_var_img(feats, small, [0, 1, 2], g.t("proj_mats")[0], g.t("planes")[0], 24)
    ref = g.np("volume41")[0]
    # a voxel whose source sample sits on the mask boundary may be counted differently by float32: its variance differs
    keep = (r["margin"] >= 1e-6).all(0).numpy()
    close(r["vol"][:9], ref[:9], "colour channels")
    close(r["vol"][9:], ref[9:], "feature variance", keep=np.broadcast_to(keep, ref[9:].shape))
    assert keep.mean() > 0.999
    assert float(r["vol"][:3, :, :24].abs().max()) == 0.0
    assert (r["count"] >= 1).all() and (r["count"] <= 3).all()


def test_march_fetch_row_and_mlp_restate_the_reference():
    g = load_golden("mvsnerf_ops.npz")
    rays = g.t("in_rays_sub")[0]
    _, z = M.ray_marcher(rays[None], 8)
    nf = g.np("near_far")
    r = F64.march_fetch_row(rays, z[0], [0, 1, 2], g.t("in_src_exts")[0], g.t("in_src_ixts")[0], H, W,
                            float(nf.min()), float(nf.max()), g.t("in_regvol")[0], g.t("in_src_inps")[0])
    ref = g.np("mlp_input")
    close(r["ndc"], g.np("ndc")[0], "ndc")
    close(r["row"][..., :3], ref[..., :3], "row ndc")
    # sin / cos of 2^k ndc: the float32 reference rounds ndc to 6e-8 and multiplies by up to 512, so its argument carries up
    # to ~3e-5 of error at k = 9; k < 5 stays within float32 accuracy
    close(r["row"][..., 3:18], ref[..., 3:18], "positional encoding sin, k < 5")
    close(r["row"][..., 33:48], ref[..., 33:48], "positional encoding cos, k < 5")
    close(r["row"][..., 3:63], ref[..., 3:63], "positional encoding", rtol=1e-4)
    close(r["vox"], ref[..., 63:71], "volume feature")
    cols = ref[..., 71:83].reshape(768, 8, 3, 4)
    close(r["rgb"], cols[..., :3], "colours")
    keep = (r["in_margin"] >= 1e-6).numpy()
    got = r["inside"].numpy()
    assert ((got == (cols[..., 3] > 0)) | ~keep).all(), "in-mask bits"
    assert keep.mean() > 0.99
    close(r["dir"], ref[..., 83:], "view direction")
    # 3-D visibility of the golden 2-D mask rays (S = 8 on in_rays_sub is not stored; the count rule is checked here)
    vkeep = (r["vis_margin"] >= 1e-6).numpy()
    m = M.E.mask_viewport(torch.from_numpy(r["xyz"].numpy().astype(np.float32))[None], g.t("in_src_exts"),
                          g.t("in_src_ixts"), torch.tensor([W - 1, H - 1], dtype=torch.float32))
    cnt = np.rint(m.numpy().reshape(768, 8) * 3)
    assert ((cnt == r["vis_count"].numpy()) | ~vkeep).all(), "visibility count"
    # the MLP in float64 on the golden input
    mlp = MvsNerfMlp().eval()
    mlp.load_state_dict({k[len("sd_nerf."):]: g.t(k) for k in g.keys() if k.startswith("sd_nerf.")}, strict=True)
    out = F64.mlp(mlp, g.t("mlp_input"))
    assert out.dtype == torch.float64
    close(out, g.np("mlp_output"), "MLP output")
