"""GPU parity of the MVSNeRF flavours (K1b, K3b, BoostMvsnerfNetwork) against the golden vectors of
the UNMODIFIED reference (tests/golden/mvsnerf_*.npz) and the CPU oracle."""
import numpy as np
import pytest
import torch

from boostmvsnerfs_b200.config import RenderConfig
from conftest import load_golden
from oracle import mvsnerf_oracle as M

pytestmark = pytest.mark.gpu
H, W = 64, 96
TRIPLE = [0, 1, 2]


def close(a, b, what, rtol=1e-4, scale=None):
    a = a.detach().float().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
    b = b.detach().float().cpu().numpy() if torch.is_tensor(b) else np.asarray(b)
    assert a.shape == b.shape, f"{what}: shape {a.shape} vs {b.shape}"
    scale = float(np.abs(b).max()) if scale is None else scale
    err = np.abs(a - b)
    bad = err > rtol * scale + rtol * np.abs(b)
    assert not bad.any(), f"{what}: {int(bad.sum())}/{a.size} outside tolerance; max abs err {err.max():.3e} (scale {scale:.3e})"


def exact(a, b, what):
    a = a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
    b = b.detach().cpu().numpy() if torch.is_tensor(b) else np.asarray(b)
    n = int((a != b).sum())
    assert a.shape == b.shape and n == 0, f"{what}: {n}/{a.size} entries differ"


@pytest.fixture(scope="module")
def ops():
    from boostmvsnerfs_b200 import ops as _ops
    return _ops


@pytest.fixture(scope="module")
def g():
    return load_golden("mvsnerf_ops.npz")


@pytest.mark.parametrize("channels_last", [False, True])
def test_cost_volume_41_vs_reference(ops, g, channels_last):
    feats = g.t("in_feats", "cuda")[0]
    if channels_last:
        feats = feats.contiguous(memory_format=torch.channels_last)
    imgs = g.t("in_src_inps", "cuda")[0]
    small = torch.nn.functional.interpolate(imgs, (H // 4, W // 4), mode="bilinear", align_corners=False)
    vol = ops.cost_volume_var_img(feats, small, TRIPLE, g.t("proj_mats", "cuda")[0], g.t("planes", "cuda")[0], 24,
                                  channels_last=channels_last)
    ref = g.np("volume41")[0]
    close(vol[9:], ref[9:], "feature variance channels")
    close(vol[:9], ref[:9], "colour channels")
    assert float(vol[:3, :, :24].abs().max()) == 0.0          # border of the reference-image channels is defined as 0
    bf = ops.cost_volume_var_img(feats, small, TRIPLE, g.t("proj_mats", "cuda")[0], g.t("planes", "cuda")[0], 24,
                                 out_dtype=torch.bfloat16, channels_last=channels_last)
    exact(bf.float(), vol.to(torch.bfloat16).float(), "bf16 volume == rn(fp32 volume)")
    close(bf, ref, "bf16 volume (BASELINE config 3 tolerance)", rtol=1e-2)
    if channels_last:
        # the warp-level kernel (dense channels-last maps, shared tap sets, 16-byte taps) is op for op the thread-per-voxel one
        planar = ops.cost_volume_var_img(g.t("in_feats", "cuda")[0], small, TRIPLE, g.t("proj_mats", "cuda")[0], g.t("planes", "cuda")[0], 24)
        exact(vol, planar, "channels-last kernel == thread-per-voxel kernel")


def test_march_fetch_vs_reference(ops, g):
    rays = g.t("in_rays_sub", "cuda")[0]
    nf = g.np("near_far")
    o = ops.mvs_march_fetch(rays, 8, TRIPLE, g.t("in_src_exts", "cuda")[0], g.t("in_src_ixts", "cuda")[0], H, W,
                            float(nf.min()), float(nf.max()), g.t("in_regvol", "cuda")[0], g.t("in_src_inps", "cuda")[0],
                            want=("mlp_in", "z_vals", "vis_mask", "vis_count"))
    close(o["z_vals"], g.np("march_z")[0], "z", rtol=2e-6)
    ref = g.np("mlp_input")
    close(o["mlp_in"][..., :3], ref[..., :3], "ndc", rtol=2e-5, scale=1.0)
    # sin/cos of 2^k * ndc: argument error grows with the frequency (512 * 1e-6 at k=9)
    close(o["mlp_in"][..., 3:63], ref[..., 3:63], "positional encoding", rtol=2e-3, scale=1.0)
    close(o["mlp_in"][..., 3:33], ref[..., 3:33], "positional encoding, k<5 sin", rtol=2e-4, scale=1.0)
    close(o["mlp_in"][..., 63:71], ref[..., 63:71], "volume feature")
    close(o["mlp_in"][..., 71:83].reshape(-1, 3, 4)[..., :3], ref[..., 71:83].reshape(-1, 3, 4)[..., :3], "colours")
    exact(o["mlp_in"][..., 71:83].reshape(-1, 3, 4)[..., 3], ref[..., 71:83].reshape(-1, 3, 4)[..., 3], "in-mask bits")
    close(o["mlp_in"][..., 83:], ref[..., 83:], "view direction", rtol=1e-5)
    exact(o["vis_mask"].reshape(-1), g.np("mask")[0, :, 0], "3-D visibility")


def test_view_selection_mask_vs_reference(ops, g):
    rays = g.t("in_rays_0", "cuda")[0]
    o = ops.mvs_march_fetch(rays, 128, TRIPLE, g.t("in_src_exts", "cuda")[0], g.t("in_src_ixts", "cuda")[0], H, W,
                            0.0, 1.0, None, None, want=("z_vals", "vis_mask"))
    m = (o["vis_mask"] / 128).unsqueeze(-1).expand(-1, -1, 4).contiguous()
    rgb, _, _ = ops.composite(m, o["z_vals"])
    close(rgb.mean(-1)[None], g.np("calc_mask"), "2-D coverage mask (S=128: warp-scan compositing)", rtol=1e-5)


@pytest.fixture()
def strict_fp32():
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _net_and_batch(gc):
    from boostmvsnerfs_b200.network_mvs import BoostMvsnerfNetwork
    net = BoostMvsnerfNetwork(preprocess=True, rc=RenderConfig.mvsnerf_eval(2, 8))
    net.load_state_dict({k[3:]: gc.t(k) for k in gc.keys() if k.startswith("sd_")}, strict=True)
    net.view_selection_outputs = {"synth_0": gc.np("k_best").tolist()}
    batch = {k[3:]: gc.t(k, "cuda") for k in gc.keys() if k.startswith("in_")}
    batch["meta"] = {"scene": ["synth"], "tar_view": torch.tensor([0])}
    return net.cuda().eval(), batch


def test_boost_mvsnerf_forward_vs_reference(strict_fp32):
    gc = load_golden("mvsnerf_chain.npz")
    net, batch = _net_and_batch(gc)
    out = net(batch)
    assert sorted(out) == sorted(k[4:] for k in gc.keys() if k.startswith("out_"))
    for k in out:
        close(out[k], gc.np(f"out_{k}"), f"chain {k}")
    for k in ("src_inps", "src_exts", "src_ixts", "near_far"):
        close(batch[k], gc.np(f"after_{k}"), f"batch[{k}] after forward", rtol=1e-7)


def test_view_selection_matches_reference():
    gc = load_golden("mvsnerf_chain.npz")
    net, batch = _net_and_batch(gc)
    sel = net.forward_view_selection(batch)
    assert sel == {"synth_0": gc.np("view_selection").tolist()}


def test_bf16_volume_chain_within_1e2(strict_fp32):
    """BASELINE config 3: bf16 cost volume feeding the 3-D CNN, 1e-2 tolerance on the frame."""
    gc = load_golden("mvsnerf_chain.npz")
    net, batch = _net_and_batch(gc)
    net.volume_dtype = torch.bfloat16
    out = net(batch)
    close(out["rgb_level0"], gc.np("out_rgb_level0"), "rgb with bf16 volume", rtol=1e-2)


@pytest.mark.parametrize("S", [32, 128])
def test_fused_mvs_render_matches_fetch_plus_mlp(S):
    """bmv_mvs_render_umma (K3b + the 6x128 MLP on tcgen05, fp16 operands) against bmv_mvs_march_fetch + the fp32
    torch module on the same inputs: z and visibility bit-exact, raw within the TF32-class bound of config 3."""
    from boostmvsnerfs_b200 import mlp_pack, ops
    from boostmvsnerfs_b200.modules_mvs import MvsNerfMlp
    from boostmvsnerfs_b200.synth import batch_to, make_scene
    H, W, N, D = 64, 96, 4, 16
    scene = batch_to(make_scene(H=H, W=W, n_views=N, seed=5, smooth=True, render_scales=(1.0,), mvs_near_far_cols=True), "cuda")
    g = torch.Generator(device="cuda").manual_seed(0)
    vol = torch.randn(8, D, H // 4 + 48, W // 4 + 48, device="cuda", generator=g)
    torch.manual_seed(2)
    mlp = MvsNerfMlp().cuda().eval()
    packed = mlp_pack.pack_mvs_weights_umma(mlp)
    rays = scene["rays_0"][0]
    views = (1, 0, 3)
    args = (rays, S, views, scene["all_src_exts"][0], scene["all_src_ixts"][0], H, W, 1.6, 9.6, vol, scene["all_src_inps"][0])
    ref = ops.mvs_march_fetch(*args, want=("mlp_in", "z_vals", "vis_mask", "vis_count"))
    with torch.no_grad():
        raw_ref = mlp(ref["mlp_in"])
    for b, n in ((0, None), (37, 1001), (1001, 1)):
        got = ops.mvs_render(*args, packed, ray_begin=b, n_rays=n, want_count=True)
        sl = slice(b, None if n is None else b + n)
        if n is None:
            full = got
        for k_ in ("raw", "z_vals", "vis_mask"):        # a sub-range is the matching slice of the full launch, bit for bit
            assert torch.equal(got[k_], full[k_][sl]), f"S={S} range=({b},{n}): {k_}"
        assert torch.equal(got["z_vals"], ref["z_vals"][sl]) and torch.equal(got["vis_count"], ref["vis_count"][sl])
        assert torch.equal(got["vis_mask"], ref["vis_mask"][sl])
        err = float((got["raw"] - raw_ref[sl]).abs().max()) / float(raw_ref.abs().max())
        assert err <= 1e-2, f"S={S} range=({b},{n}): raw differs by {err:.2e}"
        if n != 1:                                      # a mean over many rays; one ray is held by the equality above
            assert float((got["raw"] - raw_ref[sl]).abs().mean()) / float(raw_ref.abs().mean()) <= 2e-3
    # channels-last volume: same result through the 16-byte-load path
    vol_cl = vol.permute(1, 2, 3, 0).contiguous().permute(3, 0, 1, 2)
    got2 = ops.mvs_render(rays, S, views, scene["all_src_exts"][0], scene["all_src_ixts"][0], H, W, 1.6, 9.6, vol_cl,
                          scene["all_src_inps"][0], packed)
    got1 = ops.mvs_render(*args, packed)
    assert float((got2["raw"] - got1["raw"]).abs().max()) <= 1e-5


@pytest.mark.parametrize("D", [32, 128])
def test_boost_mvsnerf_forward_at_32_and_128_planes(D, strict_fp32):
    """The shipped setting (32 planes) and BASELINE config 3 (128 planes) against outputs of the UNMODIFIED reference
    (tests/golden/mvsnerf_chain_d{D}.npz; inputs, weights and selection are those of mvsnerf_chain.npz): the strict
    path at 1e-4; the config-3 engine (bf16 cost volume + the fused fp16-operand tcgen05 render) at 1e-2."""
    gc = load_golden("mvsnerf_chain.npz")
    gd = load_golden(f"mvsnerf_chain_d{D}.npz")
    net, batch = _net_and_batch(gc)
    net.rc = RenderConfig.mvsnerf_eval(2, D)
    out = net({k: (v.clone() if torch.is_tensor(v) else v) for k, v in batch.items()})
    close(out["rgb_level0"], gd.np("out_rgb_level0"), f"D={D} strict rgb")
    close(out["depth_level0"], gd.np("out_depth_level0"), f"D={D} strict depth")
    close(out["weights_level0"][:, ::8], gd.np("out_weights_level0_every8"), f"D={D} strict weights")
    net.volume_dtype = torch.bfloat16
    net.mlp_engine = "umma"
    out2 = net({k: (v.clone() if torch.is_tensor(v) else v) for k, v in batch.items()})
    close(out2["rgb_level0"], gd.np("out_rgb_level0"), f"D={D} config-3 engine rgb", rtol=1e-2)
    close(out2["depth_level0"], gd.np("out_depth_level0"), f"D={D} config-3 engine depth", rtol=1e-2)
