"""The MVSNeRF kernels beyond the 64x96 golden frame: K1b (bmv_cost_volume_var_img, both kernels), K3b
(bmv_mvs_march_fetch) and the fused tcgen05 render (bmv_mvs_render_umma) against the float64 restatement
oracle/mvsnerf_f64.py at other shapes, layouts, ray sub-ranges and tile edges, and the C3 frame (960x544, N=6, K=4,
D=128, S=128, bf16 volume, fused render).

Bars.  u = 2^-24 is the fp32 unit roundoff.  A value sampled at a coordinate is held to
    bar = c_coord * u * (coordinate magnitude scale) * (local slope)  +  c_sum * u * (sum of |terms|)
per element: the first term is the coordinate's fp32 rounding times how fast the sample changes, the second the
rounding of the weighted sum.  The constants are a factor of two above the count of roundings on each path (stated at
each bar).  Samples within that coordinate error of an in-mask or visibility threshold may flip under fp32 rounding:
they are excluded and counted, and must stay below 0.1 % of the samples compared.  Every bar is printed with the
measured maximum (`pytest -s`); each is also shown to catch a perturbed input (a one-pixel / one-voxel shift or a
swapped view)."""
import itertools

import numpy as np
import pytest
import torch

from boostmvsnerfs_b200.config import RenderConfig
from conftest import load_golden
from oracle import enerf_oracle as E
from oracle import mvsnerf_f64 as F64
from oracle import mvsnerf_oracle as M

pytestmark = pytest.mark.gpu
U = 2.0 ** -24
TABLE6 = list(itertools.combinations(range(6), 3))


def report(what, **kw):
    print(f"[measured] {what}: " + ", ".join(f"{k}={v:.3e}" if isinstance(v, float) else f"{k}={v}" for k, v in kw.items()))


def within(got, ref, bar, what, keep=None):
    """|got - ref| <= bar element-wise (where keep); returns the largest err / bar ratio and the largest error."""
    err = (got.double() - ref.double()).abs()
    bad = ~(err <= bar)
    if keep is not None:
        bad &= keep
    ratio = float(torch.where(keep if keep is not None else torch.ones_like(bad), err / bar.clamp_min(1e-300),
                              torch.zeros_like(err)).max())
    assert not bool(bad.any()), f"{what}: {int(bad.sum())}/{bad.numel()} over the bar; worst err/bar {ratio:.3g}"
    return ratio, float(err.max() if keep is None else torch.where(keep, err, torch.zeros_like(err)).max())


def over(got, ref, bar, keep=None):
    bad = ~((got.double() - ref.double()).abs() <= bar)
    if keep is not None:
        bad &= keep
    return int(bad.sum())


@pytest.fixture(scope="module")
def ops():
    from boostmvsnerfs_b200 import ops as _ops
    return _ops


@pytest.fixture(scope="module")
def golden_mlp():
    """The MVSNeRF MLP with the reference weights stored in mvsnerf_ops.npz, and its tcgen05 weight pack."""
    from boostmvsnerfs_b200 import mlp_pack
    from boostmvsnerfs_b200.modules_mvs import MvsNerfMlp
    g = load_golden("mvsnerf_ops.npz")
    mlp = MvsNerfMlp().eval()
    mlp.load_state_dict({k[len("sd_nerf."):]: g.t(k) for k in g.keys() if k.startswith("sd_nerf.")}, strict=True)
    mlp = mlp.cuda()
    return mlp, mlp_pack.pack_mvs_weights_umma(mlp)


def _scene(H, W, n_views=6, seed=3):
    from boostmvsnerfs_b200.synth import batch_to, make_scene
    return batch_to(make_scene(H=H, W=W, n_views=n_views, seed=seed, smooth=True, render_scales=(1.0,),
                               mvs_near_far_cols=True), "cuda")


def _proj(exts, ixts, triple):
    from boostmvsnerfs_b200.network_mvs import BoostMvsnerfNetwork
    return BoostMvsnerfNetwork._proj_triple(exts.cpu()[list(triple)], ixts.cpu()[list(triple)]).cuda()


# ================================================================================== host checks
def test_misaligned_rays_rgb_and_rows_are_refused(ops, golden_mlp):
    """A contiguous tensor at a storage offset of one float passes the wrappers' layout checks; the entries must refuse
    it instead of issuing 16-byte (rays, (N,H,W,4) rgb) or 8-byte (mlp_in rows) loads and stores from it."""
    from boostmvsnerfs_b200._lib import BmvError
    _, packed = golden_mlp
    sc = _scene(64, 96, n_views=4)
    rays = sc["rays_0"][0][:256].contiguous()
    exts, ixts = sc["all_src_exts"][0], sc["all_src_ixts"][0]
    inps = sc["all_src_inps"][0]
    vol = torch.zeros(8, 4, 16 + 48, 24 + 48, device="cuda")

    def off1(t):
        buf = torch.empty(t.numel() + 4, device="cuda")
        v = buf[1:1 + t.numel()].view(t.shape)
        v.copy_(t)
        assert v.is_contiguous() and v.data_ptr() % 16 == 4
        return v
    args = (3, (1, 0, 2), exts, ixts, 64, 96, 1.6, 9.6)
    with pytest.raises(BmvError, match="16-byte"):
        ops.mvs_march_fetch(off1(rays), *args, None, None, want=("z_vals",))
    with pytest.raises(BmvError, match="16-byte"):
        ops.mvs_render(off1(rays), *args, vol, inps, packed)
    rgb4 = inps.new_zeros((4, 64, 96, 4))
    with pytest.raises(BmvError, match="16-byte aligned"):
        ops.mvs_render(rays, *args, vol, off1(rgb4), packed)
    rows = torch.empty(256 * 3 * 86 + 2, device="cuda")[1:1 + 256 * 3 * 86]
    with pytest.raises(BmvError, match="8-byte"):
        ops.mvs_march_fetch(rays, *args, vol, inps, out={"mlp_in": rows})
    for b, n in ((0, 257), (250, 7), (-1, 3)):                  # a ray range outside the rays given
        with pytest.raises(BmvError, match="outside"):
            ops.mvs_march_fetch(rays, *args, vol, inps, ray_begin=b, n_rays=n)
        with pytest.raises(BmvError, match="outside"):
            ops.mvs_render(rays, *args, vol, inps, packed, ray_begin=b, n_rays=n)
    torch.cuda.synchronize()
    # the aligned calls work
    ops.mvs_render(rays, *args, vol, rgb4, packed)
    ops.mvs_march_fetch(rays, *args, vol, inps)
    torch.cuda.synchronize()


# ================================================================================== K1b
def _k1b_bars(r, h, w, V=3):
    """Per-element bars of the 41 channels against the float64 restatement (see the module docstring).
    Coordinate: ~8 roundings of its magnitude scale (dot3 + P3/d + add, two divisions, the g round trip) -> 16 u.
    Bilinear sum: a weight product and four fma -> 8 u of sum |w f|.  Variance: the per-sample errors through
    sum and sum of squares, plus 8 u of (sum f^2 / n + m^2) for the two products, the division and the cancellation.
    Measured on a B200 over every K1b case here: largest err / bar 0.054 (colour) and 0.054 (variance); largest absolute
    error 7.4e-5 (colour) and 4.9e-4 (variance), both at the C3 chain shape.  Excluded voxels: at most 55 of 423936."""
    dc = 16 * U * r["coord"][:, None]                                   # (V-1, 1, D, hp, wp) pixels
    img_bar = torch.nan_to_num(dc * r["img_slope"], nan=float("inf")) + 8 * U * r["img_absmag"] + 1e-30   # (V-1, 3, ...)
    dv = torch.nan_to_num(dc * r["feat_slope"], nan=float("inf")) + 8 * U * r["feat_absmag"]   # (V-1, C, ...)
    n = r["count"]
    fv = r["feat"]
    s1 = r["ref_feat"] + fv.sum(0)
    s2 = r["ref_feat"] ** 2 + (fv * fv).sum(0)
    m = s1 / n
    var_bar = (2 * (fv.abs() * dv).sum(0) + 2 * m.abs() * dv.sum(0)) / n + 8 * U * (s2 / n + m * m) + 1e-30
    # a voxel whose source sample is within the coordinate error of the mask boundary: its count may differ
    gerr = 2 * dc[:, 0] / (min(h, w) - 1)                                # grid units: g = 2 ix / (w - 1) - 1
    edge = (r["margin"] <= 2 * gerr).any(0)                             # (D, hp, wp)
    return img_bar.reshape(3 * (V - 1), *img_bar.shape[2:]), var_bar, edge


def _k1b_inputs(N, C, h, w, D, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    feats = torch.randn(N, C, h, w, device="cuda", generator=g)
    small = torch.rand(N, 3, h, w, device="cuda", generator=g) * 2 - 1
    return feats, small


def _feat_layout(feats, layout):
    if layout == "planar":
        return feats.contiguous()
    if layout == "channels_last":
        return feats.contiguous(memory_format=torch.channels_last)
    # strided: every other channel of a twice-as-wide channels-last tensor, one column cropped off each row end
    N, C, h, w = feats.shape
    wide = torch.zeros(N, 2 * C, h, w + 2, device="cuda").contiguous(memory_format=torch.channels_last)
    view = wide[:, ::2, :, 1:w + 1]
    view.copy_(feats)
    assert view.stride(1) == 2 and view.stride(3) == 2 * C
    return view


def _run_k1b(ops, feats, small, views, proj, planes, pad, out):
    dt = torch.bfloat16 if out == "bf16" else torch.float32
    return ops.cost_volume_var_img(feats, small, views, proj, planes, pad, out_dtype=dt, channels_last=(out != "planar"))


K1B_SHAPES = [(6, 32, 17, 29, 7, 24, (3, 1, 5)), (6, 32, 9, 13, 1, 0, (2, 0, 4)), (4, 16, 20, 28, 5, 3, (1, 2, 3))]


@pytest.mark.parametrize("layout", ["planar", "channels_last", "strided"])
@pytest.mark.parametrize("shape", K1B_SHAPES, ids=lambda s: "N{}C{}h{}w{}D{}p{}".format(*s[:6]))
def test_cost_volume_shapes_vs_float64(ops, shape, layout):
    N, C, h, w, D, pad, views = shape
    sc = _scene(4 * h, 4 * w, n_views=N, seed=N + C + h)
    proj = _proj(sc["all_src_exts"][0], sc["all_src_ixts"][0], views)
    planes = torch.linspace(1.6, 9.6, D, device="cuda") if D > 1 else torch.tensor([4.0], device="cuda")
    feats, small = _k1b_inputs(N, C, h, w, D, seed=D + pad)
    f = _feat_layout(feats, layout)
    r = F64.cost_volume_var_img(feats, small, views, proj, planes, pad)
    img_bar, var_bar, edge = _k1b_bars(r, h, w)
    thread = {o: _run_k1b(ops, feats.contiguous(), small, views, proj, planes, pad, o) for o in ("planar", "channels_last", "bf16")}
    for out in ("planar", "channels_last", "bf16"):
        vol = _run_k1b(ops, f, small, views, proj, planes, pad, out)
        # warp kernel (dense channels-last C = 32, channels-last output) and thread kernel at any strides: same bits
        assert torch.equal(vol, thread[out]), f"{layout}/{out}: differs from the thread-per-voxel kernel on planar maps"
        if out == "bf16":
            assert torch.equal(vol, thread["channels_last"].to(torch.bfloat16)), "bf16 != round-to-nearest of fp32"
            continue
        assert torch.isfinite(vol).all()
        if pad:
            assert float(vol[:3][:, ~r["in_ref"]].abs().max()) == 0.0     # border of the reference rgb is defined as 0
        assert torch.equal(vol[:3].double(), r["vol"][:3]), "reference colour channels"
        ri, ei = within(vol[3:9], r["vol"][3:9], img_bar, "warped colours")
        rv, ev = within(vol[9:], r["vol"][9:], var_bar, "variance", keep=~edge)
    n_edge = int(edge.sum())
    assert n_edge <= 1e-3 * edge.numel()
    report(f"K1b {shape[:6]} {layout}", colour_err=ei, colour_ratio=ri, var_err=ev, var_ratio=rv, excluded=n_edge,
           voxels=edge.numel())
    if layout == "planar":
        # sensitivity: a source feature map shifted by one pixel, or the two source views swapped, must fail the bars
        shifted = feats.clone()
        shifted[views[1]] = torch.roll(feats[views[1]], 1, dims=-1)
        bad = _run_k1b(ops, shifted, small, views, proj, planes, pad, "planar")
        assert over(bad[9:], r["vol"][9:], var_bar, ~edge) > 0, "a one-pixel feature shift passes the variance bar"
        sw = _run_k1b(ops, feats, small, (views[0], views[2], views[1]), proj, planes, pad, "planar")
        assert over(sw[3:9], r["vol"][3:9], img_bar) > 0, "swapped source views pass the colour bar"
        assert over(sw[9:], r["vol"][9:], var_bar, ~edge) > 0, "swapped source views pass the variance bar"


@pytest.mark.parametrize("layout", ["planar", "channels_last"])
def test_cost_volume_behind_the_source_camera(ops, layout):
    """A source camera inside the swept depth range, looking away from the scene: the near planes lie behind it
    (cam z <= 0, no clamp) and most voxels project far off its image.  Output finite and equal to float64: zero taps,
    not counted inside."""
    from boostmvsnerfs_b200.synth import _look_at
    N, C, h, w, D, pad, views = 4, 32, 12, 20, 9, 24, (0, 1, 2)
    sc = _scene(4 * h, 4 * w, n_views=N, seed=7)
    exts = sc["all_src_exts"][0].cpu().clone()
    exts[2] = torch.from_numpy(np.linalg.inv(_look_at(np.array([0.3, 0.1, 5.0]), np.array([0.5, 0.0, 12.0]))).astype(np.float32))
    proj = _proj(exts, sc["all_src_ixts"][0], views)
    planes = torch.linspace(1.6, 9.6, D, device="cuda")
    feats, small = _k1b_inputs(N, C, h, w, D, seed=11)
    r = F64.cost_volume_var_img(feats, small, views, proj, planes, pad)
    behind = r["cz"][1] <= 0
    no_taps = r["img_absmag"][1].amax(0) == 0                          # every tap off the source image
    assert int(behind.sum()) > 0 and int((no_taps & ~behind).sum()) > 0 and int(r["inside"][1].sum()) > 0
    img_bar, var_bar, edge = _k1b_bars(r, h, w)
    vol = _run_k1b(ops, _feat_layout(feats, layout), small, views, proj, planes, pad, layout)
    assert torch.isfinite(vol).all()
    ri, ei = within(vol[3:9], r["vol"][3:9], img_bar, "warped colours")
    rv, ev = within(vol[9:], r["vol"][9:], var_bar, "variance", keep=~edge)
    assert float(vol[6:9][:, no_taps].abs().max()) == 0.0             # zero taps, and not counted (variance above)
    assert int(edge.sum()) <= 1e-3 * edge.numel()
    report(f"K1b behind-camera {layout}", colour_err=ei, colour_ratio=ri, var_err=ev, var_ratio=rv,
           behind=int(behind.sum()), excluded=int(edge.sum()))


def test_cost_volume_c3_chain_shape(ops):
    """The C3 chain: N=6, C=32, 136x240 features, D=128, pad 24 (184x288 padded), bench C3's triple (1, 2, 5).
    Warp kernel (channels-last maps, channels-last bf16 and fp32 output) == thread kernel; float64 on 8 seeded planes."""
    N, C, h, w, D, pad, views = 6, 32, 136, 240, 128, 24, TABLE6[12]
    assert views[0] != 0
    sc = _scene(4 * h, 4 * w, n_views=N, seed=0)
    proj = _proj(sc["all_src_exts"][0], sc["all_src_ixts"][0], views)
    planes = torch.linspace(1.6, 9.6, D, device="cuda")
    feats, small = _k1b_inputs(N, C, h, w, D, seed=12)
    cl = feats.contiguous(memory_format=torch.channels_last)
    warp = _run_k1b(ops, cl, small, views, proj, planes, pad, "channels_last")
    thread = _run_k1b(ops, feats, small, views, proj, planes, pad, "channels_last")
    assert torch.equal(warp, thread)
    del thread
    assert torch.equal(_run_k1b(ops, cl, small, views, proj, planes, pad, "bf16"), warp.to(torch.bfloat16))
    idx = sorted({0, D - 1} | set(np.random.RandomState(5).choice(np.arange(1, D - 1), 6, replace=False).tolist()))
    r = F64.cost_volume_var_img(feats, small, views, proj, planes, pad, plane_idx=idx)
    img_bar, var_bar, edge = _k1b_bars(r, h, w)
    sub = warp[:, idx]
    assert torch.equal(sub[:3].double(), r["vol"][:3])
    ri, ei = within(sub[3:9], r["vol"][3:9], img_bar, "warped colours")
    rv, ev = within(sub[9:], r["vol"][9:], var_bar, "variance", keep=~edge)
    assert int(edge.sum()) <= 1e-3 * edge.numel()
    report("K1b C3 chain (8 planes)", colour_err=ei, colour_ratio=ri, var_err=ev, var_ratio=rv, excluded=int(edge.sum()),
           voxels=edge.numel())


# ================================================================================== K3b
KH, KW, KTRIPLE = 68, 100, (2, 0, 5)


@pytest.fixture(scope="module")
def k3b_scene():
    sc = _scene(KH, KW, n_views=6, seed=4)
    g = torch.Generator(device="cuda").manual_seed(9)
    vol = torch.randn(8, 16, KH // 4 + 48, KW // 4 + 48, device="cuda", generator=g)
    return sc, vol


def _k3b_args(sc, vol, S, channels_last=False, rgb=None):
    if channels_last:
        vol = vol.permute(1, 2, 3, 0).contiguous().permute(3, 0, 1, 2)
    # the volume spans depths 2.0 .. 8.0 while the rays march 1.6 .. 9.6: samples in front of and behind it
    return (sc["rays_0"][0], S, KTRIPLE, sc["all_src_exts"][0], sc["all_src_ixts"][0], KH, KW, 2.0, 8.0, vol,
            sc["all_src_inps"][0] if rgb is None else rgb)


@pytest.mark.parametrize("channels_last", [False, True], ids=["planar", "channels_last"])
@pytest.mark.parametrize("S", [1, 3, 8, 128])
def test_march_fetch_vs_float64(ops, k3b_scene, S, channels_last):
    sc, vol = k3b_scene
    args = _k3b_args(sc, vol, S, channels_last)
    rays = args[0]
    R = rays.shape[0]
    o = ops.mvs_march_fetch(*args, want=("mlp_in", "z_vals", "vis_mask", "vis_count"))
    # z and visibility: bit-exact against the float32 torch chain of the reference
    xyz, z = M.ray_marcher(rays[None], S)
    assert torch.equal(o["z_vals"], z[0])
    tr = list(KTRIPLE)
    vis = E.mask_viewport(xyz, sc["all_src_exts"][:, tr], sc["all_src_ixts"][:, tr],
                          torch.tensor([KW - 1.0, KH - 1.0], device="cuda")).reshape(R, S)
    assert torch.equal(o["vis_mask"], vis)
    assert torch.equal(o["vis_count"].float(), torch.round(vis * 3))
    # float64 on all rays (S <= 8) or a seeded 1024-ray subset (S = 128)
    sel = torch.arange(R, device="cuda") if S <= 8 else torch.from_numpy(np.sort(np.random.RandomState(S).choice(R, 1024, replace=False))).cuda()
    row = o["mlp_in"][sel].double()
    zz = o["z_vals"][sel]
    f = F64.march_fetch_row(rays[sel], zz, KTRIPLE, args[3], args[4], KH, KW, 2.0, 8.0, vol, args[10])
    own = F64.march_fetch_row(rays[sel], zz, KTRIPLE, args[3], args[4], KH, KW, 2.0, 8.0, vol, args[10], ndc=row[..., :3])
    # NDC: ~10 roundings of the projection's magnitude scale -> 32 u; view direction: unit vector, ~6 roundings -> 16 u.
    # Measured on a B200 (all S, both layouts): NDC err / bar 0.049, max 2.5e-7; view direction max 1.3e-7.
    rn, en = within(row[..., :3], f["ndc"], 32 * U * f["ndc_scale"], "ndc")
    rd, ed = within(row[..., 83:], f["dir"], torch.full_like(f["dir"], 16 * U), "view direction")
    # positional encoding at the kernel's own ndc (2^k x is exact): only sincosf's accuracy, a few ulps of 1.
    # Measured on a B200: max 8.7e-8.
    ep = float((row[..., 3:63] - own["pe"]).abs().max())
    assert ep <= 1e-6, f"positional encoding: max err {ep:.3e} (a fast-math sin / cos fails this)"
    # volume feature at the kernel's own ndc: index rounding ~4 u of (size - 1) per axis -> 8 u * size, 8 fma -> 16 u.
    # Measured on a B200: err / bar 0.038, max 1.1e-5.
    Dv, hv, wv = vol.shape[1:]
    vbar = 8 * U * max(Dv, hv, wv) * own["vox_slope"] + 16 * U * own["vox_absmag"] + 1e-30
    rvx, evx = within(row[..., 63:71], own["vox"], vbar, "volume feature")
    # colours at float64 projections of the kernel's z: pixel coordinate error 16 u of the projection's scale.
    # Measured on a B200: err / bar 0.10, max 6.9e-7; in-mask samples excluded at the margin: at most 9 of 393216.
    cbar = 16 * U * f["uv_scale"][..., None] * max(KW, KH) * f["rgb_slope"] + 8 * U + 1e-30
    cols = row[..., 71:83].reshape(*row.shape[:2], 3, 4)
    edge = f["in_margin"] <= 32 * U * f["uv_scale"]
    rc, ec = within(cols[..., :3], f["rgb"], cbar, "colours")
    assert bool(((cols[..., 3] > 0) == f["inside"])[~edge].all()), "in-mask bits"
    n_edge = int(edge.sum())
    assert n_edge <= 1e-3 * edge.numel()
    # volume coverage: samples outside the volume, and inside within half a voxel of a face and of the last plane
    ix = torch.stack([f["ndc"][..., 0] * (wv - 1), f["ndc"][..., 1] * (hv - 1), f["ndc"][..., 2] * (Dv - 1)], -1)
    size = torch.tensor([wv - 1, hv - 1, Dv - 1], device="cuda", dtype=torch.float64)
    inside_vol = ((ix >= 0) & (ix <= size)).all(-1)
    near_face = inside_vol & ((ix < 0.5) | (ix > size - 0.5)).any(-1)
    near_last = inside_vol & (ix[..., 2] > Dv - 1.5)
    assert int((~inside_vol).sum()) > 0
    if S == 128:                                      # the sparser marches do not reach the depth faces
        assert int(near_face.sum()) > 0 and int(near_last.sum()) > 0
    if S == 8 and not channels_last:
        # the bars catch a wrong fetch: a one-voxel shift of the volume, or the colours of a swapped view
        bad = ops.mvs_march_fetch(*_k3b_args(sc, torch.roll(vol, 1, dims=-1), S), want=("mlp_in",))["mlp_in"][sel]
        assert over(bad[..., 63:71], own["vox"], vbar) > 0
        rgb_sw = args[10][[0, 1, 5, 3, 4, 2]]
        bad = ops.mvs_march_fetch(*_k3b_args(sc, vol, S, rgb=rgb_sw), want=("mlp_in",))["mlp_in"][sel]
        assert over(bad[..., 71:83].reshape(*row.shape[:2], 3, 4)[..., :3], f["rgb"], cbar) > 0
    report(f"K3b S={S} {'cl' if channels_last else 'planar'}", ndc_ratio=rn, ndc_err=en, dir_err=ed, pe_err=ep,
           vox_err=evx, vox_ratio=rvx, rgb_err=ec, rgb_ratio=rc, excluded=n_edge, samples=edge.numel(),
           outside=int((~inside_vol).sum()), near_face=int(near_face.sum()))


@pytest.mark.parametrize("S", [1, 3, 8, 128])
def test_march_fetch_sub_ranges_and_out_slices(ops, k3b_scene, S):
    sc, vol = k3b_scene
    args = _k3b_args(sc, vol, S, channels_last=True)
    R = args[0].shape[0]
    full = ops.mvs_march_fetch(*args, want=("mlp_in", "z_vals", "vis_mask", "vis_count"))
    nan = float("nan")
    G = 3                                               # guard rows on each side of the written slice
    for b, n in ((0, R), (1, R - 1), (R - 1, 1)):
        buf = {"mlp_in": torch.full((R + 2 * G, S, 86), nan, device="cuda"), "z_vals": torch.full((R + 2 * G, S), nan, device="cuda"),
               "vis_mask": torch.full((R + 2 * G, S), nan, device="cuda")}
        cnt = torch.full((R + 2 * G, S), -7, device="cuda", dtype=torch.int32)
        o = ops.mvs_march_fetch(*args, ray_begin=b, n_rays=n,
                                out={**{k: v[G:G + n] for k, v in buf.items()}, "vis_count": cnt[G:G + n]})
        for k, v in buf.items():
            assert torch.equal(v[G:G + n], full[k][b:b + n]), f"S={S} ({b},{n}) {k}"
            assert bool(v[:G].isnan().all() and v[G + n:].isnan().all()), f"S={S} ({b},{n}) {k}: written outside its slice"
            assert o[k].data_ptr() == v[G:G + n].data_ptr()
        assert torch.equal(cnt[G:G + n], full["vis_count"][b:b + n]) and bool((cnt[:G] == -7).all() and (cnt[G + n:] == -7).all())
    # the network's chunk loop (network_mvs.py) with a 37-ray chunk, z / vis into slices of (R, S) buffers
    z = torch.full((R, S), nan, device="cuda")
    mask = torch.full((R, S), nan, device="cuda")
    rows = torch.full((R, S, 86), nan, device="cuda")
    for r0 in range(0, R, 37):
        n = min(37, R - r0)
        o = ops.mvs_march_fetch(*args, ray_begin=r0, n_rays=n, want=("mlp_in",), out={"z_vals": z[r0:r0 + n], "vis_mask": mask[r0:r0 + n]})
        rows[r0:r0 + n] = o["mlp_in"]
    assert torch.equal(z, full["z_vals"]) and torch.equal(mask, full["vis_mask"]) and torch.equal(rows, full["mlp_in"])
    # without mlp_in the kernel returns before the fetch: z and visibility unchanged
    lean = ops.mvs_march_fetch(*args, want=("z_vals", "vis_mask", "vis_count"))
    assert "mlp_in" not in lean
    for k in ("z_vals", "vis_mask", "vis_count"):
        assert torch.equal(lean[k], full[k]), k


# ================================================================================== fused render
def _nhwc4(rgb, fill=float("nan")):
    N, _, H, W = rgb.shape
    out = torch.full((N, H, W, 4), fill, device="cuda")
    out[..., :3] = rgb.permute(0, 2, 3, 1)
    return out


@pytest.mark.parametrize("size", [(64, 96), (68, 100)], ids=["64x96", "68x100"])
def test_fused_render_nhwc4_equals_planar(ops, golden_mlp, size):
    """The (N,H,W,4) colour layout the network passes (16-byte taps) gives the planar image's raw, z and visibility bit
    for bit; the 4th channel is NaN, so any read of it would show."""
    _, packed = golden_mlp
    H, W = size
    sc = _scene(H, W, n_views=6, seed=H)
    g = torch.Generator(device="cuda").manual_seed(H)
    vol = torch.randn(H // 4 + 48, W // 4 + 48, 8, 12, device="cuda", generator=g).permute(2, 3, 0, 1).contiguous()
    for S in (3, 32):
        args = (sc["rays_0"][0], S, (4, 1, 3), sc["all_src_exts"][0], sc["all_src_ixts"][0], H, W, 1.6, 9.6, vol)
        a = ops.mvs_render(*args, sc["all_src_inps"][0], packed, want_count=True)
        b = ops.mvs_render(*args, _nhwc4(sc["all_src_inps"][0]), packed, want_count=True)
        for k in ("raw", "z_vals", "vis_mask", "vis_count"):
            assert torch.equal(a[k], b[k]), f"S={S}: {k}"
        assert torch.isfinite(b["raw"]).all()


def _rel_errors(raw, ref):
    """max and mean relative error of alpha (channel 3) and of rgb (channels 0..2) separately."""
    out = {}
    for name, sl in (("alpha", slice(3, 4)), ("rgb", slice(0, 3))):
        e = (raw[..., sl].double() - ref[..., sl]).abs()
        out[name + "_max"] = float(e.max()) / float(ref[..., sl].abs().max())
        out[name + "_mean"] = float(e.mean()) / float(ref[..., sl].abs().mean())
    return out


# fp16 operands (2^-11 relative rounding on every operand of 8 layers) and fp32 accumulation, against float64.
# Measured on a B200 with the reference weights: alpha max 9.9e-4 / mean 1.14e-3, rgb max 3.0e-4 / mean 6.9e-5.  Each bar
# keeps a margin of 1.4x to 3.6x over its measurement and is tighter than the earlier bars against the fp32 module
# (max 1e-2 of max|raw|, mean 2e-3 of mean|raw|): alpha mean is the closest, 1.6e-3 against 2e-3, and its error is
# relative to mean |alpha|, which the ReLU keeps small.  The inputs are seeded and the kernel deterministic.
FUSED_BARS = {"alpha_max": 3e-3, "alpha_mean": 1.6e-3, "rgb_max": 1e-3, "rgb_mean": 2.5e-4}


def test_fused_render_vs_float64(ops, k3b_scene, golden_mlp):
    """mvs_render with the reference MLP weights against the float64 K3b row followed by the float64 MLP; a one-voxel
    volume shift and a swapped colour view must both fail the bars."""
    mlp, packed = golden_mlp
    sc, vol = k3b_scene
    S = 32
    vol_cl = vol.permute(1, 2, 3, 0).contiguous().permute(3, 0, 1, 2)
    rgb4 = _nhwc4(sc["all_src_inps"][0], 0.0)
    base = _k3b_args(sc, vol_cl, S, rgb=rgb4)
    rays = base[0]
    sel = torch.from_numpy(np.sort(np.random.RandomState(1).choice(rays.shape[0], 2048, replace=False))).cuda()
    got = ops.mvs_render(*base, packed)
    f = F64.march_fetch_row(rays[sel], got["z_vals"][sel], KTRIPLE, base[3], base[4], KH, KW, 2.0, 8.0, vol, sc["all_src_inps"][0])
    ref = F64.mlp(mlp, f["row"])
    errs = _rel_errors(got["raw"][sel], ref)
    report("fused render vs float64", **errs)
    shifted = ops.mvs_render(*_k3b_args(sc, torch.roll(vol_cl, 1, dims=-1), S, rgb=rgb4), packed)
    e_shift = _rel_errors(shifted["raw"][sel], ref)
    swapped = ops.mvs_render(*_k3b_args(sc, vol_cl, S, rgb=rgb4[[0, 1, 5, 3, 4, 2]]), packed)
    e_swap = _rel_errors(swapped["raw"][sel], ref)
    report("fused render, one-voxel volume shift", **e_shift)
    report("fused render, swapped colour view", **e_swap)
    for k, bar in FUSED_BARS.items():
        assert errs[k] <= bar, f"{k} = {errs[k]:.3e} > {bar:.1e}"
    assert any(e_shift[k] > FUSED_BARS[k] for k in FUSED_BARS), "a one-voxel volume shift passes the bars"
    assert any(e_swap[k] > FUSED_BARS[k] for k in FUSED_BARS), "a swapped colour view passes the bars"


@pytest.mark.parametrize("S,n", [(1, 1), (1, 127), (1, 128), (1, 129), (1, 255), (1, 256), (1, 257), (3, 43), (3, 85), (3, 86)])
def test_fused_render_tile_edges(ops, k3b_scene, golden_mlp, S, n):
    """n_rays * S samples around the 128-row tile and the two-tile pair: a partial tile, and pairs whose second tile is
    dead.  Written into NaN-guarded slices; equal to the slice of the full launch bit for bit."""
    _, packed = golden_mlp
    sc, vol = k3b_scene
    args = _k3b_args(sc, vol, S, channels_last=True, rgb=_nhwc4(sc["all_src_inps"][0]))
    full = ops.mvs_render(*args, packed)
    b, G = 5, 2
    nan = float("nan")
    raw = torch.full((n + 2 * G, S, 4), nan, device="cuda")
    z = torch.full((n + 2 * G, S), nan, device="cuda")
    m = torch.full((n + 2 * G, S), nan, device="cuda")
    ops.mvs_render(*args, packed, ray_begin=b, n_rays=n, out={"raw": raw[G:G + n], "z_vals": z[G:G + n], "vis_mask": m[G:G + n]})
    for name, t, k in (("raw", raw, "raw"), ("z", z, "z_vals"), ("vis", m, "vis_mask")):
        assert torch.equal(t[G:G + n], full[k][b:b + n]), name
        assert bool(t[:G].isnan().all() and t[G + n:].isnan().all()), f"{name}: written outside its slice"


def test_fused_render_frame_size_launch(ops, golden_mlp):
    """S = 128 on a C3-sized channels-last volume (8 x 128 x 184 x 288) over all 522240 C3 rays: one launch with ~1760
    tile pairs per CTA equals launches of at most 148 pairs (one pass per CTA) over seeded ray ranges, bit for bit."""
    _, packed = golden_mlp
    H, W, S = 544, 960, 128
    sc = _scene(H, W, n_views=6, seed=0)
    g = torch.Generator(device="cuda").manual_seed(3)
    vol = torch.randn(128, 184, 288, 8, device="cuda", generator=g).permute(3, 0, 1, 2)
    args = (sc["rays_0"][0], S, TABLE6[19], sc["all_src_exts"][0], sc["all_src_ixts"][0], H, W, 1.6, 9.6, vol,
            _nhwc4(sc["all_src_inps"][0], 0.0))
    R = args[0].shape[0]
    assert R == 522240
    full = ops.mvs_render(*args, packed)
    assert torch.isfinite(full["raw"]).all()
    per = 148 * 256 // S                                 # rays of 148 tile pairs
    starts = np.random.RandomState(7).choice(R - per, 6, replace=False).tolist() + [0, R - per]
    for b in starts:
        part = ops.mvs_render(*args, packed, ray_begin=b, n_rays=per)
        for k in ("raw", "z_vals", "vis_mask"):
            assert torch.equal(part[k], full[k][b:b + per]), f"rays [{b}, {b + per}): {k}"


# ================================================================================== the C3 frame
@pytest.fixture(scope="module")
def c3():
    from boostmvsnerfs_b200.network_mvs import BoostMvsnerfNetwork
    from boostmvsnerfs_b200.synth import batch_to, make_scene
    torch.manual_seed(0)
    net = BoostMvsnerfNetwork(preprocess=True, rc=RenderConfig.mvsnerf_eval(4, 128)).eval().cuda()
    net.view_selection_outputs = {"synth_0": [0, 7, 12, 19]}
    net.volume_dtype = torch.bfloat16
    net.mlp_engine = "umma"
    batch = batch_to(make_scene(H=544, W=960, n_views=6, seed=0, render_scales=(1.0,), mvs_near_far_cols=True), "cuda")
    return net, batch


@pytest.fixture()
def deterministic_cudnn():
    """Pins cuDNN to deterministic algorithms, chosen without benchmarking, so two forwards give the same bits
    (verified on a B200 with cuDNN 9.22)."""
    old = (torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
    yield
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = old


def test_c3_frame_properties_and_engines(c3, deterministic_cudnn):
    net, batch = c3
    R = 544 * 960
    out = net(dict(batch))
    rgb, depth, w = out["rgb_level0"], out["depth_level0"], out["weights_level0"]
    assert rgb.shape == (1, R, 3) and depth.shape == (1, R) and w.shape == (1, R, 128)
    for k, v in out.items():
        assert torch.isfinite(v).all(), k
    assert 0.0 <= float(rgb.min()) and float(rgb.max()) <= 1.0
    assert 1.6 - 1e-5 <= float(depth.min()) and float(depth.max()) <= 9.6 + 1e-5       # chains' z range: 2 * 0.8 .. 8 * 1.2
    assert float(w.min()) >= 0.0 and float(w.sum(-1).max()) <= 1.0 + 1e-6
    again = net(dict(batch))
    for k in out:                                       # cuDNN pinned deterministic (fixture); no atomics in libbmv
        assert torch.equal(out[k], again[k]), k
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        net.mlp_engine, net.volume_dtype = "cublas", torch.float32
        strict = net(dict(batch))
        scale = float(strict["rgb_level0"].abs().max())
        err = float((strict["rgb_level0"] - rgb).abs().max())
        report("C3 frame, config-3 engine vs strict fp32 cuBLAS engine", rgb_err=err / scale)
        assert err <= 1e-2 * scale
        # the cuBLAS engine's chunk loop: default 1 GiB chunks against a ragged 10007-ray chunk
        triples = [TABLE6[j] for j in net.view_selection_outputs["synth_0"]]
        with torch.no_grad():
            raw_a, mask_a, z_a, _, _ = net._render_chains(batch, triples)
            net.mlp_chunk_bytes = 10007 * 128 * 86 * 4
            raw_b, mask_b, z_b, _, _ = net._render_chains(batch, triples)
        assert torch.equal(z_a, z_b) and torch.equal(mask_a, mask_b)
        e = float((raw_a - raw_b).abs().max()) / float(raw_a.abs().max())
        report("C3 cuBLAS engine, 10007-ray chunks vs default", raw_rel=e)
        assert e <= 1e-6
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
        net.mlp_engine, net.volume_dtype, net.mlp_chunk_bytes = "umma", torch.bfloat16, 1 << 30


def test_c3_view_selection_matches_oracle(c3):
    net, batch = c3
    sel = net.forward_view_selection(batch)
    masks = [M.visibility_mask_2d(batch["rays_0"], batch["all_src_exts"][:, list(t)], batch["all_src_ixts"][:, list(t)],
                                  544, 960) for t in TABLE6]
    picks = M.search_k_best_views(masks, net.rc.k_best)
    # the masks forward_view_selection picks from, against the oracle's, triple by triple
    product = net.view_selection_masks(batch)
    assert product.shape == (len(TABLE6), 1, 544 * 960)
    worst = 0.0
    for t, got, ref in zip(TABLE6, product, masks):
        err = (got - ref).abs()
        worst = max(worst, float(err.max()))
        assert bool((err <= 1e-5 * (float(ref.abs().max()) + ref.abs())).all()), f"triple {t}: coverage mask differs by {float(err.max()):.3e}"
    report("C3 view selection masks", max_err=worst)
    assert sel == {"synth_0": picks}
