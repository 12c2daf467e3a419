"""bmv_render_rays_multi (all K chains in one persistent launch, lean gather) against the per-chain tensor-core kernel and
the reference op sequence: z and visibility bit-exact, raw within the MLP tolerance; ragged ranges, device-resident view
ids, both ray sources, depth_inv, K = 1..8."""
import numpy as np
import pytest
import torch

from boostmvsnerfs_b200.config import RenderConfig
from oracle import enerf_oracle as O

pytestmark = pytest.mark.gpu


def _setup(H, W, N, K, seed, smooth, depth_inv=False):
    from boostmvsnerfs_b200 import mlp_pack, ops
    from boostmvsnerfs_b200.modules import NeRF
    from boostmvsnerfs_b200.synth import batch_to, make_scene
    g = torch.Generator(device="cuda").manual_seed(seed)
    scene = batch_to(make_scene(H=H, W=W, n_views=N, seed=seed, smooth=smooth), "cuda")
    hv, wv, D = H // 2, W // 2, 8
    lo, hi = (1 / 8.0, 1 / 2.0) if depth_inv else (2.0, 8.0)
    depth = lo + (hi - lo) * torch.rand(K, hv, wv, device="cuda", generator=g)
    std = 0.05 * (hi - lo) * torch.rand(K, hv, wv, device="cuda", generator=g)
    nf = torch.stack([torch.full((K, hv, wv), hi if depth_inv else lo, device="cuda"),
                      torch.full((K, hv, wv), lo if depth_inv else hi, device="cuda")], dim=1).contiguous()
    vols = torch.randn(K, D, hv, wv, 8, device="cuda", generator=g).permute(0, 4, 1, 2, 3)
    feat = torch.randn(N, H, W, 8, device="cuda", generator=g).permute(0, 3, 1, 2)
    rgb4 = torch.zeros(N, H, W, 4, device="cuda")
    rgb4[..., :3] = scene["all_src_inps"][0].permute(0, 2, 3, 1)
    rgb = rgb4.permute(0, 3, 1, 2)[:, :3]
    cams = ops.CameraBlock(scene["all_src_exts"][0], scene["all_src_ixts"][0], scene["tar_ext"][0])
    torch.manual_seed(seed)
    nerf = NeRF(feat_ch=11, viewdir_agg=True).cuda().eval()
    packed = mlp_pack.pack_nerf_weights_mma(nerf)
    table = [(0, 1, 2), (0, 2, 3), (1, 2, 3), (0, 1, 3), (3, 1, 0), (2, 3, 1), (1, 0, 2), (3, 2, 0)]
    triples = [tuple(v % N for v in table[k % len(table)]) for k in range(K)]
    return scene, depth, std, nf, vols, feat, rgb, cams, nerf, packed, triples


def _with_samples(cases):
    """Every case at S = 1, 2, 3, 8 samples per ray.  S = 2 (the ENeRF configs, the kernels' `si >> 1` branch) keeps the
    case's plain id; the others run the general `si / S` branch, and S = 3 makes rays straddle the 32-sample rounds
    (mma) and the 128-sample tiles (tcgen05)."""
    return [pytest.param(*c, S, id="-".join(map(str, c)) + ("" if S == 2 else f"-S{S}")) for c in cases for S in (1, 2, 3, 8)]


@pytest.mark.parametrize("H,W,K,smooth,depth_inv,S", _with_samples([(64, 96, 4, True, False), (64, 96, 1, False, False),
                                                                    (96, 160, 8, False, False), (64, 96, 3, True, True)]))
def test_multi_matches_per_chain_kernel(H, W, K, smooth, depth_inv, S):
    from boostmvsnerfs_b200 import ops
    N = 4
    scene, depth, std, nf, vols, feat, rgb, cams, nerf, packed, triples = _setup(H, W, N, K, 11 + K, smooth, depth_inv)
    rays = scene["rays_1"][0]
    multi = ops.render_rays_multi(depth, std, nf, rays, H, W, depth_inv, S, vols, feat, rgb, cams, triples, packed, want_count=True)
    for k in range(K):
        one = ops.render_rays(depth[k], std[k], nf[k], rays, H, W, depth_inv, S, vols[k], feat, rgb, cams, triples[k], packed,
                              engine="mma", want_count=True)
        assert torch.equal(multi["z_vals"][k], one["z_vals"]), f"chain {k}: z"
        assert torch.equal(multi["vis_count"][k], one["vis_count"]), f"chain {k}: visibility count"
        assert torch.equal(multi["vis_mask"][k], one["vis_mask"]), f"chain {k}: visibility score"
        err = float((multi["raw"][k] - one["raw"]).abs().max()) / float(one["raw"].abs().max())
        assert err <= (3e-5 if smooth else 2e-4), f"chain {k}: raw differs by {err:.2e}"


def test_multi_device_views_ragged_range_and_generated_rays():
    from boostmvsnerfs_b200 import ops
    H, W, N, K, S = 64, 96, 4, 4, 2
    scene, depth, std, nf, vols, feat, rgb, cams, nerf, packed, triples = _setup(H, W, N, K, 5, True)
    rays = scene["rays_1"][0]
    full = ops.render_rays_multi(depth, std, nf, rays, H, W, False, S, vols, feat, rgb, cams, triples, packed)
    vdev = torch.tensor(triples, device="cuda", dtype=torch.int32)
    got = ops.render_rays_multi(depth, std, nf, rays, H, W, False, S, vols, feat, rgb, cams, None, packed, views_dev=vdev)
    for k_ in ("raw", "z_vals", "vis_mask"):
        assert torch.equal(got[k_], full[k_]), k_
    # the same launch follows a changed selection through the device buffer only
    vdev.copy_(torch.tensor(triples[::-1], device="cuda", dtype=torch.int32))
    rev = ops.render_rays_multi(depth.flip(0).contiguous(), std.flip(0).contiguous(), nf.flip(0).contiguous(), rays, H, W, False, S,
                                vols.flip(0).contiguous(memory_format=torch.channels_last_3d), feat, rgb, cams, None, packed, views_dev=vdev)
    assert torch.equal(rev["raw"].flip(0), full["raw"])
    # ragged ray range (not a multiple of 32 samples), shared near_far, generated rays
    b, n = 37, 1001
    part = ops.render_rays_multi(depth, std, nf[0], rays, H, W, False, S, vols, feat, rgb, cams, triples, packed, ray_begin=b, n_rays=n)
    assert torch.equal(part["raw"], full["raw"][:, b:b + n]) and torch.equal(part["vis_mask"], full["vis_mask"][:, b:b + n])
    gen = ops.RayGenerator.from_cameras(scene["tar_ext"][0].cpu(), scene["tar_ixt"][0].cpu(), H, W, 1.0, "cuda")
    g = ops.render_rays_multi(depth, std, nf, gen, H, W, False, S, vols, feat, rgb, cams, triples, packed)
    assert torch.equal(g["z_vals"], full["z_vals"]) and torch.equal(g["vis_mask"], full["vis_mask"])
    assert float((g["raw"] - full["raw"]).abs().max()) <= 1e-6


def test_multi_visibility_bit_exact_on_frustum_edges():
    """The approximate filter in front of the IEEE inside test must never change a decision: cameras arranged so that
    thousands of samples project within a few ulps of the image borders of the source views."""
    from boostmvsnerfs_b200 import ops
    H, W, N, K, S = 64, 96, 4, 2, 2
    scene, depth, std, nf, vols, feat, rgb, cams, nerf, packed, triples = _setup(H, W, N, K, 3, True)
    # source views = the target camera shifted by exact pixel multiples: target pixels land ON source borders
    tar_ext, tar_ixt = scene["tar_ext"][0], scene["tar_ixt"][0]
    exts = tar_ext[None].repeat(N, 1, 1).clone()
    ixts = tar_ixt[None].repeat(N, 1, 1).clone()
    for v in range(N):
        ixts[v, 0, 2] += 7.0 * (v - 1)          # principal point shifts: u_src = u_tar + 7 (v - 1) exactly at any depth
        ixts[v, 1, 2] -= 5.0 * (v - 2)
    cams2 = ops.CameraBlock(exts, ixts, tar_ext)
    rays = scene["rays_1"][0]
    multi = ops.render_rays_multi(depth, std, nf, rays, H, W, False, S, vols, feat, rgb, cams2, triples, packed, want_count=True)
    inv_scale = torch.tensor([[W - 1, H - 1]], dtype=torch.float32, device="cuda")
    o, d = rays[:, :3], rays[:, 3:6]
    for k in range(K):
        # sample positions from the kernel's own z with the reference's two separately rounded ops (o + d * z):
        # visibility is bit-exact for identical xyz (SURVEY.md 10.13); the upsampled depth may differ by 1 ulp from ATen's
        z = multi["z_vals"][k]                                              # (R,S)
        xyz = (o[:, None, :] + d[:, None, :] * z[..., None])[None]          # (1,R,S,3)
        tr = list(triples[k])
        cnt = O.visibility_count(xyz, exts[tr][None], ixts[tr][None], inv_scale).reshape(-1, S)
        assert torch.equal(multi["vis_count"][k], cnt), f"chain {k}: {(multi['vis_count'][k] != cnt).sum().item()} visibility counts differ"
        # the scene really exercises the edges: counts are neither all-in nor all-out
        assert 0 < int((cnt < 3).sum()) < cnt.numel()


def test_network_uses_the_multi_launch_and_matches_per_chain(monkeypatch):
    from boostmvsnerfs_b200 import _lib, network
    from boostmvsnerfs_b200.synth import batch_to, make_scene
    torch.manual_seed(1)
    net = network.BoostEnerfNetwork(preprocess=True, rc=RenderConfig.enerf_eval(4)).eval().cuda()
    net.view_selection_outputs = {"synth_0": [0, 7, 12, 19]}
    batch = batch_to(make_scene(H=128, W=192, n_views=6, seed=2, smooth=True), "cuda")
    calls = []
    orig = _lib.call
    monkeypatch.setattr(_lib, "call", lambda name, p, s: (calls.append(name), orig(name, p, s))[1])
    a = net(dict(batch))
    assert calls.count("bmv_render_rays_multi_umma") == 1 and "bmv_render_rays_umma" not in calls
    net.mlp_engine = "mma"
    calls.clear()
    a2 = net(dict(batch))
    assert calls.count("bmv_render_rays_multi") == 1 and "bmv_render_rays_mma" not in calls
    net.multi_chain_render = False
    calls.clear()
    b = net(dict(batch))
    assert calls.count("bmv_render_rays_mma") == 4
    for k in a:
        err = float((a2[k] - b[k]).abs().max()) / float(b[k].abs().max())
        assert err <= 2e-5, (k, err)
    for k in a:
        err = float((a[k] - b[k]).abs().max()) / float(b[k].abs().max())
        assert err <= 2e-5, (k, err)


# ------------------------------------------------------------------------------------------ tcgen05 engine
@pytest.mark.parametrize("H,W,K,smooth,depth_inv,S", _with_samples([(64, 96, 4, True, False), (64, 96, 1, False, False),
                                                                    (96, 160, 8, False, False), (64, 96, 3, True, True),
                                                                    (32, 40, 2, True, False)]))
def test_umma_engine_matches_the_mma_engine(H, W, K, smooth, depth_inv, S):
    """bmv_render_rays_multi_umma (MLP as tcgen05.mma, accumulators in tensor memory, two threads per sample row) against
    bmv_render_rays_multi: the gather is the same code (z / visibility bit-identical), the MLP the same hi / lo split
    products in another summation order.  Both engines against a ragged sub-range of their own launch, and at S = 3
    against the stand-alone fetch followed by the NeRF module in float64."""
    import copy
    from boostmvsnerfs_b200 import mlp_pack, ops
    N = 4
    scene, depth, std, nf, vols, feat, rgb, cams, nerf, packed, triples = _setup(H, W, N, K, 11 + K, smooth, depth_inv)
    packed_u = mlp_pack.pack_nerf_weights_umma(nerf)
    rays = scene["rays_1"][0]
    ref = ops.render_rays_multi(depth, std, nf, rays, H, W, depth_inv, S, vols, feat, rgb, cams, triples, packed, want_count=True)
    got = ops.render_rays_multi(depth, std, nf, rays, H, W, depth_inv, S, vols, feat, rgb, cams, triples, packed_u, want_count=True)
    for k_ in ("z_vals", "vis_count", "vis_mask"):
        assert torch.equal(got[k_], ref[k_]), k_
    for k in range(K):
        err = float((got["raw"][k] - ref["raw"][k]).abs().max()) / float(ref["raw"][k].abs().max())
        assert err <= (3e-5 if smooth else 2e-4), f"chain {k}: raw differs by {err:.2e}"
    # and against the fp32 FMA kernel (no tensor cores at all)
    packed_f = mlp_pack.pack_nerf_weights(nerf)
    one = ops.render_rays(depth[0], std[0], nf[0], rays, H, W, depth_inv, S, vols[0], feat, rgb, cams, triples[0], packed_f, engine="fma")
    err = float((got["raw"][0] - one["raw"]).abs().max()) / float(one["raw"].abs().max())
    assert err <= (3e-5 if smooth else 2e-4), f"vs fp32 FMA kernel: {err:.2e}"
    # ragged ray range: an odd first ray, and 1001 rays whose samples straddle rounds / tiles unless S divides 32
    b, n = 37, 1001
    for engine, full in (("mma", ref), ("umma", got)):
        part = ops.render_rays_multi(depth, std, nf, rays, H, W, depth_inv, S, vols, feat, rgb, cams, triples,
                                     packed if engine == "mma" else packed_u, ray_begin=b, n_rays=n, want_count=True)
        for k_ in ("raw", "z_vals", "vis_mask", "vis_count"):
            assert torch.equal(part[k_], full[k_][:, b:b + n]), f"{engine}: {k_} of rays [{b}, {b + n})"
    if S != 3 or not smooth:
        return
    # independent reference for chain 0: the stand-alone K3 fetch (pinned to the golden vectors) + the NeRF module in float64
    fetch = ops.raygen_sample_fetch(depth[0], std[0], nf[0], rays, H, W, depth_inv, S, vols[0], feat, rgb, cams, triples[0],
                                    want=("z_vals", "vox_feat", "img_feat", "vis_mask"))
    with torch.no_grad():
        raw64 = copy.deepcopy(nerf).double()(fetch["vox_feat"].double()[None], fetch["img_feat"].double()[None])[0].view(-1, S, 4)
    scale = float(raw64.abs().max())
    for engine, res in (("mma", ref), ("umma", got)):
        assert torch.equal(res["z_vals"][0], fetch["z_vals"]), f"{engine}: z vs the fetch"
        assert torch.equal(res["vis_mask"][0], fetch["vis_mask"]), f"{engine}: visibility vs the fetch"
        err = float((res["raw"][0].double() - raw64).abs().max()) / scale
        assert err <= 2e-5, f"{engine}: raw differs from the float64 MLP by {err:.2e} of range"


def test_umma_engine_device_views_ragged_range_generated_rays_and_replay():
    from boostmvsnerfs_b200 import mlp_pack, ops
    H, W, N, K, S = 64, 96, 4, 4, 2
    scene, depth, std, nf, vols, feat, rgb, cams, nerf, packed, triples = _setup(H, W, N, K, 5, True)
    packed_u = mlp_pack.pack_nerf_weights_umma(nerf)
    rays = scene["rays_1"][0]
    full = ops.render_rays_multi(depth, std, nf, rays, H, W, False, S, vols, feat, rgb, cams, triples, packed_u)
    again = ops.render_rays_multi(depth, std, nf, rays, H, W, False, S, vols, feat, rgb, cams, triples, packed_u)
    assert torch.equal(again["raw"], full["raw"]), "not deterministic"
    vdev = torch.tensor(triples, device="cuda", dtype=torch.int32)
    got = ops.render_rays_multi(depth, std, nf, rays, H, W, False, S, vols, feat, rgb, cams, None, packed_u, views_dev=vdev)
    for k_ in ("raw", "z_vals", "vis_mask"):
        assert torch.equal(got[k_], full[k_]), k_
    b, n = 37, 1001                                  # ragged: tiles with dead rows, a second tile slot without work
    part = ops.render_rays_multi(depth, std, nf[0], rays, H, W, False, S, vols, feat, rgb, cams, triples, packed_u, ray_begin=b, n_rays=n)
    assert torch.equal(part["raw"], full["raw"][:, b:b + n]) and torch.equal(part["vis_mask"], full["vis_mask"][:, b:b + n])
    tiny = ops.render_rays_multi(depth[:1], std[:1], nf[:1], rays, H, W, False, S, vols[:1], feat, rgb, cams, triples[:1], packed_u,
                                 ray_begin=5, n_rays=17)          # a single 128-sample tile: one CTA, tile slot 1 idle
    assert torch.equal(tiny["raw"][0], full["raw"][0, 5:22])
    gen = ops.RayGenerator.from_cameras(scene["tar_ext"][0].cpu(), scene["tar_ixt"][0].cpu(), H, W, 1.0, "cuda")
    g = ops.render_rays_multi(depth, std, nf, gen, H, W, False, S, vols, feat, rgb, cams, triples, packed_u)
    assert torch.equal(g["z_vals"], full["z_vals"]) and torch.equal(g["vis_mask"], full["vis_mask"])
    assert float((g["raw"] - full["raw"]).abs().max()) <= 1e-6


# ------------------------------------------------------------------------------------------ row slabs (sharded frames)
@pytest.mark.parametrize("H,W", [(64, 96), (66, 98)])
@pytest.mark.parametrize("depth_inv", [False, True])
@pytest.mark.parametrize("G", [2, 3, 4, 8])
@pytest.mark.parametrize("engine", ["mma", "umma"])
def test_row_slabs_match_the_full_grid(engine, G, depth_inv, H, W):
    """Each rank of a G-way sharded frame renders the row tile dist.row_tile from the row slab dist.slab_rows of the
    volumes and maps (ShardedFrameRenderer.render_tile: grid_rows, vol_row0, map_row0).  Every slab here sits between
    NaN guard rows, above and below each plane, so a read outside it poisons the output instead of returning a
    neighbour's finite data or vanishing under a zero weight: the tile must equal the slice of the full-grid launch bit
    for bit.  Reading the volume or the maps one row off (vol_row0 or map_row0 = y0 + 1, still inside the guards) must
    change the output."""
    from boostmvsnerfs_b200 import dist, mlp_pack, ops
    N, K, S, guard = 4, 3, 2, 2
    scene, depth, std, nf, vols, feat, rgb, cams, nerf, packed, triples = _setup(H, W, N, K, 7 + G, True, depth_inv)
    if engine == "umma":
        packed = mlp_pack.pack_nerf_weights_umma(nerf)
    _, hv, wv = depth.shape
    D = vols.shape[2]
    rays = ops.RayGenerator.from_cameras(scene["tar_ext"][0].cpu(), scene["tar_ixt"][0].cpu(), H, W, 1.0, "cuda")
    full = ops.render_rays_multi(depth, std, nf, rays, H, W, depth_inv, S, vols, feat, rgb, cams, triples, packed,
                                 want_count=True, engine=engine)
    maps_full = torch.cat([depth[:, None], std[:, None], nf], dim=1)           # (K,4,hv,wv): [depth, std, near, far]
    vol_full = vols.permute(0, 2, 3, 4, 1)                                     # (K,D,hv,wv,8) physical layout
    nan = float("nan")
    for q in range(G):
        t0, t1 = dist.row_tile(H, G, q)
        y0, y1 = dist.slab_rows(t0, t1, H, hv)
        rows = y1 - y0
        mbuf = torch.full((K, 4, rows + 2 * guard, wv), nan, device="cuda")
        mbuf[:, :, guard:guard + rows] = maps_full[:, :, y0:y1]
        maps = mbuf[:, :, guard:guard + rows]
        vbuf = torch.full((K, D, rows + 2 * guard, wv, 8), nan, device="cuda")
        vbuf[:, :, guard:guard + rows] = vol_full[:, :, y0:y1]
        slab_vols = vbuf[:, :, guard:guard + rows].permute(0, 4, 1, 2, 3)      # (K,8,D,rows,wv) channels-last-3d
        sl = slice(t0 * W, t1 * W)

        def render(vol_row0, map_row0):
            return ops.render_rays_multi(maps[:, 0], maps[:, 1], maps[:, 2:4], rays, H, W, depth_inv, S, slab_vols, feat, rgb,
                                         cams, triples, packed, ray_begin=t0 * W, n_rays=(t1 - t0) * W, want_count=True,
                                         grid_rows=hv, vol_row0=vol_row0, map_row0=map_row0, engine=engine)
        got = render(y0, y0)
        for k_ in ("raw", "z_vals", "vis_mask", "vis_count"):
            assert torch.equal(got[k_], full[k_][:, sl]), (f"rank {q}/{G}: rows [{t0}, {t1}) from slab [{y0}, {y1}): {k_} "
                                                          f"({int(got[k_].isnan().sum())} NaN)")
        # the controls: one row off (never more than the guard depth) must show
        assert not torch.equal(render(y0 + 1, y0)["raw"], full["raw"][:, sl]), f"rank {q}/{G}: a shifted volume slab went unnoticed"
        assert not torch.equal(render(y0, y0 + 1)["z_vals"], full["z_vals"][:, sl]), f"rank {q}/{G}: shifted maps went unnoticed"
