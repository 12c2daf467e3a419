"""The ENeRF cascade kernels against the float64 restatement oracle/enerf_f64.py, at the shapes of the C2, C4 and C5
workloads and at the edges where they go wrong:
  K1  bmv_cost_volume_var (every dispatch branch: v1 planar, channels-last exact coordinates, v3, v5, v6, fp16 maps) and
      bmv_cost_volume_var_multi (host chain masks and device triples, the C4 4 + 4 and C5 4 + 2 groupings);
  a3  bmv_depth_planes_first / bmv_depth_planes_next (single and batched);
  K2  bmv_depth_regression (register and generic kernels, batched with strided chains);
      bmv_volume_scale (exact exponent, placement of the maximum, inf / NaN / zero, buffer and graph re-use);
and one C4 and one C5 frame, every cascade call checked against float64 evaluated on that call's own inputs.

Every bar is per element and derived from an error model of the kernel's fp32 arithmetic, u = 2^-24 (written next to
each bar below).  Each test also shows that its bar fails for a one-pixel shift, a swapped view, the neighbouring plane
or the neighbouring plane's probability.  Run with -s to see the worst err / bar of each kernel."""
import math

import numpy as np
import pytest
import torch

from boostmvsnerfs_b200.config import RenderConfig
from oracle import enerf_f64 as E

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
WORKLOADS = {"C2": (544, 960, 4, [0, 7, 12, 19]), "C4": (1088, 1920, 8, [0, 3, 7, 9, 12, 15, 17, 19]),
             "C5": (992, 1312, 6, [0, 3, 7, 12, 15, 19])}
STATS = {}
SENS = {}


def _stat(name, ratio=0.0, err=0.0, excluded=0, total=0):
    s = STATS.setdefault(name, dict(ratio=0.0, err=0.0, excluded=0, total=0))
    s["ratio"] = max(s["ratio"], float(ratio))
    s["err"] = max(s["err"], float(err))
    s["excluded"] += int(excluded)
    s["total"] += int(total)


def _sens(name, fraction):
    """smallest fraction of the elements at which a bar rejected a deliberately wrong reference"""
    SENS[name] = min(SENS.get(name, 1.0), float(fraction))


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for k in sorted(STATS):
        s = STATS[k]
        print(f"\n[cascade] {k}: worst err/bar {s['ratio']:.3g}, max err {s['err']:.3g}, "
              f"excluded {s['excluded']}/{s['total']}", end="")
    for k in sorted(SENS):
        print(f"\n[cascade] sensitivity, {k}: rejected at >= {SENS[k]:.3f} of the elements", end="")
    print()


@pytest.fixture(scope="module")
def ops():
    from boostmvsnerfs_b200 import ops as _ops
    return _ops


def _check(got, ref, bar, what, keep=None):
    """per element |got - ref| <= bar (where keep); -> (worst err / bar, max err)."""
    err = (got.double() - ref).abs()
    ok = err <= bar
    if keep is not None:
        ok |= ~keep
    n = int((~ok).sum())
    assert n == 0, (f"{what}: {n}/{err.numel()} elements outside the bar; max err {float(err.max()):.3e}, "
                    f"worst at {np.unravel_index(int(((err - bar) * (1 if keep is None else keep)).argmax()), err.shape)}")
    m = keep if keep is not None else torch.ones_like(ok)
    ratio = torch.where(bar > 0, err / bar, torch.where(err > 0, float("inf"), 0.0))
    return float(ratio[m].max()) if bool(m.any()) else 0.0, float(err[m].max()) if bool(m.any()) else 0.0


def _fail_fraction(got, wrong, bar, keep=None, among=None):
    """fraction of the elements (where `among`) at which the bar rejects a wrong reference"""
    bad = (got.double() - wrong).abs() > bar
    sel = torch.ones_like(bad) if among is None else among
    if keep is not None:
        sel = sel & keep
    return float(bad[sel].double().mean())


# ------------------------------------------------------------------------------------------ K1 error model
def k1_bar(r, scale=1.0, fmt=torch.float32):
    """Bar of a K1 volume (C,D',R',w) against oracle result r, and the voxels kept (D',R',w).
    Sample of view s: the source pixel carries a few ulps of its magnitude scale `coord` (cam = R x + t / d rounded in
    3 to 5 operations, the reciprocals or divisions of d and cz, the normalise / unnormalise round trip: <= 10 roundings
    of coord in all) -> 16 u coord * slope; the four-tap FMA chain and the weight products -> 8 u * sum |w f|.
    Variance sum(f^2) / S - mean^2: the sample errors e_s propagate with |d var / d f_s| <= 2 (|f_s| + |mean|) / S (plus
    e_s^2 / S), the S sums, 1 / S and the final FMA add <= 8 u (sum f^2 / S + mean^2).
    Stored output scaled by s (a power of two, exact); 16-bit outputs add half an ulp of the format on s * var
    (bf16: 2^-8 relative, fp16: 2^-11 relative + 2^-25, half the fp16 subnormal spacing).
    Voxels whose cz lies within 64 u of its magnitude scale of the 1e-6 clamp are excluded (fp32 may take the other side)."""
    S = r["feat"].shape[0]
    cs = torch.where(r["slope"] > 0, r["coord"][:, None] * r["slope"], torch.zeros_like(r["slope"]))
    e = 16 * U * cs + 8 * U * r["absmag"]
    bar = (2.0 / S * (r["feat"].abs() + r["mean"].abs()) * e + e * e / S).sum(0) + 8 * U * (r["sq"] + r["mean"] ** 2)
    ref = r["var"] * scale
    bar = bar * scale
    if fmt == torch.bfloat16:
        bar = bar + 2.0 ** -8 * (ref.abs() + bar)
    elif fmt == torch.float16:
        bar = bar + 2.0 ** -11 * (ref.abs() + bar) + 2.0 ** -25
    keep = ((r["cz"] - E.CLAMP).abs() > 64 * U * r["cz_mag"]).all(0) & torch.isfinite(bar).all(0)
    return ref, bar, keep[None].expand_as(bar)


def _sub(vol, pidx, rows):
    return vol[:, pidx][:, :, rows]


def check_k1(got, feats, views, proj, planes, what, pidx=None, rows=None, hw=None, scale=1.0, name="K1 per-chain",
             sensitivity=False):
    D = planes.shape[0]
    h, w = (hw if planes.dim() == 1 else planes.shape[1:])
    pidx = list(range(D)) if pidx is None else pidx
    rows = list(range(h)) if rows is None else rows
    r = E.cost_volume_var(feats, views, proj, planes, rows=rows, plane_idx=pidx, hw=hw)
    g = _sub(got, pidx, rows)
    ref, bar, keep = k1_bar(r, scale, got.dtype)
    ratio, err = _check(g, ref, bar, what, keep)
    n_vox = keep[0].numel()
    _stat(name + (f" {str(got.dtype)[6:]} out" if got.dtype != torch.float32 else ""), ratio, err,
          n_vox - int(keep[0].sum()), n_vox)
    assert int(keep[0].sum()) >= 0.99 * n_vox, f"{what}: {n_vox - int(keep[0].sum())} voxels at the cz clamp"
    if sensitivity:
        among = ref.abs() > 1e-3 * float(ref.abs().max())
        shifted = torch.roll(feats, 1, dims=-1)
        fr = E.cost_volume_var(shifted, views, proj, planes, rows=rows, plane_idx=pidx, hw=hw)["var"] * scale
        other = next(v for v in range(feats.shape[0]) if v not in views)
        sw = E.cost_volume_var(feats, [views[0], other] + list(views[2:]), proj, planes, rows=rows, plane_idx=pidx,
                               hw=hw)["var"] * scale
        nb = [min(p + 1, D - 1) if p < D - 1 else p - 1 for p in pidx]
        pl = E.cost_volume_var(feats, views, proj, planes, rows=rows, plane_idx=nb, hw=hw)["var"] * scale
        # a swapped view leaves the voxels whose samples fall outside both maps unchanged: a lower floor for it
        for label, wrong, floor in (("one-pixel feature shift", fr, 0.5), ("swapped view", sw, 0.25),
                                    ("neighbouring plane", pl, 0.5)):
            f = _fail_fraction(g, wrong, bar, keep, among)
            _sens(f"K1 {label}", f)
            assert f > floor, f"{what}: the bar rejects only {f:.3f} of a {label}"
    return r


def _proj_synth(N, seed, sx=1.15, sy=1.1):
    """volume pixel -> source pixel at (sx, sy) with per-view translations of a few pixels (partly outside the map)"""
    g = torch.Generator().manual_seed(seed)
    proj = torch.eye(3, 4).repeat(N, 1, 1)
    proj[:, 0, 0], proj[:, 1, 1] = sx, sy
    proj[:, :, 3] = torch.randn(N, 3, generator=g) * torch.tensor([4.0, 3.0, 0.01])
    proj[:, 2, :3] += torch.randn(N, 3, generator=g) * 1e-3
    proj[:, :2, :2] += torch.randn(N, 2, 2, generator=g) * 0.02
    return proj.cuda()


def _feats(N, C, Hs, Ws, seed, smooth=False, half=False, channels_last=True):
    g = torch.Generator().manual_seed(seed)
    if smooth:
        low = torch.randn(N, C, max(Hs // 16, 2), max(Ws // 16, 2), generator=g)
        f = torch.nn.functional.interpolate(low, size=(Hs, Ws), mode="bilinear", align_corners=True)
    else:
        f = torch.randn(N, C, Hs, Ws, generator=g)
    f = f.cuda()
    if channels_last:
        f = f.contiguous(memory_format=torch.channels_last)
    return f.half() if half else f


def _planes_pp(D, h, w, seed, lo=0.5, hi=3.5):
    g = torch.Generator().manual_seed(seed)
    return torch.sort(torch.rand(D, h, w, generator=g) * (hi - lo) + lo, dim=0).values.cuda()


# ------------------------------------------------------------------------------------------ K1, every dispatch branch
# name: (C, channels-last maps and volume, exact_coords, variant, fp16 maps)
BRANCHES = {"v1_planar": (32, False, False, 0, False), "cl_exact_c32": (32, True, True, 0, False),
            "cl_exact_c16": (16, True, True, 0, False), "v3_c8": (8, True, False, 0, False),
            "v5_c16": (16, True, False, 5, False), "v5_c32": (32, True, False, 5, False),
            "v6_c16": (16, True, False, 0, False), "v6_c32": (32, True, False, 0, False),
            "v6_c32_fp16maps": (32, True, False, 0, True), "v5_c16_fp16maps": (16, True, False, 5, True)}


@pytest.mark.parametrize("S", [1, 2, 3, 4])
@pytest.mark.parametrize("branch", list(BRANCHES))
def test_k1_dispatch_branches_vs_float64(ops, branch, S):
    """Ragged shape: odd h = 37, w = 45 (not a multiple of a warp's 4 / 8 / 16 voxels nor of a CTA's), D = 7 (not a
    multiple of the plane group).  fp32 out with per-pixel planes for every S; at S = 3 also shared planes, bf16 out,
    fp16 out with a volume_scale, and the sensitivity of the bar."""
    C, cl, exact, variant, half = BRANCHES[branch]
    N, Hs, Ws, h, w, D = 5, 40, 52, 37, 45, 7
    feats = _feats(N, C, Hs, Ws, seed=C + S, half=half, channels_last=cl)
    proj = _proj_synth(N, seed=S)
    planes = _planes_pp(D, h, w, seed=S)
    views = [4, 1, 2, 0][:S]
    kw = dict(channels_last=cl, exact_coords=exact, variant=variant)
    got = ops.cost_volume_var(feats, views, proj, planes, **kw)
    check_k1(got, feats, views, proj, planes, f"{branch} S={S}", sensitivity=(S == 3))
    if S != 3:
        return
    shared = torch.linspace(0.6, 3.4, 12, device="cuda")
    got = ops.cost_volume_var_shared(feats, views, proj, shared, h, w, **kw)
    check_k1(got, feats, views, proj, shared, f"{branch} shared planes", hw=(h, w))
    got = ops.cost_volume_var(feats, views, proj, planes, out_dtype=torch.bfloat16, **kw)
    check_k1(got, feats, views, proj, planes, f"{branch} bf16 out")
    vsc = ops.volume_scale(feats)
    got = ops.cost_volume_var(feats, views, proj, planes, out_dtype=torch.float16, out_scale=vsc, **kw)
    check_k1(got, feats, views, proj, planes, f"{branch} fp16 out", scale=float(vsc[0]))


# ------------------------------------------------------------------------------------------ K1 at the workload shapes
def _workload_cams(name):
    from boostmvsnerfs_b200.network import BoostEnerfNetwork
    from boostmvsnerfs_b200.synth import make_scene
    H, W = WORKLOADS[name][:2]
    sc = make_scene(H=H, W=W, n_views=6, seed=0, render_scales=())
    rc = RenderConfig.enerf_eval()
    projs = [BoostEnerfNetwork._proj_all(sc["all_src_exts"][0], sc["all_src_ixts"][0], sc["tar_ext"][0], sc["tar_ixt"][0],
                                         rc.im_feat_scale[i], rc.volume_scale[i]).cuda() for i in range(2)]
    return H, W, projs, sc["near_far"][0].cuda()


def _edge_rows(h):
    return sorted({0, 1, h // 2, h - 2, h - 1})


@pytest.mark.parametrize("field", ["noise", "smooth"])
@pytest.mark.parametrize("level", [0, 1])
@pytest.mark.parametrize("wl", ["C2", "C4", "C5"])
def test_k1_workload_shapes_vs_float64(ops, wl, level, field):
    """The default (v6) path at each workload's level-0 (shared planes, D = 64, C = 32) and level-1 (per-pixel planes,
    D = 8, C = 16) shapes, fp32 out and fp16 out scaled by volume_scale, on the edge rows and the first, second, middle
    and last planes."""
    H, W, projs, near_far = _workload_cams(wl)
    C, fs, vs = (32, 4, 8) if level == 0 else (16, 2, 2)
    h, w = H // vs, W // vs
    feats = _feats(6, C, H // fs, W // fs, seed=level + 7, smooth=(field == "smooth"))
    if level == 0:
        planes, _ = ops.depth_planes_first(near_far, 64, h, w, True)
        hw = (h, w)
    else:
        g = torch.Generator().manual_seed(3)
        base = torch.nn.functional.interpolate(torch.rand(1, 1, 8, 8, generator=g) * 4 + 2.5, size=(h, w), mode="bilinear",
                                               align_corners=True)[0, 0].cuda()
        planes = (base[None] * (1 + 0.15 * torch.linspace(-1, 1, 8, device="cuda")).view(8, 1, 1)).contiguous()
        hw = None
    D = planes.shape[0]
    pidx, rows = sorted({0, 1, D // 2, D - 1}), _edge_rows(h)
    views = [0, 2, 5]
    run = (lambda **kw: ops.cost_volume_var_shared(feats, views, projs[level], planes, h, w, channels_last=True, **kw)) \
        if level == 0 else (lambda **kw: ops.cost_volume_var(feats, views, projs[level], planes, channels_last=True, **kw))
    got = run()
    check_k1(got, feats, views, projs[level], planes, f"{wl} l{level} {field}", pidx, rows, hw,
             sensitivity=(field == "noise"))
    vsc = ops.volume_scale(feats)
    got = run(out_dtype=torch.float16, out_scale=vsc)
    check_k1(got, feats, views, projs[level], planes, f"{wl} l{level} {field} fp16", pidx, rows, hw, scale=float(vsc[0]))


# ------------------------------------------------------------------------------------------ K1 multi-chain
MULTI = {16: [[0, 1, 2], [1, 2, 3], [0, 2, 3], [0, 1, 3]], 32: [[0, 1, 2], [3, 4, 5], [5, 6, 7], [0, 4, 7]]}


@pytest.mark.parametrize("variant", [0, 5])
@pytest.mark.parametrize("K", [1, 2, 3, 4])
@pytest.mark.parametrize("C", [16, 32])
def test_k1_multi_chain_vs_float64(ops, C, K, variant):
    """C = 16 with up to 4 unique views, C = 32 with up to 8; host chain masks and device-resident triples; fp32 out and
    fp16 out with a volume_scale; ragged 37 x 45 x 7."""
    N = 4 if C == 16 else 8
    Hs, Ws, h, w, D = 40, 52, 37, 45, 7
    feats = _feats(N, C, Hs, Ws, seed=C + K)
    proj = _proj_synth(N, seed=K + 10)
    planes = torch.linspace(0.6, 3.4, D, device="cuda")
    triples = MULTI[C][:K]
    vsc = ops.volume_scale(feats)
    for dtype in (torch.float32, torch.float16):
        for dev_triples in (False, True):
            out = torch.empty((K, D, h, w, C), device="cuda", dtype=dtype).permute(0, 4, 1, 2, 3)
            tdev = torch.tensor(triples, dtype=torch.int32, device="cuda").reshape(-1) if dev_triples else None
            sc = vsc if dtype == torch.float16 else None
            ops.cost_volume_var_shared_multi(feats, triples, proj, planes, h, w, out=out, out_scale=sc, triples_dev=tdev,
                                             variant=variant)
            for k in range(K):
                check_k1(out[k], feats, triples[k], proj, planes, f"multi C={C} K={K} chain {k} {dtype} dev={dev_triples}",
                         hw=(h, w), scale=float(vsc[0]) if sc is not None else 1.0, name="K1 multi-chain",
                         sensitivity=(k == K - 1 and dtype == torch.float32 and not dev_triples and K == 4))


@pytest.mark.parametrize("wl", ["C4", "C5"])
def test_k1_multi_chain_workload_groupings(ops, wl):
    """The level-0 volumes of C4 (8 chains: 4 + 4) and C5 (6 chains: 4 + 2) as the frame builds them: groups of <= 4
    chains per launch, fp16 out scaled by volume_scale."""
    import itertools
    H, W, projs, near_far = _workload_cams(wl)
    h, w = H // 8, W // 8
    feats = _feats(6, 32, H // 4, W // 4, seed=21)
    planes, _ = ops.depth_planes_first(near_far, 64, h, w, True)
    table = list(itertools.combinations(range(6), 3))
    triples = [list(table[i]) for i in WORKLOADS[wl][3]]
    K = len(triples)
    vsc = ops.volume_scale(feats)
    out = torch.empty((K, 64, h, w, 32), device="cuda", dtype=torch.float16).permute(0, 4, 1, 2, 3)
    groups = []
    for k0 in range(0, K, 4):
        grp = triples[k0:k0 + 4]
        groups.append(len(grp))
        ops.cost_volume_var_shared_multi(feats, grp, projs[0], planes, h, w, out=out[k0:k0 + len(grp)], out_scale=vsc)
    assert groups == ([4, 4] if wl == "C4" else [4, 2])
    for k in range(K):
        check_k1(out[k], feats, triples[k], projs[0], planes, f"{wl} chain {k}", [0, 1, 31, 63], _edge_rows(h), (h, w),
                 scale=float(vsc[0]), name="K1 multi-chain")


# ------------------------------------------------------------------------------------------ K1 geometry edges
@pytest.mark.parametrize("branch", ["v1_planar", "cl_exact_c32", "v5_c32", "v6_c32", "v6_c16"])
def test_k1_geometry_edges_vs_float64(ops, branch):
    """View 1: a camera with part of the volume behind it (cz crosses the 1e-6 clamp); view 2: projections that land
    entirely outside the map; view 0 / 3: straddling the map edges (partial zeros padding); a repeated view id in a
    triple; near-identical views (the variance cancels to rounding level)."""
    C, cl, exact, variant, half = BRANCHES[branch]
    N, Hs, Ws, h, w, D = 4, 40, 52, 37, 45, 7
    feats = _feats(N, C, Hs, Ws, seed=5, channels_last=cl)
    proj = _proj_synth(N, seed=4, sx=1.6, sy=1.5)                      # 1.6 x 45 > 52: the right part straddles / leaves
    proj[1, 2] = torch.tensor([0.021, 0.0, -0.307, 0.013], device="cuda")   # cz < 0 for x < ~14: behind the camera
    proj[2, :2, 3] += 1000.0                                           # fully outside the map
    planes = _planes_pp(D, h, w, seed=6)
    kw = dict(channels_last=cl, exact_coords=exact, variant=variant)
    for views in ([0, 1, 3], [1, 2, 3], [3, 3, 0], [2, 2], [0, 1, 2, 3]):
        got = ops.cost_volume_var(feats, views, proj, planes, **kw)
        r = check_k1(got, feats, views, proj, planes, f"{branch} edges {views}", name="K1 geometry edges")
        if 1 in views:
            assert bool((r["cz"] < 0).any()) and bool((r["cz"] > 0).any())
    # near-identical views: same camera, features 1e-3 apart
    f2 = feats.clone()
    f2[1] = feats[0] + 1e-3 * _feats(1, C, Hs, Ws, seed=8, channels_last=cl)[0]
    p2 = proj.clone()
    p2[1] = proj[0]
    got = ops.cost_volume_var(f2, [0, 1], p2, planes, **kw)
    check_k1(got, f2, [0, 1], p2, planes, f"{branch} near-identical views", name="K1 near-identical views")


# ------------------------------------------------------------------------------------------ a3
@pytest.mark.parametrize("D", [1, 8, 64])
@pytest.mark.parametrize("inv", [False, True])
def test_depth_planes_first_vs_float64(ops, inv, D):
    """Bar: the plane is 3 (uniform) or 6 (disparity) roundings of the terms summed in `mag` -> 8 u * mag."""
    nf = torch.tensor([2.0, 8.0], device="cuda")
    planes, nfo = ops.depth_planes_first(nf, D, 68, 120, inv)
    r = E.depth_planes_first(nf, D, inv)
    ratio, err = _check(planes, r["planes"], 8 * U * r["mag"], f"planes D={D} inv={inv}")
    _stat("a3 depth_planes_first", ratio, err)
    ratio, err = _check(nfo, r["nf"].view(2, 1, 1).expand(2, 68, 120), 8 * U * r["nf_mag"].view(2, 1, 1), "near_far")
    _stat("a3 depth_planes_first", ratio, err)
    if D > 1:
        f = _fail_fraction(planes, torch.roll(r["planes"], 1), 8 * U * r["mag"])
        _sens("a3 first: neighbouring plane", f)
        assert f > 0.8


def a3_next_bar(r, cur_inv):
    """Bar of depth_planes_next's planes and near / far.  Upsample: the fp32 source coordinate scale * dst carries 2 ulps
    of its magnitude -> 4 u * src * slope, the lerp weights and the two-level blend 4 u * sum |w a|.  lo = min(d + s,
    nf0) and hi = max(d - s, nf1) are 1-Lipschitz (the bar of the clamped side is the larger one) plus u |lo|; the
    inversion 1 / lo propagates e / lo^2 plus u / |lo|; the plane (3 or 6 roundings) adds 8 u * its term magnitude."""
    def up_err(k):
        v, slope, src, absmag = r[f"up_{k}"]
        return 4 * U * src * slope + 4 * U * absmag
    e_lo = torch.maximum(up_err("depth") + up_err("std") + U * r["lo"].abs(), up_err("nf0"))
    e_hi = torch.maximum(up_err("depth") + up_err("std") + U * r["hi"].abs(), up_err("nf1"))
    lo, hi = r["lo"], r["hi"]
    t = torch.linspace(0.0, 1.0, r["planes"].shape[1], device=lo.device, dtype=torch.float32).double().view(1, -1, 1, 1)
    nr, fr = (1 / lo)[:, None], (1 / hi)[:, None]
    _, mag = E._lerp_planes(nr, fr, t, cur_inv)
    if cur_inv:   # 1 / nr = lo after two more roundings; the plane 1 / disp carries e_disp / disp^2
        disp = 1 / r["planes"]
        e = ((e_lo + 2 * U * lo)[:, None] + (e_hi + 2 * U * hi)[:, None]) / disp ** 2 + 8 * U * mag
    else:
        e = (e_lo / lo ** 2 + U / lo)[:, None] + (e_hi / hi ** 2 + U / hi)[:, None] + 8 * U * mag
    ends, e_ends = r["planes"][:, [0, -1]], e[:, [0, -1]]
    e_nf = e_ends / ends ** 2 + U / ends if cur_inv else e_ends
    return e, e_nf


@pytest.mark.parametrize("cur_inv", [False, True])
@pytest.mark.parametrize("shape", [(68, 120, 272, 480), (136, 240, 544, 960), (124, 164, 496, 656), (17, 30, 68, 121)])
def test_depth_planes_next_vs_float64(ops, shape, cur_inv):
    """x4 align_corners upsample at the three workloads' level shapes and an odd 17x30 -> 68x121; two chains batched with
    shared and per-chain near / far; std pushes d + s past nf0 and d - s past nf1 at some pixels, 0 at others."""
    h0, w0, h, w = shape
    K, D = 2, 8
    g = torch.Generator().manual_seed(h0 + w0)
    depth = (torch.rand(K, h0, w0, generator=g) * 0.3 + 0.15).cuda()
    std = (torch.rand(K, h0, w0, generator=g) * 0.12).cuda()
    std[:, ::3] = 0.0
    nf_shared = torch.stack([torch.full((h0, w0), 0.5), torch.full((h0, w0), 0.125)]).cuda()
    nf_each = (nf_shared[None] * (1 + 0.1 * torch.rand(K, 2, h0, w0, generator=g).cuda())).contiguous()
    for nf in (nf_shared, nf_each):
        planes, nfo = ops.depth_planes_next_batched(depth, std, nf, D, h, w, cur_inv)
        r = E.depth_planes_next(depth, std, nf, D, h, w, cur_inv)
        clamped_lo = (r["up_depth"][0] + r["up_std"][0] >= r["up_nf0"][0])
        clamped_hi = (r["up_depth"][0] - r["up_std"][0] <= r["up_nf1"][0])
        assert bool(clamped_lo.any()) and bool((~clamped_lo).any()) and bool(clamped_hi.any()) and bool((~clamped_hi).any())
        e, e_nf = a3_next_bar(r, cur_inv)
        ratio, err = _check(planes, r["planes"], e, f"planes {shape} inv={cur_inv}")
        _stat("a3 depth_planes_next planes", ratio, err)
        ratio, err = _check(nfo, r["nf"], e_nf, f"near_far {shape} inv={cur_inv}")
        _stat("a3 depth_planes_next near_far", ratio, err)
        p1, n1 = ops.depth_planes_next(depth[1], std[1], nf if nf.dim() == 3 else nf[1], D, h, w, cur_inv)
        assert torch.equal(p1, planes[1]) and torch.equal(n1, nfo[1])
    # the bar rejects the planes of a depth map shifted by one pixel, wherever neither side is clamped
    wrong = E.depth_planes_next(torch.roll(depth, 1, dims=-1), std, nf_shared, D, h, w, cur_inv)["planes"]
    r = E.depth_planes_next(depth, std, nf_shared, D, h, w, cur_inv)
    planes, _ = ops.depth_planes_next_batched(depth, std, nf_shared, D, h, w, cur_inv)
    free = ((r["up_depth"][0] + r["up_std"][0] < r["up_nf0"][0]) & (r["up_depth"][0] - r["up_std"][0] > r["up_nf1"][0]))
    free = free[:, None].expand_as(planes)
    f = _fail_fraction(planes, wrong, a3_next_bar(r, cur_inv)[0], among=free)
    _sens("a3 one-pixel depth shift", f)
    assert f > 0.5


# ------------------------------------------------------------------------------------------ K2
def k2_bar(r):
    """Bar of depth_regression.  Probability p_d = exp(l_d - m) / den: the rounding of l_d - m is amplified by exp to
    u |l_d - m|, expf <= 2 ulp, den (D sums) D u, the division u -> relative u (|l_d - m| + D + 3), plus an absolute
    2^-126 where exp underflows.  depth = sum p v (D products and sums, D + 1 roundings; v = 1 / max(plane, 1e-6) one
    more with depth_inv): u sum p |v| (|l - m| + 2 D + 5).  var = sum p (v - depth)^2: the relative error of p, the
    D + 3 roundings of the products and sums, and the depth error (and v's) through 2 sum p |v - depth|.  std = sqrt of
    var clamped at 1e-10: |d std| <= |d var| / (std + std_low) + u std.  The first-order bounds are doubled."""
    p, v, L = r["prob"], r["vals"], r["lse_dev"]
    D = p.shape[1]
    rel = U * (L + D + 3)
    e_depth = 2 * ((U * p * v.abs() * (L + 2 * D + 5)).sum(1) + 2.0 ** -126 * v.abs().sum(1))
    dv = v - r["depth"][:, None]
    e_var = 2 * ((p * (rel + (D + 3) * U) * dv * dv).sum(1) + 2.0 ** -126 * (dv * dv).sum(1)
                 + 2 * (p * dv.abs() * (e_depth[:, None] + U * v.abs())).sum(1))
    std = r["std"]
    low = (r["var"] - e_var).clamp_min(1e-10).sqrt()
    e_std = e_var / (std + low) + U * std
    return e_depth, e_std


K2_SHAPES = {8: (544, 960), 16: (272, 480), 32: (136, 240), 64: (136, 240), 7: (124, 164), 12: (272, 480), 128: (136, 240)}


@pytest.mark.parametrize("case", ["randn", "spread60", "equal", "tiny_planes"])
@pytest.mark.parametrize("D", [8, 16, 32, 64, 7, 12, 128])
def test_depth_regression_vs_float64(ops, D, case):
    """Register kernels (D = 8, 16, 32, 64) and the generic one (7, 12, 128), three chains batched out of a wider tensor
    (chain stride (D + 3) h w > D h w).  Logits N(0, 3^2); spread over +-60 with one dominant plane (the softmax saturates
    and exp underflows); all equal; and planes at and below the 1e-6 clamp with depth_inv."""
    h, w = K2_SHAPES[D]
    K = 3
    g = torch.Generator().manual_seed(D * 7 + len(case))
    wide = torch.randn(K, D + 3, h, w, generator=g) * 3
    if case == "spread60":
        wide = torch.rand(K, D + 3, h, w, generator=g) * 120 - 60
        dom = torch.randint(1, D + 1, (K, 1, h, w), generator=g)
        wide.scatter_(1, dom, 60.0)
    elif case == "equal":
        wide = torch.full((K, D + 3, h, w), 1.7)
    logits = wide.cuda()[:, 1:D + 1]
    assert logits.stride(0) == (D + 3) * h * w
    inv = case in ("tiny_planes", "spread60")
    if case == "equal":
        planes = torch.linspace(2.0, 8.0, D, device="cuda")
    else:
        planes = torch.sort(torch.rand(K, D, h, w, generator=g) * 6 + 2, dim=1).values.cuda()
    if case == "tiny_planes":
        planes[:, 0, ::2] = E.CLAMP
        planes[:, 0, 1::4] = 3e-7
        planes[:, 0, 3::4] = 0.0
        planes = planes.contiguous()
    d, s = ops.depth_regression_batched(logits, planes, inv)
    r = E.depth_regression(logits, planes, inv)
    e_depth, e_std = k2_bar(r)
    ratio, err = _check(d, r["depth"], e_depth, f"depth D={D} {case}")
    _stat("K2 depth", ratio, err)
    ratio, err = _check(s, r["std"], e_std, f"std D={D} {case}")
    _stat("K2 std", ratio, err)
    if case in ("randn", "spread60"):
        wrong = E.depth_regression(torch.roll(logits, 1, dims=1), planes, inv)["depth"]
        f = _fail_fraction(d, wrong, e_depth)
        _sens("K2 neighbouring plane's probability", f)
        assert f > 0.5


# ------------------------------------------------------------------------------------------ volume_scale
def _expected_scale(x, target=16384.0):
    """The kernel's rule in Python: m = max |x| over the finite-or-inf values (NaN ignored, inf read as 3e38), m = f 2^e
    (frexp), target = g 2^te, k = te - 1 - 2e clamped to [-40, 40] (0 for m = 0).  Unclamped this guarantees
    2^k m^2 < 2^(te - 1) <= target (m^2 < 2^2e) and 2^k m^2 >= 2^(te - 3) > target / 8 (m >= 2^(e - 1))."""
    a = x.float().abs()
    a = a[~torch.isnan(a)]
    m = min(float(a.max()) if a.numel() else 0.0, 3.0e38)
    m = float(np.float32(m))
    if m == 0.0:
        return 0
    _, e = math.frexp(m)
    _, te = math.frexp(target)
    return max(-40, min(40, te - 1 - 2 * e))


def _check_scale(sc, k, cs=1.0):
    want = torch.tensor([2.0 ** k, 2.0 ** -k, 0.0, 0.0, 2.0 ** k * cs, 1.0 / (2.0 ** k * cs)], dtype=torch.float32)
    got = sc.cpu()
    assert torch.equal(got, want), f"volume_scale {got.tolist()} != {want.tolist()} (k = {k})"


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
def test_volume_scale_exponent_is_exact(ops, dtype):
    vec = 16 // (4 if dtype == torch.float32 else 2)
    n = 6_000_000 if dtype == torch.float32 else 12_000_000
    nvec = n // vec
    blocks = min(-(-nvec // 1024), 8 * 148)
    stride = blocks * 256                                 # vectors per grid-stride step; 4 steps per loop iteration
    g = torch.Generator().manual_seed(17)
    base = (torch.rand(n, generator=g) * 0.02 - 0.01).to(dtype).cuda()
    where = {"first element": 0, "last 16-byte vector": n - 3, "past one grid stride": stride * vec + 1,
             "past one loop iteration": 4 * stride * vec + vec - 1}
    for label, i in where.items():
        for big in (3.7, -1900.0, 1e-30 if dtype == torch.float32 else 6e-5):
            x = base.clone()
            if abs(big) < 1e-3:
                x.zero_()
            x[i] = big
            k = _expected_scale(x)
            _check_scale(ops.volume_scale(x), k)
            if abs(big) >= 1:
                s = 2.0 ** k * float(x.float().abs().max()) ** 2
                assert 16384.0 / 8 < s < 16384.0, f"{label}: 2^k max^2 = {s}"
    assert _expected_scale(torch.tensor([1e-30])) == 40               # the +40 clamp is reached (fp32 tiny maxima)
    for label, val in (("inf", float("inf")), ("nan", float("nan"))):
        x = base.clone()
        x[where["past one grid stride"]] = val
        x[5] = 2.5
        k = _expected_scale(x)
        _check_scale(ops.volume_scale(x), k)
        if label == "inf":
            assert k == -40
    _check_scale(ops.volume_scale(torch.zeros(n, dtype=dtype, device="cuda")), 0)
    _check_scale(ops.volume_scale(base, consumer_scale=0.25), _expected_scale(base), 0.25)


def test_volume_scale_buffer_reuse_eager_and_in_a_graph(ops):
    """The same out buffer for inputs with different maxima, eagerly and in a replayed CUDA graph: the scratch words
    reset after every launch, so the result follows each input."""
    x = torch.zeros(1 << 20, device="cuda")
    out = torch.zeros(6, device="cuda")
    for m in (3.0, 0.01, 700.0, 0.5):
        x.fill_(0.1)
        x[12345] = m
        ops.volume_scale(x, out=out)
        _check_scale(out, _expected_scale(x))
    x.fill_(0.1)
    x[7] = 5.0
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ops.volume_scale(x, out=out)                   # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        ops.volume_scale(x, out=out)
    for m in (5.0, 1e-3, 9000.0, 0.2):
        x.fill_(0.05)
        x[(1 << 20) - 1] = m
        graph.replay()
        torch.cuda.synchronize()
        _check_scale(out, _expected_scale(x))


# ------------------------------------------------------------------------------------------ stage-wise frame check
CASCADE_OPS = ("volume_scale", "depth_planes_first", "depth_planes_next_batched", "cost_volume_var",
               "cost_volume_var_shared", "cost_volume_var_shared_multi", "depth_regression_batched", "depth_regression")


@pytest.mark.parametrize("wl", ["C4", "C5"])
def test_frame_cascade_calls_vs_float64(ops, wl, monkeypatch):
    """One frame at the workload's size, network built as bench.py builds it (default precision: fp16 cost volumes with
    range scales).  Every cascade call is recorded and its output compared with float64 on that call's own inputs."""
    import itertools
    from boostmvsnerfs_b200 import network
    from boostmvsnerfs_b200.synth import batch_to, make_scene
    H, W, K, k_best = WORKLOADS[wl]
    calls = []

    def wrap(name, fn):
        def rec(*a, **kw):
            res = fn(*a, **kw)
            outs = res if isinstance(res, tuple) else (res,)
            calls.append((name, a, kw, tuple(o.clone() for o in outs)))
            return res
        return rec
    for name in CASCADE_OPS:
        monkeypatch.setattr(ops, name, wrap(name, getattr(ops, name)))
    old = torch.backends.cudnn.allow_tf32
    try:
        torch.backends.cudnn.allow_tf32 = True
        rc = RenderConfig.enerf_eval(K)
        torch.manual_seed(0)
        net = network.BoostEnerfNetwork(preprocess=True, rc=rc).eval().to("cuda")
        net.view_selection_outputs = {"synth_0": k_best}
        batch = batch_to(make_scene(H=H, W=W, n_views=6, seed=0), "cuda")
        with torch.no_grad():
            net(batch)
        torch.cuda.synchronize()
    finally:
        torch.backends.cudnn.allow_tf32 = old
    names = [c[0] for c in calls]
    table = list(itertools.combinations(range(6), 3))
    triples = [list(table[i]) for i in k_best]
    assert names.count("cost_volume_var_shared_multi") == 2, names       # 4 + 4 (C4) or 4 + 2 (C5) chains
    assert names.count("cost_volume_var") == K and "depth_planes_next_batched" in names
    n_regr = 0
    for name, a, kw, outs in calls:
        if name == "volume_scale":
            x = a[0]
            _check_scale(outs[0], _expected_scale(x), float(kw.get("consumer_scale", 1.0)))
        elif name == "depth_planes_first":
            near_far, D, h, w, inv = a
            r = E.depth_planes_first(near_far, D, inv)
            _stat("frame a3 first", *_check(outs[0], r["planes"], 8 * U * r["mag"], f"{wl} first planes"))
        elif name == "depth_planes_next_batched":
            depth, std, nf, D, h, w, inv = a
            r = E.depth_planes_next(depth, std, nf, D, h, w, inv)
            e, e_nf = a3_next_bar(r, inv)
            _stat("frame a3 next", *_check(outs[0], r["planes"], e, f"{wl} next planes"))
            _stat("frame a3 next", *_check(outs[1], r["nf"], e_nf, f"{wl} next near_far"))
        elif name == "cost_volume_var_shared_multi":
            f, grp, proj, planes, h, w = a
            out, vsc = kw["out"], kw.get("out_scale")
            assert out.dtype == torch.float16 and vsc is not None
            for k, t in enumerate(grp):
                check_k1(outs[0][k], f, t, proj, planes, f"{wl} frame multi chain {k}", [0, 1, 32, 63], _edge_rows(h),
                         (h, w), scale=float(vsc[0]), name="frame K1 multi-chain")
            assert [list(map(int, t)) for t in grp] in (triples[:4], triples[4:8])
        elif name == "cost_volume_var":
            f, views, proj, planes = a
            vsc = kw.get("out_scale")
            D, h, w = planes.shape
            check_k1(outs[0], f, views, proj, planes, f"{wl} frame l1 {views}", list(range(D)), _edge_rows(h),
                     scale=float(vsc[0]) if vsc is not None else 1.0, name="frame K1 per-chain")
        elif name == "depth_regression_batched":
            logits, planes, inv = a
            rows = _edge_rows(logits.shape[-2])
            pl = planes if planes.dim() == 1 else planes[:, :, rows]
            r = E.depth_regression(logits[:, :, rows], pl, inv)
            e_depth, e_std = k2_bar(r)
            _stat("frame K2 depth", *_check(outs[0][:, rows], r["depth"], e_depth, f"{wl} frame depth"))
            _stat("frame K2 std", *_check(outs[1][:, rows], r["std"], e_std, f"{wl} frame std"))
            n_regr += 1
        elif name == "depth_regression":
            logits, planes, inv = a
            rows = _edge_rows(logits.shape[-2])
            pl = planes[None] if planes.dim() == 1 else planes[None][:, :, rows]
            r = E.depth_regression(logits[None][:, :, rows], pl, inv)
            e_depth, e_std = k2_bar(r)
            _stat("frame K2 depth", *_check(outs[0][None][:, rows], r["depth"], e_depth, f"{wl} frame depth"))
            _stat("frame K2 std", *_check(outs[1][None][:, rows], r["std"], e_std, f"{wl} frame std"))
            n_regr += 1
    assert n_regr >= 2
