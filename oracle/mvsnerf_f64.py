"""ORACLE — TEST INFRASTRUCTURE ONLY.  Float64 restatement of the MVSNeRF kernels of libbmv on any torch device:
K1b (bmv_cost_volume_var_img), the K3b row (bmv_mvs_march_fetch) and the 6x128 MLP.

oracle/mvsnerf_oracle.py restates the reference operation by operation in float32 and is pinned bit-exactly to the
golden vectors; this module restates the same mathematics in float64, so that a kernel can be held to a bar derived
from its own fp32 rounding instead of to another fp32 path.  Besides the values it returns, per element, what such a
bar needs: the distance of every in-mask / visibility decision to its threshold (a sample that close may flip under
fp32 rounding), the magnitude scale of every sampling coordinate (its fp32 rounding error is a few ulps of it) and the
local slope of every bilinear / trilinear sample (how far a coordinate error moves the value).
tests/test_mvsnerf_f64.py checks it against the golden vectors on the CPU.
"""
import torch

F64 = torch.float64


def _bilinear(img, ix, iy, border):
    """grid_sample(align_corners=True) at pixel coordinates ix, iy (any shape S) of img (C,h,w), float64.
    border=False: zeros padding (a tap outside the image contributes 0; a non-finite or huge coordinate gives 0);
    border=True: coordinates clamped into the image first.
    -> value (C,*S), slope (C,*S) = bound on |dv/dix| + |dv/diy| around the point, absmag (C,*S) = sum of |w f| over the taps."""
    C, h, w = img.shape
    if border:
        ix = ix.clamp(0, w - 1)
        iy = iy.clamp(0, h - 1)
    ok = torch.isfinite(ix) & torch.isfinite(iy) & (ix.abs() < 1e9) & (iy.abs() < 1e9)
    ix = torch.where(ok, ix, torch.zeros_like(ix))
    iy = torch.where(ok, iy, torch.zeros_like(iy))
    x0, y0 = ix.floor(), iy.floor()
    fx, fy = ix - x0, iy - y0
    flat = img.reshape(C, -1)
    taps = []
    for dy in (0, 1):
        for dx in (0, 1):
            xi, yi = x0 + dx, y0 + dy
            valid = ok & (xi >= 0) & (xi <= w - 1) & (yi >= 0) & (yi <= h - 1)
            idx = (yi.clamp(0, h - 1) * w + xi.clamp(0, w - 1)).long().reshape(-1)
            f = flat[:, idx].reshape(C, *ix.shape) * valid.to(F64)
            taps.append(f)
    f00, f01, f10, f11 = taps
    wx = (1 - fx, fx)
    wy = (1 - fy, fy)
    val = wy[0] * (wx[0] * f00 + wx[1] * f01) + wy[1] * (wx[0] * f10 + wx[1] * f11)
    slope = torch.maximum((f01 - f00).abs(), (f11 - f10).abs()) + torch.maximum((f10 - f00).abs(), (f11 - f01).abs())
    absmag = (wy[0] * (wx[0] * f00.abs() + wx[1] * f01.abs()) + wy[1] * (wx[0] * f10.abs() + wx[1] * f11.abs()))
    return val, slope, absmag


def _mask_margin(gx, gy):
    """strict -1 < g < 1 in-mask test and the distance of the decision to its threshold (grid units)."""
    inside = (gx > -1) & (gx < 1) & (gy > -1) & (gy < 1)
    margin = torch.minimum(torch.minimum((gx - 1).abs(), (gx + 1).abs()), torch.minimum((gy - 1).abs(), (gy + 1).abs()))
    margin = torch.where(torch.isfinite(margin), margin, torch.full_like(margin, float("inf")))
    return inside, margin


def cost_volume_var_img(feats, imgs_small, views, proj, planes, pad=24, plane_idx=None):
    """K1b: the 41-channel MVSNeRF cost volume of one chain (reference lib/networks/mvsnerf/network.py:887-942 with
    utils.py:580-630 homo_warp), float64.
    feats (N,C,h,w), imgs_small (N,3,h,w), views: the triple (views[0] = reference), proj (V,3,4) in triple order,
    planes (D,); plane_idx: optional subset of the planes (a list of indices) to evaluate.
    Per voxel (x, y) = (xp - pad, yp - pad) and plane depth d: cam = P[:, :3] @ (x, y, 1) + P[:, 3] / d with NO clamp on
    cam.z; g = (cam.xy / cam.z) / ((w-1)/2, (h-1)/2) - 1; bilinear zeros-padding taps at ((g+1)/2)(w-1, h-1); a source view
    is counted inside on the strict -1 < g < 1 test.  Variance = sum(f^2)/n - (sum(f)/n)^2 over ALL views (a view outside
    samples zeros), n = 1 + the number of source views inside.  Reference-image colour in the border is 0.
    Returns a dict:
      vol (3V+C, D', hp, wp); inside (V-1, D', hp, wp) bool; margin (V-1, D', hp, wp) distance of g to the mask boundary;
      cz (V-1, D', hp, wp); coord (V-1, D', hp, wp) magnitude scale of the rounding error of the pixel coordinates;
      feat / feat_slope / feat_absmag (V-1, C, D', hp, wp), img_slope / img_absmag (V-1, 3, D', hp, wp) of the source
      samples; ref_feat (C, 1, hp, wp) reference features (0 in the border); count (D', hp, wp) = n."""
    dev = feats.device
    feats, imgs_small, proj, planes = feats.to(F64), imgs_small.to(F64), proj.to(F64), planes.to(F64)
    N, C, h, w = feats.shape
    V = len(views)
    if plane_idx is not None:
        planes = planes[torch.as_tensor(plane_idx, device=dev)]
    D = planes.numel()
    hp, wp = h + 2 * pad, w + 2 * pad
    ys = torch.arange(hp, device=dev, dtype=F64) - pad
    xs = torch.arange(wp, device=dev, dtype=F64) - pad
    y, x = torch.meshgrid(ys, xs, indexing="ij")
    x, y = x[None].expand(D, hp, wp), y[None].expand(D, hp, wp)
    dep = planes.view(D, 1, 1).expand(D, hp, wp)
    in_ref = (x >= 0) & (x < w) & (y >= 0) & (y < h)
    r0 = views[0]
    ref_feat = torch.zeros((C, 1, hp, wp), device=dev, dtype=F64)
    ref_feat[:, 0, pad:pad + h, pad:pad + w] = feats[r0]
    ref_img = torch.zeros((3, 1, hp, wp), device=dev, dtype=F64)
    ref_img[:, 0, pad:pad + h, pad:pad + w] = imgs_small[r0]
    vol = torch.zeros((3 * V + C, D, hp, wp), device=dev, dtype=F64)
    vol[:3] = ref_img.expand(3, D, hp, wp)
    s1 = ref_feat.expand(C, D, hp, wp).clone()
    s2 = s1 * s1
    count = torch.ones((D, hp, wp), device=dev, dtype=F64)
    out = {k: [] for k in ("inside", "margin", "cz", "coord", "feat", "feat_slope", "feat_absmag", "img_slope", "img_absmag")}
    for i in range(1, V):
        P = proj[i]
        terms = [P[r, 0] * x + P[r, 1] * y + P[r, 2] + P[r, 3] / dep for r in range(3)]
        mags = [(P[r, 0] * x).abs() + (P[r, 1] * y).abs() + P[r, 2].abs() + (P[r, 3] / dep).abs() for r in range(3)]
        cx, cy, cz = terms
        rx, ry = cx / cz, cy / cz
        gx = rx / ((w - 1) / 2.0) - 1
        gy = ry / ((h - 1) / 2.0) - 1
        inside, margin = _mask_margin(gx, gy)
        ix = (gx + 1) * 0.5 * (w - 1)
        iy = (gy + 1) * 0.5 * (h - 1)
        # relative rounding of cx, cy, cz (a few ulps of the summed magnitudes) moves r = c/cz by (|dc| + |r||dcz|)/|cz|,
        # the divisions and the (g+1)(w-1)/2 round trip add a few ulps of |r| + w
        coord = (torch.maximum(mags[0], mags[1]) + torch.maximum(rx.abs(), ry.abs()) * mags[2]) / cz.abs() \
            + torch.maximum(rx.abs(), ry.abs()) + max(w, h)
        coord = torch.where(torch.isfinite(coord), coord, torch.full_like(coord, float("inf")))
        fv, fs, fa = _bilinear(feats[views[i]], ix, iy, border=False)
        iv, isl, ia = _bilinear(imgs_small[views[i]], ix, iy, border=False)
        vol[3 * i:3 * i + 3] = iv
        s1 = s1 + fv
        s2 = s2 + fv * fv
        count = count + inside.to(F64)
        for k, v in (("inside", inside), ("margin", margin), ("cz", cz), ("coord", coord), ("feat", fv), ("feat_slope", fs),
                     ("feat_absmag", fa), ("img_slope", isl), ("img_absmag", ia)):
            out[k].append(v)
    m = s1 / count
    vol[3 * V:] = s2 / count - m * m
    res = {k: torch.stack(v) for k, v in out.items()}
    res.update(vol=vol, ref_feat=ref_feat, count=count, in_ref=in_ref)
    return res


def _project(pts, ext, K, W, H, pmag):
    """pts (...,3) world, pmag (...,3) magnitude scale of their rounding -> (u, v, qz, scale): u, v normalised by
    (W-1, H-1) as in the reference's get_ndc_coordinate; scale is the magnitude scale of the rounding error of u, v."""
    cam = pts @ ext[:3, :3].T + ext[:3, 3]
    camag = pmag @ ext[:3, :3].abs().T + ext[:3, 3].abs()
    q = cam @ K.T
    qmag = camag @ K.abs().T
    u = q[..., 0] / q[..., 2] / (W - 1)
    v = q[..., 1] / q[..., 2] / (H - 1)
    r = torch.maximum(u.abs() * (W - 1), v.abs() * (H - 1))
    scale = ((torch.maximum(qmag[..., 0], qmag[..., 1]) + r * qmag[..., 2]) / q[..., 2].abs() + r) / min(W - 1, H - 1)
    return u, v, q[..., 2], scale


def march_fetch_row(rays, z, views, src_exts, src_ixts, H, W, near, far, volume, rgb, pad=24, rgb_affine=(0.5, 0.5),
                    ndc=None):
    """The K3b row of bmv_mvs_march_fetch (reference lib/networks/mvsnerf/network.py:945-1001, utils.py:112-146 and
    300-383, renderer.py:111-137), float64.
    rays (R,8); z (R,S) the sample depths along the rays (ray param); views: the triple; src_exts (N,4,4), src_ixts
    (N,3,3) full resolution; volume (8,D,hp,wp); rgb (N,3,H,W) raw.  ndc: optional (R,S,3) coordinates at which to
    sample the volume and evaluate the positional encoding (default: the float64 NDC of the samples).
    Returns a dict:
      xyz (R,S,3); ndc (R,S,3), ndc_scale (R,S,3) magnitude scale of its rounding error; pe (R,S,60) = [sin(2^k ndc)
      k = 0..9, cos(...)] frequency-major; vox (R,S,8), vox_slope (R,S,8) bound on the sum over the axes of |d vox / d index|,
      vox_absmag (R,S,8) sum of |w f| over the corners; rgb (R,S,3,3) per view border-bilinear colour, rgb_slope
      (R,S,3,3) per pixel of coordinate; inside (R,S,3) strict in-mask bits, in_margin (R,S,3) their distance to the
      threshold (units of u, v), uv_scale (R,S,3) rounding scale of u, v; dir (R,S,3) view direction in the reference
      camera frame; vis_count (R,S) number of views with 0 <= u, v <= 1 and qz > 0, vis_margin (R,S) distance of that
      decision to its thresholds; row (R,S,86) = the MLP input."""
    dev = rays.device
    rays, z = rays.to(F64), z.to(F64)
    exts, ixts = src_exts.to(F64), src_ixts.to(F64)
    R, S = z.shape
    xyz = rays[:, None, :3] + rays[:, None, 3:6] * z[..., None]
    pmag = rays[:, None, :3].abs() + rays[:, None, 3:6].abs() * z.abs()[..., None]
    e0, k0 = exts[views[0]], ixts[views[0]]
    u, v, qz, uv0 = _project(xyz, e0, k0, W, H, pmag)
    qzmag = (pmag @ e0[:3, :3].abs().T + e0[:3, 3].abs()) @ k0[2].abs()
    ndc_scale = torch.stack([uv0, uv0, (qzmag + abs(near)) / (far - near) + 1], -1)
    dz = (qz - near) / (far - near)
    Wf, Hf = W / 4.0, H / 4.0
    v = v * Hf / (Hf + 2 * pad) + pad / (Hf + 2 * pad)
    u = u * Wf / (Wf + 2 * pad) + pad / (Wf + 2 * pad)
    own = torch.stack([u, v, dz], -1)
    nd = own if ndc is None else ndc.to(F64)
    freq = 2.0 ** torch.arange(10, device=dev, dtype=F64)
    arg = (nd[..., None, :] * freq[:, None]).reshape(R, S, 30)
    pe = torch.cat([torch.sin(arg), torch.cos(arg)], -1)
    # trilinear zeros-padding volume fetch at ndc (grid_sample align_corners=True on g = 2 ndc - 1)
    vol = volume.to(F64)
    Cv, Dv, hv, wv = vol.shape
    ix, iy, iz = nd[..., 0] * (wv - 1), nd[..., 1] * (hv - 1), nd[..., 2] * (Dv - 1)
    ok = torch.isfinite(ix) & torch.isfinite(iy) & torch.isfinite(iz) & (ix.abs() < 1e9) & (iy.abs() < 1e9) & (iz.abs() < 1e9)
    ix, iy, iz = (torch.where(ok, a, torch.zeros_like(a)) for a in (ix, iy, iz))
    x0, y0, z0 = ix.floor(), iy.floor(), iz.floor()
    fx, fy, fz = ix - x0, iy - y0, iz - z0
    flat = vol.reshape(Cv, -1)
    vox = torch.zeros((Cv, R, S), device=dev, dtype=F64)
    absmag = torch.zeros((Cv, R, S), device=dev, dtype=F64)
    corners = []
    for c in range(8):
        bx, by, bz = c & 1, (c >> 1) & 1, c >> 2
        xi, yi, zi = x0 + bx, y0 + by, z0 + bz
        valid = ok & (xi >= 0) & (xi <= wv - 1) & (yi >= 0) & (yi <= hv - 1) & (zi >= 0) & (zi <= Dv - 1)
        idx = ((zi.clamp(0, Dv - 1) * hv + yi.clamp(0, hv - 1)) * wv + xi.clamp(0, wv - 1)).long().reshape(-1)
        f = flat[:, idx].reshape(Cv, R, S) * valid.to(F64)
        wgt = (fx if bx else 1 - fx) * (fy if by else 1 - fy) * (fz if bz else 1 - fz)
        vox = vox + wgt * f
        absmag = absmag + wgt * f.abs()
        corners.append(f)
    # slope: the sum over the axes of the largest difference along that axis of the cell, per unit of grid index
    slope = torch.zeros_like(vox)
    for axis in (1, 2, 4):
        slope = slope + torch.stack([(corners[c | axis] - corners[c]).abs() for c in range(8) if not c & axis]).amax(0)
    # per view: border-bilinear colour of img * scale + shift and the strict in-mask
    img = rgb.to(F64) * rgb_affine[0] + rgb_affine[1]
    cols, cslopes, inside, in_margin, uv_scale = [], [], [], [], []
    vis_count = torch.zeros((R, S), device=dev, dtype=torch.int64)
    vis_margin = torch.full((R, S), float("inf"), device=dev, dtype=F64)
    for vi in views:
        uu, vv, qq, sc = _project(xyz, exts[vi], ixts[vi], W, H, pmag)
        gx, gy = uu * 2 - 1, vv * 2 - 1
        ins, mar = _mask_margin(gx, gy)
        inside.append(ins)
        in_margin.append(mar / 2)
        uv_scale.append(sc)
        val, sl, _ = _bilinear(img[vi], uu * (W - 1), vv * (H - 1), border=True)
        cols.append(val.permute(1, 2, 0))
        cslopes.append(sl.permute(1, 2, 0))
        vis = (uu >= 0) & (uu <= 1) & (vv >= 0) & (vv <= 1) & (qq > 0)
        vis_count += vis.long()
        vm = torch.stack([uu.abs(), (uu - 1).abs(), vv.abs(), (vv - 1).abs()]).amin(0)
        vm = torch.where(torch.isfinite(vm), vm, torch.full_like(vm, float("inf")))
        vis_margin = torch.minimum(vis_margin, vm)
    d = rays[:, 3:6] / rays[:, 3:6].norm(dim=-1, keepdim=True)
    vdir = (d @ e0[:3, :3].T)[:, None].expand(R, S, 3)
    colours = torch.stack(cols, 2)
    inside = torch.stack(inside, -1)
    row = torch.cat([nd, pe, vox.permute(1, 2, 0), torch.cat([colours, inside[..., None].to(F64)], -1).reshape(R, S, 12), vdir], -1)
    return dict(xyz=xyz, ndc=own, ndc_scale=ndc_scale, pe=pe, vox=vox.permute(1, 2, 0), vox_slope=slope.permute(1, 2, 0),
                vox_absmag=absmag.permute(1, 2, 0), rgb=colours,
                rgb_slope=torch.stack(cslopes, 2), inside=inside, in_margin=torch.stack(in_margin, -1),
                uv_scale=torch.stack(uv_scale, -1), dir=vdir, vis_count=vis_count, vis_margin=vis_margin, row=row)


def mlp(nerf, x):
    """MvsNerfMlp (the 6x128 Renderer_ours of reference lib/networks/mvsnerf/network.py:152-229) in float64 on a
    float64 copy of the module.  x (..., 86) -> (..., 4) = [rgb, alpha]."""
    import copy
    m = copy.deepcopy(nerf).to(device=x.device, dtype=F64)
    with torch.no_grad():
        return m(x.to(F64))
