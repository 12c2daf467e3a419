"""ORACLE — TEST INFRASTRUCTURE ONLY.  Float64 restatement of the ENeRF cascade kernels of libbmv on any torch device:
K1 (bmv_cost_volume_var, bmv_cost_volume_var_multi), a3 (bmv_depth_planes_first, bmv_depth_planes_next) and K2
(bmv_depth_regression).

oracle/enerf_oracle.py restates the reference operation by operation in float32 and is pinned bit-exactly to the golden
vectors; this module restates the same mathematics in float64, so that a kernel can be held to a bar derived from its own
fp32 rounding instead of to another fp32 path.  Besides the values, every function returns per element what such a bar
needs: the magnitude scale of every coordinate (its fp32 rounding error is a few ulps of it), the local slope of every
bilinear sample (how far a coordinate error moves the value), the sums of |terms| that bound the rounding of the
arithmetic, and the distance of every clamp decision to its threshold.  On the GPU it keeps frame-size references cheap;
`rows` / `plane_idx` restrict a volume to a subset.  tests/test_enerf_f64.py checks it against the golden vectors.
"""
import torch

F64 = torch.float64
# the fp32 value of 1e-6 that the reference (clamp_min on fp32 tensors) and the kernels (1e-6f) clamp to
CLAMP = float(torch.tensor(1e-6, dtype=torch.float32))


def _sample(img, ix, iy):
    """grid_sample(align_corners=True, padding_mode='zeros') of img (C,h,w) at pixel coordinates ix, iy (any shape P).
    -> value (C,*P); slope (C,*P): bound on |dv/dix| + |dv/diy| over the point's cell AND its eight neighbours (an error
    of a few ulps in the coordinate can carry the point across a cell edge, into a cell with another slope); absmag
    (C,*P) = sum over the four taps of |w f|.  A non-finite or huge coordinate samples 0 with slope 0, like ATen."""
    C, h, w = img.shape
    ok = torch.isfinite(ix) & torch.isfinite(iy) & (ix.abs() < 1e9) & (iy.abs() < 1e9)
    ix = torch.where(ok, ix, torch.full_like(ix, -10.0))      # -10: every tap of the 4x4 block is outside
    iy = torch.where(ok, iy, torch.full_like(iy, -10.0))
    x0, y0 = ix.floor(), iy.floor()
    fx, fy = ix - x0, iy - y0
    flat = img.to(F64).reshape(C, -1)
    P = ix.shape

    def tap(dx, dy):
        xi, yi = x0 + dx, y0 + dy
        valid = (xi >= 0) & (xi <= w - 1) & (yi >= 0) & (yi <= h - 1)
        idx = (yi.clamp(0, h - 1) * w + xi.clamp(0, w - 1)).long().reshape(-1)
        return flat[:, idx].reshape(C, *P) * valid.to(F64)

    rows = [[tap(dx, dy) for dx in (-1, 0, 1, 2)] for dy in (-1, 0, 1, 2)]
    f00, f01, f10, f11 = rows[1][1], rows[1][2], rows[2][1], rows[2][2]
    val = (1 - fy) * ((1 - fx) * f00 + fx * f01) + fy * ((1 - fx) * f10 + fx * f11)
    absmag = (1 - fy) * ((1 - fx) * f00.abs() + fx * f01.abs()) + fy * ((1 - fx) * f10.abs() + fx * f11.abs())
    sx = torch.zeros_like(val)
    sy = torch.zeros_like(val)
    for r in range(4):
        for c in range(3):
            sx = torch.maximum(sx, (rows[r][c + 1] - rows[r][c]).abs())
            sy = torch.maximum(sy, (rows[c + 1][r] - rows[c][r]).abs())
    return val, sx + sy, absmag


def cost_volume_var(feats, views, proj, planes, rows=None, plane_idx=None, hw=None):
    """K1: the plane-sweep variance volume of one chain (reference lib/networks/enerf/utils.py:57-95 homo_warp and
    :324-351 build_feature_volume), float64.
    feats (N,C,Hs,Ws) any dtype / layout; views: the S view ids of the chain; proj (N,3,4) indexed by view id; planes
    (D,h,w) per pixel or (D,) shared (then hw = (h, w)); rows / plane_idx: optional subsets (lists of indices).
    Per voxel (x, y, d): cam = R @ (x, y, 1) + t / d, cz clamped to >= 1e-6, the source pixel (cam.x / cz, cam.y / cz)
    (the reference's normalise to [-1, 1] and grid_sample's unnormalise cancel exactly), bilinear zeros-padding sample;
    variance = sum(f^2) / S - mean^2.
    Returns a dict, D' planes and R' rows:
      var (C,D',R',w); mean, sq (C,D',R',w): mean and sum(f^2) / S;
      feat, slope, absmag (S,C,D',R',w): the samples, their local slope (see _sample) and sum |w f|;
      coord (S,D',R',w): magnitude scale of the rounding error of the source pixel coordinates;
      cz (S,D',R',w) unclamped, cz_mag (S,D',R',w) the magnitude scale of its rounding (sum of |terms|)."""
    dev = feats.device
    N, C, Hs, Ws = feats.shape
    proj = proj.to(F64)
    planes = planes.to(F64)
    if planes.dim() == 1:
        h, w = hw
        planes = planes.view(-1, 1, 1).expand(-1, h, w)
    D, h, w = planes.shape
    pidx = torch.arange(D, device=dev) if plane_idx is None else torch.as_tensor(plane_idx, device=dev)
    ridx = torch.arange(h, device=dev) if rows is None else torch.as_tensor(rows, device=dev)
    dep = planes[pidx][:, ridx]                                        # (D',R',w)
    y = ridx.to(F64).view(1, -1, 1)
    x = torch.arange(w, device=dev, dtype=F64).view(1, 1, -1)
    out = {k: [] for k in ("feat", "slope", "absmag", "coord", "cz", "cz_mag")}
    for v in views:
        P = proj[int(v)]
        c = [P[r, 0] * x + P[r, 1] * y + P[r, 2] + P[r, 3] / dep for r in range(3)]
        mag = [(P[r, 0] * x).abs() + (P[r, 1] * y).abs() + P[r, 2].abs() + (P[r, 3] / dep).abs() for r in range(3)]
        czc = c[2].clamp_min(CLAMP)
        rx, ry = c[0] / czc, c[1] / czc
        rmax = torch.maximum(rx.abs(), ry.abs())
        # relative rounding of cam (a few ulps of the summed magnitudes) moves r = cam.xy / cz by (|dc| + |r| |dcz|) / cz;
        # the reciprocals and the normalise / unnormalise round trip add a few ulps of |r| and of the map size
        coord = (torch.maximum(mag[0], mag[1]) + rmax * mag[2]) / czc + rmax + max(Ws, Hs)
        coord = torch.where(torch.isfinite(coord), coord, torch.full_like(coord, float("inf")))
        f, s, a = _sample(feats[int(v)], rx, ry)
        for k, t in (("feat", f), ("slope", s), ("absmag", a), ("coord", coord), ("cz", c[2]), ("cz_mag", mag[2])):
            out[k].append(t)
    res = {k: torch.stack(t) for k, t in out.items()}
    S = len(views)
    mean = res["feat"].sum(0) / S
    sq = (res["feat"] ** 2).sum(0) / S
    res.update(var=sq - mean * mean, mean=mean, sq=sq)
    return res


def _lerp_planes(nr, fr, t, inv):
    """D hypotheses between nr and fr (true depths) at fractions t, uniform in depth or in disparity (inv), and the
    magnitude scale of their fp32 rounding: the sum of |terms| of every operation, propagated through the inversions."""
    if inv:
        dn, df = 1.0 / nr, 1.0 / fr
        disp = dn + t * (df - dn)
        v = 1.0 / disp
        mag = v.abs() + (dn.abs() + df.abs() + (t * (df - dn)).abs()) / disp ** 2
    else:
        v = nr + t * (fr - nr)
        mag = v.abs() + nr.abs() + (t * (fr - nr)).abs() + t * fr.abs()
    return v, mag


def depth_planes_first(near_far, D, depth_inv, t=None):
    """a3, level 0 (reference lib/networks/enerf/utils.py:103-111,149-153), float64.  near_far (2,) scene near / far;
    t: the D fractions (default torch.linspace(0, 1, D) in fp32, what the kernels read).
    -> planes (D,), mag (D,) rounding scale of each plane, nf (2,) = planes[0], planes[-1] (as disparities with
    depth_inv, after the 1e-6 clamp), nf_mag (2,)."""
    dev = near_far.device
    if t is None:
        t = torch.linspace(0.0, 1.0, D, device=dev, dtype=torch.float32)
    t = t.to(F64)
    nf = near_far.to(F64)
    v, mag = _lerp_planes(nf[0], nf[1], t, depth_inv)
    ends, emag = v[[0, -1]], mag[[0, -1]]
    if depth_inv:
        c = ends.clamp_min(CLAMP)
        ends, emag = 1.0 / c, emag / c ** 2 + 1.0 / c
    return dict(planes=v, mag=mag, nf=ends, nf_mag=emag)


def _upsample(m, h, w):
    """align_corners=True bilinear upsample of m (K,h0,w0) to (h,w) (ATen upsample_bilinear2d).
    -> value (K,h,w); slope (K,h,w) bound on |dv/dsrc_x| + |dv/dsrc_y| over the sample's cell and its neighbours;
    src (h,w) magnitude of the source coordinate, max(src_x, src_y); absmag (K,h,w) = sum of |w a| over the taps."""
    K, h0, w0 = m.shape
    m = m.to(F64)
    dev = m.device

    def axis(n_in, n_out):
        sc = (n_in - 1) / (n_out - 1) if n_out > 1 else 0.0
        src = torch.arange(n_out, device=dev, dtype=F64) * sc
        i0 = src.floor().clamp(max=n_in - 1)
        return src, i0.long(), src - i0

    sy, iy, ly = axis(h0, h)
    sx, ix, lx = axis(w0, w)

    def at(dy, dx):
        yy = (iy + dy).clamp(0, h0 - 1)
        xx = (ix + dx).clamp(0, w0 - 1)
        return m[:, yy][:, :, xx]

    blk = [[at(dy, dx) for dx in (-1, 0, 1, 2)] for dy in (-1, 0, 1, 2)]
    ly, lx = ly.view(1, -1, 1), lx.view(1, 1, -1)
    a, b, c, d = blk[1][1], blk[1][2], blk[2][1], blk[2][2]
    val = (1 - ly) * ((1 - lx) * a + lx * b) + ly * ((1 - lx) * c + lx * d)
    absmag = (1 - ly) * ((1 - lx) * a.abs() + lx * b.abs()) + ly * ((1 - lx) * c.abs() + lx * d.abs())
    s_x = torch.zeros_like(val)
    s_y = torch.zeros_like(val)
    for r in range(4):
        for q in range(3):
            s_x = torch.maximum(s_x, (blk[r][q + 1] - blk[r][q]).abs())
            s_y = torch.maximum(s_y, (blk[q + 1][r] - blk[q][r]).abs())
    src = torch.maximum(sy.view(-1, 1), sx.view(1, -1))
    return val, s_x + s_y, src, absmag


def depth_planes_next(depth, std, near_far, D, h, w, cur_inv, t=None):
    """a3, level >= 1 (reference lib/networks/enerf/utils.py:112-153 with the previous level in disparity), float64.
    depth, std (K,h0,w0); near_far (K,2,h0,w0) or shared (2,h0,w0), all disparities; t as in depth_planes_first.
    Upsample all four maps to (h,w) (align_corners), lo = min(d + s, nf0), hi = max(d - s, nf1) (the reference's
    where(), NaN-free inputs), near / far = 1 / lo, 1 / hi, D planes between them (uniform in disparity with cur_inv).
    Returns a dict: planes (K,D,h,w), nf (K,2,h,w) (planes[0], planes[-1]; as disparities with cur_inv), lo, hi
    (K,h,w); up_<name> = (value, slope, src, absmag) of each upsampled map (see _upsample)."""
    dev = depth.device
    K = depth.shape[0]
    if near_far.dim() == 3:
        near_far = near_far[None].expand(K, -1, -1, -1)
    if t is None:
        t = torch.linspace(0.0, 1.0, D, device=dev, dtype=torch.float32)
    t = t.to(F64).view(1, -1, 1, 1)
    up = {"depth": _upsample(depth, h, w), "std": _upsample(std, h, w),
          "nf0": _upsample(near_far[:, 0], h, w), "nf1": _upsample(near_far[:, 1], h, w)}
    dep, sd, n0, n1 = (up[k][0] for k in ("depth", "std", "nf0", "nf1"))
    lo = torch.minimum(dep + sd, n0)
    hi = torch.maximum(dep - sd, n1)
    nr, fr = (1.0 / lo)[:, None], (1.0 / hi)[:, None]
    planes, _ = _lerp_planes(nr, fr, t, cur_inv)
    ends = planes[:, [0, -1]]
    if cur_inv:
        ends = 1.0 / ends.clamp_min(CLAMP)
    res = {f"up_{k}": v for k, v in up.items()}
    res.update(planes=planes, nf=ends, lo=lo, hi=hi)
    return res


def depth_regression(logits, planes, depth_inv):
    """K2 (reference lib/networks/enerf/utils.py:722-727), float64.  logits (K,D,h,w); planes (K,D,h,w) or shared (D,).
    values v = planes, or 1 / max(planes, 1e-6) with depth_inv; p = softmax over D; depth = sum p v;
    var = sum p (v - depth)^2; std = sqrt(max(var, 1e-10)).
    Returns a dict: depth, var, std (K,h,w); prob, vals (K,D,h,w); dev_max (K,h,w) = max over the planes of |v - depth|;
    p_max (K,h,w) the largest probability; lse_dev (K,D,h,w) = max logit - logit (the argument of exp)."""
    lg = logits.to(F64)
    K, D, h, w = lg.shape
    pl = planes.to(F64)
    if pl.dim() == 1:
        pl = pl.view(1, D, 1, 1).expand(K, D, h, w)
    vals = 1.0 / pl.clamp_min(CLAMP) if depth_inv else pl
    prob = torch.softmax(lg, dim=1)
    depth = (prob * vals).sum(1)
    dv = vals - depth[:, None]
    var = (prob * dv * dv).sum(1)
    return dict(depth=depth, var=var, std=var.clamp_min(1e-10).sqrt(), prob=prob, vals=vals,
                dev_max=dv.abs().amax(1), p_max=prob.amax(1), lse_dev=lg.amax(1, keepdim=True) - lg)
