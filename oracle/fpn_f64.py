"""ORACLE — TEST INFRASTRUCTURE ONLY.  Float64 restatement of the feature-pyramid operations of libbmv on any torch device:
the stem (bmv_fpn_stem), the 3x3 middle layers with the 5x5 / stride-2 layers as their space-to-depth regrouped 3x3 and
conv2.1 with the fused 1x1 top layer (bmv_conv2d_k3), the top-down step up2x(prev) + lat(x) + b (bmv_fpn_topdown, the
first half of bmv_fpn_topdown_smooth) and the smoothing convolution behind it.

Every function takes the tensors the kernel takes (weights unpacked: the packed buffers are pack_* of these) and returns,
besides the value, what a per-element error bar needs:
  abs  sum |w| |x| + |b| of a convolution (a float64 convolution of |x| with |w|): the magnitude its rounding scales with;
  dw   sum |w - fp16(w)| |x|: the exact effect of rounding the weights to fp16, as the tensor-core kernels do;
  err  sum |w| e_x for a bound e_x on the error of an intermediate the kernel stores and the layer consumes;
  up   of the upsample: the value, its slope along each axis (how far a coordinate error moves it: in the sample's
       cell, and in the neighbouring cell where the error can carry the point across the edge), the source coordinates
       and sum |w tap| over the four taps.
`rows = (r0, r1)` restricts an output to rows r0 .. r1 - 1 (inputs are read with their halo), so that references at
frame size stay cheap.  tests/test_fpn_f64.py checks the composition against the stock FeatureNet.
"""
import torch
import torch.nn.functional as F

F64 = torch.float64


def band(x, r0, r1):
    """rows r0 .. r1 - 1 of x (..., H, W) as float64, zero rows outside [0, H) (the convolutions' padding)"""
    H = x.shape[-2]
    a, b = max(r0, 0), min(r1, H)
    return F.pad(x[..., a:b, :].to(F64), (0, 0, a - r0, r1 - b))


def fp16_err(w):
    """|w - fp16(w)| of fp32 weights rounded to fp16 (round to nearest, as the packing and the kernels round)"""
    w32 = w.detach().float()
    return (w32.double() - w32.half().double()).abs()


def _rows(rows, H):
    return (0, H) if rows is None else rows


def _conv_band(xb, w, b, x_err=None):
    """3x3 / pad-1 convolution of a band that already holds its one-row halo (zero outside the image)."""
    w = w.detach().to(F64)
    xa = xb.abs()
    val = F.conv2d(xb, w, None if b is None else b.detach().to(F64), padding=(0, 1))
    wa = torch.cat([w.abs(), fp16_err(w).to(w.device)])
    m = F.conv2d(xa, wa, padding=(0, 1))
    co = w.shape[0]
    res = dict(val=val, abs=m[:, :co] + (0 if b is None else b.detach().to(F64).abs().view(1, -1, 1, 1)), dw=m[:, co:])
    if x_err is not None:
        res["err"] = F.conv2d(x_err, w.abs(), padding=(0, 1))
    return res


def space_to_depth(x):
    """(N, C, 2h, 2w) -> (N, 4C, h, w), channel order (py, px, c) (inference_plan.S2DConv5x5, fpn_stem's out_s2d)"""
    N, C, H, W = x.shape
    return x.reshape(N, C, H // 2, 2, W // 2, 2).permute(0, 3, 5, 1, 2, 4).reshape(N, 4 * C, H // 2, W // 2)


def conv3x3(x, w, b=None, rows=None, relu=False, s2d=False, x_err=None):
    """3x3 / pad-1 convolution (+bias, optional ReLU) of x (N,Cin,H,W); with s2d, x is the (N,Cin/4,2H,2W) input of a 5x5 /
    stride-2 / pad-2 layer and w its space-to-depth regrouped (Cout,Cin,3,3) weight (S2DConv5x5.weight).  x_err: a bound
    on the error of x (x's shape), propagated as err.  -> dict(val, abs, dw[, err]) on `rows` of the output; val is
    the ReLU'd value with relu (abs, dw and err are the pre-activation bounds: ReLU is 1-Lipschitz)."""
    H = x.shape[-2] // 2 if s2d else x.shape[-2]
    r0, r1 = _rows(rows, H)
    if s2d:
        xb = space_to_depth(band(x, 2 * r0 - 2, 2 * r1 + 2))
        eb = None if x_err is None else space_to_depth(band(x_err, 2 * r0 - 2, 2 * r1 + 2))
    else:
        xb = band(x, r0 - 1, r1 + 1)
        eb = None if x_err is None else band(x_err, r0 - 1, r1 + 1)
    res = _conv_band(xb, w, b, eb)
    if relu:
        res["val"] = res["val"].clamp_min(0)
    return res


def stem(x, w0, b0, w1, b1, rows=None, mid_err=None):
    """bmv_fpn_stem: relu(conv3x3(relu(conv3x3(x, w0) + b0), w1) + b1) of the image x (N,3,H,W).  The kernel stores the
    intermediate as fp16 and layer 2 reads it: mid_err(mid) maps the intermediate's dict (val, abs, dw of layer 1, on
    rows r0 - 1 .. r1 clamped to the image) to a bound on its stored error, returned propagated as err."""
    H = x.shape[-2]
    r0, r1 = _rows(rows, H)
    a, b = max(r0 - 1, 0), min(r1 + 1, H)
    mid = conv3x3(x, w0, b0, (a, b), relu=True)
    pad = lambda t: F.pad(t, (0, 0, a - (r0 - 1), (r1 + 1) - b))
    out = _conv_band(pad(mid["val"]), w1, b1, None if mid_err is None else pad(mid_err(mid)))
    out["val"] = out["val"].clamp_min(0)
    return out


def conv1x1(x, w, b=None):
    """1x1 convolution of x (N,Cin,R,W) with w (Cout,Cin[,1,1]) -> dict(val, abs, dw)"""
    w = w.detach().reshape(w.shape[0], -1)
    wd = w.to(F64)
    x = x.to(F64)
    val = torch.einsum("oc,nchw->nohw", wd, x)
    ab = torch.einsum("oc,nchw->nohw", wd.abs(), x.abs())
    if b is not None:
        bd = b.detach().to(F64).view(1, -1, 1, 1)
        val, ab = val + bd, ab + bd.abs()
    return dict(val=val, abs=ab, dw=torch.einsum("oc,nchw->nohw", fp16_err(w).to(x.device), x.abs()))


def conv3x3_top(x, w, b, w1, b1, rows=None):
    """bmv_conv2d_k3 with the fused top layer: conv1x1(relu(conv3x3(x, w) + b), w1) + b1.  The kernel rounds the ReLU'd
    32 channels to fp16 (they are A fragments of the 1x1 MMA).  -> dict(val, abs, dw of the 1x1 layer; inner: the 3x3
    layer's dict; prop_abs, prop_dw = sum |w1| (abs, dw of the 3x3 layer): its errors seen through the 1x1 layer)."""
    inner = conv3x3(x, w, b, rows, relu=True)
    res = conv1x1(inner["val"], w1, b1)
    w1a = w1.detach().reshape(w1.shape[0], -1).to(F64).abs()
    res["prop_abs"] = torch.einsum("oc,nchw->nohw", w1a, inner["abs"])
    res["prop_dw"] = torch.einsum("oc,nchw->nohw", w1a, inner["dw"])
    res["inner"] = inner
    return res


def up2x(prev, H, W, rows=None, reach=2.0 ** -22):
    """bilinear upsample (align_corners=True) of prev (N,C,Hp,Wp) to (H, W), rows `rows`.  -> dict(val, slope_x, slope_y,
    src_x, src_y, absmag): src_* are the source coordinates; slope_x bounds |dv/dsrc_x| (slope_y |dv/dsrc_y|) over the
    sample's own cell and, where the point lies within reach * src of a cell edge (a coordinate rounded in fp32 can cross
    it), over the neighbouring cell too; absmag = sum over the taps of |weight tap|."""
    N, C, Hp, Wp = prev.shape
    p = prev.to(F64)
    dev = p.device
    r0, r1 = _rows(rows, H)

    def axis(n_in, n_out, lo, hi):
        src = torch.arange(lo, hi, device=dev, dtype=F64) * ((n_in - 1) / (n_out - 1))
        i0 = src.floor().clamp(max=n_in - 1)
        frac = src - i0
        tol = reach * src + 1e-300
        return src, i0.long(), (i0 + 1).clamp(max=n_in - 1).long(), frac, {-1: frac <= tol, 0: frac == frac,
                                                                            1: frac >= 1 - tol}

    sy, iy0, iy1, ly, ny = axis(Hp, H, r0, r1)
    sx, ix0, ix1, lx, nx = axis(Wp, W, 0, W)
    ly, lx = ly.view(-1, 1), lx.view(1, -1)
    top, bot = p[:, :, iy0], p[:, :, iy1]
    a, b, c, d = top[..., ix0], top[..., ix1], bot[..., ix0], bot[..., ix1]
    val = (1 - ly) * ((1 - lx) * a + lx * b) + ly * ((1 - lx) * c + lx * d)
    absmag = (1 - ly) * ((1 - lx) * a.abs() + lx * b.abs()) + ly * ((1 - lx) * c.abs() + lx * d.abs())
    # per coarse cell (i, j): the larger of its two horizontal (vertical) tap differences bounds dv/dsrc_x (dv/dsrc_y)
    # everywhere in the cell, the derivative being a convex combination of the two
    dx = F.pad((p[..., 1:] - p[..., :-1]).abs(), (0, 1))
    dy = F.pad((p[..., 1:, :] - p[..., :-1, :]).abs(), (0, 0, 0, 1))
    cell_x = torch.maximum(dx, torch.cat([dx[..., 1:, :], dx[..., -1:, :] * 0], -2))
    cell_y = torch.maximum(dy, torch.cat([dy[..., 1:], dy[..., -1:] * 0], -1))
    slope_x = torch.zeros_like(val)
    slope_y = torch.zeros_like(val)
    for di in (-1, 0, 1):
        ri = (iy0 + di).clamp(0, Hp - 1)
        for dj in (-1, 0, 1):
            cj = (ix0 + dj).clamp(0, Wp - 1)
            ok = (ny[di].view(-1, 1) & nx[dj].view(1, -1)).to(F64)
            slope_x = torch.maximum(slope_x, cell_x[:, :, ri][..., cj] * ok)
            slope_y = torch.maximum(slope_y, cell_y[:, :, ri][..., cj] * ok)
    shape = val.shape[-2:]
    return dict(val=val, slope_x=slope_x, slope_y=slope_y, src_x=sx.view(1, -1).expand(shape),
                src_y=sy.view(-1, 1).expand(shape), absmag=absmag)


def topdown(prev, lat_in, w, b, rows=None):
    """up2x(prev) + conv1x1(lat_in, w) + b (bmv_fpn_topdown, the `mid` of bmv_fpn_topdown_smooth) on `rows`.
    -> dict(val, up = up2x's dict, lat = conv1x1's dict)"""
    H, W = lat_in.shape[-2:]
    r0, r1 = _rows(rows, H)
    up = up2x(prev, H, W, (r0, r1))
    lat = conv1x1(band(lat_in, r0, r1), w, b)
    return dict(val=up["val"] + lat["val"], up=up, lat=lat)


def topdown_smooth(prev, lat_in, w, b, ws, bs, rows=None, mid_err=None):
    """bmv_fpn_topdown_smooth: out = conv3x3(mid, ws) + bs with mid = topdown(prev, lat_in, w, b).  The kernel keeps mid
    as fp16 for the convolution: mid_err(mid) maps topdown's dict (rows r0 - 1 .. r1 clamped to the image) to a bound
    on that operand's error, propagated as out's err.  -> dict(val, abs, dw[, err], mid = topdown's dict on `rows`)"""
    H = lat_in.shape[-2]
    r0, r1 = _rows(rows, H)
    a, b_ = max(r0 - 1, 0), min(r1 + 1, H)
    m = topdown(prev, lat_in, w, b, (a, b_))
    pad = lambda t: F.pad(t, (0, 0, a - (r0 - 1), (r1 + 1) - b_))
    out = _conv_band(pad(m["val"]), ws, bs, None if mid_err is None else pad(mid_err(m)))
    lo, hi = r0 - a, r0 - a + (r1 - r0)
    cut = lambda t: t[..., lo:hi, :]
    out["mid"] = dict(val=cut(m["val"]), up={k: cut(v) for k, v in m["up"].items()}, lat={k: cut(v) for k, v in m["lat"].items()})
    return out


# ------------------------------------------------------------------------------------------ the whole pyramid
def plan_params(fpn):
    """The weights the FeatureNet plan hands to the kernels, from a folded channels-last copy
    (inference_plan.folded_copy(net, torch.channels_last): BN folded, the 5x5 / stride-2 layers regrouped)."""
    cw = lambda m: (m.weight.detach(), m.bias.detach())
    return dict(stem0=cw(fpn.conv0[0].conv), stem1=cw(fpn.conv0[1].conv), c10=cw(fpn.conv1[0]), c11=cw(fpn.conv1[1].conv),
                c20=cw(fpn.conv2[0]), c21=cw(fpn.conv2[1].conv), top=cw(fpn.toplayer), lat1=cw(fpn.lat1),
                lat0=cw(fpn.lat0), smooth1=cw(fpn.smooth1), smooth0=cw(fpn.smooth0))


def feature_net(P, x):
    """The FeatureNet composed from this module's layers on plan_params P -> (quarter, level 1, level 2), float64."""
    Q = {k: (w.to(F64), b.to(F64)) for k, (w, b) in P.items()}
    x = x.to(F64)
    H, W = x.shape[-2:]
    c0 = stem(x, *Q["stem0"], *Q["stem1"])["val"]
    c1 = conv3x3(c0, *Q["c10"], relu=True, s2d=True)["val"]
    c1 = conv3x3(c1, *Q["c11"], relu=True)["val"]
    c2 = conv3x3(c1, *Q["c20"], relu=True, s2d=True)["val"]
    quarter = conv1x1(conv3x3(c2, *Q["c21"], relu=True)["val"], *Q["top"])["val"]
    l1 = topdown_smooth(quarter, c1, *Q["lat1"], *Q["smooth1"])
    l2 = topdown_smooth(l1["mid"]["val"], c0, *Q["lat0"], *Q["smooth0"])
    return quarter, l1["val"], l2["val"]
