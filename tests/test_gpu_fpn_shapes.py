"""The feature-pyramid kernels against the float64 restatement oracle/fpn_f64.py, at the image shapes of the C2, C4 and C5
workloads (N = 6 views of 544x960, 1088x1920, 992x1312) and at 68x100, whose quarter map is odd-sized (17x25):
  K9  bmv_fpn_stem (planar and channels-last images, fp32 / fp16 output, the rgb4 and space-to-depth by-products);
  K11 bmv_conv2d_k3, the four calls of the plan (conv1.0 and conv2.0 through space-to-depth, conv1.1, conv2.1 with the
      fused 1x1 top layer), each instantiation with 8- and 16-row tiles;
  K8  bmv_fpn_topdown_smooth (half- and full-resolution steps, fp16 / fp32 lateral input, fp32 / fp16 / both outputs);
      bmv_fpn_topdown (the strict-fp32 route);
and the FeatureNet plan as the network runs it, every call checked against float64 on that call's own inputs.

Bars are per element, from an error model of each kernel's arithmetic (u = 2^-24, h = 2^-11, written next to each bar):
  * an operand the kernel rounds to fp16: h |x| per element (+ 2^-25, half the fp16 subnormal spacing); weights rounded
    to fp16 enter exactly, as sum |w - fp16(w)| |x| (fpn_f64's dw), which is <= h sum |w| |x| for normal weights;
  * an fp16 store: h |y| + 2^-25;
  * fp32 accumulation on the tensor cores (mma.sync m16n8k16): ACC = 36 u * sum |w| |x| per MMA k-step.  The products
    are exact; the worst documented behaviour of the adder (the 16 products and the accumulator aligned to the largest
    exponent and truncated to fp32 precision, then normalised with truncation) loses < 2 u * max |term| <= 2 u sum |terms|
    on each of the 17 terms and 2 u on the result: 36 u.  The accumulator holds the bias and all earlier k-steps, so
    sum |terms| <= sum |w| |x| + |b| = fpn_f64's abs, and each k-step adds at most 36 u * abs.
Every kernel test shows that its bar rejects deliberately wrong references (a one-pixel shift of an input, a swapped pair
of output channels, dy/dx-transposed 3x3 weights, the (py, px) order of the space-to-depth regroup swapped,
align_corners=False, the lateral without its lo part).  Run with -s to see the worst err / bar of each kernel and the
smallest rejected fraction of each sensitivity check."""
import pytest
import torch
import torch.nn.functional as F

from oracle import fpn_f64 as P

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
H16 = 2.0 ** -11
SUB = 2.0 ** -25
ACC = 36 * U
WORKLOADS = {"C2": (6, 544, 960), "C4": (6, 1088, 1920), "C5": (6, 992, 1312), "Q68": (6, 68, 100)}
STATS = {}
SENS = {}


def _stat(name, ratio, err):
    s = STATS.setdefault(name, [0.0, 0.0])
    s[0], s[1] = max(s[0], ratio), max(s[1], err)


def _sens(name, fraction, floor, what):
    SENS[name] = min(SENS.get(name, 1.0), float(fraction))
    assert fraction > floor, f"{what}: the bar rejects only {fraction:.3f} of a {name}"


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for k in sorted(STATS):
        print(f"\n[fpn] {k}: worst err/bar {STATS[k][0]:.3g}, max err {STATS[k][1]:.3g}", end="")
    for k in sorted(SENS):
        print(f"\n[fpn] sensitivity, {k}: rejected at >= {SENS[k]:.3f} of the elements", end="")
    print()


@pytest.fixture(scope="module")
def ops():
    from boostmvsnerfs_b200 import ops as _ops
    return _ops


def _check(got, ref, bar, what, name):
    err = (got.double() - ref).abs()
    bad = ~(err <= bar)
    n = int(bad.sum())
    assert n == 0, (f"{what}: {n}/{err.numel()} elements outside the bar; max err {float(err.max()):.3e}, "
                    f"worst at {tuple(int(i) for i in torch.nonzero(bad)[0])}")
    ratio = float(torch.where(bar > 0, err / bar, torch.where(err > 0, float('inf'), 0.0)).max())
    _stat(name, ratio, float(err.max()))


def _fail_fraction(got, wrong, bar, among=None):
    bad = (got.double() - wrong).abs() > bar
    return float(bad[among].double().mean()) if among is not None else float(bad.double().mean())


def _bands(H):
    """full-resolution references of C4 / C5 in row bands at full width: the first rows, rows around a multiple of 16 near
    the middle (8- and 16-row tile seams on both sides) and the last rows (the last tile, ragged for 16-row tiles)"""
    if H <= 544:
        return [(0, H)]
    m = (H // 2) // 16 * 16
    return [(0, 10), (m - 10, m + 10), (H - 12, H)]


def _cl(t):
    return t.contiguous(memory_format=torch.channels_last)


def _gen(seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return lambda *s: torch.randn(*s, device="cuda", generator=g)


def _weights(r, shape, scale, exact):
    w = r(*shape) * scale
    return w.half().float() if exact else w


def _swapped_fraction(got, ref, bar, among):
    """fraction of channels 0 and 1 (where `among`) at which the bar rejects the reference with the two swapped"""
    return _fail_fraction(got[:, :2], ref[:, [1, 0]], bar[:, :2], among[:, :2])


# ------------------------------------------------------------------------------------------ K9 stem
def stem_bar(x_rounded, fp16_out):
    """Layer 1 (K = 27 padded to 32: 2 k-steps) -> ReLU -> fp16 intermediate: its error is 2 ACC * abs + dw (+ h abs
    + 2^-25 sum |w0| when the image is rounded) + h |mid| + 2^-25 (the store); layer 2 (8 channels x 3 x 3 = 6 k-steps)
    adds 6 ACC * abs + dw and sees the intermediate's error through |w1| (fpn_f64's err)."""
    def mid_err(m, w0sum):
        e = 2 * ACC * m["abs"] + m["dw"] + H16 * m["val"].abs() + SUB
        return e + (H16 * m["abs"] + SUB * w0sum if x_rounded else 0)

    def bar(r):
        b = 6 * ACC * r["abs"] + r["dw"] + r["err"]
        return b + H16 * (r["val"].abs() + b) + SUB if fp16_out else b
    return mid_err, bar


def check_stem(out, x, w0, b0, w1, b1, x_rounded, what, name, rows_list, sensitivity=False):
    w0sum = w0.double().abs().sum((1, 2, 3)).view(1, -1, 1, 1)
    mid_err, bar_fn = stem_bar(x_rounded, out.dtype == torch.float16)
    for rows in rows_list:
        r = P.stem(x, w0, b0, w1, b1, rows, mid_err=lambda m: mid_err(m, w0sum))
        got = out[..., rows[0]:rows[1], :]
        bar = bar_fn(r)
        _check(got, r["val"], bar, f"{what} rows {rows}", name)
        if sensitivity:
            among = r["val"].abs() > 1e-2 * float(r["val"].abs().max())
            wrong = {"one-pixel image shift": P.stem(torch.roll(x, 1, -1), w0, b0, w1, b1, rows)["val"],
                     "transposed 3x3 weights": P.stem(x, w0.transpose(-1, -2), b0, w1.transpose(-1, -2), b1, rows)["val"]}
            for k, v in wrong.items():
                _sens(f"K9 stem: {k}", _fail_fraction(got, v, bar, among), 0.5, what)
            _sens("K9 stem: swapped output channels", _swapped_fraction(got, r["val"], bar, among), 0.5, what)


@pytest.mark.parametrize("mode", ["fp16_operands", "fp32_operands"])
@pytest.mark.parametrize("wl", list(WORKLOADS))
def test_stem_workload_shapes_vs_float64(ops, wl, mode):
    """Tiles of 8 rows x 64 columns: C2 full resolution is 68 x 15 tiles, C4 136 x 30, C5 124 x 20.5 (ragged last x
    tile), 68x100 8.5 x 1.56.  Planar input (as delivered) with fp32 output, the rgb4 copy and the space-to-depth copy;
    channels-last input with fp16 output."""
    from boostmvsnerfs_b200.mlp_pack import pack_conv2d_k3_c8
    N, H, W = WORKLOADS[wl]
    exact = mode == "fp16_operands"
    r = _gen(H + W + exact)
    x = r(N, 3, H, W)
    if exact:
        x = x.half().float()
    w0, b0 = _weights(r, (8, 3, 3, 3), 0.3, exact), r(8) * 0.1
    w1, b1 = _weights(r, (8, 8, 3, 3), 0.2, exact), r(8) * 0.1
    wf = pack_conv2d_k3_c8(w1)
    out, rgb4, z = ops.fpn_stem(x, w0, b0, wf, b1, want_rgb4=True, want_s2d=True)
    assert torch.equal(rgb4[..., :3], x.permute(0, 2, 3, 1)) and bool((rgb4[..., 3] == 0).all())
    assert torch.equal(z, _cl(P.space_to_depth(out)))
    name = f"K9 stem {mode}"
    check_stem(out, x, w0, b0, w1, b1, not exact, f"{wl} stem {mode} planar", name, _bands(H),
               sensitivity=(wl in ("C5", "Q68")))
    out16 = ops.fpn_stem(_cl(x), w0, b0, wf, b1, out_dtype=torch.float16)
    assert out16.dtype == torch.float16 and out16.is_contiguous(memory_format=torch.channels_last)
    check_stem(out16, x, w0, b0, w1, b1, not exact, f"{wl} stem {mode} channels-last fp16", name + " fp16 out", _bands(H))


# ------------------------------------------------------------------------------------------ K11 middle layers
# name: (space-to-depth input, Cin of the 3x3 as the kernel sees it, Cout, fused top layer, resolution divisor of the output)
K11 = {"conv1.0_s2d": (True, 32, 16, False, 2), "conv1.1": (False, 16, 16, False, 2),
       "conv2.0_s2d": (True, 64, 32, False, 4), "conv2.1_top": (False, 32, 32, True, 4)}


def _tiles16(N, h, w):
    return -(-w // 32) * -(-h // 16) * N


def _k11_batches(h, w):
    """N = 6, and an N on the other side of the launcher's switch to 16-row tiles (>= 900 tiles of 16 x 32), if any"""
    per = _tiles16(1, h, w)
    six = 6 * per >= 900
    other = (899 // per if six else -(-900 // per)) if per < 900 else None
    return [6] + ([other] if other else [])


def k11_bar(r, ksteps, fp16_out):
    """ksteps MMA k-steps per output (3 dy x 3 dx x Cin / 16); inputs fp16 (exact operands), weights rounded: dw."""
    b = ksteps * ACC * r["abs"] + r["dw"]
    return b + H16 * (r["val"].abs() + b) + SUB if fp16_out else b


def top_bar(r, w1sum):
    """conv2.1 (18 k-steps) -> ReLU -> fp16 A fragments -> 1x1 (32 channels: 2 k-steps): the 1x1's own 2 ACC * abs + dw,
    the rounding of its operands h * abs + 2^-25 sum |w1|, and conv2.1's 18 ACC abs + dw seen through |w1| (times 1 + h:
    the operands are rounded after that error)."""
    return (2 * ACC * r["abs"] + r["dw"] + H16 * r["abs"] + SUB * w1sum
            + (1 + H16) * (18 * ACC * r["prop_abs"] + r["prop_dw"]))


@pytest.mark.parametrize("mode", ["fp16_weights", "fp32_weights"])
@pytest.mark.parametrize("layer", list(K11))
@pytest.mark.parametrize("wl", list(WORKLOADS))
def test_conv2d_k3_workload_shapes_vs_float64(ops, wl, layer, mode):
    """The four calls of the plan at each workload's shapes, fp16 inputs as the plan stores them.  Tile arithmetic:
    16-row tiles when ceil(w / 32) * ceil(h / 16) * N >= 900.  Half resolution (conv1.x): C2 272x480 is 255 tiles per
    view (N = 6: 1530, 16-row; N = 3: 765, 8-row), C4 544x960 1020 per view (16-row at any N), C5 496x656 651 per view
    (21 x 31, ragged x: N = 6 16-row, N = 1 8-row), 68x100 34x50 6 per view (8-row; N = 150: 16-row).  Quarter
    resolution (conv2.x): C2 136x240 72 per view (N = 6: 432, 8-row; N = 13: 936, 16-row), C4 272x480 255 (N = 6: 1530,
    16-row; N = 3: 765, 8-row), C5 248x328 176 (11 x 16: ragged x, and 248 = 15.5 tiles of 16 rows -- the fused top layer
    ends on a partial tile; N = 6: 1056, 16-row; N = 5: 880, 8-row), 68x100 17x25 2 per view (odd; N = 450: 16-row)."""
    from boostmvsnerfs_b200.mlp_pack import pack_conv1x1_after, pack_conv2d_k3
    s2d, cin, cout, fuse, div = K11[layer]
    _, H, W = WORKLOADS[wl]
    h, w = H // div, W // div
    exact = mode == "fp16_weights"
    r = _gen(H + cin + cout + exact)
    wgt, b = _weights(r, (cout, cin, 3, 3), 0.1, exact), r(cout) * 0.1
    w1, b1 = _weights(r, (32, 32), 0.2, exact), r(32) * 0.1
    for N in _k11_batches(h, w):
        ty = 16 if _tiles16(N, h, w) >= 900 else 8
        shape = (N, cin // 4, 2 * h, 2 * w) if s2d else (N, cin, h, w)
        x = _cl(torch.relu(r(*shape)).half())
        what = f"{wl} {layer} {mode} N={N} ({ty}-row tiles)"
        name = f"K11 {layer} {mode} {ty}-row tiles"
        if fuse:
            got = ops.conv2d_k3(x, pack_conv2d_k3(wgt), b, 32, relu=True, wfrag1x1=pack_conv1x1_after(w1), bias1x1=b1)
            res = P.conv3x3_top(x, wgt, b, w1, b1)
            bar = top_bar(res, w1.double().abs().sum(1).view(1, -1, 1, 1))
            _check(got, res["val"], bar, what, name)
        else:
            ksteps = 9 * cin // 16
            for odt in (torch.float16, torch.float32):
                got = ops.conv2d_k3(x, pack_conv2d_k3(wgt), b, cout, relu=True, s2d=s2d, out_dtype=odt)
                assert got.is_contiguous(memory_format=torch.channels_last) and got.shape == (N, cout, h, w)
                res = P.conv3x3(x, wgt, b, relu=True, s2d=s2d)
                bar = k11_bar(res, ksteps, odt == torch.float16)
                _check(got, res["val"], bar, what + f" {odt}", name)
        if N != 6 or wl not in ("C5", "Q68"):
            continue
        among = res["val"].abs() > 1e-2 * float(res["val"].abs().max())
        wrong = {"one-pixel input shift": (torch.roll(x, 1, -1), wgt), "transposed 3x3 weights": (x, wgt.transpose(-1, -2))}
        if s2d:
            wrong["(py, px) regroup order swapped"] = (x, wgt.view(cout, 2, 2, cin // 4, 3, 3).transpose(1, 2).reshape(cout, cin, 3, 3))
        for k, (xx, ww) in wrong.items():
            v = (P.conv3x3_top(xx, ww, b, w1, b1) if fuse else P.conv3x3(xx, ww, b, relu=True, s2d=s2d))["val"]
            _sens(f"K11 {k}", _fail_fraction(got, v, bar, among), 0.5, what)
        _sens("K11 swapped output channels", _swapped_fraction(got, res["val"], bar, among), 0.5, what)


# ------------------------------------------------------------------------------------------ K8 fused top-down step
LAT_FUSED = 128 * U


def mid_bar(m, lat_coef):
    """`mid` = up2x(prev) + lat(x) + b in fp32 arithmetic.  Upsample: the source coordinate fl(fl((n_in - 1) / (n_out - 1))
    * dst) is two correctly rounded operations, off by at most 2 u (1 + u) src on each axis; that moves the value by at
    most the axis's slope (up2x: the sample's cell, and the neighbouring cell where the point lies within 4 u src of an
    edge) times the offset; the weights 1 - l and their products (3 u each) and the blend's FMAs / ATen's nested sums
    (<= 6 roundings) -> 10 u sum |w tap|.  Lateral: the
    strict kernel's Cin FMAs from the bias, (Cin + 3) u * abs; the fused kernel's tensor-core hi / lo split: the hi
    product's k-step (36 u), the operands' lo parts rounded to fp16 and the dropped lo * lo term (3 * 2^-22 = 48 u), the
    lo k-steps scaled by 2^-11 and the final FMA (< 8 u): 128 u * abs (+ 2^-26 for lo parts in the fp16 subnormals)."""
    up = m["up"]
    coord = 2 * U * (1 + U) * (up["src_x"] * up["slope_x"] + up["src_y"] * up["slope_y"])
    return coord + 10 * U * up["absmag"] + lat_coef * m["lat"]["abs"] + 2.0 ** -26


def k8_bars(fp16_out):
    """out = conv3x3(fp16(mid)) + b, 32 channels x 3 x 3 = 18 k-steps: 18 ACC * abs + dw, and mid's error (mid_bar) plus its
    fp16 rounding (h |mid| + 2^-25) seen through |w| (fpn_f64's err)."""
    def mid_err(m):
        e = mid_bar(m, LAT_FUSED)
        return e + H16 * (m["val"].abs() + e) + SUB

    def bar(r):
        b = 18 * ACC * r["abs"] + r["dw"] + r["err"]
        return b + H16 * (r["val"].abs() + b) + SUB if fp16_out else b
    return mid_err, bar


def check_k8(res_out, mid, out16, prev, lat_in, wl_, bl, ws, bs, what, rows_list, sensitivity=False):
    mid_err, bar32 = k8_bars(False)
    _, bar16 = k8_bars(True)
    for rows in rows_list:
        r = P.topdown_smooth(prev, lat_in, wl_, bl, ws, bs, rows, mid_err=mid_err)
        sl = (Ellipsis, slice(rows[0], rows[1]), slice(None))
        if res_out is not None:
            _check(res_out[sl], r["val"], bar32(r), f"{what} out rows {rows}", "K8 out")
        if out16 is not None:
            _check(out16[sl], r["val"], bar16(r), f"{what} fp16 out rows {rows}", "K8 fp16 out")
        if mid is not None:
            mb = mid_bar(r["mid"], LAT_FUSED)
            _check(mid[sl], r["mid"]["val"], mb, f"{what} mid rows {rows}", "K8 mid (fp32 class)")
        if not sensitivity:
            continue
        got = res_out[sl]
        bar = bar32(r)
        among = r["val"].abs() > 1e-2 * float(r["val"].abs().max())
        H, W = lat_in.shape[-2:]
        ac_false = F.interpolate(prev.double(), scale_factor=2, mode="bilinear", align_corners=False)

        def out_of(m):          # the smoothing conv of a whole-image wrong mid, on these rows
            return P.conv3x3(m, ws, bs, rows)["val"]
        lat_full = P.conv1x1(lat_in, wl_, bl)["val"]
        wrong = {"align_corners=False": out_of(ac_false + lat_full),
                 "one-pixel prev shift": P.topdown_smooth(torch.roll(prev, 1, -1), lat_in, wl_, bl, ws, bs, rows)["val"],
                 "one-pixel lateral shift": P.topdown_smooth(prev, torch.roll(lat_in, 1, -1), wl_, bl, ws, bs, rows)["val"],
                 "transposed 3x3 weights": P.topdown_smooth(prev, lat_in, wl_, bl, ws.transpose(-1, -2), bs, rows)["val"]}
        for k, v in wrong.items():
            _sens(f"K8 out: {k}", _fail_fraction(got, v, bar, among), 0.5, what)
        _sens("K8 out: swapped output channels", _swapped_fraction(got, r["val"], bar, among), 0.5, what)
        if mid is not None:
            gm = mid[sl]
            am = r["mid"]["val"].abs() > 1e-2 * float(r["mid"]["val"].abs().max())
            wm = {"align_corners=False": (ac_false + lat_full)[sl],
                  "one-pixel prev shift": P.topdown(torch.roll(prev, 1, -1), lat_in, wl_, bl, rows)["val"],
                  "one-pixel lateral shift": P.topdown(prev, torch.roll(lat_in, 1, -1), wl_, bl, rows)["val"]}
            if lat_in.dtype == torch.float32:
                # the lateral of the fp16 hi parts only (no lo correction)
                hi = P.topdown(prev, lat_in.half().float(), wl_.half().float(), bl, rows)["val"]
                wm["lateral without its lo part"] = hi
            for k, v in wm.items():
                _sens(f"K8 mid: {k}", _fail_fraction(gm, v, mb, am), 0.5, what)


# step: (Cin of the lateral input, Cout, write_mid, resolution divisor)
K8 = {"half": (16, 16, True, 2), "full": (8, 8, False, 1)}


@pytest.mark.parametrize("lat", ["fp16", "fp32"])
@pytest.mark.parametrize("step", list(K8))
@pytest.mark.parametrize("wl", list(WORKLOADS))
def test_fpn_topdown_smooth_workload_shapes_vs_float64(ops, wl, step, lat):
    """Tiles of 8 rows x 64 columns: the last x tile is partial at C2 half resolution (480 = 7.5 tiles), C5 full (1312 =
    20.5) and half (656 = 10.25), 68x100 (100 = 1.56, 50 = 0.78).  Outputs: fp32; fp32 + fp16 (want_half=True); fp16
    only (want_half='only').  The half step also writes `mid` (fp32 class: the hi / lo lateral split)."""
    from boostmvsnerfs_b200.mlp_pack import pack_conv2d_k3_c32
    cin, cout, write_mid, div = K8[step]
    N, H, W = WORKLOADS[wl]
    H, W = H // div, W // div
    r = _gen(H + W + cin + (lat == "fp16"))
    prev = _cl(r(N, 32, H // 2, W // 2))
    lat_in = _cl(torch.relu(r(N, cin, H, W)))
    lat_in = lat_in.half() if lat == "fp16" else lat_in
    wl_, bl = r(32, cin) * 0.3, r(32) * 0.1
    ws, bs = r(cout, 32, 3, 3) * 0.1, r(cout) * 0.1
    wf = pack_conv2d_k3_c32(ws)
    mid, out = ops.fpn_topdown_smooth(prev, lat_in, wl_, bl, wf, bs, cout, write_mid)
    bands = _bands(H)
    what = f"{wl} {step} {lat} lateral"
    check_k8(out, mid, None, prev, lat_in, wl_, bl, ws, bs, what, bands,
             sensitivity=(wl in ("C5", "Q68") and (step == "half" or wl == "Q68")))
    _, out_b, out16 = ops.fpn_topdown_smooth(prev, lat_in, wl_, bl, wf, bs, cout, write_mid, want_half=True)
    assert torch.equal(out_b, out)
    _, only16 = ops.fpn_topdown_smooth(prev, lat_in, wl_, bl, wf, bs, cout, write_mid, want_half="only")
    assert only16.dtype == torch.float16 and torch.equal(only16, out16)
    check_k8(None, None, out16, prev, lat_in, wl_, bl, ws, bs, what + " want_half", bands)


@pytest.mark.parametrize("step", list(K8))
@pytest.mark.parametrize("wl", list(WORKLOADS))
def test_fpn_topdown_strict_workload_shapes_vs_float64(ops, wl, step):
    """bmv_fpn_topdown (strict-fp32 route): one thread per (pixel, 4 channels), fp32 FMAs; bar: mid_bar with the
    (Cin + 3) u lateral term."""
    cin, _, _, div = K8[step]
    N, H, W = WORKLOADS[wl]
    H, W = H // div, W // div
    r = _gen(H + W + cin + 7)
    prev = _cl(r(N, 32, H // 2, W // 2))
    lat_in = _cl(torch.relu(r(N, cin, H, W)))
    wl_, bl = r(32, cin) * 0.3, r(32) * 0.1
    got = ops.fpn_topdown(prev, lat_in, wl_, bl)
    for rows in _bands(H):
        m = P.topdown(prev, lat_in, wl_, bl, rows)
        bar = mid_bar(m, (cin + 3) * U)
        g = got[..., rows[0]:rows[1], :]
        _check(g, m["val"], bar, f"{wl} {step} strict rows {rows}", "fpn_topdown (strict fp32)")
        if wl in ("C5", "Q68"):
            among = m["val"].abs() > 1e-2 * float(m["val"].abs().max())
            wrong = {"one-pixel prev shift": P.topdown(torch.roll(prev, 1, -1), lat_in, wl_, bl, rows)["val"],
                     "one-pixel lateral shift": P.topdown(prev, torch.roll(lat_in, 1, -1), wl_, bl, rows)["val"],
                     "align_corners=False": (F.interpolate(prev.double(), scale_factor=2, mode="bilinear", align_corners=False)
                                             + P.conv1x1(lat_in, wl_, bl)["val"])[..., rows[0]:rows[1], :]}
            for k, v in wrong.items():
                _sens(f"fpn_topdown: {k}", _fail_fraction(g, v, bar, among), 0.5, f"{wl} {step} strict")


# ------------------------------------------------------------------------------------------ the plan at each workload
def _feature_net(seed=0):
    """FeatureNet with BN statistics that make the fold non-trivial (as tests/test_fpn_f64.py)"""
    from boostmvsnerfs_b200.modules import FeatureNet
    torch.manual_seed(seed)
    net = FeatureNet()
    g = torch.Generator().manual_seed(seed + 1)
    for m in net.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            c = m.num_features
            m.running_mean.copy_(torch.randn(c, generator=g) * 0.3)
            m.running_var.copy_(torch.rand(c, generator=g) * 1.5 + 0.25)
            m.weight.data.copy_(torch.rand(c, generator=g) + 0.5)
            m.bias.data.copy_(torch.randn(c, generator=g) * 0.2)
    return net.eval().cuda()


FPN_OPS = ("fpn_stem", "conv2d_k3", "fpn_topdown_smooth", "fpn_topdown")
PLAN_RUNS = {"C2": [(False, False), (True, True)], "C4": [(True, False)], "C5": [(False, True)]}


def _record(ops, monkeypatch):
    calls = []

    def wrap(name, fn):
        def rec(*a, **kw):
            res = fn(*a, **kw)
            calls.append((name, a, kw, res))
            return res
        return rec
    for name in FPN_OPS:
        monkeypatch.setattr(ops, name, wrap(name, getattr(ops, name)))
    return calls


def _same(a, b):
    return a.data_ptr() == b.data_ptr() and a.shape == b.shape


@pytest.mark.parametrize("wl,side,half", [(wl, s, h) for wl, runs in PLAN_RUNS.items() for s, h in runs])
def test_plan_calls_vs_float64(ops, monkeypatch, wl, side, half):
    """FusedTopDownFPN (tensor_core_mid, side_topdown and emit_half_features as the network sets them) on 6 views of the
    workload's size.  Routing: the seven calls come in order, each packed weight buffer is pack_* of the independently
    folded module's weight, and each call reads what the earlier calls wrote (same storage), so the plan's outputs are
    the composition of the calls.  Each call's output is then checked against float64 on its own inputs with the kernel
    tests' bars.  (tests/test_fpn_f64.py shows that the same composition in float64 is the stock FeatureNet.  A bar for
    the plan against the stock network directly, propagated through the absolute network |w|, |b|, |x|, is 1e6 to 1e7
    times the outputs at this initialisation: it would reject nothing.)"""
    from boostmvsnerfs_b200.inference_plan import PlanCache, folded_copy
    from boostmvsnerfs_b200.mlp_pack import pack_conv1x1_after, pack_conv2d_k3, pack_conv2d_k3_c8, pack_conv2d_k3_c32
    N, H, W = WORKLOADS[wl]
    net = _feature_net()
    Pw = P.plan_params(folded_copy(net, torch.channels_last))
    plan = PlanCache().get("feature_net", net, torch.channels_last)
    assert plan.tensor_core_mid
    plan.side_topdown, plan.emit_half_features = side, half
    x = torch.rand(N, 3, H, W, device="cuda") * 2 - 1
    calls = _record(ops, monkeypatch)
    old = torch.backends.cudnn.allow_tf32
    try:
        torch.backends.cudnn.allow_tf32 = True
        with torch.no_grad():
            quarter, feat1, feat0 = plan(x)
        torch.cuda.synchronize()
    finally:
        torch.backends.cudnn.allow_tf32 = old
    assert [c[0] for c in calls] == ["fpn_stem"] + ["conv2d_k3"] * 4 + ["fpn_topdown_smooth"] * 2
    (_, sa, skw, (c0, _)), k10, k11, k20, k21, t1, t0 = calls
    # routing: weights
    eq = lambda a, b: torch.equal(a.detach().float(), b.detach().float().to(a.device))
    assert sa[0] is x and eq(sa[1], Pw["stem0"][0]) and eq(sa[2], Pw["stem0"][1]) and eq(sa[4], Pw["stem1"][1])
    assert torch.equal(sa[3], pack_conv2d_k3_c8(Pw["stem1"][0]).to(sa[3].device))
    for call, key in ((k10, "c10"), (k11, "c11"), (k20, "c20"), (k21, "c21")):
        assert torch.equal(call[1][1], pack_conv2d_k3(Pw[key][0]).to("cuda")) and eq(call[1][2], Pw[key][1]), key
    assert torch.equal(k21[2]["wfrag1x1"], pack_conv1x1_after(Pw["top"][0]).to("cuda")) and eq(k21[2]["bias1x1"], Pw["top"][1])
    for call, lat, sm in ((t1, "lat1", "smooth1"), (t0, "lat0", "smooth0")):
        a = call[1]
        assert eq(a[2], Pw[lat][0]) and eq(a[3], Pw[lat][1]) and eq(a[5], Pw[sm][1])
        assert torch.equal(a[4], pack_conv2d_k3_c32(Pw[sm][0]).to("cuda"))
    # routing: each call reads the earlier calls' outputs
    assert [k10[2].get("s2d"), k11[2].get("s2d", False), k20[2].get("s2d"), k21[2].get("s2d", False)] == [True, False, True, False]
    assert _same(k10[1][0], c0) and _same(k11[1][0], k10[3]) and _same(k20[1][0], k11[3]) and _same(k21[1][0], k20[3])
    assert _same(t1[1][0], k21[3]) and _same(t1[1][1], k11[3]) and _same(t0[1][1], c0) and _same(t0[1][0], t1[3][0])
    assert t1[1][7] is True and t0[1][7] is False and (t1[2].get("want_half") == "only") == half
    assert _same(quarter, k21[3]) and _same(feat1, t1[3][1]) and _same(feat0, t0[3][1])
    assert c0.dtype == k10[3].dtype == k11[3].dtype == k20[3].dtype == torch.float16 and (feat1.dtype == torch.float16) == half
    # each call against float64 on its own inputs
    check_stem(c0, x, *Pw["stem0"], Pw["stem1"][0], Pw["stem1"][1], True, f"plan {wl} stem", "plan K9 stem", _bands(H))
    for call, key, ksteps in ((k10, "c10", 18), (k11, "c11", 9), (k20, "c20", 36)):
        res = P.conv3x3(call[1][0], *Pw[key], relu=True, s2d=call[2].get("s2d", False))
        _check(call[3], res["val"], k11_bar(res, ksteps, True), f"plan {wl} {key}", f"plan K11 {key}")
    res = P.conv3x3_top(k21[1][0], *Pw["c21"], *Pw["top"])
    _check(quarter, res["val"], top_bar(res, Pw["top"][0].double().abs().sum((1, 2, 3)).view(1, -1, 1, 1)),
           f"plan {wl} conv2.1 + top", "plan K11 conv2.1_top")
    for call, lat, sm, out in ((t1, "lat1", "smooth1", feat1), (t0, "lat0", "smooth0", feat0)):
        a = call[1]
        mid = call[3][0]
        is16 = out.dtype == torch.float16
        check_k8(None if is16 else out, mid, out if is16 else None, a[0], a[1], *Pw[lat], *Pw[sm], f"plan {wl} {lat}",
                 _bands(a[1].shape[-2]))


def test_plan_strict_fp32_calls_vs_float64(ops, monkeypatch):
    """allow_tf32 = False at C2: cuDNN fp32 convolutions and bmv_fpn_topdown; both top-down calls against float64 on their
    own inputs with the fp32 bar, and the smoothing layers' inputs are those calls' outputs."""
    from boostmvsnerfs_b200.inference_plan import PlanCache, folded_copy
    N, H, W = WORKLOADS["C2"]
    net = _feature_net(1)
    Pw = P.plan_params(folded_copy(net, torch.channels_last))
    plan = PlanCache().get("feature_net", net, torch.channels_last)
    x = torch.rand(N, 3, H, W, device="cuda") * 2 - 1
    calls = _record(ops, monkeypatch)
    old = torch.backends.cudnn.allow_tf32
    try:
        torch.backends.cudnn.allow_tf32 = False
        with torch.no_grad():
            quarter, feat1, feat0 = plan(x)
    finally:
        torch.backends.cudnn.allow_tf32 = old
    assert [c[0] for c in calls] == ["fpn_topdown"] * 2
    (_, a1, _, half), (_, a0, _, full) = calls
    assert _same(a1[0], quarter) and _same(a0[0], half)
    for a, out, lat in ((a1, half, "lat1"), (a0, full, "lat0")):
        assert torch.equal(a[2], Pw[lat][0].to("cuda")) and torch.equal(a[3], Pw[lat][1].to("cuda"))
        m = P.topdown(a[0], a[1], *Pw[lat])
        _check(out, m["val"], mid_bar(m, (a[1].shape[1] + 3) * U), f"strict {lat}", "plan strict fpn_topdown")
