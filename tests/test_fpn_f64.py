"""oracle/fpn_f64.py (the float64 restatement of the feature-pyramid kernels) on the CPU: composed on the plan's folded
weights (BN folded, the 5x5 / stride-2 layers regrouped for space-to-depth) it reproduces the stock FeatureNet evaluated
in float64, and a row band of every operation equals the same rows of the whole-image result."""
import copy

import pytest
import torch

from boostmvsnerfs_b200.inference_plan import folded_copy
from boostmvsnerfs_b200.modules import FeatureNet
from oracle import fpn_f64 as P


def _net(seed=0):
    """FeatureNet with BN statistics that make the fold non-trivial: scales 0.5 .. 2, shifts of the order of the
    activations"""
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
    return net.eval()


@pytest.mark.parametrize("hw", [(32, 48), (68, 100)])
def test_oracle_on_folded_weights_is_the_stock_feature_net(hw):
    """68 x 100: the quarter map is odd-sized (17 x 25).  Folded in float64 (the plan's fold and regroup applied to a
    float64 copy), the composition is the stock network up to float64 rounding: 1e-12 of the output's range.  With the
    plan's own fp32 fold, the folded weights carry a few fp32 ulps each (the scale's sqrt and division, the products, the
    bias's difference): an fp32-class 2^-16 of the range, which the same weights rounded to fp16 exceed."""
    net = _net()
    x = torch.randn(2, 3, *hw)
    with torch.no_grad():
        ref = copy.deepcopy(net).double()(x.double())
    p64 = P.plan_params(folded_copy(copy.deepcopy(net).double(), torch.channels_last))
    assert tuple(p64["c10"][0].shape) == (16, 32, 3, 3) and tuple(p64["c20"][0].shape) == (32, 64, 3, 3)
    assert p64["c10"][0].dtype == torch.float64
    params = P.plan_params(folded_copy(net, torch.channels_last))
    got64, got = P.feature_net(p64, x), P.feature_net(params, x)
    p16 = P.feature_net({k: (w.half().float(), b) for k, (w, b) in params.items()}, x)
    for name, a64, a, b, c in zip(("quarter", "level 1", "level 2"), got64, got, ref, p16):
        assert a.shape == b.shape, name
        rng = float(b.abs().max())
        assert float((a64 - b).abs().max()) <= 1e-12 * rng, name
        assert float((a - b).abs().max()) <= 2.0 ** -16 * rng, name
        assert float((c - b).abs().max()) > 2.0 ** -16 * rng, name
    # the fold is not the identity: the unfolded conv weights give another result
    raw = {k: (v[0], v[1]) for k, v in params.items()}
    raw["stem0"] = (net.conv0[0].conv.weight.detach(), params["stem0"][1])
    assert float((P.feature_net(raw, x)[0] - ref[0]).abs().max()) > 1e-3 * float(ref[0].abs().max())


def _fields(seed, N=2, H=20, W=28):
    g = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=g)
    return dict(x3=r(N, 3, H, W), x8=r(N, 8, H, W), x16=r(N, 16, H // 2, W // 2), prev=r(N, 32, H // 2, W // 2),
                w33=r(8, 3, 3, 3) * 0.3, w88=r(8, 8, 3, 3) * 0.2, b8=r(8), w3216=r(16, 32, 3, 3) * 0.1, b16=r(16),
                w1616=r(16, 16, 3, 3) * 0.1, wtop=r(16, 16), lat=r(32, 8), b32=r(32), ws=r(8, 32, 3, 3) * 0.1)


def _same(band_res, full_res, r0, r1, what):
    for k in ("val", "abs", "dw", "err"):
        if k in full_res:
            a, b = band_res[k], full_res[k][..., r0:r1, :]
            assert a.shape == b.shape, (what, k)
            assert torch.allclose(a, b, rtol=1e-12, atol=1e-12), (what, k, float((a - b).abs().max()))


@pytest.mark.parametrize("rows", [(0, 3), (5, 13), (17, 20), (0, 20)])
def test_row_band_equals_the_same_rows_of_the_whole_image(rows):
    f = _fields(3)
    r0, r1 = rows
    H = 20
    e = lambda m: m["abs"] * 1e-3
    full = P.stem(f["x3"], f["w33"], f["b8"], f["w88"], f["b8"], mid_err=e)
    _same(P.stem(f["x3"], f["w33"], f["b8"], f["w88"], f["b8"], rows, mid_err=e), full, r0, r1, "stem")
    err = f["x8"].abs().double() * 1e-3
    full = P.conv3x3(f["x8"], f["w88"], f["b8"], relu=True, x_err=err)
    _same(P.conv3x3(f["x8"], f["w88"], f["b8"], rows, relu=True, x_err=err), full, r0, r1, "conv3x3")
    # space-to-depth: the output has H / 2 rows
    h0, h1 = r0 // 2, max(r1 // 2, r0 // 2 + 1)
    full = P.conv3x3(f["x8"], f["w3216"], f["b16"], relu=True, s2d=True)
    _same(P.conv3x3(f["x8"], f["w3216"], f["b16"], (h0, h1), relu=True, s2d=True), full, h0, h1, "s2d")
    full = P.conv3x3_top(f["x16"], f["w1616"], f["b16"], f["wtop"], f["b16"])
    part = P.conv3x3_top(f["x16"], f["w1616"], f["b16"], f["wtop"], f["b16"], (h0, h1))
    _same(part, full, h0, h1, "conv3x3_top")
    for k in ("prop_abs", "prop_dw"):
        assert torch.allclose(part[k], full[k][..., h0:h1, :], rtol=1e-12, atol=1e-12)
    full = P.topdown_smooth(f["prev"], f["x8"], f["lat"], f["b32"], f["ws"], f["b8"], mid_err=lambda m: m["lat"]["abs"] * 1e-3)
    part = P.topdown_smooth(f["prev"], f["x8"], f["lat"], f["b32"], f["ws"], f["b8"], rows,
                            mid_err=lambda m: m["lat"]["abs"] * 1e-3)
    _same(part, full, r0, r1, "topdown_smooth")
    _same(part["mid"], full["mid"], r0, r1, "topdown mid")
    for k, a in part["mid"]["up"].items():
        assert torch.allclose(a, full["mid"]["up"][k][..., r0:r1, :], rtol=1e-12, atol=1e-12), k
    assert full["val"].shape[-2] == H


@pytest.mark.parametrize("reach", [0.0, 0.02, 0.2])
def test_upsample_value_and_slope(reach):
    """up2x's value is ATen's align_corners upsample.  Its slopes bound the change of the value when the source coordinates
    move by up to reach * src on each axis, in any direction, also where that carries the point into the next cell."""
    g = torch.Generator().manual_seed(5)
    prev = torch.randn(1, 2, 9, 13, generator=g, dtype=torch.float64)
    H, W = 18, 26
    up = P.up2x(prev, H, W, reach=reach)
    ref = torch.nn.functional.interpolate(prev, size=(H, W), mode="bilinear", align_corners=True)
    assert torch.allclose(up["val"], ref, rtol=1e-14, atol=1e-14)
    assert bool((up["absmag"] >= up["val"].abs() - 1e-14).all())
    assert float(up["src_x"].max()) == pytest.approx(12.0) and float(up["src_y"].max()) == pytest.approx(8.0)

    def sample(yy, xx):
        gy = yy / (prev.shape[-2] - 1) * 2 - 1
        gx = xx / (prev.shape[-1] - 1) * 2 - 1
        grid = torch.stack(torch.broadcast_tensors(gx, gy), -1)[None]
        return torch.nn.functional.grid_sample(prev, grid, mode="bilinear", align_corners=True, padding_mode="border")
    sy, sx = up["src_y"], up["src_x"]
    crossed = 0
    for fy, fx in ((1, 0), (-1, 0), (0, 1), (0, -1), (1, 1), (-1, 1), (1, -1), (-1, -1), (0.5, -0.3)):
        dy, dx = fy * reach * sy, fx * reach * sx
        yy, xx = (sy + dy).clamp(0, 8), (sx + dx).clamp(0, 12)
        crossed += int(((yy.floor() != sy.floor()) | (xx.floor() != sx.floor())).sum())
        moved = sample(yy, xx)
        bound = up["slope_x"] * (xx - sx).abs() + up["slope_y"] * (yy - sy).abs()
        assert bool(((moved - up["val"]).abs() <= bound + 1e-12).all()), (fy, fx)
    assert (crossed > 0) == (reach > 0)
