"""bmv_conv3d_k3 (tensor-core 3x3x3 convolution of the kept cost regularisers) against cuDNN fp32.

Two bars:  (1) with operands that are exactly representable in fp16 the kernel's only difference from an
fp32 convolution is summation order -> 1e-5 relative;  (2) with arbitrary fp32 operands the fp16 operand
rounding gives TF32-class error -> 2e-3 of the output scale (tolerances per north_star: 1e-2 wherever
reduced-precision operands are enabled)."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

SHAPES = [  # (N, Cin, Cout, D, H, W, bias, relu)
    (2, 16, 8, 8, 12, 64, True, True),
    (1, 16, 8, 5, 7, 45, True, True),        # ragged in every dimension
    (2, 32, 8, 16, 6, 40, True, True),
    (1, 32, 8, 9, 5, 33, False, False),
    (2, 8, 9, 8, 8, 64, False, False),       # merged output heads
    (1, 8, 9, 3, 9, 17, True, True),
    (1, 8, 16, 8, 4, 32, True, False),
    (2, 16, 16, 4, 8, 40, True, True),       # conv2 of the U-Nets
    (1, 16, 12, 3, 5, 19, False, False),
]


def _reference(x, w, b, relu):
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        y = torch.nn.functional.conv3d(x, w, b, padding=1)
    finally:
        torch.backends.cudnn.allow_tf32 = prev
    return torch.relu(y) if relu else y


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("exact_operands", [True, False])
def test_conv3d_k3_matches_cudnn(shape, exact_operands):
    from boostmvsnerfs_b200 import ops
    from boostmvsnerfs_b200.mlp_pack import pack_conv3d_k3
    N, Cin, Cout, D, H, W, bias, relu = shape
    g = torch.Generator().manual_seed(Cin * 100 + W)
    x = torch.randn((N, Cin, D, H, W), generator=g)
    w = torch.randn((Cout, Cin, 3, 3, 3), generator=g) * 0.1
    b = torch.randn(Cout, generator=g) if bias else None
    if exact_operands:
        x, w = x.half().float(), w.half().float()
    x = x.cuda().contiguous(memory_format=torch.channels_last_3d)
    w = w.cuda()
    b = b.cuda() if bias else None
    y = ops.conv3d_k3(x, pack_conv3d_k3(w), b, Cout, relu)
    ref = _reference(x, w, b, relu)
    assert y.shape == ref.shape and y.stride(1) == 1
    scale = ref.abs().max().item()
    tol = (1e-5 if exact_operands else 2e-3) * scale
    assert (y - ref).abs().max().item() <= tol, ((y - ref).abs().max().item(), scale)


@pytest.mark.parametrize("shape", [(2, 16, 8, 8, 64), (1, 16, 6, 10, 38), (1, 12, 5, 7, 33), (2, 16, 2, 2, 2)])
@pytest.mark.parametrize("exact_operands", [True, False])
def test_conv3d_k3_stride2_matches_cudnn(shape, exact_operands):
    from boostmvsnerfs_b200 import ops
    from boostmvsnerfs_b200.mlp_pack import pack_conv3d_k3
    N, Cout, D, H, W = shape
    g = torch.Generator().manual_seed(D * 10 + W)
    x = torch.randn((N, 8, D, H, W), generator=g)
    w = torch.randn((Cout, 8, 3, 3, 3), generator=g) * 0.1
    b = torch.randn(Cout, generator=g)
    if exact_operands:
        x, w = x.half().float(), w.half().float()
    x = x.cuda().contiguous(memory_format=torch.channels_last_3d)
    w, b = w.cuda(), b.cuda()
    y = ops.conv3d_k3(x, pack_conv3d_k3(w), b, Cout, True, stride=2)
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        ref = torch.relu(torch.nn.functional.conv3d(x, w, b, stride=2, padding=1))
    finally:
        torch.backends.cudnn.allow_tf32 = prev
    assert y.shape == ref.shape, (y.shape, ref.shape)
    scale = ref.abs().max().item()
    assert (y - ref).abs().max().item() <= (1e-5 if exact_operands else 2e-3) * scale
    # fp16 input (staged by TMA: one 9x9x66-voxel bulk copy per CTA) and fp16 output
    from boostmvsnerfs_b200 import _lib
    xh = x.half()
    yh = ops.conv3d_k3(xh, pack_conv3d_k3(w), b, Cout, True, stride=2)
    assert _lib.load().bmv_conv3d_k3_last_used_tma() == 1
    assert torch.equal(yh, ops.conv3d_k3(xh.float(), pack_conv3d_k3(w), b, Cout, True, stride=2))
    y16 = ops.conv3d_k3(xh, pack_conv3d_k3(w), b, Cout, True, stride=2, out_dtype=torch.float16)
    assert torch.equal(y16, yh.half())


def test_conv3d_k3_strided_output_and_errors():
    from boostmvsnerfs_b200 import ops
    from boostmvsnerfs_b200._lib import BmvError
    from boostmvsnerfs_b200.mlp_pack import pack_conv3d_k3
    x = torch.randn((1, 16, 4, 6, 20), device="cuda").half().float().contiguous(memory_format=torch.channels_last_3d)
    w = (torch.randn((8, 16, 3, 3, 3), device="cuda") * 0.1).half().float()
    big = torch.zeros((1, 12, 4, 6, 20), device="cuda").contiguous(memory_format=torch.channels_last_3d)
    ops.conv3d_k3(x, pack_conv3d_k3(w), None, 8, False, out=big[:, 2:10])       # channel slice of a wider volume
    ref = _reference(x, w, None, False)
    assert torch.allclose(big[:, 2:10], ref, atol=1e-5 * ref.abs().max().item())
    assert big[:, :2].abs().max().item() == 0 and big[:, 10:].abs().max().item() == 0
    # channel split: the merged heads write 8 feature channels and the depth logits to two tensors
    x8 = torch.randn((2, 8, 5, 6, 37), device="cuda").half().float().contiguous(memory_format=torch.channels_last_3d)
    w9 = (torch.randn((9, 8, 3, 3, 3), device="cuda") * 0.1).half().float()
    logits = torch.empty((2, 1, 5, 6, 37), device="cuda")
    feat = ops.conv3d_k3(x8, pack_conv3d_k3(w9), None, 9, False, out2=logits, split=8)
    ref9 = _reference(x8, w9, None, False)
    assert feat.shape == (2, 8, 5, 6, 37)
    assert torch.allclose(feat, ref9[:, :8], atol=1e-5 * ref9.abs().max().item())
    assert torch.allclose(logits, ref9[:, 8:], atol=1e-5 * ref9.abs().max().item())
    with pytest.raises(BmvError):
        ops.conv3d_k3(x.contiguous(), pack_conv3d_k3(w), None, 8, False)        # not channels-last
    with pytest.raises(ValueError):
        pack_conv3d_k3(torch.zeros(8, 24, 3, 3, 3))


@pytest.mark.parametrize("shape", [(2, 16, 8, 4, 8, 32), (1, 16, 8, 3, 5, 21), (2, 32, 16, 2, 6, 40), (1, 32, 16, 5, 3, 9)])
@pytest.mark.parametrize("exact_operands", [True, False])
@pytest.mark.parametrize("with_skip", [True, False])
def test_convT3d_k3s2_add_matches_cudnn(shape, exact_operands, with_skip):
    from boostmvsnerfs_b200 import ops
    from boostmvsnerfs_b200.mlp_pack import pack_convT3d_k3s2
    N, Cin, Cout, D, H, W = shape
    g = torch.Generator().manual_seed(Cin + W)
    x = torch.randn((N, Cin, D, H, W), generator=g)
    w = torch.randn((Cin, Cout, 3, 3, 3), generator=g) * 0.1
    b = torch.randn(Cout, generator=g)
    skip = torch.randn((N, Cout, 2 * D, 2 * H, 2 * W), generator=g)
    if exact_operands:
        x, w = x.half().float(), w.half().float()
    x = x.cuda().contiguous(memory_format=torch.channels_last_3d)
    w, b = w.cuda(), b.cuda()
    skip = skip.cuda().contiguous(memory_format=torch.channels_last_3d)
    y = ops.convT3d_k3s2_add(x, pack_convT3d_k3s2(w), b, Cout, skip=skip if with_skip else None)
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        ref = torch.nn.functional.conv_transpose3d(x, w, b, stride=2, padding=1, output_padding=1)
    finally:
        torch.backends.cudnn.allow_tf32 = prev
    if with_skip:
        ref = ref + skip
    assert y.shape == ref.shape and y.stride(1) == 1
    scale = ref.abs().max().item()
    tol = (1e-5 if exact_operands else 2e-3) * scale
    assert (y - ref).abs().max().item() <= tol, ((y - ref).abs().max().item(), scale)
    # fp16 output storage = the fp32 result rounded to fp16
    yh = ops.convT3d_k3s2_add(x, pack_convT3d_k3s2(w), b, Cout, skip=skip if with_skip else None, out_dtype=torch.float16)
    assert yh.dtype == torch.float16 and torch.equal(yh, y.half())
    # fp16 input / skip storage: same as the fp32 tensors holding the rounded values
    xh, sh = x.half(), skip.half()
    a = ops.convT3d_k3s2_add(xh, pack_convT3d_k3s2(w), b, Cout, skip=sh if with_skip else None)
    b_ = ops.convT3d_k3s2_add(xh.float(), pack_convT3d_k3s2(w), b, Cout, skip=sh.float() if with_skip else None)
    assert torch.equal(a, b_)


@pytest.mark.parametrize("minimal", [True, False])
def test_cost_reg_plan_tensor_core_convs_match_cudnn_tf32_class(minimal):
    """Whole regulariser: plan with libbmv convolutions vs the same plan on cuDNN fp32."""
    from boostmvsnerfs_b200.inference_plan import MergedHeadsCostReg, PlanCache
    from boostmvsnerfs_b200.modules import CostRegNet, MinCostRegNet
    torch.manual_seed(3)
    net = (MinCostRegNet(16) if minimal else CostRegNet(32)).eval().cuda()
    for m in net.modules():
        if isinstance(m, torch.nn.BatchNorm3d):
            m.running_mean.normal_(0, 0.1); m.running_var.uniform_(0.5, 1.5)
    plan = PlanCache().get("cr", net, torch.channels_last_3d)
    assert isinstance(plan, MergedHeadsCostReg)
    x = torch.rand((2, 16 if minimal else 32, 8, 32, 64), device="cuda").contiguous(memory_format=torch.channels_last_3d)
    prev = torch.backends.cudnn.allow_tf32
    try:
        torch.backends.cudnn.allow_tf32 = True
        with torch.no_grad():
            f_tc, d_tc = plan(x)
        torch.backends.cudnn.allow_tf32 = False
        with torch.no_grad():
            f_ref, d_ref = plan(x)
    finally:
        torch.backends.cudnn.allow_tf32 = prev
    for a, b in ((f_tc, f_ref), (d_tc, d_ref)):
        assert (a - b).abs().max().item() <= 1e-2 * b.abs().max().item()


# ------------------------------------------------------------------------------------------ fused FPN step
@pytest.mark.parametrize("cin,cout,hw", [(8, 8, (64, 96)), (16, 16, (34, 50)), (16, 8, (16, 130)), (8, 16, (10, 18))])
@pytest.mark.parametrize("write_mid", [True, False])
def test_fpn_topdown_smooth_vs_torch(cin, cout, hw, write_mid):
    from boostmvsnerfs_b200 import ops
    from boostmvsnerfs_b200.mlp_pack import pack_conv2d_k3_c32
    H, W = hw
    torch.manual_seed(cin + cout)
    prev = torch.randn(2, 32, H // 2, W // 2, device="cuda").contiguous(memory_format=torch.channels_last)
    lat_in = torch.randn(2, cin, H, W, device="cuda").contiguous(memory_format=torch.channels_last)
    lat = torch.nn.Conv2d(cin, 32, 1).cuda()
    smooth = torch.nn.Conv2d(32, cout, 3, padding=1).cuda()
    prev_flag = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():
            mid_ref = torch.nn.functional.interpolate(prev, scale_factor=2, mode="bilinear", align_corners=True) + lat(lat_in)
            out_ref = smooth(mid_ref)
    finally:
        torch.backends.cudnn.allow_tf32 = prev_flag
    mid, out = ops.fpn_topdown_smooth(prev, lat_in, lat.weight, lat.bias, pack_conv2d_k3_c32(smooth.weight), smooth.bias,
                                      cout, write_mid)
    assert (mid is not None) == write_mid
    if write_mid:                                   # the materialised intermediate is exact fp32 arithmetic
        assert torch.allclose(mid, mid_ref, rtol=1e-5, atol=1e-5 * mid_ref.abs().max().item())
    assert out.shape == out_ref.shape and out.is_contiguous(memory_format=torch.channels_last)
    assert (out - out_ref).abs().max().item() <= 2e-3 * out_ref.abs().max().item()


def test_fpn_plan_fused_smooth_matches_unfused():
    from boostmvsnerfs_b200.inference_plan import PlanCache
    from boostmvsnerfs_b200.modules import FeatureNet
    torch.manual_seed(1)
    net = FeatureNet().cuda().eval()
    x = torch.randn(3, 3, 64, 96, device="cuda").contiguous(memory_format=torch.channels_last)
    plan = PlanCache().get("feature_net", net, torch.channels_last)
    prev = torch.backends.cudnn.allow_tf32
    try:
        with torch.no_grad():
            torch.backends.cudnn.allow_tf32 = False
            ref = plan(x)
            torch.backends.cudnn.allow_tf32 = True
            got = plan(x)
    finally:
        torch.backends.cudnn.allow_tf32 = prev
    for a, b in zip(got, ref):
        assert a.shape == b.shape
        assert (a - b).abs().max().item() <= 1e-2 * b.abs().max().item()


@pytest.mark.parametrize("hw", [(64, 96), (9, 70), (33, 17)])
@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
def test_fpn_stem_vs_torch(hw, layout):
    from boostmvsnerfs_b200 import ops
    from boostmvsnerfs_b200.mlp_pack import pack_conv2d_k3_c8
    H, W = hw
    torch.manual_seed(H)
    x = torch.randn(2, 3, H, W, device="cuda")
    if layout == "nhwc":
        x = x.contiguous(memory_format=torch.channels_last)
    c0 = torch.nn.Conv2d(3, 8, 3, padding=1).cuda()
    c1 = torch.nn.Conv2d(8, 8, 3, padding=1).cuda()
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():
            ref = torch.relu(c1(torch.relu(c0(x))))
    finally:
        torch.backends.cudnn.allow_tf32 = prev
    out = ops.fpn_stem(x, c0.weight, c0.bias, pack_conv2d_k3_c8(c1.weight), c1.bias)
    assert out.shape == ref.shape and out.is_contiguous(memory_format=torch.channels_last)
    assert (out - ref).abs().max().item() <= 2e-3 * ref.abs().max().item()
    out2, rgb4 = ops.fpn_stem(x, c0.weight, c0.bias, pack_conv2d_k3_c8(c1.weight), c1.bias, want_rgb4=True)
    assert torch.equal(out2, out)
    assert torch.equal(rgb4[..., :3], x.permute(0, 2, 3, 1)) and rgb4[..., 3].abs().max().item() == 0
    if H % 2 == 0 and W % 2 == 0:
        out3, _, z = ops.fpn_stem(x, c0.weight, c0.bias, pack_conv2d_k3_c8(c1.weight), c1.bias, want_rgb4=True, want_s2d=True)
        zr = out.permute(0, 2, 3, 1).reshape(2, H // 2, 2, W // 2, 2, 8).permute(0, 1, 3, 2, 4, 5).reshape(2, H // 2, W // 2, 32)
        assert torch.equal(out3, out) and torch.equal(z.permute(0, 2, 3, 1), zr)


UMMA_SHAPES = [  # (N, Cin, Cout, D, H, W, bias, relu, out_half, split)
    (2, 8, 9, 8, 8, 64, False, False, False, 8),        # merged output heads: features + logits
    (1, 8, 9, 3, 9, 17, True, True, False, 8),          # ragged in every dimension
    (1, 8, 9, 5, 6, 300, True, False, False, 8),        # three x tiles
    (1, 8, 16, 8, 4, 140, True, False, True, 0),
    (2, 16, 8, 8, 12, 64, True, True, True, 0),         # conv0 of the level-1 U-Net
    (1, 16, 8, 5, 7, 45, True, True, False, 0),
    (2, 16, 16, 4, 8, 240, True, True, False, 0),       # conv2
    (1, 16, 12, 3, 5, 19, False, False, False, 0),
]


@pytest.mark.parametrize("shape", UMMA_SHAPES)
@pytest.mark.parametrize("exact_operands", [True, False])
def test_conv3d_k3_umma_matches_cudnn(shape, exact_operands):
    """bmv_conv3d_k3_umma (TMA + tcgen05 + TMEM) against cuDNN fp32 and against the mma.sync kernel."""
    from boostmvsnerfs_b200 import ops
    from boostmvsnerfs_b200.mlp_pack import pack_conv3d_k3, pack_conv3d_k3_umma
    N, Cin, Cout, D, H, W, bias, relu, out_half, split = shape
    g = torch.Generator().manual_seed(Cin * 100 + W + Cout)
    x = torch.randn((N, Cin, D, H, W), generator=g)
    w = torch.randn((Cout, Cin, 3, 3, 3), generator=g) * 0.1
    b = torch.randn(Cout, generator=g) if bias else None
    if exact_operands:
        x, w = x.half().float(), w.half().float()
    x = x.cuda().contiguous(memory_format=torch.channels_last_3d)
    w = w.cuda()
    b = b.cuda() if bias else None
    xh = x.half()
    ref = _reference(xh.float(), w, b, relu)
    scale = ref.abs().max().item()
    tol = (1e-5 if exact_operands else 2e-3) * scale
    kw = dict(out_dtype=torch.float16) if out_half else {}
    if split:
        out2 = torch.empty((N, Cout - split, D, H, W), device="cuda")
        y = ops.conv3d_k3(xh, pack_conv3d_k3_umma(w), b, Cout, relu, out2=out2, split=split, engine="umma")
        got = torch.cat([y, out2], dim=1)
    else:
        got = ops.conv3d_k3(xh, pack_conv3d_k3_umma(w), b, Cout, relu, engine="umma", **kw)
        assert got.stride(1) == 1
    if out_half:
        tol = max(tol, 1e-3 * scale)                            # fp16 storage of the result
    assert got.shape == ref.shape
    assert (got.float() - ref).abs().max().item() <= tol, ((got.float() - ref).abs().max().item(), scale)
    old = ops.conv3d_k3(xh, pack_conv3d_k3(w), b, Cout, relu)
    assert (got.float() - old).abs().max().item() <= max(tol, 2e-5 * scale)


UMMA_TILE = {8: (4, 4, 126), 16: (2, 4, 128)}           # (TD, TH, TW) of bmv_conv3d_k3_umma per Cin (conv3d_umma.cu)
UMMA_SMS = 148                                          # persistent grid: min(tiles, 148) CTAs
UMMA_MODE_COUT = {0: 9, 1: 8, 2: 16, 3: 12}


def _umma_tiles(cin, dhw):
    return math.prod(-(-n // t) for n, t in zip(dhw, UMMA_TILE[cin]))


def _umma_in_mode(x, wfrag, b, mode):
    """bmv_conv3d_k3_umma with an output layout that selects epilogue `mode` (conv3d_umma.cu): 0 fp32 features + channel
    8 to out2 (the merged heads), 1 fp16 with 8 channels, 2 fp32 with 16 channels, 3 per-element stores (here 12
    channels into a channel slice of a wider tensor).  Returns every output channel, and for mode 3 the whole wider
    tensor, so that stray writes into the channels around the slice are compared too."""
    from boostmvsnerfs_b200 import ops
    N, _, D, H, W = x.shape
    cout = UMMA_MODE_COUT[mode]
    if mode == 0:
        out2 = torch.empty((N, 1, D, H, W), device="cuda")
        return torch.cat([ops.conv3d_k3(x, wfrag, b, cout, False, out2=out2, split=8, engine="umma"), out2], dim=1)
    if mode == 1:
        return ops.conv3d_k3(x, wfrag, b, cout, True, out_dtype=torch.float16, engine="umma")
    if mode == 2:
        return ops.conv3d_k3(x, wfrag, b, cout, False, engine="umma")
    big = torch.full((N, 16, D, H, W), -7.0, device="cuda").contiguous(memory_format=torch.channels_last_3d)
    ops.conv3d_k3(x, wfrag, b, cout, True, out=big[:, 2:14], engine="umma")
    return big


@pytest.mark.parametrize("cin,dhw,batches", [
    (8, (4, 4, 126), (147, 148, 149, 296, 297, 445, 600)),      # one tile per volume
    (8, (3, 3, 100), (147, 148, 149, 296, 297, 445, 600)),      # one tile, ragged in every dimension
    (16, (2, 4, 128), (147, 148, 149, 296, 297, 445, 600)),
    (16, (1, 3, 77), (147, 148, 149, 296, 297, 445, 600)),
    (8, (8, 32, 252), (16,)),                                   # 32 tiles per volume: 512 tiles
], ids=["cin8", "cin8-ragged", "cin16", "cin16-ragged", "cin8-32-tiles-per-volume"])
@pytest.mark.parametrize("mode", [0, 1, 2, 3])
def test_conv3d_k3_umma_is_batch_independent(cin, dhw, batches, mode):
    """bmv_conv3d_k3_umma is persistent: min(tiles, 148) CTAs walk tiles blockIdx.x, +148, ... through a 2-slot ring (a
    staged TMA tile + a TMEM accumulator set per slot; slot = it % 2, mbarrier parity (it / 2) & 1).  A tile's MMAs and
    epilogue do not depend on the slot or the CTA that runs them, so a launch over N volumes must equal, bit for bit,
    launches over chunks of at most 148 tiles, in which every CTA runs exactly one tile.  With one-tile volumes, tile t
    is volume t and N covers one partial wave (147), the full wave (148), slot 1 first used (149), slot 0 reused with
    its parity flipped (297), several flips (445, 600) and ragged last waves.  Every epilogue mode is covered."""
    from boostmvsnerfs_b200.mlp_pack import pack_conv3d_k3_umma
    per_vol = _umma_tiles(cin, dhw)
    assert max(batches) * per_vol > 2 * UMMA_SMS               # some CTA runs >= 3 tiles (slot 0 twice)
    chunk = max(1, UMMA_SMS // per_vol)                        # volumes per reference launch: <= 148 tiles
    cout = UMMA_MODE_COUT[mode]
    g = torch.Generator().manual_seed(cin * 1000 + dhw[2] * 10 + mode)
    x = torch.randn((max(batches), cin, *dhw), generator=g).half().cuda().contiguous(memory_format=torch.channels_last_3d)
    w = (torch.randn((cout, cin, 3, 3, 3), generator=g) * 0.1).cuda()
    b = torch.randn(cout, generator=g).cuda()
    wfrag = pack_conv3d_k3_umma(w)
    for N in batches:
        xs = x[:N]
        full = _umma_in_mode(xs, wfrag, b, mode)
        ref = torch.cat([_umma_in_mode(xs[i:i + chunk], wfrag, b, mode) for i in range(0, N, chunk)])
        assert full.abs().max().item() > 0
        if mode == 3:
            assert bool((full[:, :2] == -7.0).all()) and bool((full[:, 14:] == -7.0).all()), f"N={N}: write outside the slice"
        diff = (full.float() - ref.float()).abs()
        assert torch.equal(full, ref), (f"N={N} ({N * per_vol} tiles): {int((diff > 0).sum())} outputs differ from the "
                                        f"one-tile-per-CTA launches, max {diff.max().item():.3e}")


@pytest.mark.parametrize("shape", [(4, 8, 9, 64, 68, 120), (4, 8, 9, 8, 272, 480)], ids=["level0", "level1"])
def test_conv3d_k3_umma_merged_heads_at_frame_size(shape):
    """The merged U-Net heads of a C2 frame (K = 4 chains, 960x544): level 0 is 1088 tiles, level 1 2176 (7 to 15 per
    CTA).  fp16-representable operands, so the only difference from a float64 convolution is the fp32 accumulation:
    1e-5 of the output's magnitude."""
    from boostmvsnerfs_b200 import ops
    from boostmvsnerfs_b200.mlp_pack import pack_conv3d_k3_umma
    N, Cin, Cout, D, H, W = shape
    g = torch.Generator(device="cuda").manual_seed(D + H)
    xh = torch.randn((N, Cin, D, H, W), device="cuda", generator=g).half().contiguous(memory_format=torch.channels_last_3d)
    w = (torch.randn((Cout, Cin, 3, 3, 3), device="cuda", generator=g) * 0.1).half().float()
    b = torch.randn(Cout, device="cuda", generator=g)
    out2 = torch.empty((N, 1, D, H, W), device="cuda")
    feat = ops.conv3d_k3(xh, pack_conv3d_k3_umma(w), b, Cout, False, out2=out2, split=8, engine="umma")
    got = torch.cat([feat, out2], dim=1).double()
    ref = torch.nn.functional.conv3d(xh.double(), w.double(), b.double(), padding=1)
    scale = ref.abs().max().item()
    err = (got - ref).abs().max().item()
    assert err <= 1e-5 * scale, (err, scale)


# ------------------------------------------------------------------------------------------ FPN middle layers (conv2d_mma.cu)
def _ref_conv(x, w, b, **kw):
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():
            return torch.nn.functional.conv2d(x, w, b, **kw)
    finally:
        torch.backends.cudnn.allow_tf32 = prev


@pytest.mark.parametrize("cin,cout,hw", [(16, 16, (40, 64)), (32, 32, (37, 45)), (16, 16, (5, 9))])
@pytest.mark.parametrize("out_dtype", [torch.float32, torch.float16])
def test_conv2d_k3_dense_vs_torch(cin, cout, hw, out_dtype):
    from boostmvsnerfs_b200 import ops
    from boostmvsnerfs_b200.mlp_pack import pack_conv2d_k3
    H, W = hw
    torch.manual_seed(cin + H)
    x = torch.randn(3, cin, H, W, device="cuda").half().contiguous(memory_format=torch.channels_last)
    w = (torch.randn(cout, cin, 3, 3, device="cuda") * 0.1).half().float()       # fp16-representable operands: 1e-5 class
    b = torch.randn(cout, device="cuda")
    for relu in (True, False):
        ref = _ref_conv(x.float(), w, b, padding=1)
        ref = torch.relu(ref) if relu else ref
        got = ops.conv2d_k3(x, pack_conv2d_k3(w), b, cout, relu=relu, out_dtype=out_dtype)
        assert got.shape == ref.shape and got.dtype == out_dtype and got.is_contiguous(memory_format=torch.channels_last)
        tol = 2e-5 if out_dtype == torch.float32 else 1e-3
        assert (got.float() - ref).abs().max().item() <= tol * ref.abs().max().item()


@pytest.mark.parametrize("cs,cout,hw", [(8, 16, (36, 72)), (16, 32, (20, 44)), (8, 16, (4, 8))])
@pytest.mark.parametrize("src_dtype", [torch.float32, torch.float16])
def test_conv2d_k3_space_to_depth_is_the_5x5_stride2_layer(cs, cout, hw, src_dtype):
    """fp32 source read through space-to-depth in the staging loop + S2DConv5x5's regrouped weights == the reference
    layer (5x5, stride 2, pad 2) on the fp16-rounded source."""
    from boostmvsnerfs_b200 import ops
    from boostmvsnerfs_b200.inference_plan import S2DConv5x5
    from boostmvsnerfs_b200.mlp_pack import pack_conv2d_k3
    H2, W2 = hw
    torch.manual_seed(cs + H2)
    conv = torch.nn.Conv2d(cs, cout, 5, stride=2, padding=2).cuda()
    with torch.no_grad():
        conv.weight.copy_(conv.weight.half().float())
    src = torch.randn(2, cs, H2, W2, device="cuda").contiguous(memory_format=torch.channels_last)
    ref = torch.relu(_ref_conv(src.half().float(), conv.weight, conv.bias, stride=2, padding=2))
    s2d = S2DConv5x5(conv, relu=True)
    got = ops.conv2d_k3(src.to(src_dtype), pack_conv2d_k3(s2d.weight), s2d.bias, cout, relu=True, s2d=True, out_dtype=torch.float32)
    assert got.shape == ref.shape
    assert (got - ref).abs().max().item() <= 2e-5 * ref.abs().max().item()


def test_conv2d_k3_fused_top_layer_vs_torch():
    from boostmvsnerfs_b200 import ops
    from boostmvsnerfs_b200.mlp_pack import pack_conv1x1_after, pack_conv2d_k3
    torch.manual_seed(11)
    x = torch.randn(2, 32, 35, 50, device="cuda").half().contiguous(memory_format=torch.channels_last)
    w = (torch.randn(32, 32, 3, 3, device="cuda") * 0.1).half().float()
    b = torch.randn(32, device="cuda")
    w1 = (torch.randn(32, 32, 1, 1, device="cuda") * 0.2).half().float()
    b1 = torch.randn(32, device="cuda")
    mid = torch.relu(_ref_conv(x.float(), w, b, padding=1))
    ref = _ref_conv(mid, w1, b1)
    got = ops.conv2d_k3(x, pack_conv2d_k3(w), b, 32, relu=True, wfrag1x1=pack_conv1x1_after(w1), bias1x1=b1)
    assert got.shape == ref.shape and got.dtype == torch.float32
    # the intermediate is rounded to fp16 between the two layers (TF32-class)
    assert (got - ref).abs().max().item() <= 2e-3 * ref.abs().max().item()
    ref16 = _ref_conv(mid.half().float(), w1, b1)
    assert (got - ref16).abs().max().item() <= 3e-4 * ref.abs().max().item()


def test_fpn_plan_tensor_core_mid_layers_match_cudnn_route():
    """FeatureNet plan with conv1.x / conv2.x / top layer on bmv_conv2d_k3 against the same plan with those layers on cuDNN
    (both TF32-class): all three pyramid levels."""
    from boostmvsnerfs_b200.inference_plan import PlanCache
    from boostmvsnerfs_b200.modules import FeatureNet
    torch.manual_seed(2)
    net = FeatureNet().cuda().eval()
    x = torch.randn(3, 3, 64, 96, device="cuda")
    plan = PlanCache().get("feature_net", net, torch.channels_last)
    with torch.no_grad():
        plan.tensor_core_mid = True
        got = [t.clone() for t in plan(x)]
        plan.tensor_core_mid = False
        ref = plan(x)
        prev = torch.backends.cudnn.allow_tf32
        torch.backends.cudnn.allow_tf32 = False
        try:
            strict = plan(x)
        finally:
            torch.backends.cudnn.allow_tf32 = prev
    for a, b, s in zip(got, ref, strict):
        assert a.shape == b.shape
        assert (a - s).abs().max().item() <= 1e-2 * s.abs().max().item()
        assert (a - b).abs().max().item() <= 1e-2 * s.abs().max().item()


@pytest.mark.parametrize("cin,cout,hw", [(8, 8, (64, 96)), (16, 16, (34, 50))])
def test_fpn_topdown_smooth_fp16_lateral_input(cin, cout, hw):
    """fp16 lateral input (what the stem / bmv_conv2d_k3 emit) == the fp32-input kernel on the same values: the fp16
    operand is exact, only the summation order inside the tensor core differs."""
    from boostmvsnerfs_b200 import ops
    from boostmvsnerfs_b200.mlp_pack import pack_conv2d_k3_c32
    H, W = hw
    torch.manual_seed(cin)
    prev = torch.randn(2, 32, H // 2, W // 2, device="cuda").contiguous(memory_format=torch.channels_last)
    lat16 = torch.randn(2, cin, H, W, device="cuda").half().contiguous(memory_format=torch.channels_last)
    lat = torch.nn.Conv2d(cin, 32, 1).cuda()
    smooth = torch.nn.Conv2d(32, cout, 3, padding=1).cuda()
    wf = pack_conv2d_k3_c32(smooth.weight)
    mid32, out32 = ops.fpn_topdown_smooth(prev, lat16.float(), lat.weight, lat.bias, wf, smooth.bias, cout, True)
    mid16, out16 = ops.fpn_topdown_smooth(prev, lat16, lat.weight, lat.bias, wf, smooth.bias, cout, True)
    assert (mid16 - mid32).abs().max().item() <= 2e-6 * mid32.abs().max().item()
    assert (out16 - out32).abs().max().item() <= 1e-3 * out32.abs().max().item()
    with torch.no_grad():
        prev_flag = torch.backends.cudnn.allow_tf32
        torch.backends.cudnn.allow_tf32 = False
        try:
            mid_ref = torch.nn.functional.interpolate(prev, scale_factor=2, mode="bilinear", align_corners=True) + lat(lat16.float())
        finally:
            torch.backends.cudnn.allow_tf32 = prev_flag
    assert torch.allclose(mid16, mid_ref, rtol=1e-5, atol=1e-5 * mid_ref.abs().max().item())


def test_fpn_stem_fp16_output_is_the_rounded_fp32_output():
    from boostmvsnerfs_b200 import ops
    from boostmvsnerfs_b200.mlp_pack import pack_conv2d_k3_c8
    torch.manual_seed(4)
    x = torch.randn(2, 3, 40, 72, device="cuda")
    c0 = torch.nn.Conv2d(3, 8, 3, padding=1).cuda()
    c1 = torch.nn.Conv2d(8, 8, 3, padding=1).cuda()
    wf = pack_conv2d_k3_c8(c1.weight)
    o32, rgb_a = ops.fpn_stem(x, c0.weight, c0.bias, wf, c1.bias, want_rgb4=True)
    o16, rgb_b = ops.fpn_stem(x, c0.weight, c0.bias, wf, c1.bias, want_rgb4=True, out_dtype=torch.float16)
    assert o16.dtype == torch.float16 and o16.is_contiguous(memory_format=torch.channels_last)
    assert torch.equal(o16, o32.half()) and torch.equal(rgb_a, rgb_b)


def test_conv2d_k3_large_grid_uses_the_16_row_tiles():
    """The launcher picks 8-row tiles for small grids (every other conv2d test) and 16-row tiles from 900 tiles on: the
    half-resolution layers of the C2 frame.  Same arithmetic: check both routes against torch at that size."""
    from boostmvsnerfs_b200 import ops
    from boostmvsnerfs_b200.inference_plan import S2DConv5x5
    from boostmvsnerfs_b200.mlp_pack import pack_conv2d_k3
    torch.manual_seed(21)
    x = torch.randn(4, 16, 272, 480, device="cuda").half().contiguous(memory_format=torch.channels_last)
    w = (torch.randn(16, 16, 3, 3, device="cuda") * 0.1).half().float()
    b = torch.randn(16, device="cuda")
    ref = torch.relu(_ref_conv(x.float(), w, b, padding=1))
    got = ops.conv2d_k3(x, pack_conv2d_k3(w), b, 16, relu=True, out_dtype=torch.float32)
    assert (got - ref).abs().max().item() <= 2e-5 * ref.abs().max().item()
    conv = torch.nn.Conv2d(8, 16, 5, stride=2, padding=2).cuda()
    with torch.no_grad():
        conv.weight.copy_(conv.weight.half().float())
    src = torch.randn(4, 8, 544, 960, device="cuda").half().contiguous(memory_format=torch.channels_last)
    ref = torch.relu(_ref_conv(src.float(), conv.weight, conv.bias, stride=2, padding=2))
    s2d = S2DConv5x5(conv, relu=True)
    got = ops.conv2d_k3(src, pack_conv2d_k3(s2d.weight), s2d.bias, 16, relu=True, s2d=True, out_dtype=torch.float32)
    assert (got - ref).abs().max().item() <= 2e-5 * ref.abs().max().item()
