"""CPU checks of the MMA weight packers (mlp_pack.pack_conv*): the packed words are unpacked with the
mma.sync.m16n8k16 B-fragment rule (lane = 4g+t holds b0 = B[2t, 2t+1][g], b1 = B[2t+8, 2t+9][g]) and fed
through a plain restatement of each kernel's implicit-GEMM addressing (the k-step -> (voxel offset, channel)
maps of csrc/conv3d_mma.cu, convT3d_mma.cu, fpn_fused.cu, fpn_stem.cu); the result must equal torch's
convolution on fp16-representable operands.  Runs without a GPU."""
import pytest
import torch
import torch.nn.functional as F

from boostmvsnerfs_b200 import mlp_pack


def unpack_b(words, lead):
    """words: int32 tensor [*lead][lane 32][2 regs] -> float B[*lead][k 16][n 8]."""
    h = words.view(torch.float16).float().view(*lead, 32, 2, 2)          # [.., lane, reg, elem]
    B = torch.zeros(*lead, 16, 8)
    for lane in range(32):
        g, t = lane // 4, lane % 4
        for r in range(2):
            for e in range(2):
                B[..., 2 * t + 8 * r + e, g] = h[..., lane, r, e]
    return B


def conv3d_step_sources(cin):
    """(voxel offset dx, channel) read by K index k of k-step j — restates ConvCfg::step_voxel/step_chunk."""
    if cin == 16:
        return [[(j, k) for k in range(16)] for j in range(3)]
    if cin == 32:
        return [[(j >> 1, (j & 1) * 16 + k) for k in range(16)] for j in range(6)]
    return [[(2 * j + (k >= 8), k % 8) for k in range(16)] for j in range(2)]      # cin == 8: voxel pairs


@pytest.mark.parametrize("cin,cout", [(16, 8), (16, 16), (16, 5), (32, 8), (8, 9), (8, 16)])
def test_pack_conv3d_k3_reproduces_conv3d(cin, cout):
    g = torch.Generator().manual_seed(cin * 31 + cout)
    w = (torch.randn((cout, cin, 3, 3, 3), generator=g) * 0.2).half().float()
    x = torch.randn((1, cin, 4, 5, 9), generator=g).half().float()
    steps = conv3d_step_sources(cin)
    nt = mlp_pack._conv3d_ntiles(cin, cout)
    B = unpack_b(mlp_pack.pack_conv3d_k3(w), (3, 3, len(steps), nt))     # [dz][dy][j][nt][k][n]
    xp = F.pad(x, (1, 3, 1, 1, 1, 1))[0]                                 # +2 extra on the right: Cin=8 reads x+3
    D, H, W = x.shape[2:]
    out = torch.zeros(nt * 8, D, H, W)
    for dz in range(3):
        for dy in range(3):
            for j, step in enumerate(steps):
                for k, (dx, c) in enumerate(step):
                    a = xp[c, dz:dz + D, dy:dy + H, dx:dx + W]           # A[voxel, k]
                    for t in range(nt):
                        out[t * 8:(t + 1) * 8] += B[dz, dy, j, t, k][:, None, None, None] * a
    ref = F.conv3d(x, w, padding=1)[0]
    assert torch.allclose(out[:cout], ref, atol=1e-4), (out[:cout] - ref).abs().max()
    assert out[cout:].abs().max() == 0 if cout < nt * 8 else True


def test_pack_conv3d_k3_stride2_addressing():
    """Stride 2 uses the Cin=8 packing with A rows at every second voxel (conv3d_k3s2_c8_mma_kernel)."""
    g = torch.Generator().manual_seed(5)
    w = (torch.randn((16, 8, 3, 3, 3), generator=g) * 0.2).half().float()
    x = torch.randn((1, 8, 6, 4, 10), generator=g).half().float()
    B = unpack_b(mlp_pack.pack_conv3d_k3(w), (3, 3, 2, 2))
    xp = F.pad(x, (1, 3, 1, 1, 1, 1))[0]
    Do, Ho, Wo = 3, 2, 5
    out = torch.zeros(16, Do, Ho, Wo)
    for dz in range(3):
        for dy in range(3):
            for j in range(2):
                for k in range(16):
                    dx, c = 2 * j + (k >= 8), k % 8
                    a = xp[c, dz:dz + 2 * Do:2, dy:dy + 2 * Ho:2, dx:dx + 2 * Wo:2]
                    for t in range(2):
                        out[t * 8:(t + 1) * 8] += B[dz, dy, j, t, k][:, None, None, None] * a
    ref = F.conv3d(x, w, stride=2, padding=1)[0]
    assert torch.allclose(out, ref, atol=1e-4)


@pytest.mark.parametrize("cin,cout", [(16, 8), (32, 16)])
def test_pack_convT3d_k3s2_reproduces_conv_transpose(cin, cout):
    g = torch.Generator().manual_seed(cin)
    w = (torch.randn((cin, cout, 3, 3, 3), generator=g) * 0.2).half().float()
    x = torch.randn((1, cin, 2, 3, 4), generator=g).half().float()
    kt, nt = cin // 16, cout // 8
    B = unpack_b(mlp_pack.pack_convT3d_k3s2(w), (27, kt, nt))            # [tap][kt][nt][k][n]
    D, H, W = x.shape[2:]
    xp = F.pad(x, (0, 1, 0, 1, 0, 1))[0]                                 # +1 halo on the high side
    out = torch.zeros(cout, 2 * D, 2 * H, 2 * W)
    # shift s in a dimension serves (parity 0, tap 1) and (parity 1, tap 2) when s = 0, (parity 1, tap 0) when s = 1
    opts = {0: [(0, 1), (1, 2)], 1: [(1, 0)]}
    for sz in range(2):
        for sy in range(2):
            for sx in range(2):
                a = xp[:, sz:sz + D, sy:sy + H, sx:sx + W]               # (cin, D, H, W)
                for pz, kz in opts[sz]:
                    for py, ky in opts[sy]:
                        for px, kx in opts[sx]:
                            tap = (kz * 3 + ky) * 3 + kx
                            Bt = torch.cat([torch.cat([B[tap, k, t] for t in range(nt)], dim=1) for k in range(kt)], dim=0)  # (cin, cout)
                            out[:, pz::2, py::2, px::2] += torch.einsum("cdhw,co->odhw", a, Bt)
    ref = F.conv_transpose3d(x, w, stride=2, padding=1, output_padding=1)[0]
    assert torch.allclose(out, ref, atol=1e-4), (out - ref).abs().max()


@pytest.mark.parametrize("cout", [8, 16])
def test_pack_conv2d_k3_c32_reproduces_conv2d(cout):
    g = torch.Generator().manual_seed(cout)
    w = (torch.randn((cout, 32, 3, 3), generator=g) * 0.2).half().float()
    x = torch.randn((1, 32, 5, 7), generator=g).half().float()
    nt = cout // 8
    B = unpack_b(mlp_pack.pack_conv2d_k3_c32(w), (3, 6, nt))             # [dy][j = dx*2+half][nt][k][n]
    xp = F.pad(x, (1, 1, 1, 1))[0]
    H, W = x.shape[2:]
    out = torch.zeros(cout, H, W)
    for dy in range(3):
        for j in range(6):
            dx, half = j >> 1, j & 1
            for k in range(16):
                a = xp[half * 16 + k, dy:dy + H, dx:dx + W]
                for t in range(nt):
                    out[t * 8:(t + 1) * 8] += B[dy, j, t, k][:, None, None] * a
    assert torch.allclose(out, F.conv2d(x, w, padding=1)[0], atol=1e-4)


def test_pack_conv2d_k3_c8_reproduces_conv2d():
    g = torch.Generator().manual_seed(1)
    w = (torch.randn((8, 8, 3, 3), generator=g) * 0.2).half().float()
    x = torch.randn((1, 8, 4, 6), generator=g).half().float()
    B = unpack_b(mlp_pack.pack_conv2d_k3_c8(w), (3, 2))                  # [dy][j][k][n]
    xp = F.pad(x, (1, 3, 1, 1))[0]
    H, W = x.shape[2:]
    out = torch.zeros(8, H, W)
    for dy in range(3):
        for j in range(2):
            for k in range(16):
                dx, c = 2 * j + (k >= 8), k % 8
                out += B[dy, j, k][:, None, None] * xp[c, dy:dy + H, dx:dx + W]
    assert torch.allclose(out, F.conv2d(x, w, padding=1)[0], atol=1e-4)


def test_packers_reject_uninstantiated_shapes():
    with pytest.raises(ValueError):
        mlp_pack.pack_conv3d_k3(torch.zeros(8, 24, 3, 3, 3))
    with pytest.raises(ValueError):
        mlp_pack.pack_conv3d_k3(torch.zeros(24, 16, 3, 3, 3))
    with pytest.raises(ValueError):
        mlp_pack.pack_convT3d_k3s2(torch.zeros(16, 16, 3, 3, 3))
    with pytest.raises(ValueError):
        mlp_pack.pack_conv2d_k3_c32(torch.zeros(8, 16, 3, 3))
    with pytest.raises(ValueError):
        mlp_pack.pack_conv2d_k3_c8(torch.zeros(8, 8, 5, 5))


def test_cost_reg_plan_uses_cudnn_on_cpu_and_when_tf32_is_off():
    """The tensor-core convolutions are a CUDA + allow_tf32 fast path; everywhere else the plan is the folded
    cuDNN/ATen module (and therefore runs on CPU for the host-logic tests)."""
    from boostmvsnerfs_b200.inference_plan import MergedHeadsCostReg, PlanCache
    from boostmvsnerfs_b200.modules import MinCostRegNet
    torch.manual_seed(0)
    net = MinCostRegNet(16).eval()
    plan = PlanCache().get("cr", net, None)
    assert isinstance(plan, MergedHeadsCostReg)
    x = torch.rand(1, 16, 8, 16, 16)
    assert not plan._use_tensor_core_convs(x)
    with torch.no_grad():
        feat, logits = plan(x)
        ref_feat, ref_logits = net(x)
    assert torch.allclose(feat, ref_feat, atol=1e-5) and torch.allclose(logits, ref_logits, atol=1e-5)


@pytest.mark.parametrize("cin,cout", [(8, 9), (8, 16), (16, 8), (16, 12)])
def test_umma_conv_packing_reproduces_conv3d(cin, cout):
    """pack_conv3d_k3_umma read back through the kernel's descriptor arithmetic (stacked [W(dz,2); W(dz,1); W(dz,0)]
    operands of 48 rows, K-major SWIZZLE_NONE: SBO 128 B, LBO 768 B) and applied the way csrc/conv3d_umma.cu issues its
    MMAs — input row hy feeds output rows oy = hy-2..hy with the row range starting at block 2-(hy-oy_min); Cin 8 pairs
    the taps (dx, dx+1) in one K = 16 step — gives torch's conv3d (fp16 operands)."""
    import numpy as np
    from boostmvsnerfs_b200.mlp_pack import pack_conv3d_k3_umma
    torch.manual_seed(cin + cout)
    w = (torch.randn(cout, cin, 3, 3, 3) * 0.2).half().float()
    D, H, W = 3, 5, 7
    x = torch.randn(1, cin, D, H, W).half().float()
    ref = torch.nn.functional.conv3d(x, w, padding=1)[0].numpy()
    raw = pack_conv3d_k3_umma(w).numpy().view(np.float16)
    KS = 3 if cin == 16 else 2
    assert raw.size == 3 * KS * 2 * 48 * 8

    def operand(dz, j):                                       # (48, 16) via start + (n/8)*128 + (k/8)*768 + (n%8)*16 + (k%8)*2 bytes
        base = (dz * KS + j) * 1536
        m = np.zeros((48, 16), np.float32)
        for n in range(48):
            for k in range(16):
                m[n, k] = raw[(base + (n // 8) * 128 + (k // 8) * 768 + (n % 8) * 16 + (k % 8) * 2) // 2]
        return m

    xp = np.zeros((cin, D + 2, H + 2, W + 4), np.float32)     # zero halo (what the TMA unit fills) + the pair partner of dx = 2
    xp[:, 1:-1, 1:-1, 1:W + 1] = x[0].numpy()
    TH = H
    out = np.zeros((16, D, H, W), np.float32)
    for od in range(D):
        for dz in range(3):
            for hy in range(TH + 2):
                oy_min, oy_max = max(hy - 2, 0), min(hy, TH - 1)
                cnt, b0 = oy_max - oy_min + 1, 2 - (hy - max(hy - 2, 0))
                for j in range(KS):
                    B = operand(dz, j)[16 * b0:16 * (b0 + cnt)]                   # (16 cnt, 16)
                    row = xp[:, od + dz, hy]                                      # (cin, W+4)
                    for xo in range(W):
                        a = row[:, xo + j] if cin == 16 else np.concatenate([row[:, xo + 2 * j], row[:, xo + 2 * j + 1]])
                        acc = B @ a
                        for r in range(cnt):
                            out[:, od, oy_min + r, xo] += acc[16 * r:16 * r + 16]
    assert np.abs(out[:cout] - ref).max() < 1e-4 * np.abs(ref).max()
    assert cout == 16 or np.abs(out[cout:]).max() == 0


def _conv2d_k3_emulate(x, words, cin, cout):
    """Restates csrc/conv2d_mma.cu: k-step j = dx * (Cin/16) + part reads channels part*16 .. +15 of pixel x+dx; column g
    of n-tile nt is output channel (g//2) * 2NT + 2nt + g%2.  x (Cin,H,W) -> (Cout,H,W)."""
    NT, KPD = cout // 8, cin // 16
    B = unpack_b(words, (3, 3 * KPD, NT))                                # [dy][j][nt][k][n]
    xp = F.pad(x, (1, 1, 1, 1))
    H, W = x.shape[1:]
    out = torch.zeros(cout, H, W)
    for dy in range(3):
        for j in range(3 * KPD):
            dx, part = j // KPD, j % KPD
            for k in range(16):
                a = xp[part * 16 + k, dy:dy + H, dx:dx + W]
                for nt in range(NT):
                    for n in range(8):
                        out[(n // 2) * 2 * NT + nt * 2 + n % 2] += B[dy, j, nt, k, n] * a
    return out


@pytest.mark.parametrize("cin,cout", [(16, 16), (32, 32), (32, 16), (64, 32)])
def test_pack_conv2d_k3_reproduces_conv2d(cin, cout):
    g = torch.Generator().manual_seed(cin + cout)
    w = (torch.randn((cout, cin, 3, 3), generator=g) * 0.2).half().float()
    x = torch.randn((cin, 6, 11), generator=g).half().float()
    out = _conv2d_k3_emulate(x, mlp_pack.pack_conv2d_k3(w), cin, cout)
    ref = F.conv2d(x[None], w, padding=1)[0]
    assert torch.allclose(out, ref, atol=2e-4), (out - ref).abs().max()


def test_conv2d_k3_space_to_depth_mode_is_the_5x5_stride2_layer():
    """The kernel's s2d staging (conv channel (py*2+px)*Cs + c = source pixel (2y+py, 2x+px), channel c) + the regrouped
    weights of inference_plan.S2DConv5x5 == the reference's 5x5 / stride-2 / pad-2 convolution."""
    from boostmvsnerfs_b200.inference_plan import S2DConv5x5
    g = torch.Generator().manual_seed(3)
    conv = torch.nn.Conv2d(8, 16, 5, stride=2, padding=2)
    with torch.no_grad():
        conv.weight.copy_((torch.randn(conv.weight.shape, generator=g) * 0.1).half().float())
    src = torch.randn((8, 12, 20), generator=g).half().float()
    s2d = S2DConv5x5(conv, relu=False)
    Cs, H2, W2 = src.shape
    z = torch.zeros(4 * Cs, H2 // 2, W2 // 2)
    for py in range(2):
        for px in range(2):
            z[(py * 2 + px) * Cs:(py * 2 + px + 1) * Cs] = src[:, py::2, px::2]
    out = _conv2d_k3_emulate(z, mlp_pack.pack_conv2d_k3(s2d.weight), 32, 16) + conv.bias.detach()[:, None, None]
    ref = conv(src[None])[0].detach()
    assert torch.allclose(out, ref, atol=2e-4), (out - ref).abs().max()


def test_pack_conv1x1_after_matches_the_fragment_chaining():
    """The fused top layer: A fragments = the 3x3 layer's C fragments (lane t holds channels 8t + 2nt + e of n-tile nt),
    k-step kk takes n-tiles 2kk (K 0..7) and 2kk+1 (K 8..15)."""
    g = torch.Generator().manual_seed(9)
    w1 = (torch.randn((32, 32, 1, 1), generator=g) * 0.2).half().float()
    c = torch.randn(32, generator=g).half().float()                      # one pixel's 32 channels
    B = unpack_b(mlp_pack.pack_conv1x1_after(w1), (2, 4))                 # [kk][nt][k][n]
    out = torch.zeros(32)
    for kk in range(2):
        for k in range(16):
            t, e, r = (k % 8) // 2, k % 2, k // 8
            a = c[t * 8 + (2 * kk + r) * 2 + e]                          # what the chained A fragment holds at K index k
            for nt in range(4):
                for n in range(8):
                    out[(n // 2) * 8 + nt * 2 + n % 2] += B[kk, nt, k, n] * a
    ref = w1[:, :, 0, 0] @ c
    assert torch.allclose(out, ref, atol=2e-4), (out - ref).abs().max()

