"""Host-side packing of the per-sample MLP weights for the fused kernels (csrc/nerf_mlp.cuh).

The kernel reads every weight as a 16-byte broadcast from shared memory, so each layer is stored
row by row with the row padded to a multiple of 4 floats and the row's bias (and the weight of the
following 1-output layer) appended.  Parameter names are the reference's
(lib/networks/enerf/nerf.py:6-89): agg.view_fc.0, agg.global_fc.0, agg.agg_w_fc.0, agg.fc.0, lr0.0,
sigma.0, color.0, color.2.
"""
import torch


def layout(feat_ch):
    """Offsets (in floats) of each section; mirrors MlpLayout<F> in csrc/nerf_mlp.cuh."""
    F = feat_ch
    FP = (F + 3) // 4 * 4
    FV = F + 4
    FVP = (FV + 3) // 4 * 4
    L = dict(F=F, FP=FP, FV=FV, FVP=FVP, GROW=3 * FP + 4, CROW=88 + FVP + 4)
    L["OFF_VIEW"] = 0
    L["OFF_GLOB"] = L["OFF_VIEW"] + F * 8
    L["OFF_AGGB"] = L["OFF_GLOB"] + 32 * L["GROW"]
    L["OFF_FC"] = L["OFF_AGGB"] + 4
    L["OFF_FCB"] = L["OFF_FC"] + 32 * 16
    L["OFF_LR0"] = L["OFF_FCB"] + 16
    L["OFF_SIGB"] = L["OFF_LR0"] + 64 * 28
    L["OFF_COL"] = L["OFF_SIGB"] + 4
    L["OFF_COLB"] = L["OFF_COL"] + 64 * L["CROW"]
    L["TOTAL"] = L["OFF_COLB"] + 4
    return L


def pack_nerf_weights(nerf):
    """nerf: a `modules.NeRF` (or the reference's NeRF) -> flat fp32 tensor on the module's device."""
    sd = {k: v.detach().float() for k, v in nerf.state_dict().items()}
    if "agg.view_fc.0.weight" not in sd:
        raise ValueError("fused MLP requires cfg.enerf.viewdir_agg=True (the shipped configs)")
    F = sd["agg.view_fc.0.weight"].shape[0]
    if sd["lr0.0.weight"].shape != (64, 24) or sd["color.0.weight"].shape != (64, 88 + F + 4) or len(nerf.lrs) != 0:
        raise ValueError("unexpected NeRF MLP shape")
    L = layout(F)
    dev = sd["lr0.0.weight"].device
    buf = torch.zeros(L["TOTAL"], dtype=torch.float32, device=dev)
    FP, GROW, CROW = L["FP"], L["GROW"], L["CROW"]
    view = buf[L["OFF_VIEW"]:L["OFF_GLOB"]].view(F, 8)
    view[:, :4] = sd["agg.view_fc.0.weight"]
    view[:, 4] = sd["agg.view_fc.0.bias"]
    glob = buf[L["OFF_GLOB"]:L["OFF_AGGB"]].view(32, GROW)
    wg = sd["agg.global_fc.0.weight"]                    # (32, 3F): [x | var | mean]
    glob[:, 0:F] = wg[:, 0:F]
    glob[:, FP:FP + F] = wg[:, F:2 * F]
    glob[:, 2 * FP:2 * FP + F] = wg[:, 2 * F:3 * F]
    glob[:, 3 * FP] = sd["agg.global_fc.0.bias"]
    glob[:, 3 * FP + 1] = sd["agg.agg_w_fc.0.weight"][0]
    buf[L["OFF_AGGB"]] = sd["agg.agg_w_fc.0.bias"][0]
    buf[L["OFF_FC"]:L["OFF_FCB"]].view(32, 16).copy_(sd["agg.fc.0.weight"].t())
    buf[L["OFF_FCB"]:L["OFF_LR0"]] = sd["agg.fc.0.bias"]
    lr0 = buf[L["OFF_LR0"]:L["OFF_SIGB"]].view(64, 28)
    lr0[:, :24] = sd["lr0.0.weight"]
    lr0[:, 24] = sd["lr0.0.bias"]
    lr0[:, 25] = sd["sigma.0.weight"][0]
    buf[L["OFF_SIGB"]] = sd["sigma.0.bias"][0]
    col = buf[L["OFF_COL"]:L["OFF_COLB"]].view(64, CROW)
    wc = sd["color.0.weight"]                            # (64, 88+F+4)
    col[:, :88] = wc[:, :88]
    col[:, 88:88 + F + 4] = wc[:, 88:]
    col[:, 88 + L["FVP"]] = sd["color.0.bias"]
    col[:, 88 + L["FVP"] + 1] = sd["color.2.weight"][0]
    buf[L["OFF_COLB"]] = sd["color.2.bias"][0]
    return buf


def eval_packed(packed, vox, img):
    """Torch restatement of nerf_mlp_eval() reading the PACKED buffer (layout check on CPU; the
    product path never calls this).  vox (P,8), img (P,V,F+4) -> (P,4)."""
    P, V, FV = img.shape
    F = FV - 4
    L = layout(F)
    FP = L["FP"]
    view = packed[L["OFF_VIEW"]:L["OFF_GLOB"]].view(F, 8)
    x = img[..., :F] + torch.relu(img[..., F:] @ view[:, :4].t() + view[:, 4])
    mean = x.mean(1)
    var = ((x - mean[:, None]) ** 2).sum(1) / (V - 1)
    glob = packed[L["OFF_GLOB"]:L["OFF_AGGB"]].view(32, L["GROW"])
    shared = var @ glob[:, FP:FP + F].t() + mean @ glob[:, 2 * FP:2 * FP + F].t() + glob[:, 3 * FP]
    g = torch.relu(x @ glob[:, :F].t() + shared[:, None])                     # (P,V,32)
    logit = torch.relu(g @ glob[:, 3 * FP + 1] + packed[L["OFF_AGGB"]])       # (P,V)
    w = torch.softmax(logit, dim=1)
    im = (g * w[..., None]).sum(1)
    fc = packed[L["OFF_FC"]:L["OFF_FCB"]].view(32, 16)
    pooled = torch.relu(im @ fc + packed[L["OFF_FCB"]:L["OFF_LR0"]])
    base = torch.cat([vox, pooled], -1)
    lr0 = packed[L["OFF_LR0"]:L["OFF_SIGB"]].view(64, 28)
    hid = torch.relu(base @ lr0[:, :24].t() + lr0[:, 24])
    sig = torch.nn.functional.softplus(hid @ lr0[:, 25] + packed[L["OFF_SIGB"]])
    col = packed[L["OFF_COL"]:L["OFF_COLB"]].view(64, L["CROW"])
    shared = torch.cat([hid, base], -1) @ col[:, :88].t() + col[:, 88 + L["FVP"]]
    a = torch.relu(img @ col[:, 88:88 + FV].t() + shared[:, None])
    cl = torch.relu(a @ col[:, 88 + L["FVP"] + 1] + packed[L["OFF_COLB"]])
    beta = torch.softmax(cl, dim=1)
    rgb = (img[..., F - 3:F] * beta[..., None]).sum(1)
    return torch.cat([rgb, sig[:, None]], -1)


# ------------------------------------------------------------------------------------------ tensor-core packing
MMA_BLOCKS = dict(GS=(2, 4), GV=(1, 4), FC=(2, 2), L0=(2, 8), CS=(6, 8), CV=(1, 8))   # (k-tiles, n-tiles), kernel order


def _fragment_blocks(w_pad):
    """w_pad (N, K) fp32 with N % 8 == 0 and K % 16 == 0 -> int32 tensor (K/16 * N/8 * 128,) in the
    B-fragment order of mma.sync.m16n8k16: block (kt, nt), lane = 4*g + t holds
    b0 = W[nt*8+g][kt*16 + 2t, +1], b1 = W[nt*8+g][kt*16 + 2t+8, +9]; words {b0_hi, b1_hi, b0_lo, b1_lo}
    with x = hi + lo, hi = fp16(x), lo = fp16(x - hi)."""
    N, K = w_pad.shape
    hi = w_pad.half()
    lo = (w_pad - hi.float()).half()
    KT, NT = K // 16, N // 8
    lane = torch.arange(32)
    g, t = lane // 4, lane % 4
    out = torch.empty((KT, NT, 32, 4, 2), dtype=torch.float16)
    for kt in range(KT):
        for nt in range(NT):
            n = nt * 8 + g
            k0 = kt * 16 + 2 * t
            for j, src in enumerate((hi, hi, lo, lo)):
                kk = k0 + (8 if j % 2 else 0)
                out[kt, nt, :, j, 0] = src[n, kk]
                out[kt, nt, :, j, 1] = src[n, kk + 1]
    return out.reshape(-1).view(torch.int32)


def _tensor_core_matrices(nerf):
    """The level-1 NeRF MLP (feat_ch = 11, 3 views) as the six padded (N, K) weight matrices both tensor-core
    kernels multiply by, plus the fp32 bias / 1-output vectors (400 floats) they read in the epilogues."""
    sd = {k: v.detach().float().cpu() for k, v in nerf.state_dict().items()}
    if "agg.view_fc.0.weight" not in sd:
        raise ValueError("fused MLP requires cfg.enerf.viewdir_agg=True (the shipped configs)")
    F = sd["agg.view_fc.0.weight"].shape[0]
    if F != 11 or sd["lr0.0.weight"].shape != (64, 24) or sd["color.0.weight"].shape != (64, 103):
        raise ValueError("tensor-core MLP is instantiated for feat_ch=11 (nerf_model_feat_ch=8) only")
    wg, wfc, wl, wc = sd["agg.global_fc.0.weight"], sd["agg.fc.0.weight"], sd["lr0.0.weight"], sd["color.0.weight"]
    gs = torch.zeros(32, 32); gs[:, 0:F] = wg[:, F:2 * F]; gs[:, 16:16 + F] = wg[:, 2 * F:3 * F]     # [var | mean]
    gv = torch.zeros(32, 16); gv[:, 0:F] = wg[:, 0:F]
    l0 = torch.zeros(64, 32); l0[:, 0:16] = wl[:, 8:24]; l0[:, 16:24] = wl[:, 0:8]                  # [pooled | vox]
    cs = torch.zeros(64, 96); cs[:, 0:64] = wc[:, 0:64]; cs[:, 64:80] = wc[:, 72:88]; cs[:, 80:88] = wc[:, 64:72]
    cv = torch.zeros(64, 16); cv[:, 0:15] = wc[:, 88:103]
    wv = torch.zeros(12, 4); wv[:F] = sd["agg.view_fc.0.weight"]
    bv = torch.zeros(12); bv[:F] = sd["agg.view_fc.0.bias"]
    vec = torch.cat([sd["agg.global_fc.0.bias"], sd["agg.agg_w_fc.0.weight"][0], sd["agg.fc.0.bias"], sd["lr0.0.bias"],
                     sd["sigma.0.weight"][0], sd["color.0.bias"], sd["color.2.weight"][0], wv.reshape(-1), bv,
                     torch.stack([sd["agg.agg_w_fc.0.bias"][0], sd["sigma.0.bias"][0], sd["color.2.bias"][0],
                                  torch.tensor(0.)])])
    return (gs, gv, wfc.clone(), l0, cs, cv), vec.contiguous()


def pack_nerf_weights_mma(nerf):
    """Weights of the level-1 NeRF MLP (feat_ch = 11, 3 views) for the tensor-core kernel
    (csrc/render_mma.cu): fragment-ordered split-fp16 blocks followed by the fp32 bias / 1-output
    vectors.  Returns an int32 tensor (MMA_PACK_WORDS,) on the module's device."""
    mats, vec = _tensor_core_matrices(nerf)
    blocks = torch.cat([_fragment_blocks(m) for m in mats])
    packed = torch.cat([blocks, vec.view(torch.int32)])
    return packed.to(next(nerf.parameters()).device)


UMMA_PACK_TAG = 0x414D4D55      # "UMMA"


def umma_operand(w_pad):
    """(N, K) fp32 -> (hi, lo) fp16 tensors of shape (K/8, N, 8): the SWIZZLE_NONE K-major shared-memory layout a
    tcgen05.mma descriptor with SBO = 128 B, LBO = N*16 B addresses (K-chunk c is a slab of N rows x 16 bytes)."""
    N, K = w_pad.shape
    assert K % 16 == 0 and N % 8 == 0
    hi = w_pad.half()
    lo = (w_pad - hi.float()).half()
    lay = lambda m: m.reshape(N, K // 8, 8).permute(1, 0, 2).contiguous()
    return lay(hi), lay(lo)


def pack_umma_matrix(w_pad):
    """[hi block][lo block] of one matrix as int32 words (bmv_umma_selftest's B operand)."""
    hi, lo = umma_operand(w_pad)
    return torch.cat([hi.reshape(-1), lo.reshape(-1)]).view(torch.int32)


def pack_nerf_weights_umma(nerf):
    """Weights of the level-1 NeRF MLP for the tcgen05 kernel (csrc/render_multi_umma.cu, csrc/nerf_umma_pack.cuh):
    [hi block][lo block] with the six matrices in kernel order (UW_GS .. UW_CV), each in the layout of umma_operand,
    then the fp32 vectors.
    Returns an int32 tensor (UMMA_PACK_WORDS,) on the module's device."""
    (gs, gv, wfc, l0, cs, cv), vec = _tensor_core_matrices(nerf)
    # biases ride in the MMAs: the kernel puts a 1 in a padding column of the A operand (K index 15 of
    # [var | mean], K index 24 of [pooled | vox | 1 0..], i.e. 88 of [hid | pooled | vox | 1 0..])
    gs[:, 15] = vec[0:32]            # global_fc.bias
    l0[:, 24] = vec[80:144]          # lr0.bias
    cs[:, 88] = vec[208:272]         # color.0.bias
    ops = [umma_operand(m) for m in (gs, gv, wfc, l0, cs, cv)]
    hi = torch.cat([h.reshape(-1) for h, _ in ops])
    lo = torch.cat([l.reshape(-1) for _, l in ops])
    tag = torch.tensor([UMMA_PACK_TAG, 0, 0, 0], dtype=torch.int32)    # tells this packing from the mma.sync one (same length otherwise)
    packed = torch.cat([hi.view(torch.int32), lo.view(torch.int32), vec.view(torch.int32), tag])
    return packed.to(next(nerf.parameters()).device)


# ------------------------------------------------------------------------------------------ conv3d (csrc/conv3d_mma.cu)
CONV3D_K3_SHAPES = {16: 16, 32: 8, 8: 16}    # Cin -> largest Cout instantiated


def _conv3d_ntiles(cin, cout):
    """n-tiles (of 8 output channels) of the kernel instantiation that serves (cin, cout)."""
    return 2 if cin == 8 else (cout + 7) // 8


def _conv3d_ksteps(cin):
    """k-steps of one (dz,dy) input row: list over steps of 16 (dx, channel) pairs, None = zero weight."""
    if cin == 16:
        return [[(dx, c) for c in range(16)] for dx in range(3)]
    if cin == 32:
        return [[(dx, half * 16 + c) for c in range(16)] for dx in range(3) for half in range(2)]
    if cin == 8:
        return [[(0, c) for c in range(8)] + [(1, c) for c in range(8)],
                [(2, c) for c in range(8)] + [None] * 8]
    raise ValueError(cin)


def fp16_weight_scale(weight):
    """Power of two c with max|weight| * c in [512, 1024): weights packed as fp16(weight * c) keep 11 significant bits
    down to ~1e-7 of the layer's largest weight whatever its absolute magnitude (a layer that consumes a large-valued
    input, e.g. the variance volume of large features, has correspondingly tiny weights: below 6.1e-5 they would be
    fp16 subnormals, below 6e-8 zero).  The kernel divides the result by c (bmv_conv3d_params.in_scale)."""
    import math
    m = float(weight.detach().abs().max())
    if not (m > 0.0) or not math.isfinite(m):
        return 1.0
    return 2.0 ** (9 - math.floor(math.log2(m)))


def pack_conv3d_k3(weight, scale=1.0):
    """weight (Cout, Cin, 3, 3, 3) fp32 -> int32 tensor in the order bmv_conv3d_k3 reads (values multiplied by `scale`,
    a power of two, before the fp16 rounding):
    [dz][dy][k-step j][n-tile][lane = 4g+t] x {b0, b1}; b0 = fp16 pair at K indices (2t, 2t+1) of the k-step,
    b1 at (2t+8, 2t+9), output channel n = nt*8+g (mma.sync.m16n8k16 B fragment); absent channels are zero."""
    Cout, Cin = weight.shape[:2]
    if Cin not in CONV3D_K3_SHAPES or Cout > CONV3D_K3_SHAPES[Cin] or tuple(weight.shape[2:]) != (3, 3, 3):
        raise ValueError(f"conv3d_k3 is not instantiated for weight {tuple(weight.shape)}")
    steps = _conv3d_ksteps(Cin)
    NT = _conv3d_ntiles(Cin, Cout)
    w = torch.zeros(NT * 8, Cin, 3, 3, 3)
    w[:Cout] = weight.detach().float().cpu() * float(scale)
    # B[dz][dy][j][k][n]
    B = torch.zeros(3, 3, len(steps), 16, NT * 8)
    for j, step in enumerate(steps):
        for k, src in enumerate(step):
            if src is not None:
                dx, c = src
                B[:, :, j, k, :] = w[:, c, :, :, dx].permute(1, 2, 0)
    B = B.half()
    lane = torch.arange(32)
    g, t = lane // 4, lane % 4
    out = torch.empty((3, 3, len(steps), NT, 32, 2, 2), dtype=torch.float16)
    for nt in range(NT):
        n = nt * 8 + g
        for r in range(2):
            for e in range(2):
                out[:, :, :, nt, :, r, e] = B[:, :, :, 2 * t + 8 * r + e, n]
    return out.reshape(-1).view(torch.int32).to(weight.device)


CONV3D_K3_UMMA_CIN = (8, 16)            # input channels bmv_conv3d_k3_umma is instantiated for (Cout <= 16)


def pack_conv3d_k3_umma(weight):
    """weight (Cout <= 16, Cin in {8, 16}, 3, 3, 3) fp32 -> int32 tensor in the order bmv_conv3d_k3_umma reads:
    [dz][k-step j] x one STACKED (N=48, K=16) fp16 B operand [W(dz,dy=2); W(dz,1); W(dz,0)] (16 output channels each,
    channels >= Cout zero) in the tcgen05 K-major SWIZZLE_NONE layout ((K/8, 48, 8): SBO = 128 B, LBO = 768 B) — the
    kernel multiplies an input row by a row range of it (the output rows that input row contributes to).
    Cin 16: k-step j = tap dx = j, K = the 16 channels.  Cin 8: k-step j holds taps dx = 2j (K 0..7) and dx = 2j+1
    (K 8..15; dx = 3 does not exist: zeros)."""
    Cout, Cin = weight.shape[:2]
    if Cin not in CONV3D_K3_UMMA_CIN or Cout > 16 or tuple(weight.shape[2:]) != (3, 3, 3):
        raise ValueError(f"conv3d_k3_umma is not instantiated for weight {tuple(weight.shape)}")
    w = torch.zeros(16, Cin, 3, 3, 3)
    w[:Cout] = weight.detach().float().cpu()
    KS = 3 if Cin == 16 else 2
    B = torch.zeros(3, KS, 3, 16, 16)                          # [dz][j][block b <-> dy = 2-b][n][k]
    for j in range(KS):
        for b in range(3):
            dy = 2 - b
            if Cin == 16:
                B[:, j, b] = w[:, :, :, dy, j].permute(2, 0, 1)
            else:
                for half in range(2):
                    dx = 2 * j + half
                    if dx < 3:
                        B[:, j, b, :, 8 * half:8 * half + 8] = w[:, :, :, dy, dx].permute(2, 0, 1)
    B = B.half().reshape(3 * KS, 48, 2, 8).permute(0, 2, 1, 3).contiguous()      # per (dz, j): (K/8, 48, 8)
    return B.reshape(-1).view(torch.int32).to(weight.device)


CONVT3D_K3S2_SHAPES = ((16, 8), (32, 16))


def pack_convT3d_k3s2(weight):
    """ConvTranspose3d weight (Cin, Cout, 3, 3, 3) -> int32 tensor in the order bmv_convT3d_k3s2 reads:
    [tap = (kz*3+ky)*3+kx][k-tile][n-tile][lane = 4g+t] x {b0, b1}: b0 = fp16 pair W[cin = kt*16+2t, +1][cout = nt*8+g],
    b1 the pair at cin + 8."""
    Cin, Cout = weight.shape[:2]
    if (Cin, Cout) not in CONVT3D_K3S2_SHAPES or tuple(weight.shape[2:]) != (3, 3, 3):
        raise ValueError(f"convT3d_k3s2 is not instantiated for weight {tuple(weight.shape)}")
    w = weight.detach().float().cpu().reshape(Cin, Cout, 27).half()
    KT, NT = Cin // 16, Cout // 8
    lane = torch.arange(32)
    g, t = lane // 4, lane % 4
    out = torch.empty((27, KT, NT, 32, 2, 2), dtype=torch.float16)
    for kt in range(KT):
        for nt in range(NT):
            for r in range(2):
                for e in range(2):
                    out[:, kt, nt, :, r, e] = w[kt * 16 + 2 * t + 8 * r + e, nt * 8 + g].T
    return out.reshape(-1).view(torch.int32).to(weight.device)


def pack_conv2d_k3_c32(weight):
    """Conv2d weight (Cout in {8,16}, 32, 3, 3) -> int32 tensor in the order bmv_fpn_topdown_smooth reads:
    [dy][j = dx*2 + half][n-tile][lane = 4g+t] x {b0, b1}; K index kk of k-step j is input channel half*16 + kk."""
    Cout, Cin = weight.shape[:2]
    if Cin != 32 or Cout not in (8, 16) or tuple(weight.shape[2:]) != (3, 3):
        raise ValueError(f"conv2d_k3_c32 is not instantiated for weight {tuple(weight.shape)}")
    w = weight.detach().float().cpu().half()                  # (Cout, 32, dy, dx)
    NT = Cout // 8
    lane = torch.arange(32)
    g, t = lane // 4, lane % 4
    out = torch.empty((3, 6, NT, 32, 2, 2), dtype=torch.float16)
    for j in range(6):
        dx, half = j // 2, j % 2
        for nt in range(NT):
            for r in range(2):
                for e in range(2):
                    out[:, j, nt, :, r, e] = w[nt * 8 + g, half * 16 + 2 * t + 8 * r + e, :, dx].T
    return out.reshape(-1).view(torch.int32).to(weight.device)


def pack_conv2d_k3(weight):
    """Conv2d weight (Cout, Cin, 3, 3), Cin in {16, 32, 64}, Cout in {16, 32} -> int32 tensor in the order bmv_conv2d_k3
    reads: [dy][j = dx * (Cin/16) + part][n-tile][lane = 4g+t] x {b0, b1}; K index kk of k-step j is input channel
    part*16 + kk; column g of n-tile nt is output channel (g//2) * 2NT + 2nt + g%2 (a lane's C fragments then hold 2NT
    consecutive channels of a pixel)."""
    Cout, Cin = weight.shape[:2]
    if Cin not in (16, 32, 64) or Cout not in (16, 32) or tuple(weight.shape[2:]) != (3, 3):
        raise ValueError(f"conv2d_k3 is not instantiated for weight {tuple(weight.shape)}")
    w = weight.detach().float().cpu().half()                  # (Cout, Cin, dy, dx)
    NT, KPD = Cout // 8, Cin // 16
    lane = torch.arange(32)
    g, t = lane // 4, lane % 4
    out = torch.empty((3, 3 * KPD, NT, 32, 2, 2), dtype=torch.float16)
    for j in range(3 * KPD):
        dx, part = j // KPD, j % KPD
        for nt in range(NT):
            ch = (g // 2) * (2 * NT) + nt * 2 + (g % 2)
            for r in range(2):
                for e in range(2):
                    out[:, j, nt, :, r, e] = w[ch, part * 16 + 2 * t + 8 * r + e, :, dx].T
    return out.reshape(-1).view(torch.int32).to(weight.device)


def pack_conv1x1_after(weight):
    """1x1 Conv2d weight (32, 32[, 1, 1]) applied to the output of a 32-channel bmv_conv2d_k3 layer inside its epilogue:
    [k-step kk][n-tile][lane] x {b0, b1}.  The A fragments are that layer's C fragments, so K index 2t+e (+8 for r = 1)
    of k-step kk is ITS channel t*8 + (2kk + r)*2 + e; output columns permuted like pack_conv2d_k3's."""
    w = weight.detach().float().cpu().reshape(weight.shape[0], weight.shape[1]).half()
    if tuple(w.shape) != (32, 32):
        raise ValueError(f"conv1x1_after is instantiated for 32 -> 32 channels, got {tuple(weight.shape)}")
    lane = torch.arange(32)
    g, t = lane // 4, lane % 4
    out = torch.empty((2, 4, 32, 2, 2), dtype=torch.float16)
    for kk in range(2):
        for nt in range(4):
            ch = (g // 2) * 8 + nt * 2 + (g % 2)
            for r in range(2):
                for e in range(2):
                    out[kk, nt, :, r, e] = w[ch, t * 8 + (2 * kk + r) * 2 + e]
    return out.reshape(-1).view(torch.int32).to(weight.device)


def pack_conv2d_k3_c8(weight):
    """Conv2d weight (8, 8, 3, 3) -> int32 tensor (384,) in the order bmv_fpn_stem reads: [dy][k-step j][lane] x {b0, b1};
    k-step 0 holds taps dx = 0 (K 0..7) and dx = 1 (K 8..15), k-step 1 holds dx = 2 and zeros."""
    if tuple(weight.shape) != (8, 8, 3, 3):
        raise ValueError(f"conv2d_k3_c8 needs an (8,8,3,3) weight, got {tuple(weight.shape)}")
    w = weight.detach().float().cpu()
    B = torch.zeros(3, 2, 16, 8)                              # [dy][j][k][n]
    for dx in range(3):
        j, k0 = dx // 2, (dx % 2) * 8
        B[:, j, k0:k0 + 8, :] = w[:, :, :, dx].permute(2, 1, 0)
    B = B.half()
    lane = torch.arange(32)
    g, t = lane // 4, lane % 4
    out = torch.empty((3, 2, 32, 2, 2), dtype=torch.float16)
    for r in range(2):
        for e in range(2):
            out[:, :, :, r, e] = B[:, :, 2 * t + 8 * r + e, g]
    return out.reshape(-1).view(torch.int32).to(weight.device)


# ------------------------------------------------------------------------------------------ MVSNeRF MLP (csrc/mvs_render_umma.cu)
def _umma_b(w_pad):
    """(N, K) fp32 -> fp16 (K/8, N, 8): the K-major SWIZZLE_NONE B operand (SBO 128 B, LBO N*16 B), flattened."""
    N, K = w_pad.shape
    assert K % 16 == 0 and N % 8 == 0
    return w_pad.half().reshape(N, K // 8, 8).permute(1, 0, 2).contiguous().reshape(-1)


def pack_mvs_weights_umma(mlp):
    """RendererOurs (modules_mvs.py; reference lib/networks/mvsnerf/network.py:152-229) -> the byte buffer
    bmv_mvs_render_umma streams: 16 weight panels in issue order, the bias K-steps of L1..L4 and the feature layer, the
    fp32 vectors of the CUDA-core heads.  Biases of the other layers sit in the column that multiplies the operands'
    constant 1 (pts col 63, feats col 20, views col 3)."""
    n = mlp.nerf if hasattr(mlp, 'nerf') else mlp
    f32 = lambda t: t.detach().float().cpu()
    W = [f32(l.weight) for l in n.pts_linears]
    B = [f32(l.bias) for l in n.pts_linears]
    if n.in_pts != 63 or n.in_feat != 20 or n.in_views != 3 or W[1].shape != (128, 128) or tuple(n.skips) != (4,) or len(W) != 6:
        raise ValueError("pack_mvs_weights_umma: instantiated for D=6, W=128, in_pts=63, in_feat=20, in_views=3, skips=(4,)")
    panels = []
    wg = torch.zeros(128, 32); wg[:, :20] = f32(n.pts_bias.weight); wg[:, 20] = f32(n.pts_bias.bias)
    panels.append(_umma_b(wg))
    w0 = torch.zeros(128, 64); w0[:, :63] = W[0]; w0[:, 63] = B[0]
    panels.append(_umma_b(w0))
    for i in range(1, 5):
        panels += [_umma_b(W[i][:, :64].contiguous()), _umma_b(W[i][:, 64:].contiguous())]
    w5p = torch.zeros(128, 64); w5p[:, :63] = W[5][:, :63]; w5p[:, 63] = B[5]
    panels.append(_umma_b(w5p))
    w5h = W[5][:, 63:]
    panels += [_umma_b(w5h[:, :64].contiguous()), _umma_b(w5h[:, 64:].contiguous())]
    wf = f32(n.feature_linear.weight)
    panels += [_umma_b(wf[:, :64].contiguous()), _umma_b(wf[:, 64:].contiguous())]
    wv = torch.zeros(64, 144)
    vw = f32(n.views_linears[0].weight)                     # (64, 128 + 3): [feature | views]
    wv[:, :128] = vw[:, :128]; wv[:, 128:131] = vw[:, 128:131]; wv[:, 131] = f32(n.views_linears[0].bias)
    panels.append(_umma_b(wv))
    biases = []
    for b in (B[1], B[2], B[3], B[4], f32(n.feature_linear.bias)):
        m = torch.zeros(128, 16); m[:, 4] = b                # K index 4 of the step = feats column 20 (the constant 1)
        biases.append(_umma_b(m))
    vec = torch.zeros(328)
    vec[0:128] = f32(n.alpha_linear.weight).reshape(-1)
    vec[128:320] = f32(n.rgb_linear.weight).reshape(-1)
    vec[320] = f32(n.alpha_linear.bias)[0]
    vec[321:324] = f32(n.rgb_linear.bias)
    half = torch.cat(panels + biases)
    assert half.numel() * 2 == 256000 + 5 * 4096, half.numel()
    packed = torch.cat([half.view(torch.int32), vec.view(torch.int32)])
    return packed.to(next(n.parameters()).device)
