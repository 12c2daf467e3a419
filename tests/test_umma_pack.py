"""CPU tests of the tcgen05 weight packing (mlp_pack.pack_nerf_weights_umma, csrc/nerf_umma_pack.cuh) and of the
dataflow of csrc/render_multi_umma.cu: the packed words are read back through the same shared-memory descriptor
arithmetic the kernel programs (start + (n/8)*SBO + (k/8)*LBO + (n%8)*16 + (k%8)*2 bytes, SBO = 128, LBO = N*16), and
the six matrices + vectors, applied in the kernel's phase order, reproduce the torch NeRF module."""
import numpy as np
import torch

from boostmvsnerfs_b200 import mlp_pack
from boostmvsnerfs_b200.modules import NeRF

# kernel constants (csrc/nerf_umma_pack.cuh, read by csrc/render_multi_umma.cu)
MATS = [("GS", 32, 32), ("GV", 32, 16), ("FC", 16, 32), ("L0", 64, 32), ("CS", 64, 96), ("CV", 64, 16)]
UW_BLOCK = sum(n * k * 2 for _, n, k in MATS)
UV = dict(BG=0, WA=32, BFC=64, BL=80, WS=144, BC=208, W2=272, WV=336, BV=384, SC=396, TAG=400, COUNT=404)


def _net(seed=0):
    torch.manual_seed(seed)
    net = NeRF(feat_ch=11).eval()
    for prm in net.parameters():
        if prm.dim() == 1:
            prm.data.normal_(0, 0.2)
    return net


def _read_operand(block, off, N, K):
    """(N,K) fp16 matrix as a tcgen05 K-major SWIZZLE_NONE descriptor with SBO=128, LBO=N*16 addresses it."""
    out = np.zeros((N, K), np.float16)
    h = block.view(np.float16)
    for n in range(N):
        for k in range(K):
            byte = off + (n // 8) * 128 + (k // 8) * (N * 16) + (n % 8) * 16 + (k % 8) * 2
            out[n, k] = h[byte // 2]
    return out


def _unpack(packed):
    raw = packed.cpu().numpy().view(np.uint8)
    assert raw.size == 2 * UW_BLOCK + UV["COUNT"] * 4
    hi, lo = raw[:UW_BLOCK], raw[UW_BLOCK:2 * UW_BLOCK]
    vec = raw[2 * UW_BLOCK:].view(np.float32)
    mats, off = {}, 0
    for name, N, K in MATS:
        mats[name] = (_read_operand(hi, off, N, K).astype(np.float64) + _read_operand(lo, off, N, K).astype(np.float64))
        off += N * K * 2
    return mats, vec.astype(np.float64)


def test_umma_block_size_matches_kernel_constants():
    assert UW_BLOCK == 22528
    assert mlp_pack.pack_nerf_weights_umma(_net()).numel() * 4 == 2 * UW_BLOCK + 1616


def test_umma_operand_round_trip():
    torch.manual_seed(1)
    w = torch.randn(32, 48)
    words = mlp_pack.pack_umma_matrix(w).numpy().view(np.uint8)
    half = words.size // 2
    got = (_read_operand(words[:half], 0, 32, 48).astype(np.float64) + _read_operand(words[half:], 0, 32, 48).astype(np.float64))
    assert np.abs(got - w.double().numpy()).max() < 2 ** -20 * float(w.abs().max())


def test_umma_dataflow_reproduces_the_module():
    net = _net(3)
    M, vec = _unpack(mlp_pack.pack_nerf_weights_umma(net))
    P = 64
    torch.manual_seed(7)
    vox = torch.randn(1, P, 8)
    img = torch.randn(1, P, 3, 15)
    img[..., 8:11] = torch.rand(1, P, 3, 3)
    with torch.no_grad():
        ref = net.double()(vox.double(), img.double())[0].numpy()
    f = img[0].double().numpy()                      # (P,3,15)
    vx = vox[0].double().numpy()
    relu = lambda a: np.maximum(a, 0)
    v = lambda name, n: vec[UV[name]:UV[name] + n]
    # phase A
    wv, bv = v("WV", 48).reshape(12, 4)[:11], v("BV", 12)[:11]
    x = f[:, :, :11] + relu(f[:, :, 11:15] @ wv.T + bv)          # (P,3,11)
    mean = x.mean(1)
    var = ((x - mean[:, None]) ** 2).sum(1) / 2
    pad = lambda a, n: np.concatenate([a, np.zeros(a.shape[:-1] + (n - a.shape[-1],))], -1)
    var16 = pad(var, 16); var16[:, 15] = 1.0                     # bias column of global_fc
    a_gs = np.concatenate([var16, pad(mean, 16)], -1)            # K = 32
    S = a_gs @ M["GS"].T
    G = relu(S[:, None] + pad(x, 16) @ M["GV"].T)                # (P,3,32)
    # phase B
    lg = relu(G @ v("WA", 32) + vec[UV["SC"]])
    wts = np.exp(lg - lg.max(1, keepdims=True)); wts /= wts.sum(1, keepdims=True)
    im = (G * wts[..., None]).sum(1)
    pooled = relu(im @ M["FC"].T + v("BFC", 16))
    # phase C/D
    one = np.zeros((P, 8)); one[:, 0] = 1.0                      # bias column of lr0 / color.0
    a_pv = np.concatenate([pooled, vx, one], -1)                 # K = 32
    hid = relu(a_pv @ M["L0"].T)
    sig = hid @ v("WS", 64) + vec[UV["SC"] + 1]
    sig = np.where(sig > 20, sig, np.log1p(np.exp(sig)))
    # phase E
    Sc = np.concatenate([hid, a_pv], -1) @ M["CS"].T
    Pc = pad(f, 16) @ M["CV"].T                                  # (P,3,64)
    cl = relu(relu(Sc[:, None] + Pc) @ v("W2", 64) + vec[UV["SC"] + 2])
    beta = np.exp(cl - cl.max(1, keepdims=True)); beta /= beta.sum(1, keepdims=True)
    rgb = (f[:, :, 8:11] * beta[..., None]).sum(1)
    out = np.concatenate([rgb, sig[:, None]], -1)
    assert np.abs(out - ref).max() < 2e-5 * np.abs(ref).max()
