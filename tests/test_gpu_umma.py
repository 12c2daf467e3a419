"""GPU tests of the tcgen05 (UMMA) plumbing:
  * bmv_umma_selftest (csrc/umma_selftest.cu) — one 128-row tile through the descriptor / TMEM / commit / tcgen05.ld
    helpers of umma.cuh that the tcgen05 kernels use, against a float64 matmul (isolates the tensor-memory plumbing
    from the renderers; the one-launch tcgen05 render is tested in test_gpu_render_multi.py);
  * ops.render_rays, the per-chain render, refuses the 'umma' engine."""
import pytest
import torch

from conftest import load_golden
from test_gpu_parity import H, W, TRIPLE, _cams, close

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    from boostmvsnerfs_b200 import ops as _ops
    return _ops


@pytest.fixture(scope="module")
def g():
    return load_golden("enerf_ops.npz")


@pytest.mark.parametrize("N,K", [(64, 32), (16, 32), (32, 16), (64, 96), (256, 16)])
def test_umma_selftest_matches_float64_matmul(ops, N, K):
    torch.manual_seed(N * 100 + K)
    a = torch.randn(128, K, device="cuda")
    w = torch.randn(N, K)
    d = ops.umma_selftest(a, w)
    ref = (a.double().cpu() @ w.double().T).float()
    close(d, ref, f"tcgen05 tile N={N} K={K} vs float64", rtol=2e-6)
    # rows and columns land where the layout says: a one-hot A row picks one row of W
    a1 = torch.zeros(128, K, device="cuda")
    a1[torch.arange(128), torch.arange(128) % K] = 1.0
    d1 = ops.umma_selftest(a1, w)
    close(d1, w.T[torch.arange(128) % K], "one-hot rows", rtol=2e-6)


def test_umma_render_rejects_wrong_packing(ops, g):
    from boostmvsnerfs_b200 import mlp_pack
    from boostmvsnerfs_b200._lib import BmvError
    from boostmvsnerfs_b200.modules import NeRF
    net = NeRF(feat_ch=11).eval().cuda()
    cams = _cams(ops, g)
    args = (g.t("depth_l1", "cuda")[0], g.t("std_l1", "cuda")[0], g.t("near_far_l1", "cuda")[0],
            g.t("in_rays_1", "cuda")[0], H, W, False, 2, g.t("in_regvol1", "cuda")[0], g.t("in_imfeat2", "cuda")[0],
            g.t("in_src_inps", "cuda")[0], cams, TRIPLE)
    # the per-chain render has no tcgen05 engine (render_multi_umma.cu renders all chains in one launch): 'umma' is an
    # unknown engine whatever the packing
    for packed in (mlp_pack.pack_nerf_weights_umma(net), mlp_pack.pack_nerf_weights_mma(net)):
        with pytest.raises(BmvError):
            ops.render_rays(*args, packed, engine="umma")
