"""Device SSIM (ops.frame_ssim / bmv_frame_ssim) and the two-metric evaluator sink against the float64 restatement of
skimage's structural_similarity (oracle/ssim_oracle.frame_ssim)."""
import numpy as np
import pytest
import torch

from boostmvsnerfs_b200.config import RenderConfig
from oracle import sinks_oracle as SO
from oracle import ssim_oracle as SSO

pytestmark = pytest.mark.gpu


def _images(kind, H, W, seed):
    rs = np.random.RandomState(seed)
    if kind == "random":
        return rs.rand(H, W, 3).astype(np.float32), rs.rand(H, W, 3).astype(np.float32)
    if kind == "flat":            # variance ~1e-8: the uxx - ux² cancellation
        return ((0.5 + 1e-4 * rs.randn(H, W, 3)).astype(np.float32), (0.5 + 1e-4 * rs.randn(H, W, 3)).astype(np.float32))
    gt = rs.rand(H, W, 3).astype(np.float32)
    return np.clip(gt + 0.05 * rs.randn(H, W, 3), 0, 1).astype(np.float32), gt


def _ssim(pred, gt, **kw):
    from boostmvsnerfs_b200 import ops
    H, W = pred.shape[:2]
    return ops.frame_ssim(torch.from_numpy(pred).cuda().reshape(-1, 3), torch.from_numpy(gt).cuda().reshape(-1, 3), H, W, **kw)


def _crop(H, W, center):
    return (int(H * 0.1), int(W * 0.1)) if center else (0, 0)


_CASES = [(H, W, win) for H, W in [(64, 96), (33, 47), (544, 960)] for win in (7, 11)] + [(544, 960, 101)]


@pytest.mark.parametrize("H,W,win", _CASES)
@pytest.mark.parametrize("data_range", [1.0, 2.0])
@pytest.mark.parametrize("center", [False, True])
@pytest.mark.parametrize("kind", ["random", "flat", "noisy"])
def test_frame_ssim_matches_oracle(H, W, win, data_range, center, kind):
    pred, gt = _images(kind, H, W, H * W + win)
    want = SSO.frame_ssim(pred, gt, win_size=win, data_range=data_range, eval_center=center)
    got = _ssim(pred, gt, crop=_crop(H, W, center), win_size=win, data_range=data_range)
    assert got.dtype == torch.float64 and got.shape == (1,)
    assert abs(float(got.item()) - want) <= 1e-9, (float(got.item()), want)


@pytest.mark.parametrize("H,W", [(64, 96), (544, 960)])
def test_frame_ssim_properties(H, W):
    pred, gt = _images("noisy", H, W, 7)
    assert abs(float(_ssim(gt, gt).item()) - 1.0) <= 1e-12
    a = _ssim(pred, gt, crop=_crop(H, W, True)).item()
    b = _ssim(gt, pred, crop=_crop(H, W, True)).item()
    assert abs(a - b) <= 1e-15, (a, b)
    # deterministic reduction: per-CTA partials summed in a fixed order
    assert _ssim(pred, gt, win_size=11).item() == _ssim(pred, gt, win_size=11).item()


def test_frame_ssim_graph_replay_is_bit_exact():
    from boostmvsnerfs_b200 import ops
    pred, gt = _images("noisy", 544, 960, 11)
    p, g = torch.from_numpy(pred).cuda().reshape(-1, 3), torch.from_numpy(gt).cuda().reshape(-1, 3)
    eager = ops.frame_ssim(p, g, 544, 960, crop=(54, 96)).item()
    out = torch.zeros(1, device="cuda", dtype=torch.float64)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ops.frame_ssim(p, g, 544, 960, crop=(54, 96), out=out)      # warm-up off the capturing stream
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        ops.frame_ssim(p, g, 544, 960, crop=(54, 96), out=out)
    out.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert out.item() == eager


def test_frame_ssim_rejects_bad_arguments():
    from boostmvsnerfs_b200 import ops
    from boostmvsnerfs_b200._lib import BmvError
    p = torch.rand(40 * 50, 3, device="cuda")
    g = torch.rand(40 * 50, 3, device="cuda")
    with pytest.raises(BmvError, match="win_size"):
        ops.frame_ssim(p, g, 40, 50, win_size=8)
    with pytest.raises(BmvError, match="win_size"):
        ops.frame_ssim(p, g, 40, 50, crop=(4, 5), win_size=33)    # 32 rows left after the crop
    with pytest.raises(BmvError, match="pixels"):
        ops.frame_ssim(p, g[:-1], 40, 50)
    with pytest.raises(BmvError, match="CUDA"):
        ops.frame_ssim(p.cpu(), g, 40, 50)
    with pytest.raises(BmvError, match="data_range"):
        ops.frame_ssim(p, g, 40, 50, data_range=0.0)
    assert abs(ops.frame_ssim(p, g, 40, 50, crop=(4, 5), win_size=31).item()
               - SSO.frame_ssim(p.cpu().numpy().reshape(40, 50, 3), g.cpu().numpy().reshape(40, 50, 3), 31, 2.0, True)) <= 1e-9


def test_frame_evaluator_mirrors_evaluator():
    """FrameEvaluator on a rendered frame, twice: PSNR and SSIM as the restated reference arithmetic computes them;
    PsnrAccumulator (its PSNR-only configuration) gives the same PSNR."""
    from boostmvsnerfs_b200 import network, sinks
    from boostmvsnerfs_b200.synth import batch_to, make_scene
    rc = RenderConfig.enerf_eval(2)
    torch.manual_seed(0)
    net = network.BoostEnerfNetwork(preprocess=True, rc=rc).eval().cuda()
    net.view_selection_outputs = {"synth_0": [1, 2]}
    scene = make_scene(H=64, W=96, n_views=4, seed=0, smooth=True)
    batch = batch_to(scene, "cuda")
    out = net(batch)
    rs = np.random.RandomState(0)
    gt = rs.rand(1, 64 * 96, 3).astype(np.float32)
    msk = (rs.rand(1, 64 * 96) > 0.2).astype(np.uint8)
    batch["rgb_1"], batch["msk_1"] = torch.from_numpy(gt), torch.from_numpy(msk)
    ev = sinks.FrameEvaluator(rc, eval_center=True)
    ev.evaluate(out, batch)
    ev.evaluate(out, batch)
    pa = sinks.PsnrAccumulator(rc, eval_center=True)
    pa.evaluate(out, batch)
    pred = out["rgb_level1"][0].cpu().numpy().reshape(64, 96, 3)
    gt3 = gt[0].reshape(64, 96, 3)
    want_psnr = SO.frame_psnr(pred, gt3, msk[0].reshape(64, 96), eval_center=True)
    want_ssim = SSO.frame_ssim(pred, gt3, win_size=7, data_range=2.0, eval_center=True)
    got = ev.summarize()
    assert set(got) == {"psnr", "ssim"}
    assert abs(got["psnr"] - want_psnr) < 1e-9 * abs(want_psnr) and abs(got["ssim"] - want_ssim) < 1e-9, (got, want_ssim)
    assert len(ev.scene_psnrs["synth_level1"]) == 2 and len(ev.scene_ssims["synth_level1"]) == 2
    only_psnr = pa.summarize()
    assert set(only_psnr) == {"psnr"} and abs(only_psnr["psnr"] - want_psnr) < 1e-9 * abs(want_psnr)
