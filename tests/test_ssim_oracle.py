"""oracle/ssim_oracle.frame_ssim (uniform-filter moments, the way skimage computes SSIM) against an independent
brute-force float64 evaluation: every interior pixel's own window, np.var(ddof=1) and the ddof=1 covariance."""
import numpy as np
import pytest

from oracle import ssim_oracle as SSO


def _brute_ssim(pred, gt, win, data_range, eval_center):
    h, w = pred.shape[:2]
    if eval_center:
        ch, cw = int(h * 0.1), int(w * 0.1)
        pred, gt = pred[ch:h - ch, cw:w - cw], gt[ch:h - ch, cw:w - cw]
    c1, c2 = (0.01 * data_range) ** 2, (0.03 * data_range) ** 2
    vals = []
    for c in range(3):
        x, y = pred[..., c].astype(np.float64), gt[..., c].astype(np.float64)
        s = []
        for i in range(x.shape[0] - win + 1):
            for j in range(x.shape[1] - win + 1):
                a, b = x[i:i + win, j:j + win].ravel(), y[i:i + win, j:j + win].ravel()
                ua, ub = a.mean(), b.mean()
                va, vb = np.var(a, ddof=1), np.var(b, ddof=1)
                vab = ((a - ua) * (b - ub)).sum() / (a.size - 1)
                s.append((2 * ua * ub + c1) * (2 * vab + c2) / ((ua ** 2 + ub ** 2 + c1) * (va + vb + c2)))
        vals.append(np.mean(s))
    return np.mean(vals)


@pytest.mark.parametrize("win", [3, 7, 11])
@pytest.mark.parametrize("data_range", [1.0, 2.0])
@pytest.mark.parametrize("eval_center", [False, True])
def test_frame_ssim_oracle_matches_brute_force(win, data_range, eval_center):
    rs = np.random.RandomState(win * 10 + int(data_range) + 2 * eval_center)
    gt = rs.rand(21, 27, 3).astype(np.float32)
    pred = np.clip(gt + 0.1 * rs.randn(21, 27, 3), 0, 1).astype(np.float32)
    want = _brute_ssim(pred, gt, win, data_range, eval_center)
    got = SSO.frame_ssim(pred, gt, win_size=win, data_range=data_range, eval_center=eval_center)
    assert abs(got - want) <= 1e-12, (got, want)
