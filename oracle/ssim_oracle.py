"""TEST INFRASTRUCTURE — CPU restatement (numpy / scipy, float64) of the SSIM the reference's evaluator takes from skimage.

Only tests/, tools/ and __graft_entry__.smoke() may import this module.

Parity pin: the reference's Evaluator calls skimage (lib/evaluators/enerf.py), which is not installed in this image.
`frame_ssim` restates skimage.metrics.structural_similarity(im1, im2, channel_axis=-1, win_size=w, data_range=R) with
uniform weights as scikit-image 0.19 / 0.20 compute it (the versions that still take the reference's
`multichannel=True` era of calls), in float64 throughout, with scipy.ndimage.uniform_filter, the filter skimage calls.
SURVEY.md records only "PSNR/SSIM (skimage)": the reference's win_size / data_range are not recorded, so they are
parameters here, and masks do not enter (skimage has no masked SSIM) — **parity unpinned** against the library
itself; the arithmetic is checked against a brute-force per-window float64 evaluation in tests/test_ssim_oracle.py.
"""
import numpy as np


def frame_ssim(pred, gt, win_size=7, data_range=2.0, eval_center=False):
    """pred, gt (h,w,3) float32.  The eval-centre crop (int(0.1 h), int(0.1 w) at each border) is applied first, as the
    reference slices the arrays before calling the metric.  Per channel: ux, uy, uxx, uyy, uxy = window means;
    vx = w²/(w²-1) (uxx - ux²) (sample covariance, skimage's default), likewise vy, vxy; C1 = (0.01 R)², C2 = (0.03 R)²;
    S = (2 ux uy + C1)(2 vxy + C2) / ((ux² + uy² + C1)(vx + vy + C2)), averaged in float64 over the pixels whose window
    lies inside the image (skimage drops pad = (w-1)/2 at every border); the frame's SSIM is the mean over channels.
    win_size 7 and data_range 2 are skimage's defaults for a float image (dtype_range[float32] = (-1, 1))."""
    from scipy.ndimage import uniform_filter
    h, w = pred.shape[:2]
    if eval_center:
        ch, cw = int(h * 0.1), int(w * 0.1)
        pred, gt = pred[ch:h - ch, cw:w - cw], gt[ch:h - ch, cw:w - cw]
    pad = (win_size - 1) // 2
    n = win_size * win_size
    cov_norm = n / (n - 1)
    c1, c2 = (0.01 * data_range) ** 2, (0.03 * data_range) ** 2
    vals = []
    for c in range(pred.shape[2]):
        x, y = pred[..., c].astype(np.float64), gt[..., c].astype(np.float64)
        ux, uy = uniform_filter(x, size=win_size), uniform_filter(y, size=win_size)
        uxx, uyy, uxy = (uniform_filter(a, size=win_size) for a in (x * x, y * y, x * y))
        vx, vy, vxy = cov_norm * (uxx - ux * ux), cov_norm * (uyy - uy * uy), cov_norm * (uxy - ux * uy)
        s = (2 * ux * uy + c1) * (2 * vxy + c2) / ((ux ** 2 + uy ** 2 + c1) * (vx + vy + c2))
        vals.append(s[pad:s.shape[0] - pad, pad:s.shape[1] - pad].mean(dtype=np.float64))
    return float(np.mean(vals))
