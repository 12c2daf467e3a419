"""Output sinks of the per-frame path (SURVEY.md §8 row f4): the parts of the reference's `Evaluator` and `Visualizer`
that touch every pixel of every frame, done on the device so that 4 instead of 16 bytes per pixel cross PCIe and the
host never loops over a frame.

  * `FrameEvaluator.evaluate(output, batch)`  — reference lib/evaluators/enerf.py:37-71: per rendered level, the
    prediction against `batch['rgb_{i}']` (uploaded once for both metrics) with the optional 10 % centre crop
    (`cfg.enerf.eval_center`):
      - PSNR under `batch['msk_{i}']` (>= 1), = 10 log10(1 / mse) as skimage.metrics.peak_signal_noise_ratio(data_range=1)
        computes it (float64 mean of squared differences);
      - SSIM as skimage.metrics.structural_similarity(channel_axis=-1, win_size, data_range) computes it with uniform
        weights (float64; no mask: skimage has none).  The reference does not record its SSIM arguments; the defaults
        win_size=7, data_range=2.0 are skimage's for a float image.
    Both stay on the device until `summarize()`, which reads them back and returns the means over frames of the last
    level, {'psnr', 'ssim'}, like `Evaluator.summarize` (:104-106); `scene_psnrs` / `scene_ssims` hold every level per
    scene.  `PsnrAccumulator` is its PSNR-only configuration.  LPIPS needs the VGG weights of the `lpips` package and
    stays out of scope.
  * `FrameWriter.visualize(output, batch)` — reference lib/visualizers/enerf.py:21-37: uint8 colour image and
    min/max-normalised uint8 depth image of the last level; returned as host arrays (and written as binary PPM / PGM when
    `result_dir` is given; the reference writes JPEG through imageio, a host library that is not part of the path).
"""
import math
import os

import torch

from . import ops


class FrameEvaluator:
    def __init__(self, rc, eval_center=False, ssim=True, win_size=7, data_range=2.0):
        self.rc, self.eval_center = rc, bool(eval_center)
        self.ssim, self.win_size, self.data_range = bool(ssim), int(win_size), float(data_range)
        self._pending = []            # (level, scene, device (sse, count), device ssim or None): read back in summarize()
        self.psnrs, self.scene_psnrs = [], {}
        self.ssims, self.scene_ssims = [], {}

    def evaluate(self, output, batch):
        rc = self.rc
        B, _, _, H, W = batch['src_inps'].shape
        for i in range(rc.num):
            if not rc.render_if[i]:
                continue
            h, w = int(H * rc.render_scale[i]), int(W * rc.render_scale[i])
            crop = (int(h * 0.1), int(w * 0.1)) if self.eval_center else (0, 0)
            for b in range(B):
                pred = output[f'rgb_level{i}'][b]
                gt = batch[f'rgb_{i}'][b].to(pred.device, non_blocking=True).reshape(-1, 3).float()
                msk = batch.get(f'msk_{i}')
                m8 = None if msk is None else (msk[b].to(pred.device, non_blocking=True).reshape(-1) >= 1).to(torch.uint8)
                acc = ops.frame_psnr_accumulate(pred, gt, h, w, mask=m8, crop=crop)
                ssim = ops.frame_ssim(pred, gt, h, w, crop=crop, win_size=self.win_size,
                                      data_range=self.data_range) if self.ssim else None
                self._pending.append((i, batch['meta']['scene'][b], acc, ssim))

    def _drain(self):
        for i, scene, (sse, cnt), ssim in self._pending:
            n = int(cnt.item())
            mse = float(sse.item()) / n if n else float('nan')
            psnr = 10.0 * math.log10(1.0 / mse) if mse > 0 else float('inf')
            if i == self.rc.num - 1:
                self.psnrs.append(psnr)
            self.scene_psnrs.setdefault(f'{scene}_level{i}', []).append(psnr)
            if ssim is not None:
                ssim = float(ssim.item())
                if i == self.rc.num - 1:
                    self.ssims.append(ssim)
                self.scene_ssims.setdefault(f'{scene}_level{i}', []).append(ssim)
        self._pending = []

    def summarize(self):
        self._drain()
        out = {'psnr': sum(self.psnrs) / len(self.psnrs) if self.psnrs else float('nan')}
        if self.ssim:
            out['ssim'] = sum(self.ssims) / len(self.ssims) if self.ssims else float('nan')
        return out


class PsnrAccumulator(FrameEvaluator):
    def __init__(self, rc, eval_center=False):
        super().__init__(rc, eval_center, ssim=False)


class FrameWriter:
    def __init__(self, rc, result_dir=None):
        self.rc, self.result_dir = rc, result_dir
        self.imgs, self.depths = [], []
        if result_dir:
            os.makedirs(os.path.join(result_dir, 'imgs'), exist_ok=True)

    def visualize(self, output, batch):
        rc = self.rc
        B, _, _, H, W = batch['src_inps'].shape
        if B != 1:
            raise ValueError("FrameWriter handles one frame per call (the reference asserts B == 1)")
        i = rc.num - 1
        h, w = int(H * rc.render_scale[i]), int(W * rc.render_scale[i])
        rgb_u8, dpt_u8, _ = ops.frame_to_u8(output[f'rgb_level{i}'][0], output[f'depth_level{i}'][0])
        rgb = rgb_u8.reshape(h, w, 3).cpu().numpy()
        dpt = dpt_u8.reshape(h, w).cpu().numpy()
        self.imgs.append(rgb)
        self.depths.append(dpt)
        if self.result_dir:
            fid = int(batch['meta']['frame_id'][0])
            with open(os.path.join(self.result_dir, 'imgs', f'{fid:06d}_rgb.ppm'), 'wb') as fh:
                fh.write(b'P6\n%d %d\n255\n' % (w, h) + rgb.tobytes())
            with open(os.path.join(self.result_dir, 'imgs', f'{fid:06d}_dpt.pgm'), 'wb') as fh:
                fh.write(b'P5\n%d %d\n255\n' % (w, h) + dpt.tobytes())
        return rgb, dpt
