"""Drop-in `Network` for the MVSNeRF + boost backbone (reference
lib/networks/boost_mvsnerf/network.py:11-211; single-volume baseline
lib/networks/mvsnerf/network.py:1092-1126).  Sub-module attribute names (`feature`, `cost_reg_2`,
`nerf`) are fixed by the reference checkpoints.  The cost volume (K1b), marching/fetch (K3b) and the
blend (K4) run in libbmv; the CNNs and the 6x128 MLP stay on cuDNN/cuBLAS (north_star).
The reference hard-codes B=1 on this path (boost_mvsnerf/network.py:116-117); so does this class.
"""
import itertools
import json
import os

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops
from .config import RenderConfig
from .modules_mvs import MvsCostRegNet, MvsFeatureNet, MvsNerfMlp

PAD = 24


class BoostMvsnerfNetwork(nn.Module):
    def __init__(self, preprocess=False, rc: RenderConfig = None, view_selection_file=None):
        super().__init__()
        self.rc = rc or RenderConfig.mvsnerf_eval()
        self.feature = MvsFeatureNet()
        self.cost_reg_2 = MvsCostRegNet(32 + 9)
        self.nerf = MvsNerfMlp()
        self.view_selection_outputs = {}
        self.mlp_chunk_bytes = 1 << 30         # bound on the materialised (chunk,S,86) MLP input
        self.volume_dtype = torch.float32      # torch.bfloat16: BASELINE config 3 (1e-2 tolerance)
        self.mlp_engine = 'cublas'             # 'umma': K3b + MLP fused on tcgen05 (fp16 operands: TF32-class, config 3)
        self._packed = None
        self.stage_timer = None
        if not preprocess:
            if view_selection_file is None or not os.path.exists(view_selection_file):
                raise FileNotFoundError("View selection file not found. Please run view selection first.")
            with open(view_selection_file, 'r') as fh:
                self.view_selection_outputs = json.load(fh)

    def _stage(self, name):
        from .network import _NullCtx
        return _NullCtx() if self.stage_timer is None else self.stage_timer(name)

    def _check(self, batch):
        if self.training:
            raise RuntimeError("boostmvsnerfs_b200 networks are inference-only (call .eval())")
        if batch['all_src_inps'].device.type != 'cuda':
            raise RuntimeError("boostmvsnerfs_b200 has no CPU path: move the batch and the module to a CUDA device")
        if batch['all_src_inps'].shape[0] != 1:
            raise ValueError("the MVSNeRF boost path is defined for B=1 (reference boost_mvsnerf/network.py:116-117)")

    @staticmethod
    def _proj_triple(exts, ixts):
        """reference lib/networks/mvsnerf/network.py:1070-1090 on host tensors (V,4,4),(V,3,3) -> (V,3,4)."""
        mats, ref_inv = [], None
        for i in range(exts.shape[0]):
            full = torch.eye(4)
            k = ixts[i].clone()
            k[:2] *= 0.25
            full[:3, :4] = k @ exts[i][:3, :4]
            if i == 0:
                ref_inv = torch.inverse(full)
                mats.append(torch.eye(4))
            else:
                mats.append(full @ ref_inv)
        return torch.stack(mats)[:, :3].float()

    def _render_chains(self, batch, triples):
        rc = self.rc
        inps = batch['all_src_inps'][0]
        N, _, H, W = inps.shape
        dev = inps.device
        K = len(triples)
        S = rc.num_samples[0]
        D = rc.num_samples[rc.num - 2]
        h, w = H // 4, W // 4
        with self._stage('feature'):
            feats = self.feature(batch['all_src_inps'])[0]                              # (N,32,h,w)
            small = F.interpolate(inps, (h, w), mode='bilinear', align_corners=False)   # (N,3,h,w)
        with self._stage('camera'):
            # tiny per-chain camera algebra on the host, like the ENeRF path (network.py:_camera_stage)
            exts_h, ixts_h = batch['all_src_exts'][0].cpu(), batch['all_src_ixts'][0].cpu()
            dr_h = batch['depth_ranges'][0].cpu()
            t = torch.linspace(0., 1., steps=D)
            projs, planes, nears, fars = [], [], [], []
            for tr in triples:
                idx = list(tr)
                near, far = dr_h[idx].min() * 0.8, dr_h[idx].max() * 1.2
                nears.append(near); fars.append(far)
                planes.append(near * (1. - t) + far * t)
                projs.append(self._proj_triple(exts_h[idx], ixts_h[idx]))
            projs = torch.stack(projs).to(dev)
            planes = torch.stack(planes).to(dev)
        with self._stage('cost_volume_img'):
            if self.mlp_engine == 'umma':
                # channels-last volumes: K1b's 41 stores per voxel are contiguous, cuDNN keeps the layout, and the fused
                # render kernel fetches a regularised voxel with two 16-byte loads
                vols = torch.empty((K, D, h + 2 * PAD, w + 2 * PAD, 9 + 32), device=dev, dtype=self.volume_dtype).permute(0, 4, 1, 2, 3)
            else:
                vols = torch.empty((K, 9 + 32, D, h + 2 * PAD, w + 2 * PAD), device=dev, dtype=self.volume_dtype)
            if self.mlp_engine == 'umma' and feats.shape[1] == 32:
                # dense channels-last feature maps select K1b's warp-level kernel (16-byte taps, shared tap sets)
                feats = feats.contiguous(memory_format=torch.channels_last)
            for k in range(K):
                ops.cost_volume_var_img(feats, small, triples[k], projs[k], planes[k], PAD, out=vols[k])
        with self._stage('cost_reg_2'):
            reg = self.cost_reg_2(vols.float() if vols.dtype != torch.float32 else vols)   # (K,8,D,hp,wp)
            del vols
            if self.mlp_engine == 'umma' and reg.stride(1) != 1:
                reg = reg.contiguous(memory_format=torch.channels_last_3d)
        rays = batch['rays_0'][0]
        R = rays.shape[0]
        raw = torch.empty((K, R, S, 4), device=dev)
        z = torch.empty((K, R, S), device=dev)
        mask = torch.empty((K, R, S), device=dev)
        if self.mlp_engine == 'umma':
            # nothing per-sample reaches HBM: marching, fetch and the whole MLP run in one kernel per chain
            key = tuple((q.data_ptr(), q._version) for q in self.nerf.parameters())
            if self._packed is None or self._packed[0] != key:
                from .mlp_pack import pack_mvs_weights_umma
                self._packed = (key, pack_mvs_weights_umma(self.nerf))
            rgb4 = inps.new_zeros((N, H, W, 4))                # (N,H,W,4): one 16-byte load per colour tap
            rgb4[..., :3] = inps.permute(0, 2, 3, 1)
            for k in range(K):
                with self._stage('render_fused'):
                    ops.mvs_render(rays, S, triples[k], batch['all_src_exts'][0], batch['all_src_ixts'][0], H, W,
                                   float(nears[k]), float(fars[k]), reg[k], rgb4, self._packed[1], PAD,
                                   out={'raw': raw[k], 'z_vals': z[k], 'vis_mask': mask[k]})
            return raw, mask, z, nears, fars
        chunk = max(1, min(R, self.mlp_chunk_bytes // (S * 86 * 4)))
        for k in range(K):
            for r0 in range(0, R, chunk):
                n = min(chunk, R - r0)
                with self._stage('march_fetch'):
                    o = ops.mvs_march_fetch(rays, S, triples[k], batch['all_src_exts'][0], batch['all_src_ixts'][0],
                                            H, W, float(nears[k]), float(fars[k]), reg[k], inps, PAD,
                                            ray_begin=r0, n_rays=n, want=("mlp_in",),
                                            out={'z_vals': z[k, r0:r0 + n], 'vis_mask': mask[k, r0:r0 + n]})
                with self._stage('nerf'):
                    raw[k, r0:r0 + n] = self.nerf(o['mlp_in'])
        return raw, mask, z, nears, fars

    def forward(self, batch):
        self._check(batch)
        rc = self.rc
        N = batch['all_src_inps'].shape[1]
        I, K = rc.cost_volume_input_views, rc.k_best
        table = list(itertools.combinations(range(N), I))
        key = f"{batch['meta']['scene'][0]}_{batch['meta']['tar_view'][0]}"
        k_best = self.view_selection_outputs[key][:K]
        triples = [table[int(j)] for j in k_best]
        if rc.white_bkgd:
            raise NotImplementedError
        with torch.no_grad():
            raw, mask, z, nears, fars = self._render_chains(batch, triples)
            with self._stage('composite_blend'):
                rgb, depth, weights = ops.composite_blend(list(raw.unbind(0)), list(mask.unbind(0)), list(z.unbind(0)))
            last = list(triples[-1])
            batch['near_far'] = torch.stack([nears[-1], fars[-1]]).to(rgb.device)
            batch['src_inps'] = batch['all_src_inps'][:, last]
            batch['src_exts'] = batch['all_src_exts'][:, last]
            batch['src_ixts'] = batch['all_src_ixts'][:, last]
        return {'rgb_level0': rgb[None], 'depth_level0': depth[None], 'weights_level0': weights[None]}

    # ------------------------------------------------------------------ view selection (SURVEY.md §8 f1)
    def forward_view_selection(self, batch):
        """reference lib/networks/boost_mvsnerf/network.py:23-95: for every triple of source views march
        128 uniform samples, volume-render the visibility score into a 2-D coverage mask, then pick the
        K triples greedily by newly covered area.  All on the GPU, no network involved."""
        picked = greedy_coverage(self.view_selection_masks(batch), self.rc.k_best)
        key = f"{batch['meta']['scene'][0]}_{batch['meta']['tar_view'][0]}"
        return {key: picked}

    def view_selection_masks(self, batch):
        """The 2-D coverage mask of every triple of source views (reference calc_mask,
        lib/networks/boost_mvsnerf/network.py:23-45), in the order of itertools.combinations -> (T, 1, R)."""
        self._check(batch)
        N = batch['all_src_inps'].shape[1]
        H, W = batch['all_src_inps'].shape[-2:]
        rays = batch['rays_0'][0]
        S = 128
        masks = []
        with torch.no_grad():
            for tr in itertools.combinations(range(N), 3):
                o = ops.mvs_march_fetch(rays, S, tr, batch['all_src_exts'][0], batch['all_src_ixts'][0], H, W,
                                        0.0, 1.0, None, None, want=("z_vals", "vis_mask"))
                m = (o['vis_mask'] / S).unsqueeze(-1).expand(-1, -1, 4).contiguous()
                rgbm, _, _ = ops.composite(m, o['z_vals'], self.rc.white_bkgd)
                masks.append(rgbm.mean(-1)[None])                         # (1,R)
        return torch.stack(masks)


def greedy_coverage(masks, k):
    """reference search_k_best_views (lib/networks/boost_enerf/network.py:71-95,
    lib/networks/boost_mvsnerf/network.py:47-71).  masks (T, ...) on any device -> list of <= k indices.
    One small D2H per pick (the argmax), instead of one per candidate as in the reference."""
    T = masks.shape[0]
    flat = masks.reshape(T, -1)
    hw = masks.shape[-2] * masks.shape[-1]
    prev = torch.ones_like(flat[0])
    taken = torch.zeros(T, dtype=torch.bool, device=masks.device)
    results = []
    for _ in range(k):
        ratio = (flat * prev).sum(1) / hw
        ratio = torch.where(taken, torch.full_like(ratio, -1.0), ratio)
        best_ratio, best = torch.max(ratio, dim=0)        # first maximal index, like the reference's strict '>'
        if not bool(best_ratio > 0):
            break
        b = int(best)
        prev = prev * (1 - flat[b])
        taken[b] = True
        results.append(b)
    if not results:
        results.append(0)
    return results
