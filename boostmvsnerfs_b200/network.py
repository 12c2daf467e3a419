"""Drop-in `Network` classes for the reference's plugin factory (SURVEY.md §8b).

`BoostEnerfNetwork` mirrors `lib/networks/boost_enerf/network.py:Network` of the reference:
constructor `Network(preprocess=False)` semantics, sub-module attribute names fixed by the
checkpoints (`feature_net`, `cost_reg_{i}`, `nerf_{i}`; reference lib/networks/enerf/network.py:14-22),
`forward(batch) -> {rgb,depth,weights,depth_mvs,std}_level{i}` (reference
lib/networks/boost_enerf/network.py:172-237).  The per-frame work between the kept NN modules
runs in the hand-written sm_100a kernels of libbmv (ops.py); there is no CPU / eager fallback.

B200-first differences from the reference's control flow (results unchanged):
  * the K cost-volume chains advance level by level TOGETHER, so the 3-D CNN and the MLP see one
    batched call (K volumes / K*R*S samples) instead of K small ones;
  * no gather copies of the triple's images/features: kernels take base pointers + view ids;
  * camera algebra (tiny) is hoisted to the top of the frame; nothing inside the frame syncs.
"""
import itertools
import json
import os

import torch
import torch.nn as nn

from . import ops
from .config import RenderConfig
from .inference_plan import PlanCache
from .modules import CostRegNet, FeatureNet, MinCostRegNet, NeRF


def _combinations(n, r):
    """torch.combinations(arange(n), r) as a host list (lexicographic; reference
    lib/networks/boost_enerf/network.py:176)."""
    return list(itertools.combinations(range(n), r))


class StreamedFeats(dict):
    """Feature maps of which some may still be in flight on another stream: `ready` maps a key to the event that marks
    it complete; the first access of such a key makes the CURRENT stream wait for it (a no-op for everything else)."""

    def __init__(self, *a, **k):
        super().__init__(*a, **k)
        self.ready = {}

    def _wait(self, key):
        ev = self.ready.pop(key, None)
        if ev is not None:
            torch.cuda.current_stream().wait_event(ev)

    def __getitem__(self, key):
        self._wait(key)
        return super().__getitem__(key)

    def get(self, key, default=None):
        self._wait(key)
        return super().get(key, default)

    def join(self):
        for key in list(self.ready):
            self._wait(key)


class EnerfNetwork(nn.Module):
    """Single-volume ENeRF (reference lib/networks/enerf/network.py:11-113)."""

    def __init__(self, rc: RenderConfig = None):
        super().__init__()
        self.rc = rc or RenderConfig.enerf_eval(1)
        self.feature_net = FeatureNet()
        for i in range(self.rc.num):
            ch = int(32 * (2 ** (-i)))
            setattr(self, f'cost_reg_{i}', MinCostRegNet(ch) if i == 0 else CostRegNet(ch))
            setattr(self, f'nerf_{i}', NeRF(feat_ch=self.rc.nerf_model_feat_ch[i] + 3,
                                            viewdir_agg=self.rc.viewdir_agg))
        # call-side preparation of the kept cuDNN modules (inference_plan.py); both are exact up to
        # fp32 rounding and measured in profiles/round1_conv_variants.md
        self.fold_bn = True                    # eval-mode BN folded into the convolutions
        self.channels_last = True              # NHWC / NDHWC activations, volumes emitted channels-last
        self.fused_mlp = True                  # K3+MLP in one kernel when the shape is instantiated
        self.half_feature_taps = False         # TF32-class path: the fused FPN step emits the level-1 maps in fp16 (8-byte taps in
                                               # K1: -25 us there, +22 us in the FPN kernel's half-sector stores: off by default)
        self.multi_chain_render = True         # K3+K5 of all K chains in one persistent launch (render_multi.cu)
        self._views_dev = None                 # int32 (K,3) device tensor of the frame's triples (set by FrameGraph)
        self._baked_views = False              # set when a launch took its view ids from the host (graph not re-usable
                                               # for another view selection)
        self.volume_range_scale = True         # fp16 cost volumes are stored x 2^k (ops.volume_scale), undone by conv0
        self.multi_chain_volume = True         # level 0: all K cost volumes in one launch, unique views warped once
        self.overlap_fpn_topdown = True        # FPN top-down steps on a side stream under the level-0 chain (inference_plan.py)
        # per-sample MLP engine of the fused render: 'umma' — tcgen05.mma with accumulators in tensor memory, all chains in
        # one launch (render_multi_umma.cu), per-chain fallback on mma.sync (render_mma.cu: faster than a per-chain tcgen05
        # render, profiles/round1l_tcgen05.md); 'mma' — warp-level mma.sync (render_multi.cu, render_mma.cu); 'fma' — fp32
        # FMA (render_fused.cu).  Same fp16 hi + lo split in both tensor-core engines.
        self.mlp_engine = 'umma'
        self.host_camera_algebra = True        # 4x4 inverses etc. on the host (one D2H of ~1 KB)
        self.generate_rays = False             # True: rays of full target images are generated on the device
                                               # from tar_ext/tar_ixt (SURVEY.md §8 f3); batch['rays_i'] may be absent
        self._plans = PlanCache()
        self.stage_timer = None                # optional callable(name) -> context manager
        self._packed = {}                      # level -> (param versions, packed weight tensor)
        self.keep_internals = False            # True: forward() leaves {level: per-chain visibility scores / z} of the
        self.last_internals = None             # last frame in last_internals (parity diagnostics; references, no copies)

    # ------------------------------------------------------------------ helpers
    def _check_mode(self, batch):
        if self.training:
            raise RuntimeError("boostmvsnerfs_b200 networks are inference-only (call .eval()); the "
                               "hand-written kernels have no backward")
        dev = batch['all_src_inps'].device if 'all_src_inps' in batch else batch['src_inps'].device
        if dev.type != 'cuda':
            raise RuntimeError("boostmvsnerfs_b200 has no CPU path: move the batch and the module to a CUDA device")

    def _stage(self, name):
        if self.stage_timer is None:
            return _NullCtx()
        return self.stage_timer(name)

    def invalidate_plans(self):
        """Drop the derived inference copies (folded convs, packed MLP weights).  They are rebuilt
        automatically after load_state_dict / in-place parameter updates (tensor version counters);
        call this after editing `param.data` directly, which bypasses the counters."""
        self._packed.clear()
        self._plans = PlanCache()

    def _packed_mlp(self, i, engine='fma'):
        """Packed weights of nerf_{i} for the fused kernels; re-packed when a parameter changes."""
        nerf = getattr(self, f'nerf_{i}')
        key = tuple((p.data_ptr(), p._version) for p in nerf.parameters())
        hit = self._packed.get((i, engine))
        if hit is None or hit[0] != key:
            from . import mlp_pack
            pack = {'mma': mlp_pack.pack_nerf_weights_mma, 'umma': mlp_pack.pack_nerf_weights_umma}.get(engine, mlp_pack.pack_nerf_weights)
            self._packed[(i, engine)] = (key, pack(nerf))
        return self._packed[(i, engine)][1]

    def _kept(self, name):
        """The cuDNN module `name`, through the inference plan when enabled."""
        mod = getattr(self, name)
        if not self.fold_bn:
            return mod
        fmt = None
        if self.channels_last:
            fmt = torch.channels_last if name == 'feature_net' else torch.channels_last_3d
        return self._plans.get(name, mod, fmt)

    def forward_feat(self, x, defer=False):
        """x (N,3,H,W) -> dict level_{0,1,2} of (N,C,h,w)
        (reference lib/networks/enerf/network.py:58-67, batch dim squeezed).
        defer=True (the per-frame path): the level-1 / level-2 maps may still be in flight on the FPN plan's side
        stream; the returned StreamedFeats makes the consuming stream wait at the first access of a level, and the
        caller must join() before it returns."""
        plan = self._kept('feature_net')
        fused_plan = type(plan).__name__ == 'FusedTopDownFPN'
        if fused_plan:
            plan.emit_half_features = bool(self.half_feature_taps)
            plan.side_topdown = bool(self.overlap_fpn_topdown)
            plan.scale_requests = self._volume_scale_requests(x.device)
        if self.channels_last and not fused_plan:
            x = x.contiguous(memory_format=torch.channels_last)
        quarter, half, full = plan(x)
        feats = StreamedFeats({'level_0': quarter, 'level_1': half, 'level_2': full})
        if fused_plan:
            feats.ready = dict(plan.ready or {})
            plan.ready = None
            if plan.rgb_nhwc4 is not None:
                feats['rgb_nhwc4'] = plan.rgb_nhwc4         # by-product of the stem kernel (see _render_level)
            for lvl, sc in plan.scales.items():             # range scales computed behind their level (same event)
                feats[f'vscale_{lvl}'] = sc
        if not defer:
            feats.join()
        return feats

    def _fp16_volume(self, i, C, dev):
        """Whether level i's cost volume is stored as (range-scaled) fp16: conv0 of its regulariser runs on libbmv's
        tensor-core kernel, whose operands are fp16 anyway."""
        plan = self._kept(f'cost_reg_{i}')
        return bool(self.channels_last and dev.type == 'cuda' and getattr(plan, 'tensor_core_convs', False)
                    and torch.backends.cudnn.allow_tf32 and C in (16, 32))

    def _volume_scale_requests(self, dev):
        """Levels >= 1 whose fp16 volume needs a range scale, with the consumer's weight scale (see FusedTopDownFPN)."""
        req = {}
        if self.volume_range_scale:
            for i in range(1, self.rc.num):
                if self._fp16_volume(i, int(32 * 2 ** (-i)), dev):
                    req[f'level_{i}'] = self._kept(f'cost_reg_{i}').input_weight_scale(dev)
        return req or None

    @staticmethod
    def _proj_all(exts, ixts, tar_ext, tar_ixt, src_scale, tar_scale):
        """get_proj_mats for ALL N views at once (reference lib/networks/enerf/utils.py:35-55);
        same torch ops as the reference (incl. torch.inverse of the 4x4) so the matrices match it."""
        k_src = ixts.clone()
        k_src[:, :2] *= src_scale
        p_src = k_src @ exts[:, :3]                              # (N,3,4)
        k_tar = tar_ixt.clone()
        k_tar[:2] *= tar_scale
        p_tar = k_tar @ tar_ext[:3]
        last = torch.zeros((1, 4), device=p_tar.device, dtype=p_tar.dtype)
        last[:, 3] = 1
        inv = torch.inverse(torch.cat((p_tar, last), dim=0)[None])[0]
        return (p_src @ inv).contiguous()

    def _camera_stage(self, exts, ixts, tar_ext, tar_ixt, after=None, image_hw=None):
        """All per-frame camera algebra, hoisted: homographies of every view for every cascade level
        and the camera centres.  With host_camera_algebra the ~1 KB of camera data makes one
        round trip to the host and the reference's own torch op sequence (incl. torch.inverse,
        LAPACK) runs there: ~40 tiny GPU launches and ~9 stream syncs become one copy each way."""
        rc = self.rc
        N = exts.shape[0]
        dev = exts.device
        if not self.host_camera_algebra:
            projs = [self._proj_all(exts, ixts, tar_ext, tar_ixt, rc.im_feat_scale[i], rc.volume_scale[i])
                     for i in range(rc.num)]
            gens = None
            if image_hw is not None:
                gens = [ops.RayGenerator.from_cameras(tar_ext.cpu(), tar_ixt.cpu(), image_hw[0], image_hw[1],
                                                      rc.render_scale[i], dev) for i in range(rc.num)]
            return ops.CameraBlock(exts, ixts, tar_ext), projs, gens
        if after is not None:
            if getattr(self, '_side_stream', None) is None or self._side_stream.device != dev:
                self._side_stream = torch.cuda.Stream(device=dev)
            self._side_stream.wait_event(after)
            with torch.cuda.stream(self._side_stream):
                flat = torch.cat([exts.reshape(-1), ixts.reshape(-1), tar_ext.reshape(-1), tar_ixt.reshape(-1)]).cpu()
        else:
            flat = torch.cat([exts.reshape(-1), ixts.reshape(-1), tar_ext.reshape(-1), tar_ixt.reshape(-1)]).cpu()
        packed = self._camera_host(flat, N).pin_memory().to(dev, non_blocking=True)
        gens = None
        if image_hw is not None:
            gp = self._raygen_host(flat, N).pin_memory().to(dev, non_blocking=True)
            gens = self._raygen_views(gp, image_hw)
        return self._camera_views(packed, exts, ixts) + (gens,)

    def _raygen_host(self, flat, N):
        """fp64 ray-generation parameters of every cascade level (ops.RayGenerator), (num*12,) on the host."""
        rc = self.rc
        h_text = flat[N * 25:N * 25 + 16].view(4, 4)
        h_tixt = flat[N * 25 + 16:N * 25 + 25].view(3, 3)
        return torch.cat([ops.RayGenerator.host_params(h_text.numpy(), h_tixt.numpy(), rc.render_scale[i])
                          for i in range(rc.num)])

    def _raygen_views(self, gp, image_hw):
        rc = self.rc
        return [ops.RayGenerator(int(image_hw[0] * rc.render_scale[i]) * int(image_hw[1] * rc.render_scale[i]),
                                 gp[i * 12:(i + 1) * 12]) for i in range(rc.num)]

    def _camera_host(self, flat, N):
        """Host part of the camera stage: flat = [exts (N*16), ixts (N*9), tar_ext (16), tar_ixt (9)] on the
        CPU -> packed [homographies per level (N*12 each), source centres (N*3), target centre (3)]."""
        rc = self.rc
        h_exts = flat[:N * 16].view(N, 4, 4)
        h_ixts = flat[N * 16:N * 25].view(N, 3, 3)
        h_text = flat[N * 25:N * 25 + 16].view(4, 4)
        h_tixt = flat[N * 25 + 16:N * 25 + 25].view(3, 3)
        parts = [self._proj_all(h_exts, h_ixts, h_text, h_tixt, rc.im_feat_scale[i], rc.volume_scale[i]).reshape(-1)
                 for i in range(rc.num)]
        parts.append(torch.stack([e.inverse()[:3, 3] for e in h_exts]).reshape(-1))
        parts.append(h_text.inverse()[:3, 3])
        return torch.cat(parts)

    def _camera_views(self, packed, exts, ixts):
        rc = self.rc
        N = exts.shape[0]
        projs = [packed[i * N * 12:(i + 1) * N * 12].view(N, 3, 4) for i in range(rc.num)]
        off = rc.num * N * 12
        cams = ops.CameraBlock(exts, ixts, centers=packed[off:off + N * 3].view(N, 3),
                               tar_center=packed[off + N * 3:off + N * 3 + 3])
        return cams, projs

    # ------------------------------------------------------------------ the K-chain engine
    def _render_frame(self, inps, exts, ixts, tar_ext, tar_ixt, near_far, rays_by_level, triples, camera=None):
        """One batch element.  inps (N,3,H,W); triples: list of K tuples of view ids.
        Returns per rendered level: dict(raws, masks, zs lists over K, depth/std of chain 0).
        `camera` = (cams, projs) precomputed by the caller (CUDA-graph replay, graph.py) skips the
        host round trip, which makes this function capturable."""
        rc = self.rc
        Hh, Ww = inps.shape[-2:]
        if camera is None:
            ready = torch.cuda.current_stream().record_event()      # camera tensors are valid from here on
        with self._stage('feature_net'):
            feats = self.forward_feat(inps, defer=True)
        with self._stage('camera'):
            need_gen = self.generate_rays or any(r is None for r in rays_by_level)
            if camera is not None:
                cams, projs, gens = camera
            else:
                # the host round trip runs on a side stream that only waits for `ready`, so it overlaps the FPN
                cams, projs, gens = self._camera_stage(exts, ixts, tar_ext, tar_ixt, after=ready,
                                                       image_hw=(Hh, Ww) if need_gen else None)
            if need_gen:
                rays_by_level = list(gens)
        states = self._chain_levels(feats, projs, near_far, triples, Hh, Ww)
        out = {}
        for i, st in states.items():
            out[i] = self._render_level(i, feats, inps, st, rays_by_level[i], cams, triples, Hh, Ww)
            out[i]['depth0'], out[i]['std0'] = st['depth'][0], st['std'][0]
        feats.join()                                       # every side-stream fork re-joined (a captured graph requires it)
        if self.keep_internals:
            self.last_internals = {i: {'masks': torch.stack(o['masks']), 'zs': torch.stack(o['zs'])} for i, o in out.items()}
        return out

    def _chain_levels(self, feats, projs, near_far, triples, Hh, Ww):
        """The coarse-to-fine cascade of the given cost-volume chains (reference
        lib/networks/boost_enerf/network.py:189-209): K1 -> 3-D CNN -> K2 per level, all chains of a
        level batched through the CNN.  Returns {level: dict(feat_vol (Kc,8,D,h,w), depth, std, nf
        lists)} for the levels that are rendered."""
        rc = self.rc
        K = len(triples)
        dev = feats['level_0'].device
        depth = std = nf = None              # per chain lists
        states = {}
        for i in range(rc.num):
            D, vs = rc.volume_planes[i], rc.volume_scale[i]
            h, w = int(Hh * vs), int(Ww * vs)
            f = feats[f'level_{i}']
            C = f.shape[1]
            with self._stage(f'cost_volume_l{i}'):
                # When conv0 of the regulariser runs on libbmv's tensor-core kernel its operands are rounded to
                # fp16 anyway: K1 then emits the volume in fp16 (same result, half the write + read traffic).
                plan = self._kept(f'cost_reg_{i}')
                vdt = torch.float16 if self._fp16_volume(i, C, dev) else torch.float32
                self.last_volume_dtype = vdt
                # fp16 has 5 exponent bits: store s * variance with a power of two s derived from max|feature| so the
                # volume cannot overflow and small-magnitude features stay out of the subnormals; conv0 undoes it
                vsc = None
                if vdt == torch.float16 and self.volume_range_scale:
                    vsc = feats.get(f'vscale_level_{i}')   # computed behind the FPN launch that produced the level
                    if vsc is None:
                        bufs = self.__dict__.setdefault('_vsc_bufs', {})
                        if (i, dev) not in bufs:
                            bufs[(i, dev)] = torch.zeros(6, device=dev)      # result + zeroed scratch words, re-used per frame
                        vsc = ops.volume_scale(f, consumer_scale=plan.input_weight_scale(dev), out=bufs[(i, dev)])
                if self.channels_last:
                    vols = torch.empty((K, D, h, w, C), device=dev, dtype=vdt).permute(0, 4, 1, 2, 3)
                else:
                    vols = torch.empty((K, C, D, h, w), device=dev, dtype=vdt)
                if depth is None:
                    planes0, nf0 = ops.depth_planes_first(near_far, D, h, w, rc.depth_inv[i])
                    planes = planes0                       # shared (D,)
                    nf = nf0                               # shared (2,h,w)
                    # the chains share the hypotheses and draw their views from the same N maps: warp every unique
                    # view once per group of <= 4 chains and feed all the variances it belongs to
                    vdev = self._views_dev                 # (K,3) int32 on the device, or None
                    for k0 in range(0, K, 4):
                        grp = triples[k0:k0 + 4]
                        uniq = set(range(f.shape[0])) if vdev is not None else {int(v) for t in grp for v in t}
                        if (self.channels_last and self.multi_chain_volume and f.stride(1) == 1 and len(grp) > 1
                                and len({len(t) for t in grp}) == 1 and all(len(set(t)) == len(t) for t in grp)
                                and ops.cost_volume_multi_supported(C, len(uniq), len(grp))):
                            ops.cost_volume_var_shared_multi(f, grp, projs[i], planes0, h, w, out=vols[k0:k0 + len(grp)],
                                                             out_scale=vsc,
                                                             triples_dev=None if vdev is None else vdev[k0:k0 + len(grp)])
                        else:
                            for k in range(k0, k0 + len(grp)):
                                ops.cost_volume_var_shared(f, triples[k], projs[i], planes0, h, w, out=vols[k], out_scale=vsc,
                                                           views_dev=None if vdev is None else vdev[k])
                else:                                      # all K chains' hypotheses in one launch
                    planes, nf = ops.depth_planes_next_batched(depth, std, nf, D, h, w, rc.depth_inv[i])
                    for k in range(K):                     # (f may be fp16: half_feature_taps)
                        ops.cost_volume_var(f, triples[k], projs[i], planes[k], out=vols[k], out_scale=vsc,
                                            views_dev=None if self._views_dev is None else self._views_dev[k])
            with self._stage(f'cost_reg_{i}'):
                feat_vol, logits = plan(vols, in_scale=vsc[4:6]) if vsc is not None else plan(vols)
                del vols
            with self._stage(f'depth_regression_l{i}'):
                if logits.stride(-1) == 1 and logits.stride(-2) == w and logits.stride(-3) == h * w:
                    depth, std = ops.depth_regression_batched(logits, planes, rc.depth_inv[i])   # (K,h,w) each
                else:
                    dl, sl = zip(*[ops.depth_regression(logits[k], planes if planes.dim() == 1 else planes[k],
                                                        rc.depth_inv[i]) for k in range(K)])
                    depth, std = torch.stack(dl), torch.stack(sl)
            if rc.render_if[i]:
                nf_k = [nf[k] for k in range(K)] if nf.dim() == 4 else [nf] * K
                states[i] = {'feat_vol': feat_vol, 'depth': [depth[k] for k in range(K)],
                             'std': [std[k] for k in range(K)], 'nf': nf_k,
                             'depth_all': depth, 'std_all': std, 'nf_all': nf}      # K-stacked (one-launch render)
        return states

    def _render_level(self, i, feats, inps, state, rays, cams, triples, Hh, Ww, ray_begin=0, n_rays=None):
        """K3 (+MLP) for rays [ray_begin, ray_begin+n_rays) of every chain at cascade level i
        (reference lib/networks/boost_enerf/network.py:123-161, 212-222)."""
        rc = self.rc
        K = len(triples)
        feat_vol, depth, std, nf = state['feat_vol'], state['depth'], state['std'], state['nf']
        S = rc.num_samples[i]
        rs = rc.render_scale[i]
        H, W = int(Hh * rs), int(Ww * rs)
        im_feat = feats[f'level_{rc.render_im_feat_level[i]}']
        if im_feat.dtype == torch.float16:           # maps the FPN plan keeps in fp16 for the cost volumes (half_feature_taps)
            im_feat = im_feat.float()
        up = rs / rc.im_ibr_scale[i]
        if up != 1.:   # never taken by the shipped configs (reference boost_enerf/network.py:128-131)
            im_feat = torch.nn.functional.interpolate(
                im_feat, size=(int(im_feat.shape[-2] * up), int(im_feat.shape[-1] * up)),
                align_corners=True, mode='bilinear')
        if rs == 1.:
            rgb, affine = inps, (0.5, 0.5)          # unpreprocess folded into the fetch
            if self.channels_last and inps.is_cuda:
                # (N,H,W,4) channels-last copy: one 16-byte load per bilinear tap in the fused render kernel
                rgb4 = feats.get('rgb_nhwc4')
                if rgb4 is None or rgb4.shape[:3] != (inps.shape[0], inps.shape[2], inps.shape[3]):
                    rgb4 = inps.new_zeros((inps.shape[0], inps.shape[2], inps.shape[3], 4))
                    rgb4[..., :3] = inps.permute(0, 2, 3, 1)
                rgb = rgb4.permute(0, 3, 1, 2)[:, :3]
        else:          # level-0 rendering of the pre-train configs: resized colours (enerf/utils.py:669-676)
            rgb = torch.nn.functional.interpolate(inps * 0.5 + 0.5, size=(H, W), align_corners=True, mode='bilinear')
            affine = (1.0, 0.0)
        R_all = rays.n_rays if isinstance(rays, ops.RayGenerator) else rays.shape[0]
        R = R_all - ray_begin if n_rays is None else n_rays
        dev = inps.device
        nerf = getattr(self, f'nerf_{i}')
        V, Cf, Cv = len(triples[0]), im_feat.shape[1], feat_vol.shape[1]
        raw_all = torch.empty((K, R, S, 4), device=dev)
        mask_all = torch.empty((K, R, S), device=dev)
        z_all = torch.empty((K, R, S), device=dev)
        if self.fused_mlp and rc.viewdir_agg and ops.render_rays_supported(Cv, Cf, V):
            engine = self.mlp_engine if (Cf == 8 and V == 3) else 'fma'
            if (engine in ('mma', 'umma') and self.multi_chain_render and state.get('depth_all') is not None and rs == 1.
                    and all(len(tr) == 3 for tr in triples) and ops.render_rays_multi_supported(feat_vol, im_feat, rgb, V)):
                # every chain in ONE persistent launch (csrc/render_multi.cu, or render_multi_umma.cu for the tcgen05
                # engine); view ids from device memory when the
                # caller (FrameGraph) supplies them
                packed = self._packed_mlp(i, engine)
                with self._stage(f'render_fused_l{i}'):
                    ops.render_rays_multi(state['depth_all'], state['std_all'], state['nf_all'], rays, H, W, rc.depth_inv[i], S,
                                          feat_vol, im_feat, rgb, cams, triples, packed, render_scale=rs, rgb_affine=affine,
                                          ray_begin=ray_begin, n_rays=R, views_dev=self._views_dev, engine=engine,
                                          out={'raw': raw_all, 'z_vals': z_all, 'vis_mask': mask_all})
                return {'raws': list(raw_all.unbind(0)), 'masks': list(mask_all.unbind(0)), 'zs': list(z_all.unbind(0))}
            engine = 'fma' if engine == 'fma' else 'mma'   # per chain, both tensor-core engines run the mma.sync kernel
            packed = self._packed_mlp(i, engine)
            self._baked_views = True               # the per-chain launches carry their view ids as kernel arguments
            with self._stage(f'render_fused_l{i}'):
                for k in range(K):
                    ops.render_rays(depth[k], std[k], nf[k], rays, H, W, rc.depth_inv[i], S, feat_vol[k], im_feat,
                                    rgb, cams, triples[k], packed, render_scale=rs, rgb_affine=affine,
                                    ray_begin=ray_begin, n_rays=R, engine=engine,
                                    out={'raw': raw_all[k], 'z_vals': z_all[k], 'vis_mask': mask_all[k]})
            return {'raws': list(raw_all.unbind(0)), 'masks': list(mask_all.unbind(0)), 'zs': list(z_all.unbind(0))}
        self._baked_views = True
        for r0 in range(0, R, rc.chunk_size):
            n = min(rc.chunk_size, R - r0)
            vox = torch.empty((K, n * S, Cv), device=dev)
            img = torch.empty((K, n * S, V, Cf + 7), device=dev)
            with self._stage(f'raygen_fetch_l{i}'):
                for k in range(K):
                    ops.raygen_sample_fetch(depth[k], std[k], nf[k], rays, H, W, rc.depth_inv[i], S,
                                            feat_vol[k], im_feat, rgb, cams, triples[k], render_scale=rs,
                                            rgb_affine=affine, ray_begin=ray_begin + r0, n_rays=n, want=(),
                                            out={'z_vals': z_all[k, r0:r0 + n], 'vis_mask': mask_all[k, r0:r0 + n],
                                                 'vox_feat': vox[k], 'img_feat': img[k]})
            with self._stage(f'nerf_{i}'):
                net = nerf(vox, img)                                     # (K, n*S, 4)
                del vox, img
                if n == R:
                    raw_all = net.view(K, R, S, 4)
                else:
                    raw_all[:, r0:r0 + n] = net.view(K, n, S, 4)
        return {'raws': list(raw_all.unbind(0)), 'masks': list(mask_all.unbind(0)), 'zs': list(z_all.unbind(0))}

    # ------------------------------------------------------------------ public API
    def forward(self, batch):
        self._check_mode(batch)
        rc = self.rc
        inps = batch['src_inps']
        B, N = inps.shape[:2]
        ret = {}
        per_b = []
        with torch.no_grad():
            for b in range(B):
                lv = self._render_frame(inps[b], batch['src_exts'][b], batch['src_ixts'][b], batch['tar_ext'][b],
                                        batch['tar_ixt'][b], batch['near_far'][b],
                                        [batch[f'rays_{i}'][b] if f'rays_{i}' in batch else None
                                         for i in range(rc.num)], [tuple(range(N))])
                per_b.append(lv)
            for i in range(rc.num):
                if not rc.render_if[i]:
                    continue
                rgb, dep, wts, dmvs, sd = [], [], [], [], []
                for lv in per_b:
                    with self._stage(f'composite_l{i}'):
                        r, d, w = ops.composite(lv[i]['raws'][0], lv[i]['zs'][0], rc.white_bkgd)
                    rgb.append(r); dep.append(d); wts.append(w)
                    dmvs.append(1. / lv[i]['depth0'] if rc.depth_inv[i] else lv[i]['depth0'])
                    sd.append(lv[i]['std0'])
                ret.update({f'rgb_level{i}': torch.stack(rgb), f'depth_level{i}': torch.stack(dep),
                            f'weights_level{i}': torch.stack(wts), f'depth_mvs_level{i}': torch.stack(dmvs),
                            f'std_level{i}': torch.stack(sd)})
        return ret


class BoostEnerfNetwork(EnerfNetwork):
    """ENeRF + BoostMVSNeRFs K-volume blend (reference lib/networks/boost_enerf/network.py:10-237)."""

    def __init__(self, preprocess=False, rc: RenderConfig = None, view_selection_file=None):
        super().__init__(rc or RenderConfig.enerf_eval())
        self.view_selection_outputs = {}
        if not preprocess:
            # reference lib/networks/boost_enerf/network.py:14-20: the JSON written by the
            # view-selection pre-process is mandatory (the reference `raise`s a str -> TypeError)
            if view_selection_file is None or not os.path.exists(view_selection_file):
                raise FileNotFoundError("View selection file not found. Please run view selection first.")
            with open(view_selection_file, 'r') as fh:
                self.view_selection_outputs = json.load(fh)

    def forward(self, batch):
        self._check_mode(batch)
        rc = self.rc
        inps = batch['all_src_inps']
        B, N = inps.shape[:2]
        I, K = rc.cost_volume_input_views, rc.k_best
        table = _combinations(N, I)
        scenes, views = batch['meta']['scene'], batch['meta']['tar_view']
        k_best = [self.view_selection_outputs[f'{s}_{v}'] for s, v in zip(scenes, views)]
        ret = {}
        per_b = []
        with torch.no_grad():
            for b in range(B):
                triples = [table[int(j)] for j in k_best[b][:K]]
                if len(triples) != K:
                    raise ValueError(f"view selection for {scenes[b]}_{views[b]} holds {len(triples)} volumes, "
                                     f"cfg.enerf.cas_config.k_best is {K}")
                per_b.append(self._render_frame(inps[b], batch['all_src_exts'][b], batch['all_src_ixts'][b],
                                                batch['tar_ext'][b], batch['tar_ixt'][b], batch['near_far'][b],
                                                [batch[f'rays_{i}'][b] if f'rays_{i}' in batch else None
                                                 for i in range(rc.num)], triples))
            ret = self._assemble(per_b)
            # the reference leaves the LAST triple in the batch (evaluators read batch['src_inps'].shape);
            # done last so the index upload cannot stall the kernels above
            last = [list(table[int(k_best[b][K - 1])]) for b in range(B)]
            if B == 1:
                batch['src_inps'] = inps[:, last[0]]
                batch['src_exts'] = batch['all_src_exts'][:, last[0]]
                batch['src_ixts'] = batch['all_src_ixts'][:, last[0]]
            else:
                lt = torch.tensor(last, device=inps.device)
                bidx = torch.arange(B, device=inps.device).unsqueeze(-1).expand(-1, I)
                batch['src_inps'] = inps[bidx, lt]
                batch['src_exts'] = batch['all_src_exts'][bidx, lt]
                batch['src_ixts'] = batch['all_src_ixts'][bidx, lt]
        return ret


    def _assemble(self, per_b):
        """K4 over the K chains of every batch element + the reference's output dict
        (reference lib/networks/boost_enerf/network.py:226-235)."""
        rc = self.rc
        if rc.white_bkgd:
            raise NotImplementedError   # reference lib/networks/enerf/utils.py:660-661
        ret = {}
        for i in range(rc.num):
            if not rc.render_if[i]:
                continue
            rgb, dep, wts, dmvs, sd = [], [], [], [], []
            for lv in per_b:
                with self._stage(f'composite_blend_l{i}'):
                    r, d, w = ops.composite_blend(lv[i]['raws'], lv[i]['masks'], lv[i]['zs'])
                rgb.append(r); dep.append(d); wts.append(w)
                dmvs.append(1. / lv[i]['depth0'] if rc.depth_inv[i] else lv[i]['depth0'])
                sd.append(lv[i]['std0'])
            ret.update({f'rgb_level{i}': torch.stack(rgb), f'depth_level{i}': torch.stack(dep),
                        f'weights_level{i}': torch.stack(wts), f'depth_mvs_level{i}': torch.stack(dmvs),
                        f'std_level{i}': torch.stack(sd)})
        return ret

    # ------------------------------------------------------------------ view selection (SURVEY.md §8 f1)
    def forward_view_selection(self, batch, max_chains_per_pass=32):
        """reference lib/networks/boost_enerf/network.py:22-121 (calc_mask + search_k_best_views +
        forward_view_selection): for EVERY triple of source views run the cost-volume cascade, render the
        per-sample visibility score into a 2-D coverage mask, then pick K triples greedily by newly
        covered area.  Here the FPN runs once for all views (the reference re-runs it per triple), all
        triples go through the cascade as batched chains, the MLP (whose output the reference
        discards) is skipped, and the greedy search stays on the GPU."""
        from .network_mvs import greedy_coverage
        self._check_mode(batch)
        rc = self.rc
        inps_all = batch['all_src_inps']
        B, N = inps_all.shape[:2]
        if B != 1:
            raise ValueError("view selection is defined per frame (B=1), as in the reference (network.py:118)")
        table = _combinations(N, 3)
        inps = inps_all[0]
        Hh, Ww = inps.shape[-2:]
        picked = None
        with torch.no_grad():
            feats = self.forward_feat(inps)
            cams, projs, _ = self._camera_stage(batch['all_src_exts'][0], batch['all_src_ixts'][0], batch['tar_ext'][0],
                                                batch['tar_ixt'][0])
            masks = {i: [] for i in range(rc.num) if rc.render_if[i]}
            for c0 in range(0, len(table), max_chains_per_pass):
                part = table[c0:c0 + max_chains_per_pass]
                states = self._chain_levels(feats, projs, batch['near_far'][0], part, Hh, Ww)
                for i, st in states.items():
                    S, rs = rc.num_samples[i], rc.render_scale[i]
                    H, W = int(Hh * rs), int(Ww * rs)
                    rays = batch[f'rays_{i}'][0]
                    for k, tr in enumerate(part):
                        o = ops.raygen_sample_fetch(st['depth'][k], st['std'][k], st['nf'][k], rays, H, W,
                                                    rc.depth_inv[i], S, None, None, None, cams, tr,
                                                    want=("z_vals", "vis_mask"))
                        m = (o['vis_mask'] / S).unsqueeze(-1).expand(-1, -1, 4).contiguous()
                        rgbm, _, _ = ops.composite(m, o['z_vals'], rc.white_bkgd)
                        masks[i].append(rgbm.mean(-1).view(1, H, W))
                del states
            for i in masks:                      # the reference keeps the LAST rendered level's pick
                picked = greedy_coverage(torch.stack(masks[i]), rc.k_best)
        keys = [f"{s}_{v}" for s, v in zip(batch['meta']['scene'], batch['meta']['tar_view'])]
        return {key: picked for key in keys}


class _NullCtx:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False
