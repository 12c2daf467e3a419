"""Torch-facing wrappers of the libbmv C ABI (include/bmv.h).

PyTorch is used for device memory and streams only: every function allocates its outputs with
torch, extracts raw device pointers, fills the POD params struct and enqueues the kernel on the
current CUDA stream.  Inputs must already live on the GPU; nothing here has a CPU path.
"""
import ctypes as C

import torch

from . import _lib
from ._lib import BmvError, MAX_VIEWS, MAX_VOLUMES


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _feat(t, name):
    """Source feature maps of the cost-volume kernels: CUDA float32, or float16 (half the bytes per tap; fast path only)."""
    if not (torch.is_tensor(t) and t.is_cuda and t.dtype in (torch.float32, torch.float16)):
        raise BmvError(f"{name}: expected a CUDA float32 / float16 tensor, got "
                       f"{type(t).__name__} {getattr(t, 'dtype', None)} {getattr(t, 'device', None)}")
    _on_current_device(t, name)
    return int(t.dtype == torch.float16)


def _on_current_device(t, name):
    # libbmv launches on the CURRENT device's current stream (one process per GPU): a tensor living on another
    # device would be dereferenced by the wrong GPU
    if t.device.index != torch.cuda.current_device():
        raise BmvError(f"{name}: tensor is on {t.device} but the current CUDA device is cuda:{torch.cuda.current_device()} "
                       "(call torch.cuda.set_device / use torch.cuda.device(...) around libbmv ops)")


def _f32(t, name):
    if not (torch.is_tensor(t) and t.is_cuda and t.dtype == torch.float32):
        raise BmvError(f"{name}: expected a CUDA float32 tensor, got "
                       f"{type(t).__name__} {getattr(t, 'dtype', None)} {getattr(t, 'device', None)}")
    _on_current_device(t, name)
    return t


def _cf32(t, name):
    return _f32(t, name).contiguous()


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _views(arr_type_holder, views):
    if len(views) > MAX_VIEWS:
        raise BmvError(f"at most {MAX_VIEWS} views per volume, got {len(views)}")
    for i, v in enumerate(views):
        arr_type_holder[i] = int(v)


_linspace_cache = {}


def _linspace(n, device):
    # taken from torch so that the fractions carry torch's own rounding (SURVEY.md §7)
    key = (n, str(device))
    if key not in _linspace_cache:
        _linspace_cache[key] = torch.linspace(0., 1., n, device=device, dtype=torch.float32)
    return _linspace_cache[key]


# ------------------------------------------------------------------------------------------ K1
def volume_scale(feats, target=16384.0, consumer_scale=1.0, out=None):
    """Power-of-two range scale for an fp16 cost volume built from `feats` (bmv_volume_scale): returns a device tensor
    [s, 1/s, 0, 0, s*c, 1/(s*c)] with s * max|feats|^2 <= target and c = consumer_scale (the power of two the consuming
    convolution's fp16 weights were packed with).  Pass it as `out_scale` to the cost-volume ops and `t[4:6]` as
    `in_scale` to the convolution that consumes the volume."""
    half = _feat(feats, "feats")
    n = feats.numel()
    # every element of the underlying storage span is a feature value: dense tensors only (any memory format)
    if not (feats.is_contiguous() or feats.is_contiguous(memory_format=torch.channels_last)):
        raise BmvError("volume_scale: feats must be dense (contiguous or channels_last)")
    # out: a 6-float buffer from an earlier call on this device (the kernel leaves its two scratch words zero, so it can be
    # re-used call after call in stream order: saves the fill launch of a fresh one)
    if out is not None:
        if not (out.is_cuda and out.dtype == torch.float32 and out.numel() == 6 and out.is_contiguous() and out.device == feats.device):
            raise BmvError("volume_scale: out must be a contiguous 6-float CUDA tensor on feats' device")
        sc = out
    else:
        sc = torch.zeros(6, device=feats.device)
    p = _lib.VolumeScaleParams()
    p.x, p.n, p.x_half, p.target, p.scale = feats.data_ptr(), n, half, float(target), sc.data_ptr()
    p.consumer_scale = float(consumer_scale)
    _lib.call("bmv_volume_scale", p, _stream())
    return sc


def _scale_ptr(t):
    if t is None:
        return 0
    if not (torch.is_tensor(t) and t.is_cuda and t.dtype == torch.float32 and t.numel() >= 2 and t.is_contiguous()):
        raise BmvError("scale: expected the device tensor returned by ops.volume_scale")
    return t.data_ptr()


def _views_dev_ptr(t, n):
    if t is None:
        return 0
    if not (torch.is_tensor(t) and t.is_cuda and t.dtype == torch.int32 and t.is_contiguous() and t.numel() == n):
        raise BmvError(f"views_dev: expected a contiguous int32 CUDA tensor with {n} elements")
    return t.data_ptr()


def cost_volume_var(feats, views, proj, planes, out=None, out_dtype=torch.float32, channels_last=False,
                    exact_coords=False, out_scale=None, views_dev=None, variant=0):
    """Fused plane-sweep cost volume for ONE batch element.

    feats  (N,C,Hs,Ws) feature maps of all views, any strides (NCHW or channels_last)
    views  list of S view indices forming this volume
    proj   (N,3,4) homographies of ALL views, indexed by view id like `feats`
           (get_proj_mats, reference lib/networks/enerf/utils.py:35-55)
    planes (D,h,w) per-pixel hypotheses or (D,) shared
    -> (C,D,h,w) variance volume (reference lib/networks/enerf/utils.py:324-351)
    variant 0: the fastest kernel generation the layout allows; 5: four channels per lane even where the
    eight-channels-per-lane generation applies (bit-identical; A/B tests)
    """
    feat_half = _feat(feats, "feats")
    proj = _cf32(proj, "proj")
    planes = _cf32(planes, "planes")
    N, Cc, Hs, Ws = feats.shape
    S = len(views)
    assert proj.shape == (N, 3, 4), proj.shape
    p = _lib.CostVolumeParams()
    p.feat = feats.data_ptr()
    p.feat_half = feat_half
    p.feat_view_stride, p.feat_c_stride, p.feat_y_stride, p.feat_x_stride = feats.stride()
    _views(p.view, views)
    p.S, p.C, p.Hs, p.Ws = S, Cc, Hs, Ws
    p.proj, p.planes = proj.data_ptr(), planes.data_ptr()
    if planes.dim() == 1:
        raise BmvError("shared planes need the volume size: pass planes.view(D,1,1).expand(D,h,w) "
                       "or use cost_volume_var_shared")
    D, h, w = planes.shape
    p.planes_d_stride, p.planes_pix_stride = h * w, 1
    p.D, p.h, p.w = D, h, w
    p.exact_coords = int(exact_coords)
    p.variant = int(variant)
    p.out_scale = _scale_ptr(out_scale)
    p.view_dev = _views_dev_ptr(views_dev, S)
    return _cost_volume_launch(p, Cc, D, h, w, feats.device, out, out_dtype, channels_last)


def cost_volume_var_shared(feats, views, proj, planes_d, h, w, out=None, out_dtype=torch.float32,
                           channels_last=False, exact_coords=False, out_scale=None, views_dev=None, variant=0):
    """Same as cost_volume_var with D hypotheses shared by every pixel (cascade level 0)."""
    feat_half = _feat(feats, "feats")
    proj = _cf32(proj, "proj")
    planes_d = _cf32(planes_d, "planes")
    N, Cc, Hs, Ws = feats.shape
    S = len(views)
    p = _lib.CostVolumeParams()
    p.feat = feats.data_ptr()
    p.feat_half = feat_half
    p.feat_view_stride, p.feat_c_stride, p.feat_y_stride, p.feat_x_stride = feats.stride()
    _views(p.view, views)
    p.S, p.C, p.Hs, p.Ws = S, Cc, Hs, Ws
    p.proj, p.planes = proj.data_ptr(), planes_d.data_ptr()
    D = planes_d.numel()
    p.planes_d_stride, p.planes_pix_stride = 1, 0
    p.D, p.h, p.w = D, h, w
    p.exact_coords = int(exact_coords)
    p.variant = int(variant)
    p.out_scale = _scale_ptr(out_scale)
    p.view_dev = _views_dev_ptr(views_dev, S)
    return _cost_volume_launch(p, Cc, D, h, w, feats.device, out, out_dtype, channels_last)


def cost_volume_var_shared_multi(feats, triples, proj, planes_d, h, w, out, out_scale=None, triples_dev=None, variant=0):
    """The K level-0 cost volumes (shared depth hypotheses) in one launch: every unique source view is warped once
    per (voxel, plane) and feeds the variance of each chain it belongs to (bmv_cost_volume_var_multi).
    feats (N,C,Hs,Ws) channels-last, triples: K lists of view ids (equal lengths), out (K,C,D,h,w) with
    channels-last-3d volumes (fp32 / bf16 / fp16), written in place."""
    feat_half = _feat(feats, "feats")
    proj = _cf32(proj, "proj")
    planes_d = _cf32(planes_d, "planes")
    N, Cc, Hs, Ws = feats.shape
    K, S = len(triples), len(triples[0])
    if any(len(t) != S for t in triples):
        raise BmvError("cost_volume_var_shared_multi: every chain needs the same number of views")
    # device-resident selection: every source view is a "unique view", the kernel derives the chain masks
    uniq = list(range(N)) if triples_dev is not None else sorted({int(v) for t in triples for v in t})
    D = planes_d.numel()
    if out.shape != (K, Cc, D, h, w) or out.stride(1) != 1:
        raise BmvError("cost_volume_var_shared_multi: out must be (K,C,D,h,w) with channels-last-3d volumes")
    mp = _lib.CostVolumeMultiParams()
    p = mp.b
    p.feat = feats.data_ptr()
    p.feat_half = feat_half
    p.feat_view_stride, p.feat_c_stride, p.feat_y_stride, p.feat_x_stride = feats.stride()
    _views(p.view, uniq)
    p.S, p.C, p.Hs, p.Ws = len(uniq), Cc, Hs, Ws
    p.proj, p.planes = proj.data_ptr(), planes_d.data_ptr()
    p.planes_d_stride, p.planes_pix_stride = 1, 0
    p.D, p.h, p.w = D, h, w
    p.exact_coords = 0
    p.variant = int(variant)
    p.out_scale = _scale_ptr(out_scale)
    p.out = out.data_ptr()
    p.out_c_stride, p.out_d_stride, p.out_y_stride, p.out_x_stride = out.stride(1), out.stride(2), out.stride(3), out.stride(4)
    p.out_bf16 = {torch.float32: 0, torch.bfloat16: 1, torch.float16: 2}[out.dtype]
    mp.K, mp.views_per_chain, mp.out_k_stride = K, S, out.stride(0)
    mp.triples_dev = _views_dev_ptr(triples_dev, K * S)
    for i, u in enumerate(uniq):
        mp.chain_mask[i] = sum(1 << k for k, t in enumerate(triples) if u in [int(v) for v in t])
    _lib.call("bmv_cost_volume_var_multi", mp, _stream())
    return out


def cost_volume_multi_supported(C, n_unique, K):
    return C in (16, 32) and (32 // (C // 4)) * n_unique <= 32 and 1 <= K <= 4


def _cost_volume_launch(p, Cc, D, h, w, device, out, out_dtype, channels_last):
    if out is None:
        if channels_last:   # physical (D,h,w,C), logical (C,D,h,w)
            out = torch.empty((D, h, w, Cc), device=device, dtype=out_dtype).permute(3, 0, 1, 2)
        else:
            out = torch.empty((Cc, D, h, w), device=device, dtype=out_dtype)
    assert out.shape == (Cc, D, h, w) and out.dtype in (torch.float32, torch.bfloat16, torch.float16)
    p.out = out.data_ptr()
    p.out_c_stride, p.out_d_stride, p.out_y_stride, p.out_x_stride = out.stride()
    p.out_bf16 = {torch.float32: 0, torch.bfloat16: 1, torch.float16: 2}[out.dtype]
    _lib.call("bmv_cost_volume_var", p, _stream())
    return out


# ------------------------------------------------------------------------------------------ a3
def depth_planes_first(near_far, D, h, w, depth_inv):
    """near_far (2,) -> planes (D,), near_far_out (2,h,w)
    (reference lib/networks/enerf/utils.py:103-111,149-153)."""
    near_far = _cf32(near_far, "near_far")
    dev = near_far.device
    t = _linspace(D, dev)
    planes = torch.empty(D, device=dev)
    nf = torch.empty((2, h, w), device=dev)
    p = _lib.DepthPlanesFirstParams()
    p.near_far, p.t = near_far.data_ptr(), t.data_ptr()
    p.D, p.h, p.w, p.depth_inv = D, h, w, int(depth_inv)
    p.planes, p.near_far_out = planes.data_ptr(), nf.data_ptr()
    _lib.call("bmv_depth_planes_first", p, _stream())
    return planes, nf


def depth_planes_next(depth, std, near_far, D, h, w, cur_inv):
    """depth/std (h0,w0), near_far (2,h0,w0) [disparities] -> planes (D,h,w), near_far_out (2,h,w)
    (reference lib/networks/enerf/utils.py:112-153)."""
    depth, std, near_far = _cf32(depth, "depth"), _cf32(std, "std"), _cf32(near_far, "near_far")
    dev = depth.device
    h0, w0 = depth.shape
    t = _linspace(D, dev)
    planes = torch.empty((D, h, w), device=dev)
    nf = torch.empty((2, h, w), device=dev)
    p = _lib.DepthPlanesNextParams()
    p.depth, p.std, p.near_far, p.t = depth.data_ptr(), std.data_ptr(), near_far.data_ptr(), t.data_ptr()
    p.h0, p.w0, p.h, p.w, p.D, p.cur_inv = h0, w0, h, w, D, int(cur_inv)
    p.planes, p.near_far_out = planes.data_ptr(), nf.data_ptr()
    _lib.call("bmv_depth_planes_next", p, _stream())
    return planes, nf


def depth_planes_next_batched(depth, std, near_far, D, h, w, cur_inv):
    """All K chains in one launch: depth/std (K,h0,w0), near_far (K,2,h0,w0) or shared (2,h0,w0)
    -> planes (K,D,h,w), near_far_out (K,2,h,w)."""
    depth, std, near_far = _cf32(depth, "depth"), _cf32(std, "std"), _cf32(near_far, "near_far")
    dev = depth.device
    K, h0, w0 = depth.shape
    t = _linspace(D, dev)
    planes = torch.empty((K, D, h, w), device=dev)
    nf = torch.empty((K, 2, h, w), device=dev)
    p = _lib.DepthPlanesNextParams()
    p.depth, p.std, p.near_far, p.t = depth.data_ptr(), std.data_ptr(), near_far.data_ptr(), t.data_ptr()
    p.h0, p.w0, p.h, p.w, p.D, p.cur_inv = h0, w0, h, w, D, int(cur_inv)
    p.planes, p.near_far_out = planes.data_ptr(), nf.data_ptr()
    p.batch, p.depth_b_stride, p.std_b_stride = K, h0 * w0, h0 * w0
    p.nf_b_stride = 2 * h0 * w0 if near_far.dim() == 4 else 0
    _lib.call("bmv_depth_planes_next", p, _stream())
    return planes, nf


def depth_regression_batched(logits, planes, depth_inv):
    """All K chains in one launch: logits (K,D,h,w) (any chain stride, planar within a chain); planes (K,D,h,w),
    or shared (D,) -> depth (K,h,w), std (K,h,w)."""
    _f32(logits, "logits")
    planes = _cf32(planes, "planes")
    K, D, h, w = logits.shape
    if tuple(logits.stride()[1:]) != (h * w, w, 1):
        raise BmvError("depth_regression_batched: each chain's logits must be planar-contiguous")
    dev = logits.device
    depth = torch.empty((K, h, w), device=dev)
    std = torch.empty((K, h, w), device=dev)
    p = _lib.DepthRegressionParams()
    p.logits, p.planes = logits.data_ptr(), planes.data_ptr()
    if planes.dim() == 1:
        assert planes.numel() == D
        p.planes_d_stride, p.planes_pix_stride, p.planes_b_stride = 1, 0, 0
    else:
        assert planes.shape == (K, D, h, w)
        p.planes_d_stride, p.planes_pix_stride, p.planes_b_stride = h * w, 1, D * h * w
    p.D, p.h, p.w, p.depth_inv = D, h, w, int(depth_inv)
    p.batch, p.logits_b_stride = K, logits.stride(0)
    p.depth, p.std = depth.data_ptr(), std.data_ptr()
    _lib.call("bmv_depth_regression", p, _stream())
    return depth, std


# ------------------------------------------------------------------------------------------ K2
def depth_regression(logits, planes, depth_inv):
    """logits (D,h,w); planes (D,h,w) or (D,) -> depth (h,w), std (h,w)
    (reference lib/networks/enerf/utils.py:722-727)."""
    logits, planes = _cf32(logits, "logits"), _cf32(planes, "planes")
    D, h, w = logits.shape
    dev = logits.device
    depth = torch.empty((h, w), device=dev)
    std = torch.empty((h, w), device=dev)
    p = _lib.DepthRegressionParams()
    p.logits, p.planes = logits.data_ptr(), planes.data_ptr()
    if planes.dim() == 1:
        assert planes.numel() == D
        p.planes_d_stride, p.planes_pix_stride = 1, 0
    else:
        assert planes.shape == (D, h, w)
        p.planes_d_stride, p.planes_pix_stride = h * w, 1
    p.D, p.h, p.w, p.depth_inv = D, h, w, int(depth_inv)
    p.depth, p.std = depth.data_ptr(), std.data_ptr()
    _lib.call("bmv_depth_regression", p, _stream())
    return depth, std


# ------------------------------------------------------------------------------------------ K3
class CameraBlock:
    """Device-resident camera data of one frame (all N source views + target centre).

    The centres are `inverse(ext)[:3,3]` exactly as the reference computes them
    (reference lib/networks/enerf/utils.py:771-772); pass `centers`/`tar_center` when they were
    already computed (Network hoists all camera algebra to the top of the frame)."""

    def __init__(self, src_exts, src_ixts, tar_ext=None, centers=None, tar_center=None):
        self.exts = _cf32(src_exts, "src_exts")            # (N,4,4)
        self.ixts = _cf32(src_ixts, "src_ixts")            # (N,3,3)
        if centers is None:
            centers = torch.stack([e.inverse()[:3, 3] for e in self.exts])
        if tar_center is None:
            tar_center = tar_ext.inverse()[:3, 3]
        self.centers = _cf32(centers, "centers")
        self.tar_center = _cf32(tar_center, "tar_center")


class RayGenerator:
    """On-device ray generation (SURVEY.md §8 f3): the 12 doubles the kernels need to produce ray r of a
    full target image instead of reading the (R,8) tensor the reference's loader builds on the host
    (reference lib/datasets/enerf_utils.py:25-31,62-71: origin = c2w[:3,3], direction =
    [x,y,1] @ (inv(K)^T @ R_c2w^T) in fp64, one cast to fp32).  `params` may be a slice of a larger
    device buffer (CUDA-graph replay refreshes it in place)."""

    def __init__(self, n_rays, params):
        assert params.dtype == torch.float64 and params.is_cuda and params.numel() == 12 and params.is_contiguous()
        self.n_rays, self.params = int(n_rays), params

    @staticmethod
    def host_params(tar_ext, tar_ixt, scale=1.0):
        """tar_ext (4,4), tar_ixt (3,3) host tensors/arrays -> float64 tensor (12,) on the host."""
        import numpy as np
        if torch.is_tensor(tar_ixt):
            tar_ixt = tar_ixt.detach().cpu().numpy()
        if torch.is_tensor(tar_ext):
            tar_ext = tar_ext.detach().cpu().numpy()
        ixt = np.array(tar_ixt, dtype=np.float64)
        if scale != 1.0:
            ixt[:2] *= scale
        c2w = np.linalg.inv(np.asarray(tar_ext, dtype=np.float64))
        M = np.linalg.inv(ixt).T @ c2w[:3, :3].T
        return torch.from_numpy(np.concatenate([c2w[:3, 3], M.reshape(-1)]))

    @classmethod
    def from_cameras(cls, tar_ext, tar_ixt, H, W, scale=1.0, device="cuda"):
        Hs, Ws = int(H * scale), int(W * scale)
        return cls(Hs * Ws, cls.host_params(tar_ext, tar_ixt, scale).to(device))


def _bind_rays(p, rays):
    """rays: (R,8) CUDA tensor or RayGenerator -> sets p.rays / p.ray_gen, returns (R, keepalive)."""
    if isinstance(rays, RayGenerator):
        p.ray_gen = rays.params.data_ptr()
        return rays.n_rays, rays.params
    rays = _cf32(rays, "rays")
    assert rays.shape[1] == 8
    p.rays = rays.data_ptr()
    return rays.shape[0], rays


def raygen_sample_fetch(depth, std, near_far, rays, H, W, depth_inv, S, volume, im_feat, rgb, cams, views,
                        render_scale=1.0, rgb_affine=(0.5, 0.5), ray_begin=0, n_rays=None,
                        want=("z_vals", "vox_feat", "img_feat", "vis_mask"), out=None):
    """Fused K3 for one cost-volume chain of one batch element.

    depth,std (hv,wv); near_far (2,hv,wv); rays (R,8); volume (Cv,Dv,hv,wv) any strides;
    im_feat (N,Cf,Hf,Wf) any strides; rgb (N,3,Hf,Wf) contiguous; cams CameraBlock; views triple.
    Returns a dict with the requested outputs among
    rays12 (n,12), z_vals (n,S), xyz (n,S,3), uvd (n,S,3), vox_feat (n*S,Cv), img_feat (n*S,V,Cf+7),
    vis_mask (n,S) fp32, vis_count (n,S) int32.  `out` may hold preallocated contiguous tensors for
    some of them (written in place, e.g. slices of a K-stacked buffer).
    """
    depth, std, near_far = _cf32(depth, "depth"), _cf32(std, "std"), _cf32(near_far, "near_far")
    dev = depth.device
    hv, wv = depth.shape
    V = len(views)
    p = _lib.RaygenFetchParams()
    R, _keep = _bind_rays(p, rays)
    n = R - ray_begin if n_rays is None else n_rays
    assert 0 <= ray_begin and ray_begin + n <= R
    p.depth, p.std, p.near_far = depth.data_ptr(), std.data_ptr(), near_far.data_ptr()
    p.hv, p.wv, p.H, p.W, p.depth_inv = hv, wv, H, W, int(depth_inv)
    p.ray_begin, p.n_rays = ray_begin, n
    t = _linspace(S, dev) if S > 1 else None
    p.t, p.S = (t.data_ptr() if t is not None else 0), S
    out = dict(out) if out else {}
    _fill_fetch_inputs(p, volume, im_feat, rgb, cams, views, render_scale, rgb_affine, want)
    _alloc_fetch_outputs(p, out, want, n, S, V, dev, p.Cv, p.Cf)
    _lib.call("bmv_raygen_sample_fetch", p, _stream())
    return out


def _fill_fetch_inputs(p, volume, im_feat, rgb, cams, views, render_scale, rgb_affine, want):
    V = len(views)
    p.V = V
    _views(p.view, views)
    if volume is not None:
        _f32(volume, "volume")
        p.volume = volume.data_ptr()
        p.Cv, p.Dv = volume.shape[0], volume.shape[1]
        p.vol_c_stride, p.vol_d_stride, p.vol_y_stride, p.vol_x_stride = volume.stride()
        if p.hv == 0:
            p.hv, p.wv = volume.shape[2], volume.shape[3]
    if im_feat is not None:
        _f32(im_feat, "im_feat")
        _f32(rgb, "rgb")
        p.im_feat = im_feat.data_ptr()
        p.Cf, p.Hf, p.Wf = im_feat.shape[1], im_feat.shape[2], im_feat.shape[3]
        p.imf_view_stride, p.imf_c_stride, p.imf_y_stride, p.imf_x_stride = im_feat.stride()
        assert rgb.shape[1:] == (3, p.Hf, p.Wf), (rgb.shape, p.Hf, p.Wf)
        p.rgb, p.rgb_view_stride = rgb.data_ptr(), rgb.stride(0)
        p.rgb_c_stride, p.rgb_y_stride, p.rgb_x_stride = rgb.stride(1), rgb.stride(2), rgb.stride(3)
        p.rgb_scale, p.rgb_shift = rgb_affine
        p._keep = (rgb,)
    p.src_exts, p.src_ixts = cams.exts.data_ptr(), cams.ixts.data_ptr()
    p.src_centers, p.tar_center = cams.centers.data_ptr(), cams.tar_center.data_ptr()
    p.render_scale = render_scale


def _numel(shape):
    n = 1
    for d in shape:
        n *= d
    return n


def _alloc_fetch_outputs(p, out, want, n, S, V, dev, Cv, Cf):
    def mk(name, shape, dtype=torch.float32):
        if name in out:
            t = out[name]
            if not (t.is_cuda and t.dtype == dtype and t.is_contiguous() and t.numel() == _numel(shape)):
                raise BmvError(f"preallocated output {name}: need contiguous {dtype} with {_numel(shape)} elements")
            setattr(p, name, t.data_ptr())
        elif name in want:
            out[name] = torch.empty(shape, device=dev, dtype=dtype)
            setattr(p, name, out[name].data_ptr())
    mk("rays12", (n, 12))
    mk("z_vals", (n, S))
    mk("xyz", (n, S, 3))
    mk("uvd", (n, S, 3))
    mk("vox_feat", (n * S, Cv))
    mk("img_feat", (n * S, V, Cf + 7))
    mk("vis_mask", (n, S))
    mk("vis_count", (n, S), torch.int32)


def sample_rays12(rays12, S, depth_inv, H, W, want=("xyz", "uvd", "z_vals")):
    """sample_along_depth on rays that already carry their interval
    (reference lib/networks/enerf/utils.py:424-443).  rays12 (R,12)."""
    rays12 = _cf32(rays12, "rays12")
    dev = rays12.device
    n = rays12.shape[0]
    p = _lib.RaygenFetchParams()
    p.rays12_in, p.ray_begin, p.n_rays = rays12.data_ptr(), 0, n
    p.H, p.W, p.hv, p.wv, p.depth_inv = H, W, 1, 1, int(depth_inv)
    t = _linspace(S, dev) if S > 1 else None
    p.t, p.S = (t.data_ptr() if t is not None else 0), S
    p.V = 1
    dummy = torch.zeros(16, device=dev)
    p.src_exts = p.src_ixts = dummy.data_ptr()
    out = {}
    _alloc_fetch_outputs(p, out, want, n, S, 1, dev, 0, 0)
    _lib.call("bmv_raygen_sample_fetch", p, _stream())
    return out


def fetch_points(xyz, uvd_norm, H, W, volume, im_feat, rgb, cams, views, render_scale=1.0,
                 rgb_affine=(0.5, 0.5), want=("vox_feat", "img_feat", "vis_mask")):
    """Pointwise mode: xyz (P,3) world points, uvd_norm (P,3) in [0,1] (needed for vox_feat).
    Function-level get_vox_feat / get_img_feat / mask_viewport on arbitrary points."""
    xyz = _cf32(xyz, "xyz")
    dev = xyz.device
    n = xyz.shape[0]
    p = _lib.RaygenFetchParams()
    p.xyz_in, p.n_rays, p.S = xyz.data_ptr(), n, 1
    if uvd_norm is not None:
        uvd_norm = _cf32(uvd_norm, "uvd_norm")
        p.uvd_in = uvd_norm.data_ptr()
    p.H, p.W = H, W
    out = {}
    _fill_fetch_inputs(p, volume, im_feat, rgb, cams, views, render_scale, rgb_affine, want)
    if p.hv == 0:
        p.hv = p.wv = 1
    _alloc_fetch_outputs(p, out, want, n, 1, len(views), dev, p.Cv, p.Cf)
    _lib.call("bmv_raygen_sample_fetch", p, _stream())
    return out


def mask_viewport(xyz, src_exts, src_ixts, views, inv_scale, want_count=False):
    """xyz (P,3); src_exts (N,4,4); src_ixts (N,3,3); inv_scale (W-1,H-1) ->
    fp32 mask (P,) in {0,1/V,..,1} [and int32 count] (reference lib/networks/enerf/utils.py:490-520)."""
    xyz = _cf32(xyz, "xyz")
    src_exts, src_ixts = _cf32(src_exts, "src_exts"), _cf32(src_ixts, "src_ixts")
    n = xyz.shape[0]
    dev = xyz.device
    mask = torch.empty(n, device=dev)
    count = torch.empty(n, device=dev, dtype=torch.int32) if want_count else None
    p = _lib.VisibilityParams()
    p.xyz, p.n_pts, p.V = xyz.data_ptr(), n, len(views)
    _views(p.view, views)
    p.src_exts, p.src_ixts = src_exts.data_ptr(), src_ixts.data_ptr()
    p.inv_scale_x, p.inv_scale_y = float(inv_scale[0]), float(inv_scale[1])
    p.vis_mask = mask.data_ptr()
    p.vis_count = count.data_ptr() if want_count else 0
    _lib.call("bmv_mask_viewport", p, _stream())
    return (mask, count) if want_count else mask


# ------------------------------------------------------------------------------------------ K4
def composite_blend(raws, masks, zs):
    """K-volume visibility-weighted compositing.  raws: K tensors (R,S,4); masks, zs: K tensors (R,S)
    (UN-normalised visibility scores; the 1/sum normalisation of merge_mlp_outputs happens in-kernel).
    -> rgb (R,3), depth (R,), weights (R,S)
    (reference lib/networks/boost_enerf/network.py:163-170, lib/networks/enerf/utils.py:639-667)."""
    K = len(raws)
    if not (1 <= K <= MAX_VOLUMES and len(masks) == K and len(zs) == K):
        raise BmvError(f"composite_blend: need 1..{MAX_VOLUMES} volumes with matching lists")
    raws = [_cf32(r, "raw") for r in raws]
    masks = [_cf32(m, "mask") for m in masks]
    zs = [_cf32(z, "z") for z in zs]
    R, S = raws[0].shape[0], raws[0].shape[1]
    dev = raws[0].device
    rgb = torch.empty((R, 3), device=dev)
    depth = torch.empty((R,), device=dev)
    weights = torch.empty((R, S), device=dev)
    p = _lib.CompositeBlendParams()
    p.K, p.S, p.R = K, S, R
    for k in range(K):
        assert raws[k].shape == (R, S, 4) and masks[k].shape == (R, S) and zs[k].shape == (R, S)
        p.raw[k], p.mask[k], p.z[k] = raws[k].data_ptr(), masks[k].data_ptr(), zs[k].data_ptr()
    p.rgb, p.depth, p.weights = rgb.data_ptr(), depth.data_ptr(), weights.data_ptr()
    _lib.call("bmv_composite_blend", p, _stream())
    return rgb, depth, weights


def composite(raw, z, white_bkgd=False):
    """Single-volume compositing.  raw (R,S,4), z (R,S) or None -> rgb, depth (None if z is None), weights
    (reference lib/networks/enerf/utils.py:605-637)."""
    raw = _cf32(raw, "raw")
    R, S = raw.shape[:2]
    dev = raw.device
    rgb = torch.empty((R, 3), device=dev)
    depth = torch.empty((R,), device=dev) if z is not None else None
    weights = torch.empty((R, S), device=dev)
    p = _lib.CompositeParams()
    p.S, p.R, p.raw = S, R, raw.data_ptr()
    if z is not None:
        z = _cf32(z, "z")
        p.z = z.data_ptr()
    p.white_bkgd = int(bool(white_bkgd))
    p.rgb, p.weights = rgb.data_ptr(), weights.data_ptr()
    p.depth = depth.data_ptr() if depth is not None else 0
    _lib.call("bmv_composite", p, _stream())
    return rgb, depth, weights


# ------------------------------------------------------------------------------------------ K5
def nerf_mlp(vox_feat, img_feat, packed_weights):
    """Fused per-sample MLP.  vox_feat (P,8), img_feat (P,V,feat_ch+4), packed_weights from
    mlp_pack.pack_nerf_weights -> raw (P,4) [rgb, sigma]
    (reference lib/networks/enerf/nerf.py:29-43)."""
    vox_feat, img_feat = _cf32(vox_feat, "vox_feat"), _cf32(img_feat, "img_feat")
    w = _cf32(packed_weights, "packed_weights")
    P, V, FV = img_feat.shape
    n = _lib.load().bmv_nerf_mlp_weight_count(FV - 4)
    if n != w.numel():
        raise BmvError(f"nerf_mlp: packed weight length {w.numel()} does not match feat_ch={FV - 4} (expects {n})")
    assert vox_feat.shape == (P, 8)
    raw = torch.empty((P, 4), device=vox_feat.device)
    p = _lib.NerfMlpParams()
    p.vox_feat, p.img_feat, p.weights = vox_feat.data_ptr(), img_feat.data_ptr(), w.data_ptr()
    p.P, p.feat_ch, p.V = P, FV - 4, V
    p.raw = raw.data_ptr()
    _lib.call("bmv_nerf_mlp", p, _stream())
    return raw


# ------------------------------------------------------------------------------------------ K3+K5
def render_rays_supported(Cv, Cf, V):
    return bool(_lib.load().bmv_render_rays_supported(int(Cv), int(Cf), int(V)))


def render_rays(depth, std, near_far, rays, H, W, depth_inv, S, volume, im_feat, rgb, cams, views, packed_weights,
                render_scale=1.0, rgb_affine=(0.5, 0.5), ray_begin=0, n_rays=None, out=None, want_count=False,
                engine="fma"):
    """Fused per-chain render (K3 gather + per-sample MLP, nothing materialised in HBM).
    Same inputs as raygen_sample_fetch plus the packed MLP weights.
    Returns dict(raw (n,S,4), z_vals (n,S), vis_mask (n,S) [, vis_count (n,S) int32]); `out` may
    supply preallocated contiguous tensors for any of them."""
    depth, std, near_far = _cf32(depth, "depth"), _cf32(std, "std"), _cf32(near_far, "near_far")
    if engine not in ("fma", "mma", "umma"):
        raise BmvError(f"render_rays: unknown engine {engine!r}")
    w = packed_weights
    if engine in ("mma", "umma"):
        words = getattr(_lib.load(), f"bmv_render_rays_{engine}_weight_words")()
        if not (torch.is_tensor(w) and w.is_cuda and w.dtype == torch.int32 and w.is_contiguous()
                and w.numel() == words):
            raise BmvError(f"render_rays(engine='{engine}'): weights must come from mlp_pack.pack_nerf_weights_{engine}")
    else:
        w = _cf32(w, "packed_weights")
    dev = depth.device
    rp = _lib.RenderRaysParams()
    p = rp.g
    R, _keep = _bind_rays(p, rays)
    n = R - ray_begin if n_rays is None else n_rays
    assert 0 <= ray_begin and ray_begin + n <= R
    hv, wv = depth.shape
    p.depth, p.std, p.near_far = depth.data_ptr(), std.data_ptr(), near_far.data_ptr()
    p.hv, p.wv, p.H, p.W, p.depth_inv = hv, wv, H, W, int(depth_inv)
    p.ray_begin, p.n_rays = ray_begin, n
    t = _linspace(S, dev) if S > 1 else None
    p.t, p.S = (t.data_ptr() if t is not None else 0), S
    _fill_fetch_inputs(p, volume, im_feat, rgb, cams, views, render_scale, rgb_affine, ())
    if engine == "fma" and _lib.load().bmv_nerf_mlp_weight_count(p.Cf + 3) != w.numel():
        raise BmvError(f"render_rays: packed weight length {w.numel()} does not match feat_ch={p.Cf + 3}")
    res = dict(out) if out else {}
    want = ("z_vals", "vis_mask") + (("vis_count",) if want_count else ())
    _alloc_fetch_outputs(p, res, want, n, S, len(views), dev, p.Cv, p.Cf)
    if "raw" in res:
        raw = res["raw"]
        if not (raw.is_cuda and raw.dtype == torch.float32 and raw.is_contiguous() and raw.numel() == n * S * 4):
            raise BmvError("preallocated output raw: need contiguous float32 with n*S*4 elements")
    else:
        raw = res["raw"] = torch.empty((n, S, 4), device=dev)
    rp.mlp_weights, rp.raw = w.data_ptr(), raw.data_ptr()
    _lib.call({"mma": "bmv_render_rays_mma", "umma": "bmv_render_rays_umma"}.get(engine, "bmv_render_rays"), rp, _stream())
    return res


def umma_selftest(a, w):
    """a (128,K) fp32 CUDA, w (N,K) fp32 -> a @ w.T through bmv_umma_selftest (one tcgen05 tile, split-fp16 operands)."""
    from .mlp_pack import pack_umma_matrix
    a = _cf32(a, "a")
    N, K = w.shape
    if a.shape != (128, K):
        raise BmvError(f"umma_selftest: a must be (128, {K})")
    b = pack_umma_matrix(w.detach().float().cpu()).to(a.device)
    d = torch.empty((128, N), device=a.device)
    lib = _lib.load()
    rc = lib.bmv_umma_selftest(a.data_ptr(), b.data_ptr(), d.data_ptr(), int(N), int(K), _stream())
    if rc != 0:
        raise BmvError(f"bmv_umma_selftest failed with status {rc}: {lib.bmv_last_error_string().decode()}")
    return d


# ------------------------------------------------------------------------------------------ K1b / K3b (MVSNeRF)
def cost_volume_var_img(feats, imgs_small, views, proj, planes, pad=24, out=None, out_dtype=torch.float32,
                        channels_last=False):
    """MVSNeRF 41-channel cost volume for one chain.
    feats (N,C,h,w) any strides; imgs_small (N,3,h,w) source images resized to the feature grid;
    views: the triple (views[0] = reference view); proj (V,3,4) in triple order; planes (D,)
    -> (3V+C, D, h+2pad, w+2pad)  (reference lib/networks/mvsnerf/network.py:887-942)."""
    _f32(feats, "feats")
    imgs_small, proj, planes = _cf32(imgs_small, "imgs_small"), _cf32(proj, "proj"), _cf32(planes, "planes")
    N, Cc, h, w = feats.shape
    V, D = len(views), planes.numel()
    assert imgs_small.shape == (N, 3, h, w) and proj.shape == (V, 3, 4)
    hp, wp, Ct = h + 2 * pad, w + 2 * pad, 3 * V + Cc
    if out is None:
        if channels_last:
            out = torch.empty((D, hp, wp, Ct), device=feats.device, dtype=out_dtype).permute(3, 0, 1, 2)
        else:
            out = torch.empty((Ct, D, hp, wp), device=feats.device, dtype=out_dtype)
    assert out.shape == (Ct, D, hp, wp) and out.dtype in (torch.float32, torch.bfloat16)
    p = _lib.CostVolumeImgParams()
    p.feat = feats.data_ptr()
    p.feat_view_stride, p.feat_c_stride, p.feat_y_stride, p.feat_x_stride = feats.stride()
    p.img = imgs_small.data_ptr()
    _views(p.view, views)
    p.V, p.C, p.h, p.w, p.D, p.pad = V, Cc, h, w, D, pad
    p.proj, p.planes, p.out = proj.data_ptr(), planes.data_ptr(), out.data_ptr()
    p.out_c_stride, p.out_d_stride, p.out_y_stride, p.out_x_stride = out.stride()
    p.out_bf16 = 1 if out.dtype == torch.bfloat16 else 0
    _lib.call("bmv_cost_volume_var_img", p, _stream())
    return out


def mvs_march_fetch(rays, S, views, src_exts, src_ixts, H, W, near, far, volume, rgb, pad=24,
                    rgb_affine=(0.5, 0.5), ray_begin=0, n_rays=None, want=("mlp_in", "z_vals", "vis_mask"), out=None):
    """MVSNeRF marching + fetch for one chain: rays (R,8) with near/far in columns 6,7; volume
    (8,D,h+2pad,w+2pad) any strides; rgb (N,3,H,W) raw source images.
    Returns dict with mlp_in (n,S,86), z_vals (n,S), vis_mask (n,S) [, vis_count]."""
    rays = _cf32(rays, "rays")
    src_exts, src_ixts = _cf32(src_exts, "src_exts"), _cf32(src_ixts, "src_ixts")
    dev = rays.device
    R = rays.shape[0]
    n = R - ray_begin if n_rays is None else n_rays
    if not (0 <= ray_begin and 0 <= n and ray_begin + n <= R):
        raise BmvError(f"mvs_march_fetch: rays [{ray_begin}, {ray_begin + n}) outside the {R} rays given")
    p = _lib.MvsMarchParams()
    p.rays, p.ray_begin, p.n_rays = rays.data_ptr(), ray_begin, n
    t = _linspace(S, dev)
    p.t, p.S, p.V = t.data_ptr(), S, len(views)
    _views(p.view, views)
    p.src_exts, p.src_ixts = src_exts.data_ptr(), src_ixts.data_ptr()
    p.H, p.W, p.near, p.far, p.pad = H, W, float(near), float(far), pad
    if volume is not None:
        _f32(volume, "volume")
        rgb = _cf32(rgb, "rgb")
        p.volume = volume.data_ptr()
        p.Cv, p.Dv, p.hv, p.wv = volume.shape
        p.vol_c_stride, p.vol_d_stride, p.vol_y_stride, p.vol_x_stride = volume.stride()
        p.rgb = rgb.data_ptr()
        p.rgb_scale, p.rgb_shift = rgb_affine
    res = dict(out) if out else {}

    def mk(name, shape, dtype=torch.float32):
        if name in res:
            tns = res[name]
            if not (tns.is_cuda and tns.dtype == dtype and tns.is_contiguous() and tns.numel() == _numel(shape)):
                raise BmvError(f"preallocated output {name}: need contiguous {dtype} with {_numel(shape)} elements")
            setattr(p, name, tns.data_ptr())
        elif name in want:
            res[name] = torch.empty(shape, device=dev, dtype=dtype)
            setattr(p, name, res[name].data_ptr())
    mk("mlp_in", (n, S, 86))
    mk("z_vals", (n, S))
    mk("vis_mask", (n, S))
    mk("vis_count", (n, S), torch.int32)
    _lib.call("bmv_mvs_march_fetch", p, _stream())
    return res


# ------------------------------------------------------------------------------------------ FPN top-down fusion
def fpn_topdown(prev, lateral_in, weight, bias):
    """out = bilinear_up2x(prev, align_corners=True) + conv1x1(lateral_in, weight, bias)
    (reference lib/networks/enerf/feature_net.py:24-33).  prev (N,32,H/2,W/2) and lateral_in (N,Cin,H,W)
    must be channels_last; weight (32,Cin[,1,1]); returns (N,32,H,W) channels_last."""
    _f32(prev, "prev"); _f32(lateral_in, "lateral_in")
    N, Cin, H, W = lateral_in.shape
    if not (prev.is_contiguous(memory_format=torch.channels_last) and lateral_in.is_contiguous(memory_format=torch.channels_last)):
        raise BmvError("fpn_topdown: inputs must be channels_last")
    assert prev.shape == (N, 32, H // 2, W // 2), prev.shape
    w = _cf32(weight.reshape(32, Cin), "weight")
    b = _cf32(bias, "bias") if bias is not None else None
    out = torch.empty((N, 32, H, W), device=prev.device, memory_format=torch.channels_last)
    p = _lib.FpnTopdownParams()
    p.prev, p.lateral_in, p.weight = prev.data_ptr(), lateral_in.data_ptr(), w.data_ptr()
    p.bias = b.data_ptr() if b is not None else 0
    p.N, p.H, p.W, p.Cin = N, H, W, Cin
    p.out = out.data_ptr()
    _lib.call("bmv_fpn_topdown", p, _stream())
    return out


# ------------------------------------------------------------------------------------------ tensor-core 3-D convolution
def conv3d_k3(x, wfrag, bias, cout, relu, out=None, out2=None, split=0, stride=1, no_tma=False, out_dtype=torch.float32,
              engine="mma", in_scale=None):
    """3x3x3 / stride 1 / pad 1 convolution (+bias, optional ReLU) of a channels_last_3d fp32 volume
    on tensor cores (fp16 operands, fp32 accumulation: TF32-class; reference ConvBnReLU3D / output heads,
    lib/networks/enerf/cost_reg_net.py:7-13,27-35).  x (N,Cin,D,H,W); wfrag from mlp_pack.pack_conv3d_k3;
    returns (N,cout,D,H,W) channels_last_3d (or writes `out`, any voxel-major strides).  With `out2`
    (N,cout-split,D,H,W) channels >= split go there instead (`out` then holds `split` channels).
    x may also be float16 (the operands are rounded to fp16 anyway: same result, half the read traffic).
    engine='umma': bmv_conv3d_k3_umma (TMA + tcgen05 + tensor memory; fp16 x, stride 1, Cin 8/16, wfrag from
    mlp_pack.pack_conv3d_k3_umma)."""
    if engine not in ("mma", "umma"):
        raise BmvError(f"conv3d_k3: unknown engine {engine!r}")
    if engine == "umma" and (x.dtype != torch.float16 or stride != 1):
        raise BmvError("conv3d_k3(engine='umma'): needs a float16 input and stride 1")
    if not (x.is_cuda and x.dtype in (torch.float32, torch.float16)):
        raise BmvError(f"conv3d_k3: x must be a CUDA float32/float16 tensor, got {x.dtype} on {x.device}")
    N, Cin, D, H, W = x.shape
    if x.stride(1) != 1:
        raise BmvError("conv3d_k3: x must be channels_last_3d")
    if out is None:
        Do, Ho, Wo = (((D - 1) // 2 + 1, (H - 1) // 2 + 1, (W - 1) // 2 + 1) if stride == 2 else (D, H, W))
        out = torch.empty((N, split if out2 is not None else cout, Do, Ho, Wo), device=x.device, dtype=out_dtype,
                          memory_format=torch.channels_last_3d)
    if out.stride(1) != 1 or (out2 is not None and out2.shape[1] > 1 and out2.stride(1) != 1):
        raise BmvError("conv3d_k3: out must be channels_last_3d")
    need = (_lib.load().bmv_conv3d_k3_umma_weight_words if engine == "umma" else _lib.load().bmv_conv3d_k3_weight_words)(Cin, cout)
    if need < 0 or wfrag.numel() != need or wfrag.dtype != torch.int32:
        raise BmvError(f"conv3d_k3: weight buffer does not match (Cin={Cin}, Cout={cout}, engine={engine}): {wfrag.numel()} vs {need}")
    p = _lib.Conv3dParams()
    p.x = x.data_ptr()
    p.x_n_stride, p.x_d_stride, p.x_y_stride, p.x_x_stride = x.stride(0), x.stride(2), x.stride(3), x.stride(4)
    p.wfrag = wfrag.data_ptr()
    p.bias = _cf32(bias, "bias").data_ptr() if bias is not None else 0
    p.N, p.D, p.H, p.W, p.Cin, p.Cout, p.relu = N, D, H, W, Cin, cout, int(bool(relu))
    p.stride = stride
    p.in_half = int(x.dtype == torch.float16)
    p.no_tma = int(bool(no_tma))
    p.out_half = int(out.dtype == torch.float16)
    p.in_scale = _scale_ptr(in_scale)
    p.out = out.data_ptr()
    p.o_n_stride, p.o_d_stride, p.o_y_stride, p.o_x_stride = out.stride(0), out.stride(2), out.stride(3), out.stride(4)
    if out2 is not None:
        _f32(out2, "out2")
        p.out2, p.split = out2.data_ptr(), split
        p.o2_n_stride, p.o2_d_stride, p.o2_y_stride, p.o2_x_stride = (out2.stride(0), out2.stride(2), out2.stride(3),
                                                                      out2.stride(4))
    _lib.call("bmv_conv3d_k3_umma" if engine == "umma" else "bmv_conv3d_k3", p, _stream())
    return out


def convT3d_k3s2_add(x, wfrag, bias, cout, skip=None, out_dtype=torch.float32):
    """out = skip + ConvTranspose3d(k=3, stride=2, padding=1, output_padding=1)(x) + bias on tensor cores
    (fp16 operands, fp32 accumulation; reference `x = conv0 + self.conv11(x)`,
    lib/networks/enerf/cost_reg_net.py:40-44,80-82).  x (N,Cin,D,H,W) and skip (N,cout,2D,2H,2W)
    channels_last_3d; wfrag from mlp_pack.pack_convT3d_k3s2."""
    if not (x.is_cuda and x.dtype in (torch.float32, torch.float16)):
        raise BmvError(f"convT3d_k3s2_add: x must be a CUDA float32/float16 tensor, got {x.dtype}")
    N, Cin, D, H, W = x.shape
    if x.stride(1) != 1:
        raise BmvError("convT3d_k3s2_add: x must be channels_last_3d")
    need = _lib.load().bmv_convT3d_k3s2_weight_words(Cin, cout)
    if need < 0 or wfrag.numel() != need or wfrag.dtype != torch.int32:
        raise BmvError(f"convT3d_k3s2_add: weight buffer does not match (Cin={Cin}, Cout={cout})")
    if out_dtype not in (torch.float32, torch.float16):
        raise BmvError("convT3d_k3s2_add: out_dtype must be float32 or float16")
    out = torch.empty((N, cout, 2 * D, 2 * H, 2 * W), device=x.device, dtype=out_dtype, memory_format=torch.channels_last_3d)
    p = _lib.ConvT3dParams()
    p.out_half = int(out_dtype == torch.float16)
    p.in_half = int(x.dtype == torch.float16)
    p.x = x.data_ptr()
    p.x_n_stride, p.x_d_stride, p.x_y_stride, p.x_x_stride = x.stride(0), x.stride(2), x.stride(3), x.stride(4)
    p.wfrag = wfrag.data_ptr()
    p.bias = _cf32(bias, "bias").data_ptr() if bias is not None else 0
    p.N, p.D, p.H, p.W, p.Cin, p.Cout = N, D, H, W, Cin, cout
    if skip is not None:
        if not (skip.is_cuda and skip.dtype in (torch.float32, torch.float16)):
            raise BmvError("convT3d_k3s2_add: skip must be a CUDA float32/float16 tensor")
        p.skip_half = int(skip.dtype == torch.float16)
        if tuple(skip.shape) != tuple(out.shape) or skip.stride(1) != 1:
            raise BmvError(f"convT3d_k3s2_add: skip must be channels_last_3d of shape {tuple(out.shape)}")
        p.skip = skip.data_ptr()
        p.s_n_stride, p.s_d_stride, p.s_y_stride, p.s_x_stride = skip.stride(0), skip.stride(2), skip.stride(3), skip.stride(4)
    p.out = out.data_ptr()
    p.o_n_stride, p.o_d_stride, p.o_y_stride, p.o_x_stride = out.stride(0), out.stride(2), out.stride(3), out.stride(4)
    _lib.call("bmv_convT3d_k3s2", p, _stream())
    return out


def conv3d_small(x, wfrag, bias, cout, stride=1, relu=True, transposed=False, skip=None, out_dtype=torch.float16):
    """3x3x3 convolution (+bias, +ReLU) — or ConvTranspose3d(k3, s2, p1, op1) + bias + skip with transposed=True — for
    the low-resolution core of the cost regularisers (bmv_conv3d_small; fp16 operands, fp32 accumulation).  x fp16
    channels_last_3d (N,Cin,D,H,W); wfrag from mlp_pack.pack_conv3d_small; skip fp16, dense, of the output's shape."""
    if not (torch.is_tensor(x) and x.is_cuda and x.dtype == torch.float16 and x.dim() == 5 and x.stride(1) == 1):
        raise BmvError("conv3d_small: x must be a channels_last_3d fp16 CUDA tensor (N,C,D,H,W)")
    _on_current_device(x, "x")
    N, Cin, D, H, W = x.shape
    need = _lib.load().bmv_conv3d_small_weight_words(Cin, cout, int(transposed))
    if need < 0 or wfrag.dtype != torch.int32 or wfrag.numel() != need:
        raise BmvError(f"conv3d_small: ({Cin} -> {cout}, transposed={transposed}) not instantiated or wfrag does not match")
    if transposed:
        stride = 2
        osz = (2 * D, 2 * H, 2 * W)
    else:
        osz = ((D - 1) // stride + 1, (H - 1) // stride + 1, (W - 1) // stride + 1)
    out = torch.empty((N, cout) + osz, device=x.device, dtype=out_dtype, memory_format=torch.channels_last_3d)
    p = _lib.Conv3dSmallParams()
    p.x = x.data_ptr()
    p.x_n_stride, p.x_d_stride, p.x_y_stride, p.x_x_stride = x.stride(0), x.stride(2), x.stride(3), x.stride(4)
    p.N, p.D, p.H, p.W, p.Cin, p.Cout = N, D, H, W, Cin, cout
    p.stride, p.transposed, p.relu, p.out_half = stride, int(transposed), int(relu), int(out_dtype == torch.float16)
    p.wfrag = wfrag.data_ptr()
    p.bias = _cf32(bias, "bias").data_ptr() if bias is not None else 0
    if skip is not None:
        if not (skip.is_cuda and skip.dtype == torch.float16 and tuple(skip.shape) == tuple(out.shape)
                and skip.is_contiguous(memory_format=torch.channels_last_3d)):
            raise BmvError(f"conv3d_small: skip must be a dense channels_last_3d fp16 tensor of shape {tuple(out.shape)}")
        p.skip = skip.data_ptr()
    p.out = out.data_ptr()
    _lib.call("bmv_conv3d_small", p, _stream())
    return out


def fpn_topdown_smooth(prev, lateral_in, lat_weight, lat_bias, smooth_wfrag, smooth_bias, cout, write_mid, want_half=False):
    """mid = up2x(prev) + conv1x1(lateral_in) + lat_bias; out = conv3x3(mid) + smooth_bias in ONE launch
    (reference lib/networks/enerf/feature_net.py:24-47; the 3x3 runs on tensor cores with fp16 operands).
    Returns (mid or None, out); tensors channels_last, smooth_wfrag from mlp_pack.pack_conv2d_k3_c32.
    want_half: True = also write an fp16 copy of out (returned as a third value) for the cost-volume kernel's fp16
    taps; 'only' = write out in fp16 ONLY (returned in place of out).  lateral_in: fp32 or fp16 (what fpn_stem /
    conv2d_k3 emit with out_dtype=float16: the 1x1 lateral then takes it as an exact tensor-core operand)."""
    _f32(prev, "prev")
    if lateral_in.dtype != torch.float16:
        _f32(lateral_in, "lateral_in")
    elif not lateral_in.is_cuda:
        raise BmvError("fpn_topdown_smooth: lateral_in must be a CUDA tensor")
    N, Cin, H, W = lateral_in.shape
    if not (prev.is_contiguous(memory_format=torch.channels_last) and lateral_in.is_contiguous(memory_format=torch.channels_last)):
        raise BmvError("fpn_topdown_smooth: inputs must be channels_last")
    assert prev.shape == (N, 32, H // 2, W // 2), prev.shape
    if smooth_wfrag.dtype != torch.int32 or smooth_wfrag.numel() != _lib.load().bmv_fpn_topdown_smooth_weight_words(cout):
        raise BmvError(f"fpn_topdown_smooth: weight buffer does not match Cout={cout}")
    w = _cf32(lat_weight.reshape(32, Cin), "lat_weight")
    lb = _cf32(lat_bias, "lat_bias") if lat_bias is not None else None
    sb = _cf32(smooth_bias, "smooth_bias") if smooth_bias is not None else None
    out = None if want_half == 'only' else torch.empty((N, cout, H, W), device=prev.device, memory_format=torch.channels_last)
    mid = torch.empty((N, 32, H, W), device=prev.device, memory_format=torch.channels_last) if write_mid else None
    p = _lib.FpnFusedParams()
    p.prev, p.lateral_in, p.lat_weight = prev.data_ptr(), lateral_in.data_ptr(), w.data_ptr()
    p.lat_bias = lb.data_ptr() if lb is not None else 0
    p.wfrag = smooth_wfrag.data_ptr()
    p.bias = sb.data_ptr() if sb is not None else 0
    p.N, p.H, p.W, p.Cin, p.Cout = N, H, W, Cin, cout
    p.lat_half = int(lateral_in.dtype == torch.float16)
    p.mid = mid.data_ptr() if mid is not None else 0
    p.out = out.data_ptr() if out is not None else 0
    out16 = torch.empty((N, cout, H, W), device=prev.device, dtype=torch.float16, memory_format=torch.channels_last) if want_half else None
    p.out16 = out16.data_ptr() if want_half else 0
    _lib.call("bmv_fpn_topdown_smooth", p, _stream())
    if want_half == 'only':
        return mid, out16
    return (mid, out, out16) if want_half else (mid, out)


def fpn_stem(x, w0, b0, wfrag1, b1, want_rgb4=False, want_s2d=False, out_dtype=torch.float32):
    """relu(conv3x3_{8->8}(relu(conv3x3_{3->8}(x) + b0)) + b1) in one launch (reference
    lib/networks/enerf/feature_net.py:7-9; BN already folded into w/b).  x (N,3,H,W) fp32, any strides;
    returns (N,8,H,W) channels_last — and, with want_rgb4, also x as an (N,H,W,4) [r,g,b,0] tensor (the layout
    the render kernels fetch colours from with one 16-byte load per tap); with want_s2d (implies the 3-tuple
    return) also the space-to-depth(2) copy of the output, (N,32,H/2,W/2) channels_last with channel order
    (py, px, c) — the input layout of the regrouped 5x5/stride-2 layer (inference_plan.S2DConv5x5)."""
    _f32(x, "x")
    N, C, H, W = x.shape
    if C != 3:
        raise BmvError("fpn_stem: x must have 3 channels")
    if wfrag1.dtype != torch.int32 or wfrag1.numel() != 384:
        raise BmvError("fpn_stem: wfrag1 must come from mlp_pack.pack_conv2d_k3_c8")
    w0c, b0c, b1c = _cf32(w0.reshape(8, 27), "w0"), _cf32(b0, "b0"), _cf32(b1, "b1")
    if out_dtype not in (torch.float32, torch.float16) or (out_dtype == torch.float16 and want_s2d):
        raise BmvError("fpn_stem: out_dtype is fp32 or fp16 (fp16 without the space-to-depth copy)")
    out = torch.empty((N, 8, H, W), device=x.device, dtype=out_dtype, memory_format=torch.channels_last)
    p = _lib.FpnStemParams()
    p.out_half = int(out_dtype == torch.float16)
    p.x = x.data_ptr()
    p.x_n_stride, p.x_c_stride, p.x_y_stride, p.x_x_stride = x.stride()
    p.w0, p.b0, p.wfrag1, p.b1 = w0c.data_ptr(), b0c.data_ptr(), wfrag1.data_ptr(), b1c.data_ptr()
    p.N, p.H, p.W = N, H, W
    p.out = out.data_ptr()
    rgb4 = torch.empty((N, H, W, 4), device=x.device) if want_rgb4 else None
    p.rgb4 = rgb4.data_ptr() if want_rgb4 else 0
    s2d = None
    if want_s2d:
        if H % 2 or W % 2:
            raise BmvError("fpn_stem: space-to-depth output needs even H and W")
        s2d = torch.empty((N, 32, H // 2, W // 2), device=x.device, memory_format=torch.channels_last)
        p.out_s2d = s2d.data_ptr()
    _lib.call("bmv_fpn_stem", p, _stream())
    if want_s2d:
        return out, rgb4, s2d
    return (out, rgb4) if want_rgb4 else out


def conv2d_k3(x, wfrag, bias, cout, relu=True, s2d=False, out_dtype=torch.float32, wfrag1x1=None, bias1x1=None, cout1x1=32):
    """3x3 / pad-1 convolution (+bias, +ReLU) of the FPN's middle layers on tensor cores (bmv_conv2d_k3; fp16 operands,
    fp32 accumulation: TF32-class).  x channels-last: fp16 (N,Cin,H,W), or with s2d=True fp32 (N,Cin/4,2H,2W) read
    through space-to-depth(2) (a 5x5 / stride-2 layer regrouped by inference_plan.S2DConv5x5).  wfrag from
    mlp_pack.pack_conv2d_k3.  With wfrag1x1 (mlp_pack.pack_conv1x1_after) a 1x1 convolution is applied to the ReLU'd
    result inside the epilogue and only ITS output (fp32) is written."""
    if not (torch.is_tensor(x) and x.is_cuda and x.dim() == 4 and x.stride(1) == 1):
        raise BmvError("conv2d_k3: x must be a channels-last CUDA tensor (N,C,H,W)")
    _on_current_device(x, "x")
    if s2d:
        if x.dtype not in (torch.float32, torch.float16) or x.shape[2] % 2 or x.shape[3] % 2:
            raise BmvError("conv2d_k3: the space-to-depth mode reads an fp32 / fp16 tensor with even H and W")
        N, cin, H, W = x.shape[0], 4 * x.shape[1], x.shape[2] // 2, x.shape[3] // 2
    else:
        if x.dtype != torch.float16:
            raise BmvError("conv2d_k3: the dense mode reads fp16")
        N, cin, H, W = x.shape
    words = _lib.load().bmv_conv2d_k3_weight_words(cin, cout)
    if words < 0 or wfrag.dtype != torch.int32 or wfrag.numel() != words:
        raise BmvError(f"conv2d_k3: ({cin} -> {cout}) not instantiated or wfrag is not from mlp_pack.pack_conv2d_k3")
    fuse = wfrag1x1 is not None
    co = cout1x1 if fuse else cout
    if fuse and out_dtype != torch.float32:
        raise BmvError("conv2d_k3: the fused 1x1 layer writes fp32")
    out = torch.empty((N, co, H, W), device=x.device, dtype=out_dtype, memory_format=torch.channels_last)
    p = _lib.Conv2dParams()
    p.x = x.data_ptr()
    p.x_n_stride, p.x_y_stride, p.x_x_stride = x.stride(0), x.stride(2), x.stride(3)
    p.N, p.H, p.W, p.Cin, p.Cout = N, H, W, cin, cout
    p.s2d, p.in_half, p.out_half, p.relu = int(s2d), int(x.dtype == torch.float16), int(out_dtype == torch.float16), int(relu)
    p.wfrag = wfrag.data_ptr()
    p.bias = _cf32(bias, "bias").data_ptr() if bias is not None else 0
    p.out = out.data_ptr()
    p.o_n_stride, p.o_y_stride, p.o_x_stride = out.stride(0), out.stride(2), out.stride(3)
    if fuse:
        if wfrag1x1.dtype != torch.int32 or wfrag1x1.numel() != 2 * 4 * 32 * 2:
            raise BmvError("conv2d_k3: wfrag1x1 must come from mlp_pack.pack_conv1x1_after")
        p.wfrag1x1 = wfrag1x1.data_ptr()
        p.bias1x1 = _cf32(bias1x1, "bias1x1").data_ptr() if bias1x1 is not None else 0
        p.C1x1_out = cout1x1
    _lib.call("bmv_conv2d_k3", p, _stream())
    return out


# ------------------------------------------------------------------------------------------ f4: output sinks
def frame_psnr_accumulate(pred, gt, H, W, mask=None, crop=(0, 0), acc=None):
    """Adds the masked / centre-cropped squared error of one frame to `acc` = (sse float64[1], count int64[1]) on the
    device (allocated when None) and returns it (reference lib/evaluators/enerf.py:45-71).  pred, gt: (H*W,3) fp32;
    mask: (H*W) uint8 or None; crop = (crop_h, crop_w) rows / columns dropped at each border."""
    pred, gt = _cf32(pred.reshape(-1, 3), "pred"), _cf32(gt.reshape(-1, 3), "gt")
    if pred.shape[0] != H * W or gt.shape[0] != H * W:
        raise BmvError(f"frame_psnr_accumulate: expected {H * W} pixels, got {pred.shape[0]} / {gt.shape[0]}")
    if acc is None:
        acc = (torch.zeros(1, device=pred.device, dtype=torch.float64), torch.zeros(1, device=pred.device, dtype=torch.int64))
    p = _lib.FramePsnrParams()
    p.pred, p.gt = pred.data_ptr(), gt.data_ptr()
    if mask is not None:
        if not (mask.is_cuda and mask.dtype == torch.uint8 and mask.numel() == H * W and mask.is_contiguous()):
            raise BmvError("frame_psnr_accumulate: mask must be a contiguous CUDA uint8 tensor with H*W elements")
        p.mask = mask.data_ptr()
    p.H, p.W, p.crop_h, p.crop_w = H, W, int(crop[0]), int(crop[1])
    p.sse, p.count = acc[0].data_ptr(), acc[1].data_ptr()
    _lib.call("bmv_frame_psnr_accumulate", p, _stream())
    return acc


def frame_ssim(pred, gt, H, W, crop=(0, 0), win_size=7, data_range=2.0, out=None):
    """SSIM of one frame, skimage.metrics.structural_similarity(gt, pred, channel_axis=-1, win_size=win_size,
    data_range=data_range) with uniform weights, in float64 on the device (bmv_frame_ssim).  pred, gt: (H*W,3) fp32;
    crop = (crop_h, crop_w) rows / columns dropped at each border before the metric sees the image.  Returns `out`, a
    1-element float64 device tensor (allocated when None); nothing is read back.

    The reference does not record the arguments its evaluator passes to skimage: the defaults are skimage's for a float
    image (scikit-image <= 0.20: win_size 7, data_range 2 = the span of dtype_range[float32] = (-1, 1))."""
    pred, gt = _cf32(pred.reshape(-1, 3), "pred"), _cf32(gt.reshape(-1, 3), "gt")
    if pred.shape[0] != H * W or gt.shape[0] != H * W:
        raise BmvError(f"frame_ssim: expected {H * W} pixels, got {pred.shape[0]} / {gt.shape[0]}")
    if out is None:
        out = torch.empty(1, device=pred.device, dtype=torch.float64)
    elif not (torch.is_tensor(out) and out.is_cuda and out.dtype == torch.float64 and out.numel() == 1):
        raise BmvError("frame_ssim: out must be a 1-element CUDA float64 tensor")
    _on_current_device(out, "out")
    scratch = torch.empty(_lib.FRAME_SSIM_SCRATCH_WORDS, device=pred.device, dtype=torch.float64)
    p = _lib.FrameSsimParams()
    p.pred, p.gt = pred.data_ptr(), gt.data_ptr()
    p.H, p.W, p.crop_h, p.crop_w = H, W, int(crop[0]), int(crop[1])
    p.win_size, p.data_range = int(win_size), float(data_range)
    p.scratch, p.ssim = scratch.data_ptr(), out.data_ptr()
    _lib.call("bmv_frame_ssim", p, _stream())
    return out


def frame_to_u8(rgb=None, depth=None):
    """rgb (R,3) fp32 -> uint8 `(rgb*255).astype(uint8)`; depth (R,) fp32 -> uint8 `((d-min)/(max-min)*255).astype(uint8)`
    (reference lib/visualizers/enerf.py:27-37).  Returns (rgb_u8 or None, depth_u8 or None, minmax (2,) fp32 or None)."""
    if rgb is None and depth is None:
        raise BmvError("frame_to_u8: nothing to convert")
    p = _lib.FrameToU8Params()
    rgb_u8 = depth_u8 = minmax = None
    if rgb is not None:
        rgb = _cf32(rgb.reshape(-1, 3), "rgb")
        rgb_u8 = torch.empty(rgb.shape, device=rgb.device, dtype=torch.uint8)
        p.R, p.rgb, p.rgb_u8 = rgb.shape[0], rgb.data_ptr(), rgb_u8.data_ptr()
    if depth is not None:
        depth = _cf32(depth.reshape(-1), "depth")
        if rgb is not None and depth.numel() != rgb.shape[0]:
            raise BmvError("frame_to_u8: rgb and depth must cover the same rays")
        depth_u8 = torch.empty(depth.shape, device=depth.device, dtype=torch.uint8)
        scratch = torch.empty(2, device=depth.device, dtype=torch.int32)
        minmax = torch.empty(2, device=depth.device)
        p.R, p.depth, p.depth_u8 = depth.numel(), depth.data_ptr(), depth_u8.data_ptr()
        p.minmax_ord, p.minmax = scratch.data_ptr(), minmax.data_ptr()
    _lib.call("bmv_frame_to_u8", p, _stream())
    return rgb_u8, depth_u8, minmax


# ------------------------------------------------------------------------------------------ K3+K5, all chains in one launch
def render_rays_multi_supported(volumes, im_feat, rgb, V):
    """Layouts bmv_render_rays_multi is instantiated for: (K,8,D,h,w) dense channels-last-3d volumes, (N,8,Hf,Wf)
    dense channels-last feature maps, (N,3,Hf,Wf) colours viewed from an (N,Hf,Wf,4) tensor, triples."""
    if not (V == 3 and volumes.dim() == 5 and volumes.shape[1] == 8 and im_feat.shape[1] == 8 and volumes.shape[0] <= MAX_VOLUMES):
        return False
    K, _, D, h, w = volumes.shape
    N, _, Hf, Wf = im_feat.shape
    return (volumes.dtype == torch.float32 and tuple(volumes.stride()[1:]) == (1, h * w * 8, w * 8, 8) and volumes.stride(0) % 8 == 0
            and volumes.data_ptr() % 32 == 0 and im_feat.data_ptr() % 32 == 0
            and im_feat.dtype == torch.float32 and tuple(im_feat.stride()[1:]) == (1, Wf * 8, 8) and im_feat.stride(0) % 8 == 0
            and rgb.dtype == torch.float32 and tuple(rgb.stride()[1:]) == (1, Wf * 4, 4) and rgb.stride(0) % 4 == 0
            and N <= MAX_VIEWS and D * h * w * 8 < 2 ** 31 and Hf * Wf * 8 < 2 ** 31)


def _rows_f32(t, name):
    """CUDA fp32 tensor whose trailing (rows, w) block is contiguous (any leading strides: slices of a stacked buffer)."""
    _f32(t, name)
    if t.stride(-1) != 1 or t.stride(-2) != t.shape[-1]:
        t = t.contiguous()
    return t


def render_rays_multi(depth, std, near_far, rays, H, W, depth_inv, S, volumes, im_feat, rgb, cams, triples, packed_weights,
                      render_scale=1.0, rgb_affine=(0.5, 0.5), ray_begin=0, n_rays=None, out=None, want_count=False,
                      views_dev=None, grid_rows=None, vol_row0=0, map_row0=0, engine=None):
    """K3 + per-sample MLP of ALL K chains in one persistent launch: bmv_render_rays_multi (engine 'mma': warp-level
    mma.sync MLP, weights from mlp_pack.pack_nerf_weights_mma) or bmv_render_rays_multi_umma (engine 'umma': tcgen05 MLP
    with accumulators in tensor memory, weights from mlp_pack.pack_nerf_weights_umma).  engine=None: told by the packing.
    depth, std (K,hv,wv); near_far (K,2,hv,wv) or shared (2,hv,wv); volumes (K,8,D,hv,wv) channels-last-3d; triples: K
    view triples (host list) — or views_dev, an int32 CUDA tensor (K,3) read by the kernel (graph-replay friendly);
    packed_weights from mlp_pack.pack_nerf_weights_mma.
    Row slabs (multi-GPU row tiles): depth / std / near_far hold map rows [map_row0, map_row0 + rows) and volumes volume
    rows [vol_row0, ...) of a grid with `grid_rows` rows; the rays of [ray_begin, ray_begin + n_rays) must only touch them.
    Returns dict(raw (K,n,S,4), z_vals (K,n,S), vis_mask (K,n,S) [, vis_count]); `out` may supply them."""
    depth, std, near_far = _rows_f32(depth, "depth"), _rows_f32(std, "std"), _rows_f32(near_far, "near_far")
    K, map_rows, wv = depth.shape
    hv = map_rows if grid_rows is None else int(grid_rows)
    if std.shape != depth.shape or near_far.shape[-2:] != depth.shape[-2:]:
        raise BmvError("render_rays_multi: depth / std / near_far must cover the same rows")
    w = packed_weights
    words = {"mma": _lib.load().bmv_render_rays_mma_weight_words(), "umma": _lib.load().bmv_render_rays_umma_weight_words()}
    if not (torch.is_tensor(w) and w.is_cuda and w.dtype == torch.int32 and w.is_contiguous()):
        raise BmvError("render_rays_multi: weights must be a contiguous int32 CUDA tensor from mlp_pack")
    if engine is None:
        engine = next((e for e, n_ in words.items() if w.numel() == n_), None)
    if engine not in words or w.numel() != words[engine]:
        raise BmvError("render_rays_multi: weights must come from mlp_pack.pack_nerf_weights_mma (engine 'mma') or "
                       "pack_nerf_weights_umma (engine 'umma')")
    if volumes.shape[0] != K or std.shape != depth.shape:
        raise BmvError("render_rays_multi: depth / std / volumes must agree on K")
    dev = depth.device
    mp = _lib.RenderMultiParams()
    p = mp.g
    R, _keep = _bind_rays(p, rays)
    n = R - ray_begin if n_rays is None else n_rays
    assert 0 <= ray_begin and ray_begin + n <= R
    p.hv, p.wv, p.H, p.W, p.depth_inv = hv, wv, H, W, int(depth_inv)
    p.ray_begin, p.n_rays = ray_begin, n
    t = _linspace(S, dev) if S > 1 else None
    p.t, p.S = (t.data_ptr() if t is not None else 0), S
    V = 3
    _fill_fetch_inputs(p, volumes[0], im_feat, rgb, cams, (0, 0, 0), render_scale, rgb_affine, ())
    mp.K, mp.n_views = K, im_feat.shape[0]
    mp.depth, mp.depth_k_stride = depth.data_ptr(), depth.stride(0)
    mp.std, mp.std_k_stride = std.data_ptr(), std.stride(0)
    if near_far.dim() == 4:
        if near_far.shape[0] != K:
            raise BmvError("render_rays_multi: near_far must be (K,2,hv,wv) or (2,hv,wv)")
        mp.near_far, mp.nf_k_stride, mp.nf_plane_stride = near_far.data_ptr(), near_far.stride(0), near_far.stride(1)
    else:
        mp.near_far, mp.nf_k_stride, mp.nf_plane_stride = near_far.data_ptr(), 0, near_far.stride(0)
    mp.vol_row0, mp.map_row0 = int(vol_row0), int(map_row0)
    mp.volume, mp.vol_k_stride = volumes.data_ptr(), volumes.stride(0)
    if views_dev is not None:
        if not (views_dev.is_cuda and views_dev.dtype == torch.int32 and views_dev.is_contiguous() and views_dev.numel() == K * V):
            raise BmvError("render_rays_multi: views_dev must be a contiguous int32 CUDA tensor with K*3 elements")
        mp.views = views_dev.data_ptr()
    else:
        if len(triples) != K or any(len(tr) != V for tr in triples):
            raise BmvError("render_rays_multi: need K view triples")
        for i, v in enumerate(v for tr in triples for v in tr):
            mp.views_host[i] = int(v)
    res = dict(out) if out else {}

    def mk(name, shape, dtype=torch.float32):
        if name in res:
            tns = res[name]
            if not (tns.is_cuda and tns.dtype == dtype and tns.is_contiguous() and tns.numel() == _numel(shape)):
                raise BmvError(f"preallocated output {name}: need contiguous {dtype} with {_numel(shape)} elements")
        else:
            res[name] = torch.empty(shape, device=dev, dtype=dtype)
        return res[name].data_ptr()
    mp.raw = mk("raw", (K, n, S, 4))
    mp.z_vals = mk("z_vals", (K, n, S))
    mp.vis_mask = mk("vis_mask", (K, n, S))
    if want_count or "vis_count" in res:
        mp.vis_count = mk("vis_count", (K, n, S), torch.int32)
    mp.mlp_weights = w.data_ptr()
    _lib.call("bmv_render_rays_multi_umma" if engine == "umma" else "bmv_render_rays_multi", mp, _stream())
    return res


# ------------------------------------------------------------------------------------------ K3b + MLP fused (MVSNeRF)
def mvs_render(rays, S, views, src_exts, src_ixts, H, W, near, far, volume, rgb, packed_weights, pad=24,
               rgb_affine=(0.5, 0.5), ray_begin=0, n_rays=None, out=None, want_count=False):
    """MVSNeRF marching + fetch + the 6x128 MLP in one tcgen05 kernel (bmv_mvs_render_umma): same inputs as
    mvs_march_fetch plus mlp_pack.pack_mvs_weights_umma(nerf); nothing per-sample is materialised.
    Returns dict(raw (n,S,4), z_vals (n,S), vis_mask (n,S) [, vis_count]).  TF32-class (fp16 operands)."""
    rays = _cf32(rays, "rays")
    src_exts, src_ixts = _cf32(src_exts, "src_exts"), _cf32(src_ixts, "src_ixts")
    _f32(volume, "volume")
    rgb = _cf32(rgb, "rgb")                                  # (N,3,H,W) planar, or (N,H,W,4) [r,g,b,x]
    nhwc4 = rgb.dim() == 4 and rgb.shape[-1] == 4 and rgb.shape[1] == H and rgb.shape[2] == W
    if not nhwc4 and tuple(rgb.shape[1:]) != (3, H, W):
        raise BmvError(f"mvs_render: rgb must be (N,3,{H},{W}) or (N,{H},{W},4), got {tuple(rgb.shape)}")
    dev = rays.device
    R = rays.shape[0]
    n = R - ray_begin if n_rays is None else n_rays
    if not (0 <= ray_begin and 0 <= n and ray_begin + n <= R):
        raise BmvError(f"mvs_render: rays [{ray_begin}, {ray_begin + n}) outside the {R} rays given")
    w = packed_weights
    if not (torch.is_tensor(w) and w.is_cuda and w.dtype == torch.int32 and w.is_contiguous()
            and w.numel() * 4 == _lib.load().bmv_mvs_render_umma_weight_bytes()):
        raise BmvError("mvs_render: weights must come from mlp_pack.pack_mvs_weights_umma")
    rp = _lib.MvsRenderParams()
    p = rp.g
    p.rays, p.ray_begin, p.n_rays = rays.data_ptr(), ray_begin, n
    t = _linspace(S, dev)
    p.t, p.S, p.V = t.data_ptr(), S, len(views)
    _views(p.view, views)
    p.src_exts, p.src_ixts = src_exts.data_ptr(), src_ixts.data_ptr()
    p.H, p.W, p.near, p.far, p.pad = H, W, float(near), float(far), pad
    p.volume = volume.data_ptr()
    p.Cv, p.Dv, p.hv, p.wv = volume.shape
    p.vol_c_stride, p.vol_d_stride, p.vol_y_stride, p.vol_x_stride = volume.stride()
    p.rgb = rgb.data_ptr()
    p.rgb_nhwc4 = int(nhwc4)
    p.rgb_scale, p.rgb_shift = rgb_affine
    res = dict(out) if out else {}

    def mk(name, shape, dtype=torch.float32):
        if name in res:
            tns = res[name]
            if not (tns.is_cuda and tns.dtype == dtype and tns.is_contiguous() and tns.numel() == _numel(shape)):
                raise BmvError(f"preallocated output {name}: need contiguous {dtype} with {_numel(shape)} elements")
        else:
            res[name] = torch.empty(shape, device=dev, dtype=dtype)
        return res[name].data_ptr()
    rp.raw = mk("raw", (n, S, 4))
    p.z_vals = mk("z_vals", (n, S))
    p.vis_mask = mk("vis_mask", (n, S))
    if want_count or "vis_count" in res:
        p.vis_count = mk("vis_count", (n, S), torch.int32)
    rp.weights = w.data_ptr()
    _lib.call("bmv_mvs_render_umma", rp, _stream())
    return res
