"""ctypes binding of libbmv.so — a 1:1 mirror of include/bmv.h.

There is NO fallback: if the shared library is missing or an entry point fails, an exception is
raised (north_star: "no CPU fallback, no multi-backend dispatch").
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libbmv.so")

MAX_VIEWS = 8
MAX_VOLUMES = 16
FRAME_SSIM_SCRATCH_WORDS = 2048

f32p = C.POINTER(C.c_float)
i32p = C.POINTER(C.c_int32)
i64, i32, f32 = C.c_int64, C.c_int32, C.c_float


class CostVolumeParams(C.Structure):
    _fields_ = [("feat", C.c_void_p), ("feat_view_stride", i64),
                ("feat_c_stride", i64), ("feat_y_stride", i64), ("feat_x_stride", i64),
                ("view", i32 * MAX_VIEWS), ("S", i32), ("C", i32), ("Hs", i32), ("Ws", i32),
                ("proj", C.c_void_p), ("planes", C.c_void_p),
                ("planes_d_stride", i64), ("planes_pix_stride", i64),
                ("D", i32), ("h", i32), ("w", i32),
                ("out", C.c_void_p),
                ("out_c_stride", i64), ("out_d_stride", i64), ("out_y_stride", i64), ("out_x_stride", i64),
                ("out_bf16", i32), ("exact_coords", i32), ("feat_half", i32), ("variant", i32),
                ("out_scale", C.c_void_p), ("view_dev", C.c_void_p)]


class CostVolumeMultiParams(C.Structure):
    _fields_ = [("b", CostVolumeParams), ("K", i32), ("views_per_chain", i32), ("chain_mask", i32 * MAX_VIEWS),
                ("out_k_stride", i64), ("triples_dev", C.c_void_p)]


class VolumeScaleParams(C.Structure):
    _fields_ = [("x", C.c_void_p), ("n", i64), ("x_half", i32), ("target", f32), ("scale", C.c_void_p),
                ("consumer_scale", f32), ("reserved0", i32)]


class DepthPlanesFirstParams(C.Structure):
    _fields_ = [("near_far", C.c_void_p), ("t", C.c_void_p),
                ("D", i32), ("h", i32), ("w", i32), ("depth_inv", i32),
                ("planes", C.c_void_p), ("near_far_out", C.c_void_p)]


class DepthPlanesNextParams(C.Structure):
    _fields_ = [("depth", C.c_void_p), ("std", C.c_void_p), ("near_far", C.c_void_p), ("t", C.c_void_p),
                ("h0", i32), ("w0", i32), ("h", i32), ("w", i32), ("D", i32), ("cur_inv", i32),
                ("planes", C.c_void_p), ("near_far_out", C.c_void_p),
                ("batch", i32), ("depth_b_stride", i64), ("std_b_stride", i64), ("nf_b_stride", i64)]


class DepthRegressionParams(C.Structure):
    _fields_ = [("logits", C.c_void_p), ("planes", C.c_void_p),
                ("planes_d_stride", i64), ("planes_pix_stride", i64),
                ("D", i32), ("h", i32), ("w", i32), ("depth_inv", i32),
                ("depth", C.c_void_p), ("std", C.c_void_p),
                ("batch", i32), ("logits_b_stride", i64), ("planes_b_stride", i64)]


class RaygenFetchParams(C.Structure):
    _fields_ = [("depth", C.c_void_p), ("std", C.c_void_p), ("near_far", C.c_void_p),
                ("hv", i32), ("wv", i32), ("H", i32), ("W", i32), ("depth_inv", i32),
                ("rays", C.c_void_p), ("ray_begin", i64), ("n_rays", i64),
                ("rays12_in", C.c_void_p), ("xyz_in", C.c_void_p), ("uvd_in", C.c_void_p), ("ray_gen", C.c_void_p),
                ("t", C.c_void_p), ("S", i32),
                ("volume", C.c_void_p), ("Cv", i32), ("Dv", i32),
                ("vol_c_stride", i64), ("vol_d_stride", i64), ("vol_y_stride", i64), ("vol_x_stride", i64),
                ("V", i32), ("view", i32 * MAX_VIEWS),
                ("im_feat", C.c_void_p), ("Cf", i32), ("Hf", i32), ("Wf", i32),
                ("imf_view_stride", i64), ("imf_c_stride", i64), ("imf_y_stride", i64), ("imf_x_stride", i64),
                ("rgb", C.c_void_p), ("rgb_view_stride", i64), ("rgb_scale", f32), ("rgb_shift", f32),
                ("src_exts", C.c_void_p), ("src_ixts", C.c_void_p), ("src_centers", C.c_void_p),
                ("tar_center", C.c_void_p), ("render_scale", f32),
                ("rays12", C.c_void_p), ("z_vals", C.c_void_p), ("xyz", C.c_void_p), ("uvd", C.c_void_p),
                ("vox_feat", C.c_void_p), ("img_feat", C.c_void_p),
                ("vis_mask", C.c_void_p), ("vis_count", C.c_void_p),
                ("rgb_c_stride", i64), ("rgb_y_stride", i64), ("rgb_x_stride", i64)]


class VisibilityParams(C.Structure):
    _fields_ = [("xyz", C.c_void_p), ("n_pts", i64), ("V", i32), ("view", i32 * MAX_VIEWS),
                ("src_exts", C.c_void_p), ("src_ixts", C.c_void_p),
                ("inv_scale_x", f32), ("inv_scale_y", f32),
                ("vis_mask", C.c_void_p), ("vis_count", C.c_void_p)]


class CompositeBlendParams(C.Structure):
    _fields_ = [("K", i32), ("S", i32), ("R", i64),
                ("raw", C.c_void_p * MAX_VOLUMES), ("mask", C.c_void_p * MAX_VOLUMES),
                ("z", C.c_void_p * MAX_VOLUMES),
                ("rgb", C.c_void_p), ("depth", C.c_void_p), ("weights", C.c_void_p)]


class CompositeParams(C.Structure):
    _fields_ = [("S", i32), ("R", i64), ("raw", C.c_void_p), ("z", C.c_void_p), ("white_bkgd", i32),
                ("rgb", C.c_void_p), ("depth", C.c_void_p), ("weights", C.c_void_p)]


class NerfMlpParams(C.Structure):
    _fields_ = [("vox_feat", C.c_void_p), ("img_feat", C.c_void_p), ("weights", C.c_void_p),
                ("P", i64), ("feat_ch", i32), ("V", i32), ("raw", C.c_void_p)]


class RenderRaysParams(C.Structure):
    _fields_ = [("g", RaygenFetchParams), ("mlp_weights", C.c_void_p), ("raw", C.c_void_p)]


class RenderMultiParams(C.Structure):
    _fields_ = [("g", RaygenFetchParams), ("K", i32), ("n_views", i32),
                ("depth", C.c_void_p), ("depth_k_stride", i64), ("std", C.c_void_p), ("std_k_stride", i64),
                ("near_far", C.c_void_p), ("nf_k_stride", i64), ("volume", C.c_void_p), ("vol_k_stride", i64),
                ("views", C.c_void_p), ("views_host", i32 * (MAX_VOLUMES * 3)),
                ("mlp_weights", C.c_void_p), ("raw", C.c_void_p), ("z_vals", C.c_void_p), ("vis_mask", C.c_void_p),
                ("vis_count", C.c_void_p), ("vol_row0", i32), ("map_row0", i32), ("nf_plane_stride", i64)]


class CostVolumeImgParams(C.Structure):
    _fields_ = [("feat", C.c_void_p), ("feat_view_stride", i64), ("feat_c_stride", i64), ("feat_y_stride", i64),
                ("feat_x_stride", i64), ("img", C.c_void_p), ("view", i32 * MAX_VIEWS),
                ("V", i32), ("C", i32), ("h", i32), ("w", i32), ("D", i32), ("pad", i32),
                ("proj", C.c_void_p), ("planes", C.c_void_p), ("out", C.c_void_p),
                ("out_c_stride", i64), ("out_d_stride", i64), ("out_y_stride", i64), ("out_x_stride", i64),
                ("out_bf16", i32)]


class MvsMarchParams(C.Structure):
    _fields_ = [("rays", C.c_void_p), ("ray_begin", i64), ("n_rays", i64), ("t", C.c_void_p), ("S", i32),
                ("V", i32), ("view", i32 * MAX_VIEWS), ("src_exts", C.c_void_p), ("src_ixts", C.c_void_p),
                ("H", i32), ("W", i32), ("near", f32), ("far", f32), ("pad", i32),
                ("volume", C.c_void_p), ("Cv", i32), ("Dv", i32), ("hv", i32), ("wv", i32),
                ("vol_c_stride", i64), ("vol_d_stride", i64), ("vol_y_stride", i64), ("vol_x_stride", i64),
                ("rgb", C.c_void_p), ("rgb_scale", f32), ("rgb_shift", f32),
                ("mlp_in", C.c_void_p), ("z_vals", C.c_void_p), ("vis_mask", C.c_void_p), ("vis_count", C.c_void_p),
                ("rgb_nhwc4", i32), ("reserved0", i32)]


class MvsRenderParams(C.Structure):
    _fields_ = [("g", MvsMarchParams), ("weights", C.c_void_p), ("raw", C.c_void_p)]


class FpnTopdownParams(C.Structure):
    _fields_ = [("prev", C.c_void_p), ("lateral_in", C.c_void_p), ("weight", C.c_void_p), ("bias", C.c_void_p),
                ("N", i32), ("H", i32), ("W", i32), ("Cin", i32), ("out", C.c_void_p)]


class Conv3dParams(C.Structure):
    _fields_ = [("x", C.c_void_p), ("x_n_stride", i64), ("x_d_stride", i64), ("x_y_stride", i64), ("x_x_stride", i64),
                ("wfrag", C.c_void_p), ("bias", C.c_void_p),
                ("N", i32), ("D", i32), ("H", i32), ("W", i32), ("Cin", i32), ("Cout", i32), ("relu", i32),
                ("out", C.c_void_p), ("o_n_stride", i64), ("o_d_stride", i64), ("o_y_stride", i64), ("o_x_stride", i64),
                ("out2", C.c_void_p), ("o2_n_stride", i64), ("o2_d_stride", i64), ("o2_y_stride", i64),
                ("o2_x_stride", i64), ("split", i32), ("stride", i32), ("in_half", i32), ("no_tma", i32), ("out_half", i32),
                ("reserved0", i32), ("in_scale", C.c_void_p)]


class ConvT3dParams(C.Structure):
    _fields_ = [("x", C.c_void_p), ("x_n_stride", i64), ("x_d_stride", i64), ("x_y_stride", i64), ("x_x_stride", i64),
                ("wfrag", C.c_void_p), ("bias", C.c_void_p),
                ("N", i32), ("D", i32), ("H", i32), ("W", i32), ("Cin", i32), ("Cout", i32),
                ("skip", C.c_void_p), ("s_n_stride", i64), ("s_d_stride", i64), ("s_y_stride", i64), ("s_x_stride", i64),
                ("out", C.c_void_p), ("o_n_stride", i64), ("o_d_stride", i64), ("o_y_stride", i64), ("o_x_stride", i64),
                ("out_half", i32), ("skip_half", i32), ("in_half", i32)]


class FpnFusedParams(C.Structure):
    _fields_ = [("prev", C.c_void_p), ("lateral_in", C.c_void_p), ("lat_weight", C.c_void_p), ("lat_bias", C.c_void_p),
                ("wfrag", C.c_void_p), ("bias", C.c_void_p),
                ("N", i32), ("H", i32), ("W", i32), ("Cin", i32), ("Cout", i32),
                ("mid", C.c_void_p), ("out", C.c_void_p), ("out16", C.c_void_p), ("lat_half", i32), ("reserved0", i32)]


class Conv2dParams(C.Structure):
    _fields_ = [("x", C.c_void_p), ("x_n_stride", i64), ("x_y_stride", i64), ("x_x_stride", i64),
                ("N", i32), ("H", i32), ("W", i32), ("Cin", i32), ("Cout", i32),
                ("s2d", i32), ("in_half", i32), ("out_half", i32), ("relu", i32), ("C1x1_out", i32),
                ("wfrag", C.c_void_p), ("bias", C.c_void_p),
                ("out", C.c_void_p), ("o_n_stride", i64), ("o_y_stride", i64), ("o_x_stride", i64),
                ("wfrag1x1", C.c_void_p), ("bias1x1", C.c_void_p)]


class FpnStemParams(C.Structure):
    _fields_ = [("x", C.c_void_p), ("x_n_stride", i64), ("x_c_stride", i64), ("x_y_stride", i64), ("x_x_stride", i64),
                ("w0", C.c_void_p), ("b0", C.c_void_p), ("wfrag1", C.c_void_p), ("b1", C.c_void_p),
                ("N", i32), ("H", i32), ("W", i32), ("out", C.c_void_p), ("rgb4", C.c_void_p),
                ("out_s2d", C.c_void_p), ("out_half", i32), ("reserved0", i32)]


class FramePsnrParams(C.Structure):
    _fields_ = [("pred", C.c_void_p), ("gt", C.c_void_p), ("mask", C.c_void_p),
                ("H", i32), ("W", i32), ("crop_h", i32), ("crop_w", i32), ("sse", C.c_void_p), ("count", C.c_void_p)]


class FrameToU8Params(C.Structure):
    _fields_ = [("R", i64), ("rgb", C.c_void_p), ("rgb_u8", C.c_void_p), ("depth", C.c_void_p), ("depth_u8", C.c_void_p),
                ("minmax_ord", C.c_void_p), ("minmax", C.c_void_p)]


class FrameSsimParams(C.Structure):
    _fields_ = [("pred", C.c_void_p), ("gt", C.c_void_p), ("H", i32), ("W", i32), ("crop_h", i32), ("crop_w", i32),
                ("win_size", i32), ("reserved0", i32), ("data_range", C.c_double),
                ("scratch", C.c_void_p), ("ssim", C.c_void_p)]


ENTRY_POINTS = {
    "bmv_cost_volume_var": CostVolumeParams,
    "bmv_cost_volume_var_multi": CostVolumeMultiParams,
    "bmv_volume_scale": VolumeScaleParams,
    "bmv_depth_planes_first": DepthPlanesFirstParams,
    "bmv_depth_planes_next": DepthPlanesNextParams,
    "bmv_depth_regression": DepthRegressionParams,
    "bmv_raygen_sample_fetch": RaygenFetchParams,
    "bmv_mask_viewport": VisibilityParams,
    "bmv_composite_blend": CompositeBlendParams,
    "bmv_composite": CompositeParams,
    "bmv_nerf_mlp": NerfMlpParams,
    "bmv_render_rays": RenderRaysParams,
    "bmv_render_rays_mma": RenderRaysParams,
    "bmv_render_rays_multi": RenderMultiParams,
    "bmv_render_rays_multi_umma": RenderMultiParams,
    "bmv_cost_volume_var_img": CostVolumeImgParams,
    "bmv_mvs_march_fetch": MvsMarchParams,
    "bmv_mvs_render_umma": MvsRenderParams,
    "bmv_fpn_topdown": FpnTopdownParams,
    "bmv_conv3d_k3": Conv3dParams,
    "bmv_conv3d_k3_umma": Conv3dParams,
    "bmv_convT3d_k3s2": ConvT3dParams,
    "bmv_fpn_topdown_smooth": FpnFusedParams,
    "bmv_fpn_stem": FpnStemParams,
    "bmv_conv2d_k3": Conv2dParams,
    "bmv_frame_psnr_accumulate": FramePsnrParams,
    "bmv_frame_to_u8": FrameToU8Params,
    "bmv_frame_ssim": FrameSsimParams,
}
PLAIN_SYMBOLS = ("bmv_version", "bmv_last_error_string", "bmv_launch_count", "bmv_sizeof_params",
                 "bmv_nerf_mlp_weight_count", "bmv_render_rays_supported", "bmv_render_rays_mma_weight_words",
                 "bmv_render_rays_umma_weight_words", "bmv_umma_selftest",
                 "bmv_conv3d_k3_weight_words", "bmv_conv3d_k3_umma_weight_words", "bmv_conv3d_k3_last_used_tma", "bmv_convT3d_k3s2_weight_words",
                 "bmv_fpn_topdown_smooth_weight_words", "bmv_mvs_render_umma_weight_bytes", "bmv_conv2d_k3_weight_words")

_lib = None


class BmvError(RuntimeError):
    pass


def load():
    """dlopen libbmv.so (raises if it has not been built: `python -m boostmvsnerfs_b200.build`)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BmvError(f"{LIB_PATH} not found — build it with `python -m boostmvsnerfs_b200.build`; "
                       "there is no CPU fallback for the rendering kernels")
    lib = C.CDLL(LIB_PATH)
    lib.bmv_version.restype = C.c_int
    lib.bmv_last_error_string.restype = C.c_char_p
    lib.bmv_launch_count.restype = C.c_uint64
    lib.bmv_nerf_mlp_weight_count.restype = C.c_int
    lib.bmv_nerf_mlp_weight_count.argtypes = [C.c_int]
    lib.bmv_render_rays_mma_weight_words.restype = C.c_int
    lib.bmv_render_rays_umma_weight_words.restype = C.c_int
    lib.bmv_umma_selftest.restype = C.c_int
    lib.bmv_umma_selftest.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    lib.bmv_render_rays_supported.restype = C.c_int
    lib.bmv_render_rays_supported.argtypes = [C.c_int, C.c_int, C.c_int]
    lib.bmv_conv3d_k3_weight_words.restype = C.c_int
    lib.bmv_conv3d_k3_weight_words.argtypes = [C.c_int, C.c_int]
    lib.bmv_conv3d_k3_last_used_tma.restype = C.c_int
    lib.bmv_conv3d_k3_umma_weight_words.restype = C.c_int
    lib.bmv_conv3d_k3_umma_weight_words.argtypes = [C.c_int, C.c_int]
    lib.bmv_convT3d_k3s2_weight_words.restype = C.c_int
    lib.bmv_convT3d_k3s2_weight_words.argtypes = [C.c_int, C.c_int]
    lib.bmv_fpn_topdown_smooth_weight_words.restype = C.c_int
    lib.bmv_conv2d_k3_weight_words.restype = C.c_int
    lib.bmv_conv2d_k3_weight_words.argtypes = [C.c_int, C.c_int]
    lib.bmv_fpn_topdown_smooth_weight_words.argtypes = [C.c_int]
    lib.bmv_mvs_render_umma_weight_bytes.restype = C.c_int
    lib.bmv_sizeof_params.restype = C.c_int
    lib.bmv_sizeof_params.argtypes = [C.c_char_p]
    for name, struct in ENTRY_POINTS.items():
        fn = getattr(lib, name)
        fn.argtypes = [C.POINTER(struct), C.c_void_p]
        fn.restype = C.c_int
        native = lib.bmv_sizeof_params(name.encode())
        if native != C.sizeof(struct):
            raise BmvError(f"ABI mismatch for {name}: library struct is {native} B, binding is {C.sizeof(struct)} B")
    _lib = lib
    return lib


# Optional per-launch profiler: an object with before(name) / after(name) called right around the
# enqueue (bench.py records CUDA events there, so a kernel's time excludes host-side gaps).
kernel_timer = None


def call(name, params, stream):
    lib = load()
    if kernel_timer is not None:
        kernel_timer.before(name)
    rc = getattr(lib, name)(C.byref(params), C.c_void_p(stream))
    if kernel_timer is not None:
        kernel_timer.after(name)
    if rc != 0:
        raise BmvError(f"{name} failed with status {rc}: {lib.bmv_last_error_string().decode()}")


def launch_count():
    return int(load().bmv_launch_count())
