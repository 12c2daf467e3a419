// libbmv: version / error plumbing of the C ABI (include/bmv.h).
#include <stdarg.h>
#include <string.h>

#include "bmv_internal.cuh"

namespace bmv {
static thread_local char g_err[512] = "";
std::atomic<uint64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
}  // namespace bmv

extern "C" BMV_API int bmv_version(void) { return BMV_VERSION; }
extern "C" BMV_API const char* bmv_last_error_string(void) { return bmv::g_err; }
extern "C" BMV_API uint64_t bmv_launch_count(void) { return bmv::g_launches.load(); }

// sizeof() of every params struct, so a foreign-language binding can verify its layout at load time.
extern "C" BMV_API int bmv_sizeof_params(const char* entry) {
  if (!entry) return -1;
  if (!strcmp(entry, "bmv_cost_volume_var")) return (int)sizeof(bmv_cost_volume_params);
  if (!strcmp(entry, "bmv_cost_volume_var_multi")) return (int)sizeof(bmv_cost_volume_multi_params);
  if (!strcmp(entry, "bmv_volume_scale")) return (int)sizeof(bmv_volume_scale_params);
  if (!strcmp(entry, "bmv_depth_planes_first")) return (int)sizeof(bmv_depth_planes_first_params);
  if (!strcmp(entry, "bmv_depth_planes_next")) return (int)sizeof(bmv_depth_planes_next_params);
  if (!strcmp(entry, "bmv_depth_regression")) return (int)sizeof(bmv_depth_regression_params);
  if (!strcmp(entry, "bmv_raygen_sample_fetch")) return (int)sizeof(bmv_raygen_fetch_params);
  if (!strcmp(entry, "bmv_mask_viewport")) return (int)sizeof(bmv_visibility_params);
  if (!strcmp(entry, "bmv_composite_blend")) return (int)sizeof(bmv_composite_blend_params);
  if (!strcmp(entry, "bmv_composite")) return (int)sizeof(bmv_composite_params);
  if (!strcmp(entry, "bmv_nerf_mlp")) return (int)sizeof(bmv_nerf_mlp_params);
  if (!strcmp(entry, "bmv_render_rays")) return (int)sizeof(bmv_render_rays_params);
  if (!strcmp(entry, "bmv_render_rays_mma")) return (int)sizeof(bmv_render_rays_params);
  if (!strcmp(entry, "bmv_render_rays_umma")) return (int)sizeof(bmv_render_rays_params);
  if (!strcmp(entry, "bmv_cost_volume_var_img")) return (int)sizeof(bmv_cost_volume_img_params);
  if (!strcmp(entry, "bmv_mvs_march_fetch")) return (int)sizeof(bmv_mvs_march_params);
  if (!strcmp(entry, "bmv_fpn_topdown")) return (int)sizeof(bmv_fpn_topdown_params);
  if (!strcmp(entry, "bmv_conv3d_k3")) return (int)sizeof(bmv_conv3d_params);
  if (!strcmp(entry, "bmv_conv3d_k3_umma")) return (int)sizeof(bmv_conv3d_params);
  if (!strcmp(entry, "bmv_convT3d_k3s2")) return (int)sizeof(bmv_convT3d_params);
  if (!strcmp(entry, "bmv_fpn_topdown_smooth")) return (int)sizeof(bmv_fpn_fused_params);
  if (!strcmp(entry, "bmv_fpn_stem")) return (int)sizeof(bmv_fpn_stem_params);
  if (!strcmp(entry, "bmv_conv2d_k3")) return (int)sizeof(bmv_conv2d_params);
  if (!strcmp(entry, "bmv_conv3d_small")) return (int)sizeof(bmv_conv3d_small_params);
  if (!strcmp(entry, "bmv_mvs_render_umma")) return (int)sizeof(bmv_mvs_render_params);
  if (!strcmp(entry, "bmv_render_rays_multi")) return (int)sizeof(bmv_render_multi_params);
  if (!strcmp(entry, "bmv_render_rays_multi_umma")) return (int)sizeof(bmv_render_multi_params);
  if (!strcmp(entry, "bmv_frame_psnr_accumulate")) return (int)sizeof(bmv_frame_psnr_params);
  if (!strcmp(entry, "bmv_frame_to_u8")) return (int)sizeof(bmv_frame_to_u8_params);
  if (!strcmp(entry, "bmv_frame_ssim")) return (int)sizeof(bmv_frame_ssim_params);
  return -1;
}
