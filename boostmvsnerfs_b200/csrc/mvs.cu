// MVSNeRF flavours of the hot path (SURVEY.md §8 rows a17, a18):
//   K1b bmv_cost_volume_var_img — 41-channel plane-sweep volume: [ref rgb | warped src rgb | feature variance]
//       reference lib/networks/mvsnerf/network.py:887-942 (build_volume_costvar_img),
//       lib/networks/mvsnerf/utils.py:580-630 (homo_warp, pad=24, NO clamp on z)
//   K3b bmv_mvs_march_fetch — uniform ray marching, NDC in the padded reference frustum, trilinear
//       volume fetch, per-view colour + in-mask, positional encoding, view direction -> the 86-wide
//       MLP input, plus z and the 3-D visibility score
//       reference lib/networks/mvsnerf/network.py:945-1001, lib/networks/mvsnerf/utils.py:112-146,300-383,
//       lib/networks/mvsnerf/renderer.py:111-137, lib/networks/boost_mvsnerf/network.py:97-135
#include "raygen_common.cuh"

namespace bmv {

struct MvsTap { int off[4]; float w[4]; bool inside; };

// homo_warp of the MVSNeRF flavour: pixel coords are (x-pad, y-pad), z is NOT clamped, the in-mask
// is the strict -1 < g < 1 test on the normalised grid.
__device__ __forceinline__ MvsTap mvs_taps(const float* __restrict__ P, float x, float y, float dep, int h, int w,
                                           int64_t ys, int64_t xs) {
  const float cx = add_rn(dot3_gemm(P[0], P[1], P[2], x, y, 1.f), div_rn(P[3], dep));
  const float cy = add_rn(dot3_gemm(P[4], P[5], P[6], x, y, 1.f), div_rn(P[7], dep));
  const float cz = add_rn(dot3_gemm(P[8], P[9], P[10], x, y, 1.f), div_rn(P[11], dep));
  const float gx = sub_rn(div_rn(div_rn(cx, cz), (float)(w - 1) / 2.f), 1.f);
  const float gy = sub_rn(div_rn(div_rn(cy, cz), (float)(h - 1) / 2.f), 1.f);
  MvsTap t;
  t.inside = (gx > -1.f) && (gx < 1.f) && (gy > -1.f) && (gy < 1.f);
  const float ix = unnormalize_ac(gx, w), iy = unnormalize_ac(gy, h);
  if (!(coord_ok(ix) && coord_ok(iy))) {
#pragma unroll
    for (int i = 0; i < 4; ++i) { t.off[i] = 0; t.w[i] = 0.f; }
    return t;
  }
  const float x0 = floorf(ix), y0 = floorf(iy), x1 = x0 + 1.f, y1 = y0 + 1.f;
  const float wx1 = ix - x0, wx0 = x1 - ix, wy1 = iy - y0, wy0 = y1 - iy;
  const bool vx0 = x0 >= 0.f && x0 <= (float)(w - 1), vx1 = x1 >= 0.f && x1 <= (float)(w - 1);
  const bool vy0 = y0 >= 0.f && y0 <= (float)(h - 1), vy1 = y1 >= 0.f && y1 <= (float)(h - 1);
  const int ix0 = min(max((int)x0, 0), w - 1), ix1 = min(max((int)x1, 0), w - 1);
  const int iy0 = min(max((int)y0, 0), h - 1), iy1 = min(max((int)y1, 0), h - 1);
  t.off[0] = (int)(iy0 * ys + ix0 * xs); t.w[0] = (vx0 && vy0) ? wx0 * wy0 : 0.f;
  t.off[1] = (int)(iy0 * ys + ix1 * xs); t.w[1] = (vx1 && vy0) ? wx1 * wy0 : 0.f;
  t.off[2] = (int)(iy1 * ys + ix0 * xs); t.w[2] = (vx0 && vy1) ? wx0 * wy1 : 0.f;
  t.off[3] = (int)(iy1 * ys + ix1 * xs); t.w[3] = (vx1 && vy1) ? wx1 * wy1 : 0.f;
  return t;
}

template <typename OutT>
__device__ __forceinline__ void put(OutT* p, float v);
template <>
__device__ __forceinline__ void put<float>(float* p, float v) { *p = v; }
template <>
__device__ __forceinline__ void put<__nv_bfloat16>(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }

// One thread per voxel of the padded volume (flat over D*hp*wp, x fastest).
template <int V, typename OutT>
__global__ void __launch_bounds__(256) cost_volume_var_img_kernel(bmv_cost_volume_img_params p) {
  __shared__ float sP[V * 12];
  if (threadIdx.x < V * 12) sP[threadIdx.x] = p.proj[threadIdx.x];
  __syncthreads();
  const int hp = p.h + 2 * p.pad, wp = p.w + 2 * p.pad;
  const int64_t nvox = (int64_t)p.D * hp * wp;
  const int64_t vox = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (vox >= nvox) return;
  const int xp = (int)(vox % wp), yp = (int)((vox / wp) % hp), d = (int)(vox / ((int64_t)wp * hp));
  const int x = xp - p.pad, y = yp - p.pad;
  const float dep = __ldg(p.planes + d);
  const bool in_ref = x >= 0 && x < p.w && y >= 0 && y < p.h;
  MvsTap tap[V];
  float cnt = 1.f;
#pragma unroll
  for (int i = 1; i < V; ++i) {
    tap[i] = mvs_taps(sP + i * 12, (float)x, (float)y, dep, p.h, p.w, p.feat_y_stride, p.feat_x_stride);
    cnt = add_rn(cnt, tap[i].inside ? 1.f : 0.f);
  }
  const float inv_cnt = div_rn(1.f, cnt);
  OutT* out = reinterpret_cast<OutT*>(p.out) + (int64_t)d * p.out_d_stride + (int64_t)yp * p.out_y_stride +
              (int64_t)xp * p.out_x_stride;
  // ---- colour channels: reference image (zero in the border), then each source image warped
  const int64_t plane = (int64_t)p.h * p.w;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float v = in_ref ? __ldg(p.img + ((int64_t)p.view[0] * 3 + c) * plane + (int64_t)y * p.w + x) : 0.f;
    put<OutT>(out + (int64_t)c * p.out_c_stride, v);
  }
#pragma unroll
  for (int i = 1; i < V; ++i) {
    // the image taps use the planar (h,w) layout of the resized images
    MvsTap ti = mvs_taps(sP + i * 12, (float)x, (float)y, dep, p.h, p.w, p.w, 1);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float* f = p.img + ((int64_t)p.view[i] * 3 + c) * plane;
      float v = ti.w[0] * __ldg(f + ti.off[0]);
      v = fmaf(ti.w[1], __ldg(f + ti.off[1]), v);
      v = fmaf(ti.w[2], __ldg(f + ti.off[2]), v);
      v = fmaf(ti.w[3], __ldg(f + ti.off[3]), v);
      put<OutT>(out + (int64_t)(3 * i + c) * p.out_c_stride, v);
    }
  }
  // ---- feature variance over the views that see the voxel
  const int64_t ref_off = in_ref ? (int64_t)y * p.feat_y_stride + (int64_t)x * p.feat_x_stride : 0;
  const float* fref = p.feat + (int64_t)p.view[0] * p.feat_view_stride;
#pragma unroll 2
  for (int c = 0; c < p.C; ++c) {
    const float r = in_ref ? __ldg(fref + (int64_t)c * p.feat_c_stride + ref_off) : 0.f;
    float sum = r, sq = mul_rn(r, r);
#pragma unroll
    for (int i = 1; i < V; ++i) {
      const float* f = p.feat + (int64_t)p.view[i] * p.feat_view_stride + (int64_t)c * p.feat_c_stride;
      float v = tap[i].w[0] * __ldg(f + tap[i].off[0]);
      v = fmaf(tap[i].w[1], __ldg(f + tap[i].off[1]), v);
      v = fmaf(tap[i].w[2], __ldg(f + tap[i].off[2]), v);
      v = fmaf(tap[i].w[3], __ldg(f + tap[i].off[3]), v);
      sum = add_rn(sum, v);
      sq = add_rn(sq, mul_rn(v, v));
    }
    const float m = mul_rn(sum, inv_cnt);
    put<OutT>(out + (int64_t)(3 * V + c) * p.out_c_stride, sub_rn(mul_rn(sq, inv_cnt), mul_rn(m, m)));
  }
}

// Channels-last variant (C = 32 dense (N,h,w,32) feature maps, channels-last output): a warp = 4 consecutive voxels x 8
// lanes of 4 channels.  The tap set of a (voxel, source view) — nine IEEE divisions in mvs_taps — is computed by ONE of
// the voxel's lanes and handed to the others with warp shuffles; a feature tap is one 16-byte load per lane (a whole
// 128-byte texel per voxel and tap); the nine colour channels are spread over the voxel's lanes.  Same arithmetic, op for
// op, as the thread-per-voxel kernel above (bit-identical output; tests/test_gpu_mvs.py).
// The thread-per-voxel kernel did 32 scalar loads per tap: 2.2 ms per chain at C3 (D = 128, 184 x 288 padded grid).
template <typename OutT>
__global__ void __launch_bounds__(256) cost_volume_var_img_cl_kernel(bmv_cost_volume_img_params p) {
  constexpr int V = 3, C = 32;
  __shared__ float sP[V * 12];
  if (threadIdx.x < V * 12) sP[threadIdx.x] = p.proj[threadIdx.x];
  __syncthreads();
  const int hp = p.h + 2 * p.pad, wp = p.w + 2 * p.pad;
  const int lane = threadIdx.x & 31, cg = lane & 7;
  const int xp_raw = blockIdx.x * 32 + (threadIdx.x >> 3);
  const bool live = xp_raw < wp;
  const int xp = live ? xp_raw : wp - 1, yp = blockIdx.y, d = blockIdx.z;
  const int x = xp - p.pad, y = yp - p.pad;
  const float dep = __ldg(p.planes + d);
  const bool in_ref = x >= 0 && x < p.w && y >= 0 && y < p.h;
  // lane cg = i (1, 2) of a voxel computes the taps of source view i; everybody receives both sets
  MvsTap mine;
  {
    const int i = (cg == 2) ? 2 : 1;
    mine = mvs_taps(sP + i * 12, (float)x, (float)y, dep, p.h, p.w, (int64_t)p.w * C, C);
  }
  MvsTap tap[V];
  float cnt = 1.f;
#pragma unroll
  for (int i = 1; i < V; ++i) {
    const int src = (lane & ~7) + i;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      tap[i].off[j] = __shfl_sync(0xffffffffu, mine.off[j], src);
      tap[i].w[j] = __shfl_sync(0xffffffffu, mine.w[j], src);
    }
    tap[i].inside = __shfl_sync(0xffffffffu, mine.inside ? 1 : 0, src) != 0;
    cnt = add_rn(cnt, tap[i].inside ? 1.f : 0.f);
  }
  const float inv_cnt = div_rn(1.f, cnt);
  OutT* out = reinterpret_cast<OutT*>(p.out) + (int64_t)d * p.out_d_stride + (int64_t)yp * p.out_y_stride + (int64_t)xp * p.out_x_stride;
  // ---- colour channels 0..8 (reference rgb, then each source image warped): lane cg takes channel cg, lane 0 also 8
  const int64_t plane = (int64_t)p.h * p.w;
#pragma unroll
  for (int rep = 0; rep < 2; ++rep) {
    const int ch = rep == 0 ? cg : 8;
    if (rep == 1 && cg != 0) break;
    float v;
    if (ch < 3) {
      v = in_ref ? __ldg(p.img + ((int64_t)p.view[0] * 3 + ch) * plane + (int64_t)y * p.w + x) : 0.f;
    } else {
      const int i = 1 + (ch - 3) / 3, c = (ch - 3) % 3;
      const MvsTap& ti = tap[i == 1 ? 1 : 2];
      const float* f = p.img + ((int64_t)p.view[i] * 3 + c) * plane;     // planar (h,w): offset = feature offset / C
      v = ti.w[0] * __ldg(f + (ti.off[0] >> 5));
      v = fmaf(ti.w[1], __ldg(f + (ti.off[1] >> 5)), v);
      v = fmaf(ti.w[2], __ldg(f + (ti.off[2] >> 5)), v);
      v = fmaf(ti.w[3], __ldg(f + (ti.off[3] >> 5)), v);
    }
    if (live) put<OutT>(out + ch, v);
  }
  // ---- feature variance over the views that see the voxel: this lane's 4 channels
  const float* fref = p.feat + (int64_t)p.view[0] * p.feat_view_stride + cg * 4;
  const float4 r4 = in_ref ? ldg4(fref + ((int64_t)y * p.w + x) * C) : make_float4(0.f, 0.f, 0.f, 0.f);
  const float r[4] = {r4.x, r4.y, r4.z, r4.w};
  float sum[4], sq[4];
#pragma unroll
  for (int c = 0; c < 4; ++c) { sum[c] = r[c]; sq[c] = mul_rn(r[c], r[c]); }
#pragma unroll
  for (int i = 1; i < V; ++i) {
    const float* f = p.feat + (int64_t)p.view[i] * p.feat_view_stride + cg * 4;
    const float4 a = ldg4(f + tap[i].off[0]), b = ldg4(f + tap[i].off[1]), cc = ldg4(f + tap[i].off[2]), dd = ldg4(f + tap[i].off[3]);
    const float t0[4] = {a.x, a.y, a.z, a.w}, t1[4] = {b.x, b.y, b.z, b.w}, t2[4] = {cc.x, cc.y, cc.z, cc.w}, t3[4] = {dd.x, dd.y, dd.z, dd.w};
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      float v = tap[i].w[0] * t0[c];
      v = fmaf(tap[i].w[1], t1[c], v);
      v = fmaf(tap[i].w[2], t2[c], v);
      v = fmaf(tap[i].w[3], t3[c], v);
      sum[c] = add_rn(sum[c], v);
      sq[c] = add_rn(sq[c], mul_rn(v, v));
    }
  }
  if (live) {
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const float m = mul_rn(sum[c], inv_cnt);
      put<OutT>(out + 3 * V + cg * 4 + c, sub_rn(mul_rn(sq[c], inv_cnt), mul_rn(m, m)));
    }
  }
}

// ---------------------------------------------------------------- K3b
// One thread per sample.  Output row (86 floats): [ndc(3), sin(2^k ndc) k=0..9 (30), cos (30),
// vox(8), (rgb,in)x3 (12), dir(3)].
template <int V>
__global__ void __launch_bounds__(128) mvs_march_fetch_kernel(bmv_mvs_march_params p) {
  __shared__ ViewCam cams[V];
  if (threadIdx.x < 32) {
    for (int v = 0; v < V; ++v) load_cam(&cams[v], p.src_exts, p.src_ixts, nullptr, p.view[v], threadIdx.x);
  }
  __syncthreads();
  // the 86-float rows of a warp's 32 consecutive samples are contiguous in the output: stage them in
  // shared memory (stride 87: conflict-free) and write them back with coalesced 8-byte stores
  __shared__ float s_rows[128][87];
  const int64_t total = p.n_rays * p.S;
  const int64_t i_raw = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = i_raw < total;
  const int64_t i = live ? i_raw : total - 1;
  const int64_t li = i / p.S;
  const int s = (int)(i % p.S);
  const int64_t r = p.ray_begin + li;
  const float4 ra = __ldg(reinterpret_cast<const float4*>(p.rays + r * 8));
  const float4 rb = __ldg(reinterpret_cast<const float4*>(p.rays + r * 8 + 4));
  const float near = rb.z, far = rb.w;                   // ray columns 6,7 (SURVEY.md §10.1)
  const float t = __ldg(p.t + s);
  const float z = add_rn(mul_rn(near, sub_rn(1.f, t)), mul_rn(far, t));
  const float x = add_rn(ra.x, mul_rn(ra.w, z)), y = add_rn(ra.y, mul_rn(rb.x, z)), zz = add_rn(ra.z, mul_rn(rb.y, z));
  if (p.z_vals && live) p.z_vals[li * p.S + s] = z;
  const float isx = (float)(p.W - 1), isy = (float)(p.H - 1);
  // ---- visibility over the triple (same arithmetic as the ENeRF path)
  int cnt = 0;
#pragma unroll
  for (int v = 0; v < V; ++v) cnt += point_visible(cams[v], x, y, zz, isx, isy) ? 1 : 0;
  if (p.vis_mask && live) p.vis_mask[li * p.S + s] = div_rn((float)cnt, (float)V);
  if (p.vis_count && live) p.vis_count[li * p.S + s] = cnt;
  if (!p.mlp_in) return;
  float* o = s_rows[threadIdx.x];
  // ---- NDC in the padded frustum of reference view 0: matmul(R^T)+T, @K^T, /z, /inv_scale, pad rescale
  const ViewCam& c0 = cams[0];
  float ndc[3];
  {
    const float cx = add_rn(dot3_gemm(x, y, zz, c0.E[0], c0.E[1], c0.E[2]), c0.E[3]);
    const float cy = add_rn(dot3_gemm(x, y, zz, c0.E[4], c0.E[5], c0.E[6]), c0.E[7]);
    const float cz = add_rn(dot3_gemm(x, y, zz, c0.E[8], c0.E[9], c0.E[10]), c0.E[11]);
    const float qx = dot3_gemm(cx, cy, cz, c0.K[0], c0.K[1], c0.K[2]);
    const float qy = dot3_gemm(cx, cy, cz, c0.K[3], c0.K[4], c0.K[5]);
    const float qz = dot3_gemm(cx, cy, cz, c0.K[6], c0.K[7], c0.K[8]);
    float u = div_rn(add_rn(div_rn(qx, qz), 0.f), isx), w = div_rn(add_rn(div_rn(qy, qz), 0.f), isy);
    const float dz = div_rn(sub_rn(qz, p.near), sub_rn(p.far, p.near));
    const float Wf = div_rn(add_rn(isx, 1.f), 4.f), Hf = div_rn(add_rn(isy, 1.f), 4.f);
    const float pad2 = (float)(p.pad * 2), padf = (float)p.pad;
    w = add_rn(div_rn(mul_rn(w, Hf), add_rn(Hf, pad2)), div_rn(padf, add_rn(Hf, pad2)));
    u = add_rn(div_rn(mul_rn(u, Wf), add_rn(Wf, pad2)), div_rn(padf, add_rn(Wf, pad2)));
    ndc[0] = u; ndc[1] = w; ndc[2] = dz;
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) o[k] = ndc[k];
  {
    float f = 1.f;
#pragma unroll
    for (int k = 0; k < 10; ++k) {
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        const float arg = mul_rn(ndc[a], f);
        float sn, cs;
        sincosf(arg, &sn, &cs);                 // same accuracy as sinf/cosf, one range reduction
        o[3 + k * 3 + a] = sn;
        o[33 + k * 3 + a] = cs;
      }
      f *= 2.f;
    }
  }
  // ---- trilinear volume fetch at ndc (zeros padding)
  {
    const int wp = p.wv, hp = p.hv;
    const float gx = sub_rn(mul_rn(ndc[0], 2.f), 1.f), gy = sub_rn(mul_rn(ndc[1], 2.f), 1.f), gz = sub_rn(mul_rn(ndc[2], 2.f), 1.f);
    const float ix = unnormalize_ac(gx, wp), iy = unnormalize_ac(gy, hp), iz = unnormalize_ac(gz, p.Dv);
    float acc[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[c] = 0.f;
    if (coord_ok(ix) && coord_ok(iy) && coord_ok(iz)) {
      const float x0 = floorf(ix), y0 = floorf(iy), z0 = floorf(iz);
      const float fx1 = ix - x0, fy1 = iy - y0, fz1 = iz - z0;
      const float fx0 = (x0 + 1.f) - ix, fy0 = (y0 + 1.f) - iy, fz0 = (z0 + 1.f) - iz;
#pragma unroll
      for (int corner = 0; corner < 8; ++corner) {
        const int bx = corner & 1, by = (corner >> 1) & 1, bz = corner >> 2;
        const float cxf = x0 + bx, cyf = y0 + by, czf = z0 + bz;
        const bool ok = cxf >= 0.f && cxf <= (float)(wp - 1) && cyf >= 0.f && cyf <= (float)(hp - 1) &&
                        czf >= 0.f && czf <= (float)(p.Dv - 1);
        if (!ok) continue;
        const float wgt = (bx ? fx1 : fx0) * (by ? fy1 : fy0) * (bz ? fz1 : fz0);
        const float* src = p.volume + (int64_t)czf * p.vol_d_stride + (int64_t)cyf * p.vol_y_stride +
                           (int64_t)cxf * p.vol_x_stride;
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[c] = fmaf(wgt, __ldg(src + (int64_t)c * p.vol_c_stride), acc[c]);
      }
    }
#pragma unroll
    for (int c = 0; c < 8; ++c) o[63 + c] = acc[c];
  }
  // ---- per view: border-bilinear colour (img*scale+shift) and strict in-mask
  const int64_t plane = (int64_t)p.H * p.W;
#pragma unroll
  for (int v = 0; v < V; ++v) {
    const ViewCam& cam = cams[v];
    const float cx = add_rn(dot3_gemm(x, y, zz, cam.E[0], cam.E[1], cam.E[2]), cam.E[3]);
    const float cy = add_rn(dot3_gemm(x, y, zz, cam.E[4], cam.E[5], cam.E[6]), cam.E[7]);
    const float cz = add_rn(dot3_gemm(x, y, zz, cam.E[8], cam.E[9], cam.E[10]), cam.E[11]);
    const float qx = dot3_gemm(cx, cy, cz, cam.K[0], cam.K[1], cam.K[2]);
    const float qy = dot3_gemm(cx, cy, cz, cam.K[3], cam.K[4], cam.K[5]);
    const float qz = dot3_gemm(cx, cy, cz, cam.K[6], cam.K[7], cam.K[8]);
    const float u = div_rn(add_rn(div_rn(qx, qz), 0.f), isx), w = div_rn(add_rn(div_rn(qy, qz), 0.f), isy);
    const float gx = sub_rn(mul_rn(u, 2.f), 1.f), gy = sub_rn(mul_rn(w, 2.f), 1.f);
    const bool inside = (gx > -1.f) && (gx < 1.f) && (gy > -1.f) && (gy < 1.f);
    const Tap2 tp = border_taps(gx, gy, p.H, p.W, p.W, 1);
    const float* f = p.rgb + (int64_t)p.view[v] * 3 * plane;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float* fc = f + c * plane;
      float val = tp.w00 * fmaf(__ldg(fc + tp.o00), p.rgb_scale, p.rgb_shift);
      val = fmaf(tp.w01, fmaf(__ldg(fc + tp.o01), p.rgb_scale, p.rgb_shift), val);
      val = fmaf(tp.w10, fmaf(__ldg(fc + tp.o10), p.rgb_scale, p.rgb_shift), val);
      val = fmaf(tp.w11, fmaf(__ldg(fc + tp.o11), p.rgb_scale, p.rgb_shift), val);
      o[71 + v * 4 + c] = val;
    }
    o[71 + v * 4 + 3] = inside ? 1.f : 0.f;
  }
  // ---- view direction in the reference camera frame: (d/|d|) @ R0^T
  {
    const float n = sqrtf(ra.w * ra.w + rb.x * rb.x + rb.y * rb.y);
    const float ux = div_rn(ra.w, n), uy = div_rn(rb.x, n), uz = div_rn(rb.y, n);
    o[83] = dot3_gemm(ux, uy, uz, c0.E[0], c0.E[1], c0.E[2]);
    o[84] = dot3_gemm(ux, uy, uz, c0.E[4], c0.E[5], c0.E[6]);
    o[85] = dot3_gemm(ux, uy, uz, c0.E[8], c0.E[9], c0.E[10]);
  }
  __syncwarp();
  {
    const int lane = threadIdx.x & 31, wbase = threadIdx.x & ~31;
    const int64_t i0 = (int64_t)blockIdx.x * blockDim.x + wbase;            // first sample of this warp
    const int rows = (int)min((int64_t)32, total - i0);
    float2* dst = reinterpret_cast<float2*>(p.mlp_in + i0 * 86);             // 344 B rows: 8-byte aligned
    for (int j = lane; j < rows * 43; j += 32) {
      const int e = 2 * j, r = e / 86, c = e - r * 86;
      dst[j] = make_float2(s_rows[wbase + r][c], s_rows[wbase + r][c + 1]);
    }
  }
}

}  // namespace bmv

extern "C" BMV_API int bmv_cost_volume_var_img(const bmv_cost_volume_img_params* p, bmv_stream_t stream) {
  BMV_NVTX_RANGE("bmv_cost_volume_var_img");
  using namespace bmv;
  BMV_REQUIRE(p != nullptr, BMV_ERR_INVALID_ARGUMENT, "bmv_cost_volume_var_img: null params");
  BMV_REQUIRE(p->feat && p->img && p->proj && p->planes && p->out, BMV_ERR_INVALID_ARGUMENT,
              "bmv_cost_volume_var_img: null device pointer");
  BMV_REQUIRE(p->V == 3, BMV_ERR_UNSUPPORTED_SHAPE, "bmv_cost_volume_var_img: V=%d views not instantiated (3)", p->V);
  BMV_REQUIRE(p->C >= 1 && p->h >= 2 && p->w >= 2 && p->D >= 1 && p->pad >= 0, BMV_ERR_INVALID_ARGUMENT,
              "bmv_cost_volume_var_img: bad size");
  BMV_REQUIRE((int64_t)p->h * llabs(p->feat_y_stride) + (int64_t)p->w * llabs(p->feat_x_stride) < (1ll << 31),
              BMV_ERR_UNSUPPORTED_SHAPE, "bmv_cost_volume_var_img: feature map too large for 32-bit tap offsets");
  const int64_t nvox = (int64_t)p->D * (p->h + 2 * p->pad) * (p->w + 2 * p->pad);
  const unsigned blocks = (unsigned)ceil_div64(nvox, 256);
  cudaStream_t st = (cudaStream_t)stream;
  // dense channels-last features and a channels-last volume: warp-level tap sharing, 16-byte taps
  const int hp = p->h + 2 * p->pad, wp = p->w + 2 * p->pad;
  if (p->C == 32 && p->feat_c_stride == 1 && p->feat_x_stride == 32 && p->feat_y_stride == (int64_t)p->w * 32 &&
      p->feat_view_stride % 4 == 0 && ((uintptr_t)p->feat & 15) == 0 && p->out_c_stride == 1 && hp <= 65535 && p->D <= 65535 &&
      (int64_t)p->h * p->w * 32 < (1ll << 31)) {
    const dim3 grid((unsigned)((wp + 31) / 32), (unsigned)hp, (unsigned)p->D);
    if (p->out_bf16) cost_volume_var_img_cl_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(*p);
    else cost_volume_var_img_cl_kernel<float><<<grid, 256, 0, st>>>(*p);
    return check_launch("bmv_cost_volume_var_img");
  }
  if (p->out_bf16) cost_volume_var_img_kernel<3, __nv_bfloat16><<<blocks, 256, 0, st>>>(*p);
  else cost_volume_var_img_kernel<3, float><<<blocks, 256, 0, st>>>(*p);
  return check_launch("bmv_cost_volume_var_img");
}

extern "C" BMV_API int bmv_mvs_march_fetch(const bmv_mvs_march_params* p, bmv_stream_t stream) {
  BMV_NVTX_RANGE("bmv_mvs_march_fetch");
  using namespace bmv;
  BMV_REQUIRE(p != nullptr, BMV_ERR_INVALID_ARGUMENT, "bmv_mvs_march_fetch: null params");
  BMV_REQUIRE(p->n_rays >= 0 && p->ray_begin >= 0 && p->S >= 1, BMV_ERR_INVALID_ARGUMENT, "bmv_mvs_march_fetch: bad range");
  if (p->n_rays == 0) return BMV_OK;
  BMV_REQUIRE(p->rays && p->t && p->src_exts && p->src_ixts, BMV_ERR_INVALID_ARGUMENT, "bmv_mvs_march_fetch: null input");
  BMV_REQUIRE(p->V == 3, BMV_ERR_UNSUPPORTED_SHAPE, "bmv_mvs_march_fetch: V=%d views not instantiated (3)", p->V);
  // a ray is read as two float4, and the staged 86-float rows are stored as float2
  BMV_REQUIRE(((uintptr_t)p->rays & 15) == 0 && ((uintptr_t)p->mlp_in & 7) == 0, BMV_ERR_INVALID_ARGUMENT,
              "bmv_mvs_march_fetch: rays must be 16-byte aligned and mlp_in 8-byte aligned");
  if (p->mlp_in)
    BMV_REQUIRE(p->volume && p->rgb && p->Cv == 8 && p->Dv >= 1 && p->hv >= 1 && p->wv >= 1 && p->H >= 2 && p->W >= 2,
                BMV_ERR_INVALID_ARGUMENT, "bmv_mvs_march_fetch: volume/rgb inputs missing or Cv != 8");
  const unsigned blocks = (unsigned)ceil_div64(p->n_rays * p->S, 128);
  mvs_march_fetch_kernel<3><<<blocks, 128, 0, (cudaStream_t)stream>>>(*p);
  return check_launch("bmv_mvs_march_fetch");
}
