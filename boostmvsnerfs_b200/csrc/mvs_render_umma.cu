// K3b + the 6x128 MVSNeRF MLP ("Renderer_ours", reference lib/networks/mvsnerf/network.py:152-229) in ONE kernel on the
// 5th-generation tensor cores: the (chunk, S, 86) MLP input — > 90 % of the C3 frame's HBM traffic in the reference
// (SURVEY.md §11: 45.5 KB per ray) — and every activation stay on chip.
//
// Arithmetic class: fp16 operands, fp32 accumulation in tensor memory, ONE MMA per product (no hi/lo split): this is
// the TF32-class engine of BASELINE config 3 (bf16 cost volume, 1e-2 tolerance).  The strict path keeps the fp32
// cuBLAS module (network_mvs.py).
//
// Structure (one CTA per SM, persistent, 18 warps):
//   warps 0-7 / 8-15 own the 128 sample rows of tile 0 / tile 1, TWO threads per row (warp w and w + 4 of a tile read the
//                    same TMEM lane quarter): the gather is split between them (march + NDC by both; visibility,
//                    positional encoding and view direction by half 0; trilinear volume fetch and per-view colours by
//                    half 1), each writes its K-chunks of the layer's A operand (fp16, UMMA K-major SWIZZLE_NONE: chunk c =
//                    128 rows x 16 B) and handles 64 of the 128 accumulator columns in the epilogues (tcgen05.ld, gate *
//                    ReLU); partial alpha / rgb sums meet in shared memory.  (First version: one thread per row, 8
//                    row-owner warps: issue 20 %, tensor pipe 15 %, long scoreboard 8 per issue — latency bound.)
//   warp 16          issues every tcgen05.mma (M = 128, N = 128 / 64, K = 16) of both tiles, ping-pong: while tile 0 is
//                    in its epilogue the tensor core works on tile 1;
//   warp 17          streams the weights (256 KB per pass, more than fits) through a 4-slot ring of 18 KB panels with
//                    cp.async.bulk + mbarrier transaction counts; a panel is used by BOTH tiles before its slot is
//                    released by tcgen05.commit.
// Layers as MMAs (biases ride on constant-1 columns of the operands):
//   gate  = feats20 . Wg           K 32   (F chunks, col 20 = 1)              -> TMEM cols 128..255 of the tile, kept
//   L0    = PE63 . W0              K 64   (P chunks, col 63 = 1)              -> cols 0..127;  h = relu(acc * gate)
//   L1-4  = h . Wi + 1 . bi        K 128 + 16 (bias K-step: F cols 16..31)     ;  h = relu(acc * gate)
//   L5    = PE63 . W5p + h . W5h   K 64 + 128 (skip connection)               ;  h = relu(acc * gate), alpha = relu(wa.h + ba)
//   FL    = h . Wf + 1 . bf        K 128 + 16                                 ;  feature (no activation)
//   VL    = [feature | dir3 1] . Wv  K 128 + 16, N 64                         ;  rgb = sigmoid(Wr . relu(acc) + br)
#include <stdlib.h>

#include "raygen_common.cuh"
#include "umma.cuh"

namespace bmv {

constexpr int MR_CHUNK = 2048;                        // one K-chunk (8 fp16) of a 128-row A operand
constexpr int MR_P = 0, MR_F = 8, MR_V = 12, MR_H = 14, MR_TILE_CHUNKS = 30;
constexpr int MR_TILE_BYTES = MR_TILE_CHUNKS * MR_CHUNK;        // 61440
constexpr int MR_SLOT = 18432, MR_SLOTS = 4;
constexpr int MR_NPANEL = 16;
constexpr int MR_PANEL_BYTES_TOTAL = 8192 + 14 * 16384 + 18432;  // 256000
constexpr int MR_BIAS_BYTES = 5 * 4096;                           // bias K-steps of L1..L4, FL: (K 16, N 128) each
constexpr int MR_VEC_FLOATS = 328;                                // wa[128], Wr[3][64], ba, br[3], pad
constexpr int MR_V_WA = 0, MR_V_WR = 128, MR_V_BA = 320, MR_V_BR = 321;
constexpr int MR_PACK_BYTES = MR_PANEL_BYTES_TOTAL + MR_BIAS_BYTES + MR_VEC_FLOATS * 4;
constexpr int MR_THREADS = 576;                       // 16 row-owner warps + MMA issuer + weight producer
constexpr size_t MR_SMEM = (size_t)2 * MR_TILE_BYTES + (size_t)MR_SLOTS * MR_SLOT + MR_BIAS_BYTES + MR_VEC_FLOATS * 4 + 128;

__host__ __device__ constexpr int mr_panel_bytes(int p) { return p == 0 ? 8192 : (p == 15 ? 18432 : 16384); }
__host__ __device__ constexpr int mr_panel_offset(int p) { return p == 0 ? 0 : 8192 + (p - 1) * 16384; }

// n_ksteps K = 16 steps: D (+)= A[chunks a0, a0+1, ...] . B[chunks b0, ...]
__device__ __forceinline__ void mr_issue(uint32_t d_tmem, uint32_t a_addr, uint32_t b_addr, uint32_t b_chunk, int n_ksteps,
                                         uint32_t idesc, bool acc_first) {
  for (int ks = 0; ks < n_ksteps; ++ks) {
    const uint64_t ad = umma_desc(a_addr + ks * 2 * MR_CHUNK, MR_CHUNK, 128);
    const uint64_t bd = umma_desc(b_addr + ks * 2 * b_chunk, b_chunk, 128);
    umma_f16(d_tmem, ad, bd, idesc, (acc_first || ks) ? 1u : 0u);
  }
}

// this row's 8 values of K-chunk `chunk`
__device__ __forceinline__ void mr_put(unsigned char* tile, int chunk, int row, const float* v) {
  uint4 q;
  q.x = pack_half2_sat(v[0], v[1]); q.y = pack_half2_sat(v[2], v[3]);
  q.z = pack_half2_sat(v[4], v[5]); q.w = pack_half2_sat(v[6], v[7]);
  *reinterpret_cast<uint4*>(tile + chunk * MR_CHUNK + row * 16) = q;
}

// ---- the per-sample gather of bmv_mvs_march_fetch (same arithmetic; the positional encoding by angle doubling:
// sin / cos of 2^k x from those of x, error < 2^k ulp, far below the fp16 rounding of the operand)
// part 0: visibility + outputs, P and V operands; part 1: F operand (volume fetch, colours).  Both recompute the march
// and the NDC coordinates (cheap) instead of exchanging them.
template <int V>
__device__ __forceinline__ void mr_gather(const bmv_mvs_march_params& p, const ViewCam* cams, const int* views, int64_t i, bool live,
                                          unsigned char* tile, int row, int part) {
  const int64_t li = i / p.S;
  const int s = (int)(i - li * p.S);
  const int64_t r = p.ray_begin + li;
  const float4 ra = __ldg(reinterpret_cast<const float4*>(p.rays + r * 8));
  const float4 rb = __ldg(reinterpret_cast<const float4*>(p.rays + r * 8 + 4));
  const float near = rb.z, far = rb.w;
  const float t = __ldg(p.t + s);
  const float z = add_rn(mul_rn(near, sub_rn(1.f, t)), mul_rn(far, t));
  const float x = add_rn(ra.x, mul_rn(ra.w, z)), y = add_rn(ra.y, mul_rn(rb.x, z)), zz = add_rn(ra.z, mul_rn(rb.y, z));
  const float isx = (float)(p.W - 1), isy = (float)(p.H - 1);
  if (part == 0) {
    int cnt = 0;
#pragma unroll
    for (int v = 0; v < V; ++v) cnt += point_visible(cams[v], x, y, zz, isx, isy) ? 1 : 0;
    if (live) {
      if (p.z_vals) p.z_vals[i] = z;
      if (p.vis_mask) p.vis_mask[i] = div_rn((float)cnt, (float)V);
      if (p.vis_count) p.vis_count[i] = cnt;
    }
  }
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
  // ---- P operand: [ndc(3), sin(2^k ndc) k = 0..9 (30), cos (30), 1]
  if (part == 0) {
    float pe[64];
    pe[0] = ndc[0]; pe[1] = ndc[1]; pe[2] = ndc[2];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      float sn, cs;
      sincosf(ndc[a], &sn, &cs);
      pe[3 + a] = sn; pe[33 + a] = cs;
#pragma unroll
      for (int k = 1; k < 10; ++k) {
        const float s2 = 2.f * sn * cs, c2 = fmaf(-2.f * sn, sn, 1.f);
        sn = s2; cs = c2;
        pe[3 + k * 3 + a] = sn; pe[33 + k * 3 + a] = cs;
      }
    }
    pe[63] = 1.f;
#pragma unroll
    for (int c = 0; c < 8; ++c) mr_put(tile, MR_P + c, row, pe + 8 * c);
  }
  if (part == 0) {
    // ---- V operand: view direction in the reference camera frame, then the constant 1
    float vd[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) vd[c] = 0.f;
    const float n = sqrtf(ra.w * ra.w + rb.x * rb.x + rb.y * rb.y);
    const float ux = div_rn(ra.w, n), uy = div_rn(rb.x, n), uz = div_rn(rb.y, n);
    vd[0] = dot3_gemm(ux, uy, uz, c0.E[0], c0.E[1], c0.E[2]);
    vd[1] = dot3_gemm(ux, uy, uz, c0.E[4], c0.E[5], c0.E[6]);
    vd[2] = dot3_gemm(ux, uy, uz, c0.E[8], c0.E[9], c0.E[10]);
    vd[3] = 1.f;
    mr_put(tile, MR_V, row, vd);
    mr_put(tile, MR_V + 1, row, vd + 8);
    return;
  }
  // ---- F operand: [vox(8), (rgb, in) x 3 (12), 1, 0 ...]
  float f[32];
#pragma unroll
  for (int c = 0; c < 32; ++c) f[c] = 0.f;
  f[20] = 1.f;
  {
    const int wp = p.wv, hp = p.hv;
    const float gx = sub_rn(mul_rn(ndc[0], 2.f), 1.f), gy = sub_rn(mul_rn(ndc[1], 2.f), 1.f), gz = sub_rn(mul_rn(ndc[2], 2.f), 1.f);
    const float ix = unnormalize_ac(gx, wp), iy = unnormalize_ac(gy, hp), iz = unnormalize_ac(gz, p.Dv);
    // branch-free: validity folded into the weights, invalid corners read a clamped (valid) address with weight 0 — all 16
    // loads of a channels-last voxel set are in flight together (with `if (!ok) continue` per corner they were eight
    // dependent round trips: 30 % of this kernel's stall samples, ncu round2j)
    const bool fin = coord_ok(ix) && coord_ok(iy) && coord_ok(iz);
    const float x0 = floorf(ix), y0 = floorf(iy), z0 = floorf(iz);
    const float fx1 = ix - x0, fy1 = iy - y0, fz1 = iz - z0;
    const float fx0 = (x0 + 1.f) - ix, fy0 = (y0 + 1.f) - iy, fz0 = (z0 + 1.f) - iz;
    const float wm = (float)(wp - 1), hm = (float)(hp - 1), dm = (float)(p.Dv - 1);
    const bool vx0 = fin && x0 >= 0.f && x0 <= wm, vx1 = fin && x0 + 1.f >= 0.f && x0 + 1.f <= wm;
    const bool vy0 = fin && y0 >= 0.f && y0 <= hm, vy1 = fin && y0 + 1.f >= 0.f && y0 + 1.f <= hm;
    const bool vz0 = fin && z0 >= 0.f && z0 <= dm, vz1 = fin && z0 + 1.f >= 0.f && z0 + 1.f <= dm;
    const float wx[2] = {vx0 ? fx0 : 0.f, vx1 ? fx1 : 0.f};
    const float wy[2] = {vy0 ? fy0 : 0.f, vy1 ? fy1 : 0.f};
    const float wz[2] = {vz0 ? fz0 : 0.f, vz1 ? fz1 : 0.f};
    const int64_t xi = fin ? (int64_t)fminf(fmaxf(x0, 0.f), wm) : 0, yi = fin ? (int64_t)fminf(fmaxf(y0, 0.f), hm) : 0;
    const int64_t zi = fin ? (int64_t)fminf(fmaxf(z0, 0.f), dm) : 0;
    const int64_t ox1 = (vx0 && vx1) ? p.vol_x_stride : 0, oy1 = (vy0 && vy1) ? p.vol_y_stride : 0, oz1 = (vz0 && vz1) ? p.vol_d_stride : 0;
    const float* b000 = p.volume + zi * p.vol_d_stride + yi * p.vol_y_stride + xi * p.vol_x_stride;
    if (p.vol_c_stride == 1) {                            // channels-last volume: two 16-byte loads per corner
      float4 va[8], vb[8];
#pragma unroll
      for (int corner = 0; corner < 8; ++corner) {
        const float* src = b000 + ((corner & 1) ? ox1 : 0) + (((corner >> 1) & 1) ? oy1 : 0) + ((corner >> 2) ? oz1 : 0);
        va[corner] = ldg4(src); vb[corner] = ldg4(src + 4);
      }
#pragma unroll
      for (int corner = 0; corner < 8; ++corner) {
        const float wgt = (wx[corner & 1] * wy[(corner >> 1) & 1]) * wz[corner >> 2];
        const float4 a = va[corner], b = vb[corner];
        f[0] = fmaf(wgt, a.x, f[0]); f[1] = fmaf(wgt, a.y, f[1]); f[2] = fmaf(wgt, a.z, f[2]); f[3] = fmaf(wgt, a.w, f[3]);
        f[4] = fmaf(wgt, b.x, f[4]); f[5] = fmaf(wgt, b.y, f[5]); f[6] = fmaf(wgt, b.z, f[6]); f[7] = fmaf(wgt, b.w, f[7]);
      }
    } else {
#pragma unroll
      for (int corner = 0; corner < 8; ++corner) {
        const float wgt = (wx[corner & 1] * wy[(corner >> 1) & 1]) * wz[corner >> 2];
        const float* src = b000 + ((corner & 1) ? ox1 : 0) + (((corner >> 1) & 1) ? oy1 : 0) + ((corner >> 2) ? oz1 : 0);
#pragma unroll
        for (int c = 0; c < 8; ++c) f[c] = fmaf(wgt, __ldg(src + (int64_t)c * p.vol_c_stride), f[c]);
      }
    }
  }
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
    if (p.rgb_nhwc4) {                                     // (N,H,W,4): one 16-byte load per tap
      const Tap2 tp = border_taps(gx, gy, p.H, p.W, (int64_t)p.W * 4, 4);
      const float* fi = p.rgb + (int64_t)views[v] * 4 * plane;
      const float4 a = ldg4(fi + tp.o00), b = ldg4(fi + tp.o01), cc = ldg4(fi + tp.o10), d = ldg4(fi + tp.o11);
      const float sc = p.rgb_scale, sf = p.rgb_shift;
      f[8 + v * 4 + 0] = fmaf(tp.w11, fmaf(d.x, sc, sf), fmaf(tp.w10, fmaf(cc.x, sc, sf), fmaf(tp.w01, fmaf(b.x, sc, sf), tp.w00 * fmaf(a.x, sc, sf))));
      f[8 + v * 4 + 1] = fmaf(tp.w11, fmaf(d.y, sc, sf), fmaf(tp.w10, fmaf(cc.y, sc, sf), fmaf(tp.w01, fmaf(b.y, sc, sf), tp.w00 * fmaf(a.y, sc, sf))));
      f[8 + v * 4 + 2] = fmaf(tp.w11, fmaf(d.z, sc, sf), fmaf(tp.w10, fmaf(cc.z, sc, sf), fmaf(tp.w01, fmaf(b.z, sc, sf), tp.w00 * fmaf(a.z, sc, sf))));
      f[8 + v * 4 + 3] = inside ? 1.f : 0.f;
      continue;
    }
    const Tap2 tp = border_taps(gx, gy, p.H, p.W, p.W, 1);
    const float* fi = p.rgb + (int64_t)views[v] * 3 * plane;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float* fc = fi + c * plane;
      float val = tp.w00 * fmaf(__ldg(fc + tp.o00), p.rgb_scale, p.rgb_shift);
      val = fmaf(tp.w01, fmaf(__ldg(fc + tp.o01), p.rgb_scale, p.rgb_shift), val);
      val = fmaf(tp.w10, fmaf(__ldg(fc + tp.o10), p.rgb_scale, p.rgb_shift), val);
      val = fmaf(tp.w11, fmaf(__ldg(fc + tp.o11), p.rgb_scale, p.rgb_shift), val);
      f[8 + v * 4 + c] = val;
    }
    f[8 + v * 4 + 3] = inside ? 1.f : 0.f;
  }
#pragma unroll
  for (int c = 0; c < 4; ++c) mr_put(tile, MR_F + c, row, f + 8 * c);
}

// dbg_panel_bytes (environment BMV_MR_DEBUG_PANEL, measurement only: WRONG results) takes the kernel apart: low 20 bits > 0:
// copy only that many bytes of every weight panel; bit 20: skip the gather; bit 21: skip the MMAs (commits only); bit 22:
// skip the epilogue arithmetic
__global__ void __launch_bounds__(MR_THREADS, 1) mvs_render_umma_kernel(bmv_mvs_render_params rp, int dbg_panel_bytes) {
  constexpr int V = 3;
  const bmv_mvs_march_params& p = rp.g;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>(((uintptr_t)smem_raw + 127) & ~(uintptr_t)127);
  unsigned char* sA = smem;                                           // 2 operand tiles
  unsigned char* sRing = smem + 2 * MR_TILE_BYTES;                    // weight panel ring
  unsigned char* sBias = sRing + MR_SLOTS * MR_SLOT;                  // resident bias K-steps
  const float* sVec = reinterpret_cast<const float*>(sBias + MR_BIAS_BYTES);
  __shared__ ViewCam cams[V];
  __shared__ int s_view[V];
  __shared__ __align__(8) uint64_t s_full[MR_SLOTS], s_empty[MR_SLOTS], s_acc[2], s_aready[2];
  __shared__ uint32_t s_tmem;
  __shared__ float s_alpha[2][2][128];                 // [tile][half][row]: partial alpha dots over 64 columns each
  __shared__ __align__(16) float s_rgb[2][128][4];                   // [tile][row]: half 1's partial rgb sums

  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const unsigned char* gw = reinterpret_cast<const unsigned char*>(rp.weights);
  // resident part: bias K-steps + fp32 vectors
  for (int i = tid * 16; i < MR_BIAS_BYTES + MR_VEC_FLOATS * 4; i += MR_THREADS * 16)
    *reinterpret_cast<uint4*>(sBias + i) = __ldg(reinterpret_cast<const uint4*>(gw + MR_PANEL_BYTES_TOTAL + i));
  if (tid < V) s_view[tid] = p.view[tid];
  if (tid == 0) {
    for (int s = 0; s < MR_SLOTS; ++s) { mbar_init(smem_u32(&s_full[s]), 1); mbar_init(smem_u32(&s_empty[s]), 1); }
    for (int w = 0; w < 2; ++w) { mbar_init(smem_u32(&s_acc[w]), 1); mbar_init(smem_u32(&s_aready[w]), 256); }
  }
  __syncwarp();
  if (warp == 16) tmem_alloc_512(smem_u32(&s_tmem));
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (tid < 32) for (int v = 0; v < V; ++v) load_cam(&cams[v], p.src_exts, p.src_ixts, nullptr, s_view[v], tid);
  __syncthreads();

  const uint32_t tmem_base = s_tmem;
  const int64_t n_samples = p.n_rays * p.S;
  const int64_t n_tiles = (n_samples + 127) / 128;
  const int64_t n_pairs = (n_tiles + 1) / 2;
  const uint32_t idesc128 = umma_idesc(128), idesc64 = umma_idesc(64);

  if (warp < 16) {
    // =============================================================== row owners: gather + epilogues
    const int tile_id = warp >> 3, half = (warp >> 2) & 1, row = (warp & 3) * 32 + (tid & 31);
    unsigned char* tile = sA + tile_id * MR_TILE_BYTES;
    const uint32_t acc_col = tmem_base + (uint32_t)(tile_id * 256) + ((uint32_t)((warp & 3) * 32) << 16);
    const uint32_t gate_col = acc_col + 128;
    const uint32_t mb_acc = smem_u32(&s_acc[tile_id]), mb_ready = smem_u32(&s_aready[tile_id]);
    uint32_t par_acc = 0;
    for (int64_t pair = blockIdx.x; pair < n_pairs; pair += gridDim.x) {
      const int64_t si_raw = (pair * 2 + tile_id) * 128 + row;
      const bool live = si_raw < n_samples;
      const int64_t si = live ? si_raw : n_samples - 1;
      if (!(dbg_panel_bytes & (1 << 20))) mr_gather<V>(p, cams, s_view, si, live, tile, row, half);
      proxy_fence_async();
      mbar_arrive(mb_ready);
#pragma unroll 1
      for (int phase = 0; phase < 8; ++phase) {
        mbar_wait(mb_acc, par_acc); par_acc ^= 1u;
        __syncwarp();
        tc_fence_after();
        if (phase < 7) {
          float dot = 0.f;
#pragma unroll 1
          for (int c4 = 2 * half; c4 < 2 * half + 2 && !(dbg_panel_bytes & (4 << 20)); ++c4) {      // this thread's 64 of the 128 columns
            float a[32];
            tmem_ld32(acc_col + 32 * c4, a);
            if (phase < 6) {
              float g[32];
              tmem_ld32(gate_col + 32 * c4, g);
#pragma unroll
              for (int j = 0; j < 32; ++j) a[j] = fmaxf(a[j] * g[j], 0.f);
              if (phase == 5) {
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                  const float4 w = *reinterpret_cast<const float4*>(sVec + MR_V_WA + 32 * c4 + j);
                  dot = fmaf(w.x, a[j], dot); dot = fmaf(w.y, a[j + 1], dot); dot = fmaf(w.z, a[j + 2], dot); dot = fmaf(w.w, a[j + 3], dot);
                }
              }
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) mr_put(tile, MR_H + 4 * c4 + q, row, a + 8 * q);
          }
          if (phase == 5) s_alpha[tile_id][half][row] = dot;
          proxy_fence_async();
          tc_fence_before();
          mbar_arrive(mb_ready);
        } else {
          // 64 output columns: 32 per thread, partial rgb sums meet in shared memory
          float r0 = 0.f, r1 = 0.f, r2 = 0.f;
          {
            float a[32];
            tmem_ld32(acc_col + 32 * half, a);
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const float4 w0 = *reinterpret_cast<const float4*>(sVec + MR_V_WR + 32 * half + j);
              const float4 w1 = *reinterpret_cast<const float4*>(sVec + MR_V_WR + 64 + 32 * half + j);
              const float4 w2 = *reinterpret_cast<const float4*>(sVec + MR_V_WR + 128 + 32 * half + j);
              const float v0 = fmaxf(a[j], 0.f), v1 = fmaxf(a[j + 1], 0.f), v2 = fmaxf(a[j + 2], 0.f), v3 = fmaxf(a[j + 3], 0.f);
              r0 = fmaf(w0.w, v3, fmaf(w0.z, v2, fmaf(w0.y, v1, fmaf(w0.x, v0, r0))));
              r1 = fmaf(w1.w, v3, fmaf(w1.z, v2, fmaf(w1.y, v1, fmaf(w1.x, v0, r1))));
              r2 = fmaf(w2.w, v3, fmaf(w2.z, v2, fmaf(w2.y, v1, fmaf(w2.x, v0, r2))));
            }
          }
          tc_fence_before();
          if (half == 1) *reinterpret_cast<float4*>(s_rgb[tile_id][row]) = make_float4(r0, r1, r2, 0.f);
          bar_sync_named(1 + tile_id, 256);                  // the two halves of every row of this tile
          if (half == 0 && live) {
            const float4 q = *reinterpret_cast<const float4*>(s_rgb[tile_id][row]);
            r0 += q.x + sVec[MR_V_BR]; r1 += q.y + sVec[MR_V_BR + 1]; r2 += q.z + sVec[MR_V_BR + 2];
            float4 o;
            o.x = 1.f / (1.f + expf(-r0)); o.y = 1.f / (1.f + expf(-r1)); o.z = 1.f / (1.f + expf(-r2));
            o.w = fmaxf(s_alpha[tile_id][0][row] + s_alpha[tile_id][1][row] + sVec[MR_V_BA], 0.f);
            reinterpret_cast<float4*>(rp.raw)[si] = o;
          }
          bar_sync_named(1 + tile_id, 256);                  // s_rgb / s_alpha are rewritten by the next pass
        }
      }
    }
  } else if (warp == 16) {
    // =============================================================== MMA issuer
    // The whole warp walks the issue code on warp-uniform values and ONE elected lane executes the MMAs; every descriptor
    // is a (low word, constant high word) pair whose low word is computed OUTSIDE the elected branch (uniform datapath)
    // and only advanced by compile-time constants inside it (the first version built the 64-bit descriptors inside
    // `if (elected)`: R2UR / elect sequences per operand).
    // Dissection (BMV_MR_DEBUG_PANEL, tools/mvs_render_dissect.py, clk per tile pair): all 41.9 k | no gather 28.5 k |
    // no MMAs 33.4 k | no epilogue arithmetic 39.7 k | empty pipeline 15.5 k, the same with 1 KB weight panels (so the
    // 256 KB weight pass per pair is not what bounds it).  Issuing from the last-publishing row-owner warp instead of this
    // polling warp (as render_multi_umma.cu does) took the empty pipeline to 10.4 k and left the full kernel at 42.9 k:
    // the parts add up whatever the hand-shake costs, because what they share is the L1 / shared-memory data pipe
    // (tensor-core operand reads ~9 k + operand stores ~4.6 k + weight ring ~2 k + gather ~9 k wavefronts of the 42 k clk).
    const bool elected = elect_one();
    constexpr uint32_t HI = (128u >> 4) | (1u << 14);                   // SBO = 128 B, descriptor version 1, SWIZZLE_NONE
    constexpr uint32_t LBO_A = (uint32_t)(MR_CHUNK >> 4) << 16;         // K-chunks of an A operand are 2048 B apart
    constexpr uint32_t LBO_B128 = (2048u >> 4) << 16, LBO_B64 = (1024u >> 4) << 16;
    uint32_t par_ready[2] = {0u, 0u};
    uint32_t panel_n = 0;                                               // panels consumed so far (ring position)
    const uint32_t ring = smem_u32(sRing);
    const uint32_t bias_lo = ((smem_u32(sBias) & 0x3FFFFu) >> 4) | LBO_B128;
    uint32_t aP[2], aF[2], aFb[2], aV[2], aH[2], aH2[2];
#pragma unroll
    for (int w = 0; w < 2; ++w) {
      const uint32_t base = smem_u32(sA + w * MR_TILE_BYTES);
      aP[w] = (((base + MR_P * MR_CHUNK) & 0x3FFFFu) >> 4) | LBO_A;
      aF[w] = (((base + MR_F * MR_CHUNK) & 0x3FFFFu) >> 4) | LBO_A;
      aFb[w] = (((base + (MR_F + 2) * MR_CHUNK) & 0x3FFFFu) >> 4) | LBO_A;
      aV[w] = (((base + MR_V * MR_CHUNK) & 0x3FFFFu) >> 4) | LBO_A;
      aH[w] = (((base + MR_H * MR_CHUNK) & 0x3FFFFu) >> 4) | LBO_A;
      aH2[w] = (((base + (MR_H + 8) * MR_CHUNK) & 0x3FFFFu) >> 4) | LBO_A;
    }
    const int ph_count[8] = {2, 2, 2, 2, 2, 3, 2, 1};
    for (int64_t pair = blockIdx.x; pair < n_pairs; pair += gridDim.x) {
#pragma unroll 1
      for (int phase = 0; phase < 8; ++phase) {
        // ring slots of this phase's panels as descriptor low words (uniform: the shuffle pins it for the compiler)
        const uint32_t pn = __shfl_sync(0xffffffffu, panel_n, 0);
        const uint32_t s0 = (((ring + ((pn + 0) % MR_SLOTS) * MR_SLOT) & 0x3FFFFu) >> 4);
        const uint32_t s1 = (((ring + ((pn + 1) % MR_SLOTS) * MR_SLOT) & 0x3FFFFu) >> 4);
        const uint32_t s2 = (((ring + ((pn + 2) % MR_SLOTS) * MR_SLOT) & 0x3FFFFu) >> 4);
        const uint32_t bias_p = bias_lo + (uint32_t)(((phase == 6 ? 4 : phase - 1) * 4096) >> 4);
#pragma unroll 1
        for (int w = 0; w < 2; ++w) {
          mbar_wait(smem_u32(&s_aready[w]), par_ready[w]); par_ready[w] ^= 1u;
          if (w == 0) {
            for (int q = 0; q < ph_count[phase]; ++q) {
              const uint32_t n = pn + q;
              mbar_wait(smem_u32(&s_full[n % MR_SLOTS]), (n / MR_SLOTS) & 1u);
            }
          }
          __syncwarp();
          tc_fence_after();
          const uint32_t acc = tmem_base + (uint32_t)(w * 256), gate = acc + 128;
          const uint32_t ap = aP[w], af = aF[w], afb = aFb[w], av = aV[w], ah = aH[w], ah2 = aH2[w];
          if (elected && (dbg_panel_bytes & (2 << 20))) {
            umma_commit(smem_u32(&s_acc[w]));
            if (w == 1) {
              umma_commit(smem_u32(&s_empty[(pn + 0) % MR_SLOTS]));
              if (ph_count[phase] > 1) umma_commit(smem_u32(&s_empty[(pn + 1) % MR_SLOTS]));
              if (ph_count[phase] > 2) umma_commit(smem_u32(&s_empty[(pn + 2) % MR_SLOTS]));
            }
          } else if (elected) {
            if (phase == 0) {
              umma_f16_lohi<false>(gate, af, HI, s0 | LBO_B128, HI, idesc128);
              umma_f16_lohi<true>(gate, af + 256, HI, (s0 | LBO_B128) + 256, HI, idesc128);
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) {
                if (ks == 0) umma_f16_lohi<false>(acc, ap, HI, s1 | LBO_B128, HI, idesc128);
                else umma_f16_lohi<true>(acc, ap + 256 * ks, HI, (s1 | LBO_B128) + 256 * ks, HI, idesc128);
              }
            } else if (phase == 5) {
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) {
                if (ks == 0) umma_f16_lohi<false>(acc, ap, HI, s0 | LBO_B128, HI, idesc128);
                else umma_f16_lohi<true>(acc, ap + 256 * ks, HI, (s0 | LBO_B128) + 256 * ks, HI, idesc128);
              }
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) umma_f16_lohi<true>(acc, ah + 256 * ks, HI, (s1 | LBO_B128) + 256 * ks, HI, idesc128);
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) umma_f16_lohi<true>(acc, ah2 + 256 * ks, HI, (s2 | LBO_B128) + 256 * ks, HI, idesc128);
            } else if (phase == 7) {
#pragma unroll
              for (int ks = 0; ks < 8; ++ks) {
                if (ks == 0) umma_f16_lohi<false>(acc, ah, HI, s0 | LBO_B64, HI, idesc64);
                else umma_f16_lohi<true>(acc, ah + 256 * ks, HI, (s0 | LBO_B64) + 128 * ks, HI, idesc64);
              }
              umma_f16_lohi<true>(acc, av, HI, (s0 | LBO_B64) + 128 * 8, HI, idesc64);
            } else {                                        // L1..L4 and the feature layer: h . W + 1 . b
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) {
                if (ks == 0) umma_f16_lohi<false>(acc, ah, HI, s0 | LBO_B128, HI, idesc128);
                else umma_f16_lohi<true>(acc, ah + 256 * ks, HI, (s0 | LBO_B128) + 256 * ks, HI, idesc128);
              }
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) umma_f16_lohi<true>(acc, ah2 + 256 * ks, HI, (s1 | LBO_B128) + 256 * ks, HI, idesc128);
              umma_f16_lohi<true>(acc, afb, HI, bias_p, HI, idesc128);
            }
            umma_commit(smem_u32(&s_acc[w]));
            if (w == 1) {                                   // both tiles have read this phase's panels
              umma_commit(smem_u32(&s_empty[(pn + 0) % MR_SLOTS]));
              if (ph_count[phase] > 1) umma_commit(smem_u32(&s_empty[(pn + 1) % MR_SLOTS]));
              if (ph_count[phase] > 2) umma_commit(smem_u32(&s_empty[(pn + 2) % MR_SLOTS]));
            }
          }
          __syncwarp();
        }
        panel_n += ph_count[phase];
      }
    }
  } else {
    // =============================================================== weight producer
    if (elect_one()) {
      uint32_t n = 0;
      for (int64_t pair = blockIdx.x; pair < n_pairs; pair += gridDim.x) {
        for (int q = 0; q < MR_NPANEL; ++q, ++n) {
          const uint32_t s = n % MR_SLOTS;
          if (n >= MR_SLOTS) {                               // back off between polls: this lane only feeds the ring
            const uint32_t mb = smem_u32(&s_empty[s]), par = ((n / MR_SLOTS) - 1) & 1u;
            uint32_t done = 0;
            while (true) {
              asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
                           : "=r"(done) : "r"(mb), "r"(par) : "memory");
              if (done) break;
              __nanosleep(64);
            }
          }
          const uint32_t bytes = (dbg_panel_bytes & 0xFFFFF) > 0 ? (uint32_t)(dbg_panel_bytes & 0xFFFFF) : (uint32_t)mr_panel_bytes(q);
          mbar_expect_tx(smem_u32(&s_full[s]), bytes);
          bulk_g2s(smem_u32(sRing + s * MR_SLOT), gw + mr_panel_offset(q), bytes, smem_u32(&s_full[s]));
        }
      }
    }
    __syncwarp();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 16) tmem_dealloc_512(tmem_base);
}

}  // namespace bmv

extern "C" BMV_API int bmv_mvs_render_umma_weight_bytes(void) { return bmv::MR_PACK_BYTES; }

extern "C" BMV_API int bmv_mvs_render_umma(const bmv_mvs_render_params* rp, bmv_stream_t stream) {
  BMV_NVTX_RANGE("bmv_mvs_render_umma");
  using namespace bmv;
  BMV_REQUIRE(rp != nullptr, BMV_ERR_INVALID_ARGUMENT, "bmv_mvs_render_umma: null params");
  const bmv_mvs_march_params* p = &rp->g;
  BMV_REQUIRE(p->n_rays >= 0 && p->ray_begin >= 0 && p->S >= 1, BMV_ERR_INVALID_ARGUMENT, "bmv_mvs_render_umma: bad range");
  if (p->n_rays == 0) return BMV_OK;
  BMV_REQUIRE(p->rays && p->t && p->src_exts && p->src_ixts && p->volume && p->rgb && rp->weights && rp->raw,
              BMV_ERR_INVALID_ARGUMENT, "bmv_mvs_render_umma: null device pointer");
  BMV_REQUIRE(p->V == 3 && p->Cv == 8, BMV_ERR_UNSUPPORTED_SHAPE, "bmv_mvs_render_umma: V=%d, Cv=%d not instantiated (3, 8)", p->V, p->Cv);
  BMV_REQUIRE(p->Dv >= 1 && p->hv >= 1 && p->wv >= 1 && p->H >= 2 && p->W >= 2, BMV_ERR_INVALID_ARGUMENT, "bmv_mvs_render_umma: bad grid size");
  BMV_REQUIRE(((uintptr_t)rp->weights & 15) == 0 && ((uintptr_t)rp->raw & 15) == 0 && ((uintptr_t)p->rays & 15) == 0,
              BMV_ERR_INVALID_ARGUMENT, "bmv_mvs_render_umma: weights / raw / rays must be 16-byte aligned");
  BMV_REQUIRE(!p->rgb_nhwc4 || ((uintptr_t)p->rgb & 15) == 0, BMV_ERR_INVALID_ARGUMENT,
              "bmv_mvs_render_umma: an (N,H,W,4) rgb image must be 16-byte aligned");
  BMV_REQUIRE(p->vol_c_stride != 1 || (((uintptr_t)p->volume & 15) == 0 && p->vol_x_stride % 4 == 0 && p->vol_y_stride % 4 == 0 &&
                                       p->vol_d_stride % 4 == 0),
              BMV_ERR_INVALID_ARGUMENT, "bmv_mvs_render_umma: a channels-last volume must have 16-byte aligned voxels");
  static DeviceOnce configured;
  if (const int cfg_dev = configured.needed(); cfg_dev >= 0) {
    cudaError_t e = cudaFuncSetAttribute(mvs_render_umma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)MR_SMEM);
    if (e != cudaSuccess) {
      set_error("bmv_mvs_render_umma: cannot reserve %zu B shared memory: %s", MR_SMEM, cudaGetErrorString(e));
      return BMV_ERR_CUDA_LAUNCH;
    }
    configured.done(cfg_dev);
  }
  const int64_t pairs = ceil_div64(ceil_div64(p->n_rays * p->S, 128), 2);
  const unsigned blocks = (unsigned)(pairs < kNumSMs ? pairs : kNumSMs);   // persistent: the CTA owns all 512 TMEM columns
  static const int dbg_panel = getenv("BMV_MR_DEBUG_PANEL") ? atoi(getenv("BMV_MR_DEBUG_PANEL")) : 0;
  mvs_render_umma_kernel<<<blocks, MR_THREADS, MR_SMEM, (cudaStream_t)stream>>>(*rp, dbg_panel);
  return check_launch("bmv_mvs_render_umma");
}
