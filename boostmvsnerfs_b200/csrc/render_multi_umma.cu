// K3+K5 for ALL K cost-volume chains of a frame in ONE persistent launch with the per-sample MLP on the 5th-generation
// tensor cores (tcgen05.mma, accumulators in tensor memory): the lean gather of render_multi.cu (lean_gather.cuh) in
// front of the UMMA formulation of render_umma.cu, restructured around what bounded those two kernels.
//
// What was measured (profiles/round2c_ncu_render_multi.csv, BMV_RM_DEBUG dissection of render_multi.cu at C2: 1.51 ms
// = 0.42 ms gather + 1.06 ms mma.sync MLP, the two do NOT overlap: both are issue-slot work of the same 16 warps; and
// the first tcgen05 version, render_umma.cu: 510 us per chain with ~100 MMAs per 128-sample tile each costing ~290 clk
// of descriptor construction inside the elected branch, i.e. the single issuing thread bounded it):
//   * the MMAs of a phase are issued by the LAST warp of the tile to publish its operand rows (all arrive on an mbarrier,
//     a shared-memory counter elects the last): warp-uniform code, one elected lane; every descriptor is a (low word, constant high word) pair
//     with the low words advanced by compile-time constants (2 uniform-datapath instructions per MMA).  No issuer warp:
//     a 17th warp costs a whole 4-warp register allocation (96 instead of 128 registers per thread for the gather), its
//     polling loop costs issue slots, and the extra hop costs latency on a chain that is latency-bound (measured: the
//     first version with a polling issuer warp spent 8 k of its 32 k clk per tile waiting on the hand-shakes).  The
//     two tiles of a CTA are independent chains and drift apart: while one waits for its MMAs the other gathers;
//   * TWO threads per sample row (warps w and w + 4 of a tile read the same TMEM lane quarter): 16 row-owner warps per
//     SM instead of 8.  The gather is split by CHANNEL, not by view — half 0: the 8 image-feature channels of the three
//     views, visibility and the z / visibility outputs; half 1: colours, direction features and the trilinear volume
//     fetch — so x_v = f_v + relu(view_fc(dir_v)) and its mean / variance over the views stay thread-local (both halves
//     project the point into the three views: ~25 % duplicated gather arithmetic, no exchange, no barrier).  In the
//     epilogues each half owns half of the accumulator columns; the three partial dot products that span a row (view
//     attention logits, sigma, colour logits) meet through shared memory behind a 64-thread named barrier per warp pair;
//   * colour layer: the part shared by the views ([hid | pooled | vox | 1] . Wcs, K = 96) is computed ONCE into its own
//     accumulator and added to the per-view parts (f_v . Wcv) in the epilogue: 27 MMAs instead of 63.
// Measured (profiles/round2s_render_tcgen05.md): on a par with the mma.sync kernel (1.59 vs 1.58 ms for the 4 chains of
// C2); two further restructurings — gather warps handing samples over through tensor memory, and the next unit's gather
// software-pipelined into the MMA waits — are parity-green and slower (git history).  All formulations sit at ~65 % of
// the L1 data pipe (global taps ~5 k + operand STS / weight LDS ~2 k + tensor-core operand reads ~3 k wavefronts per
// 128-sample tile): that pipe, not the tensor pipe (10 %) or the issue slots (34 %), is what they share.
// Arithmetic: operands fp16 hi + lo (22 significant bits), three MMAs per product (lo.hi + hi.lo + hi.hi), fp32
// accumulation — the same split as render_mma.cu / render_multi.cu, so raw agrees with the fp32 kernels to ~1e-5; z and
// visibility are bit-identical to render_multi.cu (same code).
//
// Operands.  The A operands of phases 0..2 (global_fc, agg.fc, lr0: 13 of the 22 K-steps) go to tensor memory with
// tcgen05.st and the MMAs read them from there (the TS form; only the weights come from shared memory): the rows come
// out of TMEM (tcgen05.ld) into registers for ReLU / soft-max anyway, and st.shared + the tensor core's shared-memory
// reads of A were the largest shared-memory traffic of a tile.  Phase 3 (color.0, 27 MMAs) keeps A in shared memory:
// its accumulators fill all 256 TMEM columns of the tile (shared 64 + 3 views x 64), and its A operands (hid, pooled,
// vox | 1, f_v) would need another 224.  Measured (profiles/round4_render_tmem_operands.md, B200 at 1000 W): 1.497 ->
// 1.347 ms for the 4 chains of the C2 frame, bit-identical raw.
// Shared memory: packed weights (mlp_pack.pack_nerf_weights_umma, nerf_umma_pack.cuh) + two operand tiles of 18 K-chunks
// (chunk = 128 rows x 16 B hi slab + the same for lo; UMMA K-major SWIZZLE_NONE: SBO = 128 B, LBO = 4096 B), all A of color.0:
//   0..7 hid      8+2v,9+2v f_v = [feat8 | rgb3 dir4 0]      14,15 pooled (before that: the phase-B exchange)
//   16 vox      17 (1, 0, ...): bias column of color.0
// TMEM (512 columns, 256 per tile; an A slab = one K = 16 step = hi 8 columns + lo 8 columns, two fp16 per column):
//   phase 0: G_v 32v (accumulators) | A: var 96, mean 112, x_v 128 + 16v, [vox | 1 0 ...] 176..191 (bias column of lr0)
//   phase 1: A: im 96..127 (over var, mean) | fc 128..143 (over x_0)
//   phase 2: A: pooled 96..111 (over im), [vox | 1] 176 | lr0 112..175
//   phase 3: colour: shared 0..63, per view 64 + 64v (A in shared memory)
// Each reused column range was last read by an MMA that has completed (the epilogue waited on its commit) or by
// tcgen05.ld of all 8 warps (retired before they arrive on `ready`).  The exception is the next unit's operand slabs
// over the colour accumulators: the half-0 warp stores its slabs right after phase E's pair barrier, so the half-1
// warp of the same lane quarter retires its tcgen05.ld of those columns before that barrier.
#include <stdlib.h>

#include "lean_gather.cuh"
#include "mlp_mma_tile.cuh"
#include "nerf_umma_pack.cuh"
#include "render_multi_check.cuh"
#include "umma.cuh"

namespace bmv {

constexpr int RU_CHUNK = 4096, RU_LO = 2048;               // bytes per K-chunk (hi slab + lo slab), offset of the lo slab
constexpr int RU_HID = 0, RU_F = 8, RU_POOLED = 14, RU_VOX = 16, RU_ONE = 17;
constexpr int RU_TILE_BYTES = 18 * RU_CHUNK;               // 73728
constexpr int RU_ROW_WARPS = 16;
constexpr int RU_THREADS = RU_ROW_WARPS * 32;
constexpr int RU_PACK_PADDED = (UMMA_PACK_BYTES + 127) / 128 * 128;
constexpr size_t RU_SMEM = (size_t)RU_PACK_PADDED + 2 * (size_t)RU_TILE_BYTES + 128;
// TMEM columns within a tile's 256: accumulators and the A slabs of phases 0..2 (16 columns each: hi 8 + lo 8)
constexpr int RU_T_G = 0, RU_T_VAR = 96, RU_T_MEAN = 112, RU_T_X = 128, RU_T_VOX = 176;            // phase 0
constexpr int RU_T_IM = 96, RU_T_FC = 128, RU_T_POOLED = 96, RU_T_L0 = 112, RU_T_CS = 0, RU_T_CV = 64;

// this row's 8 values of one K-chunk as fp16 hi / lo pairs
struct RuWords {
  uint32_t hi[4], lo[4];
};
__device__ __forceinline__ RuWords ru_split(float v0, float v1, float v2, float v3, float v4, float v5, float v6, float v7) {
  RuWords w;
  split_pack(v0, v1, w.hi[0], w.lo[0]); split_pack(v2, v3, w.hi[1], w.lo[1]);
  split_pack(v4, v5, w.hi[2], w.lo[2]); split_pack(v6, v7, w.hi[3], w.lo[3]);
  return w;
}
__device__ __forceinline__ RuWords ru_split(const float* v) { return ru_split(v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7]); }
// shared-memory K-chunk `chunk`: 16 B into the hi slab, 16 B into the lo slab
__device__ __forceinline__ void ru_put(unsigned char* tile, int chunk, int row, const RuWords& w) {
  unsigned char* q = tile + chunk * RU_CHUNK + row * 16;
  *reinterpret_cast<uint4*>(q) = make_uint4(w.hi[0], w.hi[1], w.hi[2], w.hi[3]);
  *reinterpret_cast<uint4*>(q + RU_LO) = make_uint4(w.lo[0], w.lo[1], w.lo[2], w.lo[3]);
}
// TMEM: K-chunk j (0 | 1) of the slab at column c is taddr = c + 4 j: hi words there, lo words 8 columns further
__device__ __forceinline__ void ru_put_tm(uint32_t taddr, const RuWords& w) {
  tmem_st4(taddr, w.hi);
  tmem_st4(taddr + 8, w.lo);
}

// one K = 16 step of a split product: D (+)= A_lo B_hi + A_hi B_lo + A_hi B_hi; a: TMEM address of the A slab (hi
// columns, lo 8 further) or descriptor low word of the shared hi operand (lo a chunk's lo offset further); b: descriptor
// low word of the hi weights (start address >> 4 | LBO field), the lo block a constant further
template <bool ACC, bool A_TMEM>
__device__ __forceinline__ void ru_kstep(uint32_t d, uint32_t a, uint32_t b, uint32_t idesc) {
  constexpr uint32_t HI = (128u >> 4) | (1u << 14);        // SBO = 128 B, descriptor version 1, SWIZZLE_NONE
  if constexpr (A_TMEM) {
    umma_f16_ts<ACC>(d, a + 8, b, HI, idesc);
    umma_f16_ts<true>(d, a, b + (UW_BLOCK >> 4), HI, idesc);
    umma_f16_ts<true>(d, a, b, HI, idesc);
  } else {
    umma_f16_lohi<ACC>(d, a + (RU_LO >> 4), HI, b, HI, idesc);
    umma_f16_lohi<true>(d, a, HI, b + (UW_BLOCK >> 4), HI, idesc);
    umma_f16_lohi<true>(d, a, HI, b, HI, idesc);
  }
}

// every tcgen05.mma of one phase of one tile (executed by one elected lane); acc: the tile's TMEM base, a: descriptor low
// word of the tile's shared chunk 0, wB: shared-memory address of the packed weights
template <int PHASE>
__device__ __forceinline__ void ru_issue_phase(uint32_t acc, uint32_t a, uint32_t wB) {
  constexpr uint32_t CH = RU_CHUNK >> 4;                   // one K-chunk in descriptor address units
  auto desc_lo = [](uint32_t saddr, uint32_t lbo_bytes) { return ((saddr & 0x3FFFFu) >> 4) | ((lbo_bytes >> 4) << 16); };
  if constexpr (PHASE == 0) {                              // global_fc: G_v = [var | mean] Wgs + x_v Wgv (+ bias, folded)
    const uint32_t id = umma_idesc(32), bGS = desc_lo(wB + UW_GS, 32 * 16), bGV = desc_lo(wB + UW_GV, 32 * 16);
#pragma unroll
    for (int v = 0; v < 3; ++v) {
      const uint32_t d = acc + RU_T_G + 32 * v;
      ru_kstep<false, true>(d, acc + RU_T_VAR, bGS, id);
      ru_kstep<true, true>(d, acc + RU_T_MEAN, bGS + 2 * 32, id);
      ru_kstep<true, true>(d, acc + RU_T_X + 16 * v, bGV, id);
    }
  } else if constexpr (PHASE == 1) {                       // agg.fc: im (K = 32) -> 16
    const uint32_t id = umma_idesc(16), bFC = desc_lo(wB + UW_FC, 16 * 16);
    ru_kstep<false, true>(acc + RU_T_FC, acc + RU_T_IM, bFC, id);
    ru_kstep<true, true>(acc + RU_T_FC, acc + RU_T_IM + 16, bFC + 2 * 16, id);
  } else if constexpr (PHASE == 2) {                       // lr0: [pooled | vox 1] (K = 32) -> 64
    const uint32_t id = umma_idesc(64), bL0 = desc_lo(wB + UW_L0, 64 * 16);
    ru_kstep<false, true>(acc + RU_T_L0, acc + RU_T_POOLED, bL0, id);
    ru_kstep<true, true>(acc + RU_T_L0, acc + RU_T_VOX, bL0 + 2 * 64, id);
  } else {                                                 // color.0: shared part once, per-view parts next to it
    const uint32_t id = umma_idesc(64), bCS = desc_lo(wB + UW_CS, 64 * 16), bCV = desc_lo(wB + UW_CV, 64 * 16);
    ru_kstep<false, false>(acc + RU_T_CS, a + RU_HID * CH, bCS, id);
#pragma unroll
    for (int ks = 1; ks < 4; ++ks) ru_kstep<true, false>(acc + RU_T_CS, a + (RU_HID + 2 * ks) * CH, bCS + ks * 2 * 64, id);
    ru_kstep<true, false>(acc + RU_T_CS, a + RU_POOLED * CH, bCS + 4 * 2 * 64, id);
    ru_kstep<true, false>(acc + RU_T_CS, a + RU_VOX * CH, bCS + 5 * 2 * 64, id);
#pragma unroll
    for (int v = 0; v < 3; ++v) ru_kstep<false, false>(acc + RU_T_CV + 64 * v, a + (RU_F + 2 * v) * CH, bCV, id);
  }
}

// All 8 warps of a tile: publish the operand rows just written (and retire the TMEM loads of the columns about to be
// overwritten) by arriving on the tile's `ready` barrier; the warp that arrives LAST (a shared-memory counter elects it)
// waits for that barrier — complete by then: the wait is the acquire side of the 256 arrivals — issues the phase's MMAs
// and commits them to the tile's accumulator barrier.
template <int PHASE>
__device__ __forceinline__ void ru_publish_and_issue(uint32_t* cnt, uint32_t mb_ready, uint32_t& par_ready, uint32_t mb_acc, uint32_t acc,
                                                     uint32_t a, uint32_t wB, bool no_mma, int lane) {
  if constexpr (PHASE < 3) tmem_wait_st();    // this phase's A slabs (tcgen05.st) complete
  if constexpr (PHASE != 1) proxy_fence_async();   // st.shared of phase 3's operands -> visible to the tensor core (async proxy)
  tc_fence_before();
  mbar_arrive(mb_ready);
  __syncwarp();
  uint32_t last = 0;
  if (lane == 0) last = atomicAdd(cnt, 1u) == (uint32_t)(RU_ROW_WARPS / 2 - 1);
  last = __shfl_sync(0xffffffffu, last, 0);
  if (last) {                          // warp-uniform
    if (lane == 0) *cnt = 0u;          // nobody arrives again before these MMAs have completed
    mbar_wait(mb_ready, par_ready);
    __syncwarp();
    tc_fence_after();
    if (elect_one()) {
      if (!no_mma) ru_issue_phase<PHASE>(acc, a, wB);
      umma_commit(mb_acc);
    }
    __syncwarp();
  }
  par_ready ^= 1u;
}

// dbg (environment BMV_RU_DEBUG, measurement only — bits 0..2 give WRONG results): bit 0 skips the gather arithmetic,
// bit 1 the MMAs (commits only), bit 2 the epilogue arithmetic; bit 3 starts both tiles together (no initial skew)
template <bool GEN, bool INV>
__global__ void __launch_bounds__(RU_THREADS, 1) render_multi_umma_kernel(bmv_render_multi_params mp, int dbg) {
  constexpr int V = 3;
  const bmv_raygen_fetch_params& p = mp.g;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>(((uintptr_t)smem_raw + 127) & ~(uintptr_t)127);
  unsigned char* sW = smem;                                              // hi block, lo block
  const float* sV = reinterpret_cast<const float*>(smem + 2 * UW_BLOCK);  // fp32 vectors
  unsigned char* sA = smem + RU_PACK_PADDED;                             // two operand tiles
  __shared__ LeanCam cams[BMV_MAX_VIEWS];
  __shared__ float s_tar_c[4];
  __shared__ int s_view[BMV_MAX_VOLUMES * V];
  __shared__ __align__(16) float4 s_xe[2][128];                          // phase-E exchange: half 0's partial sums
  __shared__ __align__(8) uint64_t s_acc[2], s_ready[2], s_skew;
  __shared__ uint32_t s_cnt[2];                                          // warps of a tile that have published the current phase
  __shared__ uint32_t s_tmem;

  const int tid = threadIdx.x, lane = tid & 31, warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  for (int i = tid * 16; i < UMMA_PACK_BYTES; i += RU_THREADS * 16)
    *reinterpret_cast<uint4*>(smem + i) = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const unsigned char*>(mp.mlp_weights) + i));
  if (tid < mp.K * V) {                                    // device-resident ids are clamped: they index shared memory
    const int id = mp.views ? __ldg(mp.views + tid) : mp.views_host[tid];
    s_view[tid] = min(max(id, 0), mp.n_views - 1);
  }
  if (tid < mp.n_views) cams[tid] = lean_cam_load(p, tid);
  if (tid < 3) s_tar_c[tid] = p.tar_center[tid];
  if (tid == 0) {
    for (int w = 0; w < 2; ++w) { mbar_init(smem_u32(&s_acc[w]), 1); mbar_init(smem_u32(&s_ready[w]), 256); s_cnt[w] = 0u; }
    mbar_init(smem_u32(&s_skew), 256);
  }
  if (tid < 256) {                                         // the constant K-chunk (1, 0, ..., 0) of both tiles
    unsigned char* q = sA + (tid >> 7) * RU_TILE_BYTES + RU_ONE * RU_CHUNK + (tid & 127) * 16;
    *reinterpret_cast<uint4*>(q) = make_uint4(0x00003C00u, 0, 0, 0);
    *reinterpret_cast<uint4*>(q + RU_LO) = make_uint4(0, 0, 0, 0);
  }
  __syncwarp();
  if (warp == 0) tmem_alloc_512(smem_u32(&s_tmem));
  proxy_fence_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  const uint32_t tmem_base = s_tmem;
  const uint32_t S = (uint32_t)p.S;
  const uint32_t n_samples = (uint32_t)(p.n_rays * p.S);
  const uint32_t tiles = (n_samples + 127u) / 128u;        // per chain
  const uint32_t total = tiles * (uint32_t)mp.K;           // work units: (chain, 128-sample tile)

  {
    // every warp owns 32 sample rows of a tile (as one of two halves): gather, operand rows, MMA issue, epilogues
    const int tile_id = warp >> 3, half = (warp >> 2) & 1, wq = warp & 3, row = wq * 32 + lane;
    unsigned char* tile = sA + tile_id * RU_TILE_BYTES;
    const uint32_t tcol = tmem_base + (uint32_t)(tile_id * 256) + ((uint32_t)(wq * 32) << 16);
    const uint32_t mb_acc = smem_u32(&s_acc[tile_id]), mb_ready = smem_u32(&s_ready[tile_id]);
    uint32_t* cnt = &s_cnt[tile_id];
    uint32_t par_ready = 0;
    const uint32_t acc_t = tmem_base + (uint32_t)(tile_id * 256);
    const uint32_t a_lo = ((smem_u32(tile) & 0x3FFFFu) >> 4) | ((uint32_t)(RU_CHUNK >> 4) << 16), wB = smem_u32(sW);
    const bool no_mma = dbg & 2;
    const int pair_bar = 1 + tile_id * 4 + wq;             // named barrier of the two warps that share this lane quarter
    float4* xb = reinterpret_cast<float4*>(tile + RU_POOLED * RU_CHUNK + row * 16);   // phase-B exchange, + half * RU_LO
    const RmCtx c = lean_ctx(p, mp.nf_plane_stride);
    const bool unit_scale = p.render_scale == 1.f;
    const int vol_row0 = mp.vol_row0, map_row0 = mp.map_row0;
    const bool skip_gather = dbg & 1, skip_epi = dbg & 4;
    uint32_t par_acc = 0;
    bool first = true;
    for (uint32_t u = blockIdx.x * 2u + (uint32_t)tile_id; u < total; u += gridDim.x * 2u) {
      const uint32_t k = u / tiles;                        // chain (uniform over the tile's warps)
      const uint32_t base = (u - k * tiles) * 128u;
      const int* views = s_view + k * V;
      const int64_t out0 = (int64_t)k * n_samples;
      const uint32_t si_raw = base + (uint32_t)row;
      const bool live = si_raw < n_samples;
      const uint32_t si = live ? si_raw : n_samples - 1u;
      if (first && tile_id == 1 && !(dbg & 8)) mbar_wait(smem_u32(&s_skew), 0);   // tile 1 starts half a period late
      // ------------------------------------------------------------ gather + phase A operand rows
      float rgbv[V][3];                                    // half 1: the views' colours, blended in phase E
      if (!skip_gather) {
        const uint32_t li = S == 2u ? (si >> 1) : si / S;
        const int s = (int)(si - li * S);
        const LeanPoint q = lean_sample_point<GEN, INV>(p, c, (uint32_t)p.ray_begin + li, s, mp.depth + (int64_t)k * mp.depth_k_stride,
                                                        mp.std + (int64_t)k * mp.std_k_stride, mp.near_far + (int64_t)k * mp.nf_k_stride,
                                                        map_row0);
        const float3 tt = lean_target_dir(q, s_tar_c);
        if (half == 0) {
          // feature channels 0..7: x = f + relu(view_fc(dir)), mean / unbiased variance over the views
          float x[V][8];
          int cnt = 0;
#pragma unroll
          for (int v = 0; v < V; ++v) {
            const int view = views[v];
            const LeanCam& cam = cams[view];
            const LeanTaps tp = lean_project(p, c, cam, q, unit_scale);
            cnt += tp.visible ? 1 : 0;
            float f[8], d[4];
            lean_fetch_feat(p, view, tp, f);
            lean_dir_feat(cam, q, tt, d);
            ru_put(tile, RU_F + 2 * v, row, ru_split(f));
#pragma unroll
            for (int ch = 0; ch < 8; ++ch) {
              const float4 w = *reinterpret_cast<const float4*>(sV + UV_WV + ch * 4);
              const float e = fmaf(w.w, d[3], fmaf(w.z, d[2], fmaf(w.y, d[1], fmaf(w.x, d[0], sV[UV_BV + ch]))));
              x[v][ch] = f[ch] + fmaxf(e, 0.f);
            }
          }
          float var[8], mean[8];
#pragma unroll
          for (int ch = 0; ch < 8; ++ch) {
            const float m = (x[0][ch] + x[1][ch] + x[2][ch]) * (1.f / 3.f);
            const float e0 = x[0][ch] - m, e1 = x[1][ch] - m, e2 = x[2][ch] - m;
            mean[ch] = m;
            var[ch] = fmaf(e2, e2, fmaf(e1, e1, e0 * e0)) * 0.5f;
          }
          __syncwarp();                                    // tcgen05.st is warp-collective
#pragma unroll
          for (int v = 0; v < V; ++v) ru_put_tm(tcol + RU_T_X + 16 * v, ru_split(x[v]));
          ru_put_tm(tcol + RU_T_VAR, ru_split(var));
          ru_put_tm(tcol + RU_T_MEAN, ru_split(mean));
          if (live) {
            const int64_t oi = out0 + si;
            if (mp.z_vals) mp.z_vals[oi] = q.z;
            if (mp.vis_mask) mp.vis_mask[oi] = lean_vis_score3(cnt);
            if (mp.vis_count) mp.vis_count[oi] = cnt;
          }
        } else {
          // trilinear volume fetch; colours (channels 8..10) and direction features of the views
          RuWords vox;
          {
            float vf[8];
            lean_vox_fetch(p, c, mp.volume + (int64_t)k * mp.vol_k_stride, vol_row0, q, vf);
            vox = ru_split(vf);
            ru_put(tile, RU_VOX, row, vox);                // phase 3 reads vox from shared memory, phase 2 from TMEM
          }
          float x[V][3];
#pragma unroll
          for (int v = 0; v < V; ++v) {
            const int view = views[v];
            const LeanCam& cam = cams[view];
            const LeanTaps tp = lean_project(p, c, cam, q, unit_scale);
            float d[4];
            lean_fetch_rgb(p, view, tp, rgbv[v]);
            lean_dir_feat(cam, q, tt, d);
            ru_put(tile, RU_F + 2 * v + 1, row, ru_split(rgbv[v][0], rgbv[v][1], rgbv[v][2], d[0], d[1], d[2], d[3], 0.f));
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) {
              const float4 w = *reinterpret_cast<const float4*>(sV + UV_WV + (8 + ch) * 4);
              const float e = fmaf(w.w, d[3], fmaf(w.z, d[2], fmaf(w.y, d[1], fmaf(w.x, d[0], sV[UV_BV + 8 + ch]))));
              x[v][ch] = rgbv[v][ch] + fmaxf(e, 0.f);
            }
          }
          float var[3], mean[3];
#pragma unroll
          for (int ch = 0; ch < 3; ++ch) {
            const float m = (x[0][ch] + x[1][ch] + x[2][ch]) * (1.f / 3.f);
            const float e0 = x[0][ch] - m, e1 = x[1][ch] - m, e2 = x[2][ch] - m;
            mean[ch] = m;
            var[ch] = fmaf(e2, e2, fmaf(e1, e1, e0 * e0)) * 0.5f;
          }
          __syncwarp();                                    // tcgen05.st is warp-collective
#pragma unroll
          for (int v = 0; v < V; ++v) ru_put_tm(tcol + RU_T_X + 16 * v + 4, ru_split(x[v][0], x[v][1], x[v][2], 0.f, 0.f, 0.f, 0.f, 0.f));
          ru_put_tm(tcol + RU_T_VAR + 4, ru_split(var[0], var[1], var[2], 0.f, 0.f, 0.f, 0.f, 1.f));   // K index 15: global_fc bias column
          ru_put_tm(tcol + RU_T_MEAN + 4, ru_split(mean[0], mean[1], mean[2], 0.f, 0.f, 0.f, 0.f, 0.f));
          // the whole [vox | 1 0 ... 0] slab of lr0 (K index 24: its bias column); phase 3 overwrites these columns
          const uint32_t vs[16] = {vox.hi[0], vox.hi[1], vox.hi[2], vox.hi[3], 0x00003C00u, 0u, 0u, 0u,
                                   vox.lo[0], vox.lo[1], vox.lo[2], vox.lo[3], 0u, 0u, 0u, 0u};
          tmem_st16(tcol + RU_T_VOX, vs);
        }
      } else {
#pragma unroll
        for (int v = 0; v < V; ++v) rgbv[v][0] = rgbv[v][1] = rgbv[v][2] = 0.f;
      }
      ru_publish_and_issue<0>(cnt, mb_ready, par_ready, mb_acc, acc_t, a_lo, wB, no_mma, lane);
      if (first && tile_id == 0) mbar_arrive(smem_u32(&s_skew));
      first = false;
      // ------------------------------------------------------------ phase B: ReLU, view soft-max, im = input of agg.fc
      mbar_wait(mb_acc, par_acc); par_acc ^= 1u;
      __syncwarp();
      tc_fence_after();
      if (!skip_epi) {
        float g[V][16], pl[V];
#pragma unroll
        for (int v = 0; v < V; ++v) {
          tmem_ld16(tcol + RU_T_G + 32 * v + 16 * half, g[v]);
          float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
          for (int j = 0; j < 16; j += 4) {
            const float4 w = *reinterpret_cast<const float4*>(sV + UV_WA + 16 * half + j);
            g[v][j] = fmaxf(g[v][j], 0.f); g[v][j + 1] = fmaxf(g[v][j + 1], 0.f);
            g[v][j + 2] = fmaxf(g[v][j + 2], 0.f); g[v][j + 3] = fmaxf(g[v][j + 3], 0.f);
            a0 = fmaf(w.x, g[v][j], a0); a1 = fmaf(w.y, g[v][j + 1], a1); a2 = fmaf(w.z, g[v][j + 2], a2); a3 = fmaf(w.w, g[v][j + 3], a3);
          }
          pl[v] = (a0 + a1) + (a2 + a3);
        }
        xb[half * (RU_LO / 16)] = make_float4(pl[0], pl[1], pl[2], 0.f);
        bar_sync_named(pair_bar, 64);
        const float4 po = xb[(half ^ 1) * (RU_LO / 16)];
        const float ba = sV[UV_SC];                        // bias scalars are read where used: fewer live registers
        // both halves add (columns 0..15) + (columns 16..31) in this order: identical soft-max weights in both
        const float l0 = fmaxf((half ? po.x + pl[0] : pl[0] + po.x) + ba, 0.f);
        const float l1 = fmaxf((half ? po.y + pl[1] : pl[1] + po.y) + ba, 0.f);
        const float l2 = fmaxf((half ? po.z + pl[2] : pl[2] + po.z) + ba, 0.f);
        const float mx = fmaxf(l0, fmaxf(l1, l2));
        const float e0 = expf(l0 - mx), e1 = expf(l1 - mx), e2 = expf(l2 - mx);
        const float inv = 1.f / (e0 + e1 + e2);
        const float w0 = e0 * inv, w1 = e1 * inv, w2 = e2 * inv;
        float im[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) im[j] = fmaf(w2, g[2][j], fmaf(w1, g[1][j], w0 * g[0][j]));
        uint32_t s[16];                                    // this half's K = 16 slab of agg.fc: hi 8 columns, lo 8
#pragma unroll
        for (int j = 0; j < 8; ++j) split_pack(im[2 * j], im[2 * j + 1], s[j], s[8 + j]);
        tmem_st16(tcol + RU_T_IM + 16 * half, s);
      }
      ru_publish_and_issue<1>(cnt, mb_ready, par_ready, mb_acc, acc_t, a_lo, wB, no_mma, lane);
      // ------------------------------------------------------------ phase C: pooled = relu(fc + b)
      mbar_wait(mb_acc, par_acc); par_acc ^= 1u;
      __syncwarp();
      tc_fence_after();
      if (!skip_epi) {
        float pc[8];
        tmem_ld8(tcol + RU_T_FC + 8 * half, pc);
        const float4 b0 = *reinterpret_cast<const float4*>(sV + UV_BFC + 8 * half), b1 = *reinterpret_cast<const float4*>(sV + UV_BFC + 8 * half + 4);
        const RuWords pw = ru_split(fmaxf(pc[0] + b0.x, 0.f), fmaxf(pc[1] + b0.y, 0.f), fmaxf(pc[2] + b0.z, 0.f), fmaxf(pc[3] + b0.w, 0.f),
                                    fmaxf(pc[4] + b1.x, 0.f), fmaxf(pc[5] + b1.y, 0.f), fmaxf(pc[6] + b1.z, 0.f), fmaxf(pc[7] + b1.w, 0.f));
        ru_put_tm(tcol + RU_T_POOLED + 4 * half, pw);      // A of lr0
        ru_put(tile, RU_POOLED + half, row, pw);           // A of color.0 (shared-memory operand)
      }
      ru_publish_and_issue<2>(cnt, mb_ready, par_ready, mb_acc, acc_t, a_lo, wB, no_mma, lane);
      // ------------------------------------------------------------ phase D: hid = relu(lr0), partial sigma
      mbar_wait(mb_acc, par_acc); par_acc ^= 1u;
      __syncwarp();
      tc_fence_after();
      float sig_part = 0.f;
      if (!skip_epi) {
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
        for (int cb = 0; cb < 2; ++cb) {
          float h[16];
          tmem_ld16(tcol + RU_T_L0 + 32 * half + 16 * cb, h);
#pragma unroll
          for (int j = 0; j < 16; j += 4) {
            const float4 w = *reinterpret_cast<const float4*>(sV + UV_WS + 32 * half + 16 * cb + j);
            h[j] = fmaxf(h[j], 0.f); h[j + 1] = fmaxf(h[j + 1], 0.f); h[j + 2] = fmaxf(h[j + 2], 0.f); h[j + 3] = fmaxf(h[j + 3], 0.f);
            a0 = fmaf(w.x, h[j], a0); a1 = fmaf(w.y, h[j + 1], a1); a2 = fmaf(w.z, h[j + 2], a2); a3 = fmaf(w.w, h[j + 3], a3);
          }
          ru_put(tile, RU_HID + 4 * half + 2 * cb, row, ru_split(h));
          ru_put(tile, RU_HID + 4 * half + 2 * cb + 1, row, ru_split(h + 8));
        }
        sig_part = (a0 + a1) + (a2 + a3);
      }
      ru_publish_and_issue<3>(cnt, mb_ready, par_ready, mb_acc, acc_t, a_lo, wB, no_mma, lane);
      // ------------------------------------------------------------ phase E: color.2 logits, view soft-max, rgb, sigma
      mbar_wait(mb_acc, par_acc); par_acc ^= 1u;
      __syncwarp();
      tc_fence_after();
      float cl[V] = {0.f, 0.f, 0.f};
      if (!skip_epi) {
#pragma unroll
        for (int cb = 0; cb < 2; ++cb) {
          float sh[16];
          tmem_ld16(tcol + RU_T_CS + 32 * half + 16 * cb, sh);
#pragma unroll
          for (int v = 0; v < V; ++v) {
            float cv[16];
            tmem_ld16(tcol + RU_T_CV + 64 * v + 32 * half + 16 * cb, cv);
            float a0 = 0.f, a1 = 0.f;
#pragma unroll
            for (int j = 0; j < 16; j += 4) {
              const float4 w = *reinterpret_cast<const float4*>(sV + UV_W2 + 32 * half + 16 * cb + j);
              a0 = fmaf(w.x, fmaxf(sh[j] + cv[j], 0.f), a0); a1 = fmaf(w.y, fmaxf(sh[j + 1] + cv[j + 1], 0.f), a1);
              a0 = fmaf(w.z, fmaxf(sh[j + 2] + cv[j + 2], 0.f), a0); a1 = fmaf(w.w, fmaxf(sh[j + 3] + cv[j + 3], 0.f), a1);
            }
            cl[v] += a0 + a1;
          }
        }
      }
      // the pair barrier also orders half 1's colour-accumulator loads before half 0's tcgen05.st of the next unit's
      // operand slabs into the same lanes and columns
      tc_fence_before();
      if (half == 0) s_xe[tile_id][row] = make_float4(cl[0], cl[1], cl[2], sig_part);
      bar_sync_named(pair_bar, 64);
      tc_fence_after();
      if (half == 1 && live) {
        const float4 o0 = s_xe[tile_id][row];
        const float bs = sV[UV_SC + 1], b2 = sV[UV_SC + 2];
        const float c0 = fmaxf((o0.x + cl[0]) + b2, 0.f), c1 = fmaxf((o0.y + cl[1]) + b2, 0.f), c2 = fmaxf((o0.z + cl[2]) + b2, 0.f);
        const float mx = fmaxf(c0, fmaxf(c1, c2));
        const float e0 = expf(c0 - mx), e1 = expf(c1 - mx), e2 = expf(c2 - mx);
        const float inv = 1.f / (e0 + e1 + e2);
        float sig = (o0.w + sig_part) + bs;
        sig = sig > 20.f ? sig : log1pf(expf(sig));
        float4 o;
        o.x = (e0 * rgbv[0][0] + e1 * rgbv[1][0] + e2 * rgbv[2][0]) * inv;
        o.y = (e0 * rgbv[0][1] + e1 * rgbv[1][1] + e2 * rgbv[2][1]) * inv;
        o.z = (e0 * rgbv[0][2] + e1 * rgbv[1][2] + e2 * rgbv[2][2]) * inv;
        o.w = sig;
        reinterpret_cast<float4*>(mp.raw)[out0 + si] = o;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc_512(tmem_base);
}


}  // namespace bmv

extern "C" BMV_API int bmv_render_rays_multi_umma(const bmv_render_multi_params* mp, bmv_stream_t stream) {
  BMV_NVTX_RANGE("bmv_render_rays_multi_umma");
  using namespace bmv;
  if (const int rc = render_multi_validate(mp, "bmv_render_rays_multi_umma"); rc != BMV_OK) return rc;
  const bmv_raygen_fetch_params* p = &mp->g;
  if (p->n_rays == 0) return BMV_OK;
  const bool gen = p->ray_gen && !p->rays, invd = p->depth_inv != 0;
  static DeviceOnce configured;
  if (const int cfg_dev = configured.needed(); cfg_dev >= 0) {
    const int smem = (int)RU_SMEM;
    cudaError_t e = cudaFuncSetAttribute(render_multi_umma_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(render_multi_umma_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(render_multi_umma_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(render_multi_umma_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) {
      set_error("bmv_render_rays_multi_umma: cannot reserve %zu B shared memory: %s", RU_SMEM, cudaGetErrorString(e));
      return BMV_ERR_CUDA_LAUNCH;
    }
    configured.done(cfg_dev);
  }
  // persistent: one CTA per SM owns all 512 TMEM columns (the shared-memory footprint keeps it alone on the SM)
  const int64_t units = ceil_div64(p->n_rays * p->S, 128) * mp->K;
  const int64_t want = ceil_div64(units, 2);
  const unsigned blocks = (unsigned)(want < kNumSMs ? want : kNumSMs);
  cudaStream_t st = (cudaStream_t)stream;
  static const int dbg = getenv("BMV_RU_DEBUG") ? atoi(getenv("BMV_RU_DEBUG")) : 0;
  if (gen && invd) render_multi_umma_kernel<true, true><<<blocks, RU_THREADS, RU_SMEM, st>>>(*mp, dbg);
  else if (gen) render_multi_umma_kernel<true, false><<<blocks, RU_THREADS, RU_SMEM, st>>>(*mp, dbg);
  else if (invd) render_multi_umma_kernel<false, true><<<blocks, RU_THREADS, RU_SMEM, st>>>(*mp, dbg);
  else render_multi_umma_kernel<false, false><<<blocks, RU_THREADS, RU_SMEM, st>>>(*mp, dbg);
  return check_launch("bmv_render_rays_multi_umma");
}
