// Output sinks of a rendered frame (SURVEY.md §8 row f4), so that what leaves the GPU is what the reference's
// evaluator / visualiser actually consume instead of the fp32 frame:
//   * bmv_frame_psnr_accumulate: masked (and optionally centre-cropped) sum of squared errors + element count of a
//     predicted frame against the ground truth (reference lib/evaluators/enerf.py:45-71: pred/gt reshaped to
//     (h,w,3), `eval_center` crop of 10 %, `gt[mask]` vs `pred[mask]` into skimage's PSNR = 10 log10(1 / mse),
//     mse accumulated in float64);
//   * bmv_frame_to_u8: rgb -> uint8 with numpy's `(x * 255).astype(uint8)` truncation, depth min / max, and
//     depth -> uint8 `(d - min) / (max - min) * 255` (reference lib/visualizers/enerf.py:21-37);
//   * bmv_frame_ssim: skimage's structural_similarity(channel_axis=-1, win_size=w, data_range=R) with uniform
//     weights, moments and formula in float64, over the optionally centre-cropped frame.
// All are single-pass HBM streams (16 / 28 / 24 bytes per pixel); the D2H copy shrinks from 16 to 4 bytes per pixel.
#include <float.h>

#include "bmv_internal.cuh"

namespace bmv {

__global__ void __launch_bounds__(256) frame_psnr_kernel(bmv_frame_psnr_params p) {
  double sse = 0.0;
  unsigned long long cnt = 0;
  const int64_t n = (int64_t)p.H * p.W;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int y = (int)(i / p.W), x = (int)(i % p.W);
    if (y < p.crop_h || y >= p.H - p.crop_h || x < p.crop_w || x >= p.W - p.crop_w) continue;
    if (p.mask && !(__ldg(p.mask + i) >= 1)) continue;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const double d = (double)__ldg(p.gt + i * 3 + c) - (double)__ldg(p.pred + i * 3 + c);
      sse = fma(d, d, sse);
    }
    cnt += 3;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    sse += __shfl_xor_sync(0xffffffffu, sse, o);
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  }
  __shared__ double s_sse[8];
  __shared__ unsigned long long s_cnt[8];
  if ((threadIdx.x & 31) == 0) { s_sse[threadIdx.x >> 5] = sse; s_cnt[threadIdx.x >> 5] = cnt; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < 8; ++i) { sse += s_sse[i]; cnt += s_cnt[i]; }
    atomicAdd(p.sse, sse);
    atomicAdd(p.count, cnt);
  }
}

// order-preserving map float -> uint32 for atomicMin / atomicMax on floats of either sign
__device__ __forceinline__ unsigned f2ord(float f) {
  const unsigned u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord2f(unsigned u) {
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

__global__ void minmax_init_kernel(unsigned* s) {
  s[0] = 0xff800000u;   // ord(+inf): running minimum
  s[1] = 0x007fffffu;   // ord(-inf): running maximum
}

__global__ void __launch_bounds__(256) frame_rgb_u8_minmax_kernel(bmv_frame_to_u8_params p) {
  float mn = INFINITY, mx = -INFINITY;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < p.R; i += (int64_t)gridDim.x * blockDim.x) {
    if (p.rgb_u8) {
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        // numpy: (pred * 255).astype(np.uint8) — fp32 multiply, truncation toward zero; values are convex
        // combinations of source colours in [0, 1], the clamp only guards the undefined out-of-range cast
        const float v = mul_rn(__ldg(p.rgb + i * 3 + c), 255.f);
        p.rgb_u8[i * 3 + c] = (uint8_t)(int)fminf(fmaxf(v, 0.f), 255.f);
      }
    }
    if (p.depth) {
      const float d = __ldg(p.depth + i);
      mn = fminf(mn, d);
      mx = fmaxf(mx, d);
    }
  }
  if (!p.depth) return;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  if ((threadIdx.x & 31) == 0) {
    atomicMin(p.minmax_ord, f2ord(mn));
    atomicMax(p.minmax_ord + 1, f2ord(mx));
  }
}

__global__ void __launch_bounds__(256) frame_depth_u8_kernel(bmv_frame_to_u8_params p) {
  const float mn = ord2f(p.minmax_ord[0]), mx = ord2f(p.minmax_ord[1]);
  const float span = sub_rn(mx, mn);
  if (blockIdx.x == 0 && threadIdx.x == 0 && p.minmax) { p.minmax[0] = mn; p.minmax[1] = mx; }
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < p.R; i += (int64_t)gridDim.x * blockDim.x) {
    // ((depth - depth.min()) / (depth.max() - depth.min()) * 255).astype(np.uint8): three separately rounded fp32 ops
    const float v = mul_rn(div_rn(sub_rn(__ldg(p.depth + i), mn), span), 255.f);
    p.depth_u8[i] = (uint8_t)(int)fminf(fmaxf(v, 0.f), 255.f);
  }
}

// ---------------------------------------------------------------------------------------------- SSIM
// Work item = (strip of up to `tw` output columns, segment of up to `th` output rows, channel); a CTA loops over items
// with a stride of gridDim.x, so the grid (and the scratch it writes) is bounded whatever the frame size.  Output pixel
// (r, x) of the interior (cropped-image coordinates of its window's top-left corner) has the box sum
// A_r(x + w) - A_r(x), where A_r(q) sums the five moments x, y, x², y², xy over the window's rows r .. r+w-1 and the
// strip's columns [0, q).  One thread per output column keeps A_r(x) and A_r(x + w) in registers; stepping to row r+1
// adds the column prefix sums of row(r+w) - row(r), taken by a block-wide scan over the strip's tw + w - 1 input
// columns in chunks of 256.  The first row of a segment scans the w-row column sums instead.  Cost per pixel is
// independent of w; every sum runs in a fixed order, so the result is bit-reproducible.
constexpr int kSsimThreads = 256;
constexpr int kSsimWarps = kSsimThreads / 32;

struct SsimGeom {
  int out_h, out_w;   // interior size: cropped size - w + 1
  int tw, th;         // output columns / rows per item
  int strips;         // items per channel and segment
  int64_t items;
};

__global__ void __launch_bounds__(kSsimThreads) frame_ssim_kernel(bmv_frame_ssim_params p, SsimGeom g) {
  __shared__ double s_pre[5][kSsimThreads];    // inclusive column prefix of the current chunk, carry included
  __shared__ double s_warp[5][kSsimWarps];
  __shared__ double s_red[kSsimWarps];
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5, w = p.win_size;
  const double np = (double)w * (double)w;
  const double inv_np = 1.0 / np, cov_norm = np / (np - 1.0);
  const double c1 = (0.01 * p.data_range) * (0.01 * p.data_range), c2 = (0.03 * p.data_range) * (0.03 * p.data_range);
  double acc = 0.0;
  for (int64_t item = blockIdx.x; item < g.items; item += gridDim.x) {
    const int c = (int)(item % 3);
    const int64_t tile = item / 3;
    const int xs = (int)(tile % g.strips) * g.tw, r0 = (int)(tile / g.strips) * g.th;
    const int ntw = min(g.tw, g.out_w - xs), nth = min(g.th, g.out_h - r0), nc = ntw + w - 1;
    // element (row i, strip column j) of channel c sits at base[(i * W + j) * 3]
    const int64_t base = ((int64_t)p.crop_h * p.W + p.crop_w + xs) * 3 + c;
    const float* __restrict__ xp = p.pred + base;
    const float* __restrict__ yp = p.gt + base;
    double a1[5] = {0, 0, 0, 0, 0}, a2[5] = {0, 0, 0, 0, 0};
    for (int r = r0; r < r0 + nth; ++r) {
      double d1[5] = {0, 0, 0, 0, 0}, d2[5] = {0, 0, 0, 0, 0}, carry[5] = {0, 0, 0, 0, 0};
      for (int k = 0; k * kSsimThreads < nc; ++k) {
        const int j = k * kSsimThreads + t;
        double v[5] = {0, 0, 0, 0, 0};
        if (j < nc) {
          if (r == r0) {
#pragma unroll 4
            for (int i = r; i < r + w; ++i) {
              const double x = (double)__ldg(xp + ((int64_t)i * p.W + j) * 3), y = (double)__ldg(yp + ((int64_t)i * p.W + j) * 3);
              v[0] += x; v[1] += y; v[2] += x * x; v[3] += y * y; v[4] += x * y;   // products of fp32 values are exact
            }
          } else {
            const int64_t in = ((int64_t)(r + w - 1) * p.W + j) * 3, out = ((int64_t)(r - 1) * p.W + j) * 3;
            const double x = (double)__ldg(xp + in), y = (double)__ldg(yp + in);
            const double xo = (double)__ldg(xp + out), yo = (double)__ldg(yp + out);
            v[0] = x - xo; v[1] = y - yo; v[2] = x * x - xo * xo; v[3] = y * y - yo * yo; v[4] = x * y - xo * yo;
          }
        }
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
#pragma unroll
          for (int q = 0; q < 5; ++q) {
            const double u = __shfl_up_sync(0xffffffffu, v[q], o);
            if (lane >= o) v[q] += u;
          }
        }
        if (lane == 31) {
#pragma unroll
          for (int q = 0; q < 5; ++q) s_warp[q][warp] = v[q];
        }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < 5; ++q) {
          double off = carry[q];
          for (int u = 0; u < warp; ++u) off += s_warp[q][u];
          s_pre[q][t] = off + v[q];
        }
        __syncthreads();
        // A(x) = inclusive prefix of column x-1 (0 for x = 0), always in chunk 0; A(x+w) = that of column x+w-1
        const int q2 = t + w - 1;
#pragma unroll
        for (int q = 0; q < 5; ++q) {
          if (k == 0 && t >= 1) d1[q] = s_pre[q][t - 1];
          if ((q2 / kSsimThreads) == k) d2[q] = s_pre[q][q2 % kSsimThreads];
          carry[q] = s_pre[q][kSsimThreads - 1];
        }
      }
#pragma unroll
      for (int q = 0; q < 5; ++q) {
        a1[q] += d1[q];
        a2[q] += d2[q];
      }
      if (t < ntw) {
        // skimage: ux = filter(X), vx = cov_norm * (filter(X*X) - ux*ux), S = A1*A2 / (B1*B2).  Explicit roundings (no
        // contraction), so exchanging pred and gt exchanges x and y and reproduces every value bit for bit.
        const double ux = __dmul_rn(__dsub_rn(a2[0], a1[0]), inv_np), uy = __dmul_rn(__dsub_rn(a2[1], a1[1]), inv_np);
        const double uxx = __dmul_rn(__dsub_rn(a2[2], a1[2]), inv_np), uyy = __dmul_rn(__dsub_rn(a2[3], a1[3]), inv_np);
        const double uxy = __dmul_rn(__dsub_rn(a2[4], a1[4]), inv_np);
        const double vx = __dmul_rn(cov_norm, __dsub_rn(uxx, __dmul_rn(ux, ux)));
        const double vy = __dmul_rn(cov_norm, __dsub_rn(uyy, __dmul_rn(uy, uy)));
        const double vxy = __dmul_rn(cov_norm, __dsub_rn(uxy, __dmul_rn(ux, uy)));
        const double n1 = __dadd_rn(__dmul_rn(2.0 * ux, uy), c1), n2 = __dadd_rn(2.0 * vxy, c2);
        const double e1 = __dadd_rn(__dadd_rn(__dmul_rn(ux, ux), __dmul_rn(uy, uy)), c1), e2 = __dadd_rn(__dadd_rn(vx, vy), c2);
        acc += __ddiv_rn(__dmul_rn(n1, n2), __dmul_rn(e1, e2));
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) s_red[warp] = acc;
  __syncthreads();
  if (t == 0) {
    for (int u = 1; u < kSsimWarps; ++u) acc += s_red[u];
    p.scratch[blockIdx.x] = acc;
  }
}

// Fixed-order sum of the per-CTA partials: mean over the interior of all three channels (equal pixel counts, so this
// is the mean of the three channel means).
__global__ void __launch_bounds__(kSsimThreads) frame_ssim_finish_kernel(bmv_frame_ssim_params p, int parts, double count) {
  __shared__ double s_red[kSsimWarps];
  double acc = 0.0;
  for (int i = threadIdx.x; i < parts; i += kSsimThreads) acc += p.scratch[i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int u = 1; u < kSsimWarps; ++u) acc += s_red[u];
    *p.ssim = acc / count;
  }
}

}  // namespace bmv

extern "C" BMV_API int bmv_frame_psnr_accumulate(const bmv_frame_psnr_params* p, bmv_stream_t stream) {
  BMV_NVTX_RANGE("bmv_frame_psnr_accumulate");
  using namespace bmv;
  BMV_REQUIRE(p && p->pred && p->gt && p->sse && p->count, BMV_ERR_INVALID_ARGUMENT, "bmv_frame_psnr_accumulate: null pointer");
  BMV_REQUIRE(p->H >= 1 && p->W >= 1 && p->crop_h >= 0 && p->crop_w >= 0 && 2 * p->crop_h < p->H && 2 * p->crop_w < p->W,
              BMV_ERR_INVALID_ARGUMENT, "bmv_frame_psnr_accumulate: bad size / crop");
  const int64_t want = ceil_div64((int64_t)p->H * p->W, 256 * 4);
  const unsigned blocks = (unsigned)(want < 4 * kNumSMs ? want : 4 * kNumSMs);
  frame_psnr_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(*p);
  return check_launch("bmv_frame_psnr_accumulate");
}

extern "C" BMV_API int bmv_frame_to_u8(const bmv_frame_to_u8_params* p, bmv_stream_t stream) {
  BMV_NVTX_RANGE("bmv_frame_to_u8");
  using namespace bmv;
  BMV_REQUIRE(p && p->R >= 1, BMV_ERR_INVALID_ARGUMENT, "bmv_frame_to_u8: null params / empty frame");
  BMV_REQUIRE((p->rgb && p->rgb_u8) || (p->depth && p->depth_u8), BMV_ERR_INVALID_ARGUMENT, "bmv_frame_to_u8: nothing to convert");
  BMV_REQUIRE(!p->rgb_u8 || p->rgb, BMV_ERR_INVALID_ARGUMENT, "bmv_frame_to_u8: rgb_u8 without rgb");
  BMV_REQUIRE(!p->depth || (p->depth_u8 && p->minmax_ord), BMV_ERR_INVALID_ARGUMENT,
              "bmv_frame_to_u8: depth needs depth_u8 and the 2-word minmax_ord scratch");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t want = ceil_div64(p->R, 256 * 4);
  const unsigned blocks = (unsigned)(want < 4 * kNumSMs ? want : 4 * kNumSMs);
  if (p->depth) minmax_init_kernel<<<1, 1, 0, st>>>(p->minmax_ord);   // a kernel, not a copy: graph-capturable
  frame_rgb_u8_minmax_kernel<<<blocks, 256, 0, st>>>(*p);
  if (p->depth) frame_depth_u8_kernel<<<blocks, 256, 0, st>>>(*p);
  return check_launch("bmv_frame_to_u8");
}

extern "C" BMV_API int bmv_frame_ssim(const bmv_frame_ssim_params* p, bmv_stream_t stream) {
  BMV_NVTX_RANGE("bmv_frame_ssim");
  using namespace bmv;
  BMV_REQUIRE(p && p->pred && p->gt && p->scratch && p->ssim, BMV_ERR_INVALID_ARGUMENT, "bmv_frame_ssim: null pointer");
  BMV_REQUIRE(p->H >= 1 && p->W >= 1 && p->crop_h >= 0 && p->crop_w >= 0 && 2 * p->crop_h < p->H && 2 * p->crop_w < p->W,
              BMV_ERR_INVALID_ARGUMENT, "bmv_frame_ssim: bad size / crop");
  const int hc = p->H - 2 * p->crop_h, wc = p->W - 2 * p->crop_w, w = p->win_size;
  BMV_REQUIRE(w >= 3 && (w & 1) && w <= hc && w <= wc, BMV_ERR_INVALID_ARGUMENT,
              "bmv_frame_ssim: win_size %d must be odd, >= 3 and fit the %d x %d (cropped) image", w, hc, wc);
  BMV_REQUIRE(p->data_range > 0.0 && p->data_range <= DBL_MAX, BMV_ERR_INVALID_ARGUMENT,
              "bmv_frame_ssim: data_range must be positive and finite");
  SsimGeom g;
  g.out_h = hc - w + 1;
  g.out_w = wc - w + 1;
  // one 256-column scan chunk per row step while the halo leaves at least half the chunk to outputs
  g.tw = w - 1 < kSsimThreads / 2 ? kSsimThreads - (w - 1) : kSsimThreads;
  g.strips = (int)ceil_div64(g.out_w, g.tw);
  // each item re-reads w - 1 halo rows: take the tallest segments (up to 64 rows) that still leave ~2 items per SM
  g.th = 8;
  while (g.th < 64 && 3 * g.strips * ceil_div64(g.out_h, 2 * g.th) >= 2 * kNumSMs) g.th *= 2;
  g.items = 3 * g.strips * ceil_div64(g.out_h, g.th);
  const int grid = (int)(g.items < BMV_FRAME_SSIM_SCRATCH_WORDS ? g.items : BMV_FRAME_SSIM_SCRATCH_WORDS);
  cudaStream_t st = (cudaStream_t)stream;
  frame_ssim_kernel<<<grid, kSsimThreads, 0, st>>>(*p, g);
  frame_ssim_finish_kernel<<<1, kSsimThreads, 0, st>>>(*p, grid, 3.0 * g.out_h * g.out_w);
  return check_launch("bmv_frame_ssim");
}
