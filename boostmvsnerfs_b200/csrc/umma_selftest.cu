// Isolated check of the tcgen05 plumbing in umma.cuh (shared-memory descriptors, TMEM allocation, commit to an
// mbarrier, tcgen05.ld) that render_multi_umma.cu, mvs_render_umma.cu and conv3d_umma.cu rely on: one 128-row tile of
// D = A . B^T with the operands split into fp16 hi + lo like the render kernels' (tests/test_gpu_umma.py compares it
// with float64).
#include "bmv_internal.cuh"
#include "umma.cuh"

namespace bmv {

constexpr int kChunkBytes = 4096;                         // one K-chunk of 8: hi slab (128 rows x 16 B) + lo slab

// x = hi + lo with hi = fp16(x), lo = fp16(x - hi), two values per 32-bit word
__device__ __forceinline__ void split2(float v0, float v1, uint32_t& hi, uint32_t& lo) {
  __half2 hh = __floats2half2_rn(v0, v1);
  const float2 back = __half22float2(hh);
  __half2 ll = __floats2half2_rn(v0 - back.x, v1 - back.y);
  hi = *reinterpret_cast<uint32_t*>(&hh);
  lo = *reinterpret_cast<uint32_t*>(&ll);
}
// this row's 8 values of K-chunk `chunk`: 16 B into the hi slab, 16 B into the lo slab
__device__ __forceinline__ void put_chunk(unsigned char* tile, int chunk, int row, float v0, float v1, float v2, float v3,
                                          float v4, float v5, float v6, float v7) {
  uint4 hi, lo;
  split2(v0, v1, hi.x, lo.x); split2(v2, v3, hi.y, lo.y); split2(v4, v5, hi.z, lo.z); split2(v6, v7, hi.w, lo.w);
  unsigned char* q = tile + chunk * kChunkBytes + row * 16;
  *reinterpret_cast<uint4*>(q) = hi;
  *reinterpret_cast<uint4*>(q + 2048) = lo;
}

// D (128 x N, fp32) = A (128 x K, fp32, row-major) . B^T with B given in the packed [hi block][lo block]
// layout ([K/8][N][8] fp16 each): one CTA, A in the UMMA K-major SWIZZLE_NONE layout (SBO = 128 B, LBO = kChunkBytes).
__global__ void __launch_bounds__(128, 1) umma_selftest_kernel(const float* __restrict__ A, const uint4* __restrict__ Bp,
                                                               float* __restrict__ D, int N, int K) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>(((uintptr_t)smem_raw + 127) & ~(uintptr_t)127);
  __shared__ __align__(8) uint64_t s_mbar;
  __shared__ uint32_t s_tmem;
  const int tid = threadIdx.x, warp = tid >> 5;
  const int chunks = K / 8;
  unsigned char* sAop = smem;                               // chunks x 4096
  unsigned char* sB = smem + chunks * kChunkBytes;          // hi block, lo block of chunks x N x 16
  const int bblock = chunks * N * 16;
  for (int i = tid; i < 2 * bblock / 16; i += 128) reinterpret_cast<uint4*>(sB)[i] = Bp[i];
  for (int c = 0; c < chunks; ++c) {
    const float* a = A + (int64_t)tid * K + 8 * c;
    put_chunk(sAop, c, tid, a[0], a[1], a[2], a[3], a[4], a[5], a[6], a[7]);
  }
  if (tid == 0) mbar_init(smem_u32(&s_mbar), 1);
  __syncwarp();
  if (warp == 0) tmem_alloc_512(smem_u32(&s_tmem));
  proxy_fence_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = s_tmem;
  if (tid == 0) {
    const uint32_t id = umma_idesc(N);
    for (int ks = 0; ks < K / 16; ++ks)
      umma_kstep(tmem_base, smem_u32(sAop) + ks * 2 * kChunkBytes, kChunkBytes, 2048, smem_u32(sB) + ks * 2 * N * 16, N * 16, bblock, id, ks ? 1u : 0u);
    umma_commit(smem_u32(&s_mbar));
  }
  mbar_wait(smem_u32(&s_mbar), 0);
  __syncwarp();
  tc_fence_after();
  const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16);
  for (int c = 0; c < N / 16; ++c) {
    float v[16];
    tmem_ld16(trow + 16 * c, v);
    for (int j = 0; j < 16; ++j) D[(int64_t)tid * N + 16 * c + j] = v[j];
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc_512(tmem_base);
}

}  // namespace bmv

extern "C" BMV_API int bmv_umma_selftest(const float* A, const void* B_packed, float* D, int N, int K, bmv_stream_t stream) {
  BMV_NVTX_RANGE("bmv_umma_selftest");
  using namespace bmv;
  BMV_REQUIRE(A && B_packed && D, BMV_ERR_INVALID_ARGUMENT, "bmv_umma_selftest: null pointer");
  BMV_REQUIRE(N >= 16 && N <= 256 && N % 16 == 0 && K >= 16 && K <= 96 && K % 16 == 0, BMV_ERR_UNSUPPORTED_SHAPE,
              "bmv_umma_selftest: N=%d K=%d unsupported", N, K);
  const size_t smem = (size_t)(K / 8) * kChunkBytes + (size_t)2 * (K / 8) * N * 16 + 128;
  cudaError_t e = cudaFuncSetAttribute(umma_selftest_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) {
    set_error("bmv_umma_selftest: cannot reserve %zu B shared memory: %s", smem, cudaGetErrorString(e));
    return BMV_ERR_CUDA_LAUNCH;
  }
  umma_selftest_kernel<<<1, 128, smem, (cudaStream_t)stream>>>(A, reinterpret_cast<const uint4*>(B_packed), D, N, K);
  return check_launch("bmv_umma_selftest");
}
