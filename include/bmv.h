/*
 * bmv.h — C ABI of the B200-native (sm_100a) BoostMVSNeRFs per-frame rendering kernels.
 *
 * Drop-in boundary (SURVEY.md §8b): the reference has no native code; its "operator interface" for
 * this path is the set of pure Python renderer functions in lib/networks/enerf/utils.py and
 * lib/networks/boost_enerf/network.py.  Each entry point below replaces one or more of those
 * functions (cited per entry as reference file:line) and is what a ctypes binding on the reference
 * side would bind (see INTEGRATION.md).
 *
 * Conventions
 *  - plain C: raw DEVICE pointers, sizes, element strides and scalars; no torch types.
 *  - the caller owns every buffer; the library never allocates, frees or keeps a pointer after
 *    the enqueue returns.
 *  - work is enqueued on `stream` (a cudaStream_t passed as void*); no host syncs; every entry
 *    is CUDA-graph capturable; the caller selects the device (cudaSetDevice) beforehand.
 *  - return value: BMV_OK (0) or a negative bmv_status; bmv_last_error_string() gives detail
 *    (thread-local).  No C++ exception crosses the ABI.
 *  - all tensors are fp32 and contiguous in the stated layout unless strides are given.
 *    Strides are in ELEMENTS.
 *  - camera matrices are read from DEVICE memory (they change every frame; keeping them out of
 *    the kernel parameters keeps a captured graph replayable).
 */
#ifndef BMV_H_
#define BMV_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define BMV_API __attribute__((visibility("default")))
#else
#define BMV_API
#endif

#define BMV_VERSION 100          /* 0.1.0 */
#define BMV_MAX_VIEWS 8          /* source views per cost volume (reference uses 3) */
#define BMV_MAX_VOLUMES 16       /* K cost volumes blended per frame */

typedef enum bmv_status {
  BMV_OK = 0,
  BMV_ERR_INVALID_ARGUMENT = -1,
  BMV_ERR_UNSUPPORTED_SHAPE = -2,
  BMV_ERR_CUDA_LAUNCH = -3,
  BMV_ERR_NOT_IMPLEMENTED = -4
} bmv_status;

typedef void* bmv_stream_t;      /* cudaStream_t */

BMV_API int bmv_version(void);
BMV_API const char* bmv_last_error_string(void);
/* Number of kernel launches enqueued by this library in the calling process so far
 * (bench.py reports the per-step delta as "gpu_launches"). */
BMV_API uint64_t bmv_launch_count(void);
/* sizeof() of the params struct of entry point `entry` ("bmv_cost_volume_var", ...), -1 if unknown:
 * lets a foreign-language binding verify its struct layout at load time. */
BMV_API int bmv_sizeof_params(const char* entry);

/* ------------------------------------------------------------------------------------------
 * K1  cost-volume build: per-plane homography warp of S source feature maps + variance.
 * Replaces homo_warp + build_feature_volume (reference lib/networks/enerf/utils.py:57-95,324-351).
 *   vol[c,d,y,x] = (sum_s f_s^2)/S - ((sum_s f_s)/S)^2,
 *   f_s = bilinear_zeros(feat_s[c], homography_s(x, y, planes[d,y,x]))
 * The S maps are addressed as feat + view[s]*feat_view_stride (no gather copy of the triple,
 * cf. reference lib/networks/boost_enerf/network.py:196-201).
 */
typedef struct bmv_cost_volume_params {
  const float* feat;            /* source feature maps of ALL views */
  int64_t feat_view_stride;     /* elements between consecutive views */
  int64_t feat_c_stride, feat_y_stride, feat_x_stride; /* NCHW: Hs*Ws, Ws, 1; NHWC: 1, Ws*C, C */
  int32_t view[BMV_MAX_VIEWS];  /* which views form this volume */
  int32_t S, C, Hs, Ws;         /* views per volume, channels, source map size */
  const float* proj;            /* DEVICE (N,3,4) row-major, indexed by view[s] like feat:
                                   src_proj @ inv(tar_proj) of get_proj_mats */
  const float* planes;          /* DEVICE depth hypotheses */
  int64_t planes_d_stride;      /* h*w for per-pixel planes (B,D,h,w); 1 with planes_pix_stride 0 for (D,) */
  int64_t planes_pix_stride;    /* 1 for per-pixel planes, 0 when every pixel shares the D values */
  int32_t D, h, w;              /* volume size */
  float* out;                   /* (C,D,h,w) with the strides below */
  int64_t out_c_stride, out_d_stride, out_y_stride, out_x_stride;
  int32_t out_bf16;             /* 0: fp32 out, 1: out points to bf16 storage, 2: fp16 storage (round-to-nearest-even) */
  int32_t exact_coords;         /* 1: reproduce the reference's coordinate arithmetic op for op (IEEE divisions,
                                   slower); 0: reciprocal-multiply form, coordinates within 2 ulp (default) */
  int32_t feat_half;            /* 1: feat points to fp16 storage (strides in fp16 elements): half the bytes per bilinear tap.
                                   TF32-class (the maps come out of TF32-class convolutions): channels-last fast path only */
  int32_t variant;              /* 0: the fastest kernel generation that fits the layout; 5: the four-channels-per-lane
                                   generation (v5) even where the eight-channels-per-lane one (v6) applies (A/B tests:
                                   the two are bit-identical) */
  const float* out_scale;       /* DEVICE or NULL: every stored variance is multiplied by out_scale[0] (a power of two from
                                   bmv_volume_scale): keeps an fp16 volume inside the fp16 range whatever the feature
                                   magnitude; the consuming convolution undoes it (bmv_conv3d_params.in_scale) */
  const int32_t* view_dev;      /* DEVICE or NULL: S view ids read by the kernel instead of view[] — a captured CUDA graph
                                   then follows a changed view selection by rewriting S ints (channels-last fast paths) */
} bmv_cost_volume_params;
BMV_API int bmv_cost_volume_var(const bmv_cost_volume_params* p, bmv_stream_t stream);

/* Range scale for an fp16 cost volume (no counterpart in the reference, which stores fp32): the variance of S values in
 * [-m, m] is at most m^2, so with m = max|x| over the level's feature maps scale = 2^k, k = floor(log2(target / m^2)),
 * bounds every stored variance by `target` (default use: 16384 of the 65504 fp16 maximum) and moves small-magnitude
 * features up out of the fp16 subnormals.  One launch: block maxima -> atomicMax -> the last block writes
 * scale[0] = 2^k, scale[1] = 2^-k, and scale[4] = 2^k * consumer_scale, scale[5] = 1 / scale[4] for a consumer whose fp16
 * weights were themselves packed pre-multiplied by consumer_scale (bmv_conv3d_params.in_scale = scale + 4; 0 is read
 * as 1).  scale has 6 floats; scale[2..3] are scratch words that must be zero before the first use; the kernel
 * leaves them zero.  x: fp32 or fp16 (x_half), n elements, 16-byte aligned, n % 4 == 0 (fp32) / 8 (fp16). */
typedef struct bmv_volume_scale_params {
  const void* x; int64_t n; int32_t x_half; float target;
  float* scale;
  float consumer_scale; int32_t reserved0;
} bmv_volume_scale_params;
BMV_API int bmv_volume_scale(const bmv_volume_scale_params* p, bmv_stream_t stream);

/* The K cost volumes of one cascade level in ONE launch when they share the depth hypotheses (level 0 of the boost
 * path: reference lib/networks/boost_enerf/network.py:189-201 builds them one chain at a time).  A warped source
 * feature is identical in every chain that uses the view, so each UNIQUE view is gathered once per (voxel, plane).
 * b: as above with view[0..S) = the unique views, planes common to all chains, out = the volume of chain 0;
 * chain_mask[u] bit k = unique view u belongs to chain k; every chain has views_per_chain views; the volume of chain k
 * starts out_k_stride elements after chain k-1's.  Channels-last tensors, C in {16, 32}, K <= 4, exact_coords = 0. */
typedef struct bmv_cost_volume_multi_params {
  bmv_cost_volume_params b;
  int32_t K, views_per_chain;
  int32_t chain_mask[BMV_MAX_VIEWS];
  int64_t out_k_stride;
  const int32_t* triples_dev;   /* DEVICE (K, views_per_chain) or NULL.  When set: b.S = the number of source views N,
                                   "unique view" u IS source view u (b.view / chain_mask ignored) and the chain masks are
                                   derived in the kernel from this table; views used by no chain are skipped. */
} bmv_cost_volume_multi_params;
BMV_API int bmv_cost_volume_var_multi(const bmv_cost_volume_multi_params* p, bmv_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * a3  depth hypotheses.
 * bmv_depth_planes_first: reference lib/networks/enerf/utils.py:103-111,149-153 — D planes shared by
 *   all pixels: planes (D,) and near_far (2,h,w).  `t` = torch.linspace(0,1,D) (DEVICE, taken from
 *   torch rather than recomputed so both sides share the same rounding).
 * bmv_depth_planes_next: reference lib/networks/enerf/utils.py:112-153 — bilinear (align_corners)
 *   upsample of the previous level's depth/std/near_far (disparities), clamp, invert, per-pixel planes.
 */
typedef struct bmv_depth_planes_first_params {
  const float* near_far;        /* DEVICE (2,) scene near, far */
  const float* t;               /* DEVICE (D,) */
  int32_t D, h, w, depth_inv;
  float* planes;                /* (D,) */
  float* near_far_out;          /* (2,h,w) */
} bmv_depth_planes_first_params;
BMV_API int bmv_depth_planes_first(const bmv_depth_planes_first_params* p, bmv_stream_t stream);

typedef struct bmv_depth_planes_next_params {
  const float* depth;           /* (h0,w0) previous level expectation (a disparity) */
  const float* std;             /* (h0,w0) */
  const float* near_far;        /* (2,h0,w0) previous level near/far (disparities) */
  const float* t;               /* DEVICE (D,) */
  int32_t h0, w0, h, w, D, cur_inv;
  float* planes;                /* (D,h,w) */
  float* near_far_out;          /* (2,h,w) */
  /* batch > 1: `batch` chains in one launch; chain b reads depth + b*depth_b_stride, std + b*std_b_stride,
   * near_far + b*nf_b_stride (0 = shared) and writes planes + b*D*h*w, near_far_out + b*2*h*w.  0/1 = single. */
  int32_t batch;
  int64_t depth_b_stride, std_b_stride, nf_b_stride;
} bmv_depth_planes_next_params;
BMV_API int bmv_depth_planes_next(const bmv_depth_planes_next_params* p, bmv_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * K2  depth regression: softmax over D, expectation and standard deviation.
 * Replaces depth_regression (reference lib/networks/enerf/utils.py:722-727).
 */
typedef struct bmv_depth_regression_params {
  const float* logits;          /* (D,h,w) */
  const float* planes;          /* per-pixel (D,h,w) or shared (D,) */
  int64_t planes_d_stride, planes_pix_stride;
  int32_t D, h, w, depth_inv;
  float* depth;                 /* (h,w) */
  float* std;                   /* (h,w) */
  /* batch > 1: `batch` chains in one launch; chain b reads logits + b*logits_b_stride and planes +
   * b*planes_b_stride (0 = shared) and writes depth + b*h*w, std + b*h*w.  0/1 = single. */
  int32_t batch;
  int64_t logits_b_stride, planes_b_stride;
} bmv_depth_regression_params;
BMV_API int bmv_depth_regression(const bmv_depth_regression_params* p, bmv_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * K3  depth-guided ray generation + sampling + feature fetch + 3-D visibility, fused.
 * Replaces build_rays, sample_along_depth, get_vox_feat, unpreprocess(scale 1), get_img_feat,
 * get_ndc_coords, mask_viewport (reference lib/networks/enerf/utils.py:392-443,458-460,490-520,
 * 669-676,753-786) and the glue of render_rays (reference lib/networks/boost_enerf/network.py:123-149).
 * One launch handles rays [ray_begin, ray_begin+n_rays) of one cost-volume chain.
 */
typedef struct bmv_raygen_fetch_params {
  /* per-pixel maps at VOLUME resolution (hv,wv), upsampled on the fly to the render grid (H,W) */
  const float* depth; const float* std; const float* near_far;   /* (hv,wv),(hv,wv),(2,hv,wv) */
  int32_t hv, wv, H, W;         /* H,W = render grid = int(H_img*render_scale) */
  int32_t depth_inv;            /* cfg.enerf.cas_config.depth_inv[level] */
  const float* rays;            /* (R,8) [o,d,x,y] */
  int64_t ray_begin, n_rays;
  /* alternative input modes for function-level use (normally NULL):
   *   rays12_in (R,12): rays that already carry [ray_near ray_far vol_near vol_far] (sample_along_depth)
   *   xyz_in (n_rays,3) [+ uvd_in (n_rays,3) normalised to [0,1]]: explicit points, one per "ray", S ignored
   *     (get_vox_feat / get_img_feat / mask_viewport on arbitrary points) */
  const float* rays12_in; const float* xyz_in; const float* uvd_in;
  /* on-device ray generation (SURVEY.md §8 f3; replaces the (R,8) tensor of
   * lib/datasets/enerf_utils.py:62-71 when rays == NULL): DEVICE, 12 doubles = camera origin (3) followed
   * by the 3x3 matrix M = inv(K)^T R_c2w^T (row-major); ray r is pixel (x, y) = (r % W, r / W) of the
   * render grid, direction = [x, y, 1] M evaluated in fp64 and rounded once to fp32 like the loader. */
  const double* ray_gen;
  const float* t; int32_t S;    /* DEVICE (S,) sample fractions; S==1 -> midpoint (t ignored) */
  /* regularised feature volume (Cv=8 channels) */
  const float* volume; int32_t Cv, Dv;                 /* spatial size = (hv,wv) */
  int64_t vol_c_stride, vol_d_stride, vol_y_stride, vol_x_stride;
  /* per-view image features + colours */
  int32_t V; int32_t view[BMV_MAX_VIEWS];
  const float* im_feat; int32_t Cf; int32_t Hf, Wf;    /* (N,Cf,Hf,Wf)-like with strides below */
  int64_t imf_view_stride, imf_c_stride, imf_y_stride, imf_x_stride;
  const float* rgb;             /* (N,3,Hf,Wf); strides: rgb_view_stride + rgb_{c,y,x}_stride at the end of the struct */
  int64_t rgb_view_stride;
  float rgb_scale, rgb_shift;   /* colour = rgb*scale+shift (0.5,0.5 folds unpreprocess; 1,0 if pre-resized) */
  /* cameras, DEVICE memory */
  const float* src_exts;        /* (N,4,4) world->cam */
  const float* src_ixts;        /* (N,3,3) full-resolution intrinsics (visibility uses them unscaled) */
  const float* src_centers;     /* (N,3) = inverse(ext)[:3,3] */
  const float* tar_center;      /* (3,) */
  float render_scale;           /* intrinsics rows 0,1 scaled by this for the colour fetch */
  /* outputs (any may be NULL to skip) */
  float* rays12;                /* (n_rays,12)  build_rays output */
  float* z_vals;                /* (n_rays,S) */
  float* xyz;                   /* (n_rays,S,3) */
  float* uvd;                   /* (n_rays,S,3) [pixel x, pixel y, normalised depth] */
  float* vox_feat;              /* (n_rays*S,Cv) */
  float* img_feat;              /* (n_rays*S,V,Cf+3+4) */
  float* vis_mask;              /* (n_rays,S) fp32 count/V */
  int32_t* vis_count;           /* (n_rays,S) integer count */
  /* rgb element strides (floats).  All zero = planar contiguous (c: Hf*Wf, y: Wf, x: 1).  A channels-last
   * (N,H,W,4) image (c: 1, x: 4) lets the fused render kernels fetch a tap with one 16-byte load. */
  int64_t rgb_c_stride, rgb_y_stride, rgb_x_stride;
} bmv_raygen_fetch_params;
BMV_API int bmv_raygen_sample_fetch(const bmv_raygen_fetch_params* p, bmv_stream_t stream);

/* Stand-alone 3-D visibility of given world points (op-level parity with mask_viewport,
 * reference lib/networks/enerf/utils.py:490-520). */
typedef struct bmv_visibility_params {
  const float* xyz; int64_t n_pts;                     /* (n_pts,3) */
  int32_t V; int32_t view[BMV_MAX_VIEWS];
  const float* src_exts; const float* src_ixts;        /* (N,4,4), (N,3,3) DEVICE */
  float inv_scale_x, inv_scale_y;                      /* (W-1, H-1) */
  float* vis_mask; int32_t* vis_count;                 /* (n_pts,) each, either may be NULL */
} bmv_visibility_params;
BMV_API int bmv_mask_viewport(const bmv_visibility_params* p, bmv_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * K4  alpha compositing.
 * bmv_composite_blend replaces merge_mlp_outputs + raw2outputs_blend (reference
 *   lib/networks/boost_enerf/network.py:163-170, lib/networks/enerf/utils.py:639-667): takes K
 *   pointers, no stacking.  Also emits the visibility-weighted 2-D coverage when asked.
 * bmv_composite replaces raw2outputs (reference lib/networks/enerf/utils.py:605-637).
 */
typedef struct bmv_composite_blend_params {
  int32_t K, S; int64_t R;
  const float* raw[BMV_MAX_VOLUMES];    /* each (R,S,4) [rgb,sigma] */
  const float* mask[BMV_MAX_VOLUMES];   /* each (R,S) un-normalised visibility score */
  const float* z[BMV_MAX_VOLUMES];      /* each (R,S) */
  float* rgb;                           /* (R,3) */
  float* depth;                         /* (R,) */
  float* weights;                       /* (R,S) */
} bmv_composite_blend_params;
BMV_API int bmv_composite_blend(const bmv_composite_blend_params* p, bmv_stream_t stream);

typedef struct bmv_composite_params {
  int32_t S; int64_t R;
  const float* raw;                     /* (R,S,4) */
  const float* z;                       /* (R,S) or NULL */
  int32_t white_bkgd;
  float* rgb; float* depth; float* weights;
} bmv_composite_params;
BMV_API int bmv_composite(const bmv_composite_params* p, bmv_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * K5  fused per-sample MLP (SURVEY.md §8 row f2).
 * Replaces NeRF.forward + Agg.forward (reference lib/networks/enerf/nerf.py:29-43,73-89) for
 * feat_ch = nerf_model_feat_ch+3 and V views: one thread per sample, fp32 FMA, weights packed by the
 * host (layout in csrc/nerf_mlp.cuh; bmv_nerf_mlp_weight_count gives the packed length or -1).
 */
typedef struct bmv_nerf_mlp_params {
  const float* vox_feat;        /* (P,8) */
  const float* img_feat;        /* (P,V,feat_ch+4) */
  const float* weights;         /* packed, DEVICE, 16-byte aligned */
  int64_t P; int32_t feat_ch, V;
  float* raw;                   /* (P,4) [r,g,b,sigma] */
} bmv_nerf_mlp_params;
BMV_API int bmv_nerf_mlp(const bmv_nerf_mlp_params* p, bmv_stream_t stream);
BMV_API int bmv_nerf_mlp_weight_count(int feat_ch);

/* ------------------------------------------------------------------------------------------
 * K3+K5 fused per-chain render: ray generation + sampling + gather + visibility + MLP in one launch
 * (replaces render_rays, reference lib/networks/boost_enerf/network.py:123-149, without ever
 * materialising vox_feat / img_feat_rgb_dir).  `g` carries the K3 inputs (fused or rays12_in mode);
 * of its outputs only z_vals, vis_mask and vis_count are honoured.  raw is (n_rays,S,4).
 * bmv_render_rays_supported tells whether a (Cv,Cf,V) combination is instantiated; callers fall
 * back to bmv_raygen_sample_fetch + the cuBLAS modules otherwise.
 */
typedef struct bmv_render_rays_params {
  bmv_raygen_fetch_params g;
  const float* mlp_weights;     /* packed (csrc/nerf_mlp.cuh), DEVICE, 16-byte aligned */
  float* raw;                   /* (n_rays,S,4) [r,g,b,sigma], 16-byte aligned */
} bmv_render_rays_params;
BMV_API int bmv_render_rays(const bmv_render_rays_params* p, bmv_stream_t stream);
BMV_API int bmv_render_rays_supported(int Cv, int Cf, int V);
/* Tensor-core variant (csrc/render_mma.cu): same contract, every Linear layer on warp-level MMAs
 * (fp16 hi/lo split operands, fp32 accumulate, ~1e-6 agreement with the fp32-FMA kernel);
 * mlp_weights must come from the MMA packing (bmv_render_rays_mma_weight_words 32-bit words).
 * Instantiated for Cv=8, Cf=8, V=3 (the ENeRF level-1 MLP). */
BMV_API int bmv_render_rays_mma(const bmv_render_rays_params* p, bmv_stream_t stream);
BMV_API int bmv_render_rays_mma_weight_words(void);
/* 5th-generation tensor-core variant (csrc/render_umma.cu): same contract and the same split-fp16 arithmetic,
 * every Linear layer issued as tcgen05.mma on 128-sample tiles (operands in shared memory in the UMMA
 * K-major layout, accumulators in tensor memory, read back with tcgen05.ld); two tiles ping-pong per CTA.
 * mlp_weights must come from the UMMA packing (bmv_render_rays_umma_weight_words 32-bit words). */
BMV_API int bmv_render_rays_umma(const bmv_render_rays_params* p, bmv_stream_t stream);
BMV_API int bmv_render_rays_umma_weight_words(void);
/* Unit test hook for the tcgen05 plumbing (descriptors, TMEM allocation, commit, tcgen05.ld):
 * D (128,N) fp32 = A (128,K) fp32 . B^T, B (N,K) given as [hi block][lo block] of (K/8,N,8) fp16
 * (mlp_pack.pack_umma_matrix); N % 16 == 0, 16 <= N <= 256, K % 16 == 0, K <= 96.  Device pointers. */
BMV_API int bmv_umma_selftest(const float* A, const void* B_packed, float* D, int N, int K, bmv_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * K1b  MVSNeRF cost volume with colour channels.
 * Replaces build_volume_costvar_img + homo_warp(pad) (reference lib/networks/mvsnerf/network.py:887-942,
 * lib/networks/mvsnerf/utils.py:580-630).  View view[0] is the reference view (unwarped, zero-padded by
 * `pad` pixels); out = (3V + C, D, h+2pad, w+2pad): [ref rgb | warped src rgb x(V-1) | feature variance
 * over the views whose strict in-mask holds].  Channels 0:3 are 0 in the border (the reference leaves
 * them uninitialised, SURVEY.md §10.12).
 */
typedef struct bmv_cost_volume_img_params {
  const float* feat;            /* (N,C,h,w)-like feature maps, strides below */
  int64_t feat_view_stride, feat_c_stride, feat_y_stride, feat_x_stride;
  const float* img;             /* (N,3,h,w) planar: source images resized to the feature grid */
  int32_t view[BMV_MAX_VIEWS];
  int32_t V, C, h, w, D, pad;
  const float* proj;            /* DEVICE (V,3,4) in TRIPLE order; row 0 (reference) unused */
  const float* planes;          /* DEVICE (D,) */
  float* out;
  int64_t out_c_stride, out_d_stride, out_y_stride, out_x_stride;
  int32_t out_bf16;
} bmv_cost_volume_img_params;
BMV_API int bmv_cost_volume_var_img(const bmv_cost_volume_img_params* p, bmv_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * K3b  MVSNeRF ray marching + fetch: builds the 86-wide MLP input of every sample.
 * Replaces ray_marcher, get_ndc_coordinate(pad), index_point_feature, build_color_volume,
 * gen_dir_feature, Embedder.embed, run_network_mvs and mask_viewport (reference
 * lib/networks/mvsnerf/network.py:945-1001, utils.py:112-146,300-383, renderer.py:111-137,
 * lib/networks/boost_mvsnerf/network.py:97-135).  near/far of a ray are its columns 6,7.
 */
typedef struct bmv_mvs_march_params {
  const float* rays;            /* (R,8) */
  int64_t ray_begin, n_rays;
  const float* t; int32_t S;    /* DEVICE (S,) = torch.linspace(0,1,S) */
  int32_t V; int32_t view[BMV_MAX_VIEWS];              /* view[0] = reference view of the volume */
  const float* src_exts; const float* src_ixts;        /* (N,4,4), (N,3,3) DEVICE */
  int32_t H, W;                 /* image size (render scale 1) */
  float near, far;              /* volume depth range of this chain (NDC z normalisation) */
  int32_t pad;
  const float* volume; int32_t Cv, Dv, hv, wv;         /* regularised volume (8, D, h+2pad, w+2pad) */
  int64_t vol_c_stride, vol_d_stride, vol_y_stride, vol_x_stride;
  const float* rgb;             /* (N,3,H,W) planar source images */
  float rgb_scale, rgb_shift;   /* 0.5,0.5 folds unpreprocess */
  float* mlp_in;                /* (n_rays,S,86) or NULL */
  float* z_vals;                /* (n_rays,S) or NULL */
  float* vis_mask;              /* (n_rays,S) or NULL */
  int32_t* vis_count;           /* (n_rays,S) or NULL */
  int32_t rgb_nhwc4;            /* 1: rgb is (N,H,W,4) [r,g,b,x] instead of planar (one 16-byte load per bilinear tap);
                                   honoured by bmv_mvs_render_umma only */
  int32_t reserved0;
} bmv_mvs_march_params;
BMV_API int bmv_mvs_march_fetch(const bmv_mvs_march_params* p, bmv_stream_t stream);

/* K3b fused with the 6x128 MLP of the MVSNeRF backbone (reference lib/networks/mvsnerf/network.py:152-229 Renderer_ours,
 * :945-1001 marcher, lib/networks/mvsnerf/renderer.py:111-137 feature assembly) on tcgen05 tensor cores: the
 * (n_rays, S, 86) MLP input of bmv_mvs_march_fetch is never materialised.  g as for bmv_mvs_march_fetch (mlp_in ignored;
 * z_vals / vis_mask / vis_count optional); raw (n_rays, S, 4) = [sigmoid rgb (3), relu alpha (1)].
 * fp16 operands, fp32 accumulation, one MMA per product: TF32-class (BASELINE config 3, 1e-2).
 * weights: bmv_mvs_render_umma_weight_bytes() bytes from mlp_pack.pack_mvs_weights_umma. */
typedef struct bmv_mvs_render_params {
  bmv_mvs_march_params g;
  const uint32_t* weights;
  float* raw;
} bmv_mvs_render_params;
BMV_API int bmv_mvs_render_umma(const bmv_mvs_render_params* p, bmv_stream_t stream);
BMV_API int bmv_mvs_render_umma_weight_bytes(void);

/* ------------------------------------------------------------------------------------------
 * Fused top-down step of the feature pyramid: out = up2x(prev) + conv1x1(lateral_in) + bias
 * (`_upsample_add(x, lat(c))`, reference lib/networks/enerf/feature_net.py:24-33).  All tensors
 * channels-last (N,H,W,C) fp32, 32 output channels; prev is (N,H/2,W/2,32); weight (32,Cin) row-major.
 */
typedef struct bmv_fpn_topdown_params {
  const float* prev; const float* lateral_in; const float* weight; const float* bias;
  int32_t N, H, W, Cin;
  float* out;                   /* (N,H,W,32) */
} bmv_fpn_topdown_params;
BMV_API int bmv_fpn_topdown(const bmv_fpn_topdown_params* p, bmv_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Tensor-core 3x3x3 / stride 1 / padding 1 convolution (+bias, optional ReLU) for the full-resolution
 * layers of the kept 3-D cost regularisers: conv0 = ConvBnReLU3D(C,8) and the output heads
 * (reference lib/networks/enerf/cost_reg_net.py:7-13,27-35 MinCostRegNet, 39-62 CostRegNet; BN folded).
 * Operands rounded to fp16, fp32 accumulation: TF32-class accuracy, so hosts route a layer here only
 * where the framework would use TF32 convolutions (torch.backends.cudnn.allow_tf32).
 * x (N,D,H,W,Cin) channels-last fp32 via strides (in floats, multiples of 4); out likewise (any
 * strides, Cout channels written at out + ... + c).  wfrag: bmv_conv3d_k3_weight_words(Cin,Cout)
 * uint32 words in mma B-fragment order [dz][dy][k-step][n-tile][lane][2] (mlp_pack.pack_conv3d_k3; the
 * k-steps of each Cin are described in csrc/conv3d_mma.cu).
 * Instantiated (Cin,Cout<=): (16,8) (16,16) (32,8) (8,16).
 */
typedef struct bmv_conv3d_params {
  const float* x; int64_t x_n_stride, x_d_stride, x_y_stride, x_x_stride;
  const uint32_t* wfrag; const float* bias;   /* bias (Cout) or NULL */
  int32_t N, D, H, W, Cin, Cout, relu;
  float* out; int64_t o_n_stride, o_d_stride, o_y_stride, o_x_stride;
  float* out2; int64_t o2_n_stride, o2_d_stride, o2_y_stride, o2_x_stride;   /* optional: channels >= split */
  int32_t split;                /* with out2: channel c >= split is written to out2 at channel c - split */
  int32_t stride;               /* 0/1: stride 1.  2: stride-2 convolution (Cin=8, Cout<=16; ConvBnReLU3D(8,16,stride=2),
                                   cost_reg_net.py:14,53), out is (N, (D-1)/2+1, (H-1)/2+1, (W-1)/2+1, Cout) */
  int32_t in_half;              /* 1: x points to fp16 storage (strides in fp16 elements, multiples of 8).
                                   The operands are rounded to fp16 in any case, so results are identical.  With
                                   Cin 16 / 32, Cout <= 8 and voxels contiguous along x the input tile is staged by TMA
                                   (one 5-D bulk-tensor copy per CTA, hardware zero fill = the padding). */
  int32_t no_tma;               /* 1: force the register-staged path (A/B testing) */
  int32_t out_half;             /* 1: out points to fp16 storage (strides in fp16 elements; even Cout, no out2): for results
                                   that only feed other fp16-operand libbmv convolutions */
  int32_t reserved0;
  const float* in_scale;        /* DEVICE or NULL: [s, 1/s] written by bmv_volume_scale — x holds s * (the real input); the
                                   accumulator starts at s*bias and the result is multiplied by 1/s (exact: s is a power
                                   of two).  Stride-1 mma.sync kernel only. */
} bmv_conv3d_params;
BMV_API int bmv_conv3d_k3(const bmv_conv3d_params* p, bmv_stream_t stream);
BMV_API int bmv_conv3d_k3_weight_words(int Cin, int Cout);
BMV_API int bmv_conv3d_k3_last_used_tma(void);   /* 1 if this thread's last stride-1 launch staged its tile with TMA */
/* The same convolution on the 5th-generation tensor cores (csrc/conv3d_umma.cu): the halo tile is staged by one
 * 5-D TMA copy, every tap is a tcgen05.mma whose A operand is that tile addressed through a shifted shared-memory
 * descriptor (M = 128 x voxels, N = 16, K = 16), accumulators live in tensor memory.  Same params struct and
 * arithmetic class; requires in_half = 1, stride 1, x_x_stride == Cin, Cin in {8, 16}, Cout <= 16.
 * wfrag: bmv_conv3d_k3_umma_weight_words(Cin,Cout) words in operand order (mlp_pack.pack_conv3d_k3_umma). */
BMV_API int bmv_conv3d_k3_umma(const bmv_conv3d_params* p, bmv_stream_t stream);
BMV_API int bmv_conv3d_k3_umma_weight_words(int Cin, int Cout);

/* ------------------------------------------------------------------------------------------
 * Tensor-core ConvTranspose3d(k=3, stride=2, padding=1, output_padding=1) + bias + skip add:
 *     out = skip + convT(x) + bias
 * the decoder steps `x = conv0 + self.conv11(x)` / `x = conv2 + self.conv9(x)` of the kept cost
 * regularisers (reference lib/networks/enerf/cost_reg_net.py:23-31,40-44,62-70,80-82; BN folded).
 * x (N,D,H,W,Cin) channels-last fp32 (strides in floats); skip/out (N,2D,2H,2W,Cout) channels-last.
 * fp16 operands, fp32 accumulation (TF32-class; same gating as bmv_conv3d_k3).
 * wfrag: bmv_convT3d_k3s2_weight_words(Cin,Cout) words, B-fragment order [tap][k-tile][n-tile][lane][2]
 * (mlp_pack.pack_convT3d_k3s2).  Instantiated (Cin,Cout): (16,8) (32,16).
 */
typedef struct bmv_convT3d_params {
  const float* x; int64_t x_n_stride, x_d_stride, x_y_stride, x_x_stride;
  const uint32_t* wfrag; const float* bias;   /* bias (Cout) or NULL */
  int32_t N, D, H, W, Cin, Cout;              /* D,H,W: INPUT size */
  const float* skip; int64_t s_n_stride, s_d_stride, s_y_stride, s_x_stride;   /* or NULL */
  float* out; int64_t o_n_stride, o_d_stride, o_y_stride, o_x_stride;
  int32_t out_half;             /* 1: out points to fp16 storage (strides in fp16 elements): the result only feeds another
                                   fp16-operand convolution (the merged heads), so nothing is lost */
  int32_t skip_half;            /* 1: skip points to fp16 storage (strides in fp16 elements) */
  int32_t in_half;              /* 1: x points to fp16 storage (strides in fp16 elements, multiples of 8) */
} bmv_convT3d_params;
BMV_API int bmv_convT3d_k3s2(const bmv_convT3d_params* p, bmv_stream_t stream);
BMV_API int bmv_convT3d_k3s2_weight_words(int Cin, int Cout);

/* ------------------------------------------------------------------------------------------
 * 3x3x3 convolutions of the LOW-RESOLUTION core of the 3-D cost regularisers on tensor cores (fp16 operands, fp32
 * accumulation: TF32-class, same gating as bmv_conv3d_k3): conv3 / conv4 / conv5 / conv6 (padding 1, stride 1 or 2,
 * + bias, + ReLU) and the transposed conv7 (kernel 3, stride 2, padding 1, output_padding 1, + bias, + skip)
 * (reference lib/networks/enerf/cost_reg_net.py:14-24,58-75; BN folded by the caller).  Volumes of a few 10 k voxels: a
 * direct implicit GEMM without a staged tile (csrc/conv3d_small.cu).
 *   x     fp16 channels-last-3d (N,D,H,W,Cin) via strides (elements)
 *   out   DENSE channels-last-3d (N,Do,Ho,Wo,Cout), fp16 (out_half) or fp32; Do = (D-1)/stride + 1, transposed: 2D
 *   skip  optional DENSE fp16 tensor of out's shape, added after the bias (before the ReLU), or NULL
 *   wfrag bmv_conv3d_small_weight_words(Cin, Cout, transposed) words, order [tap = (kd*3+ky)*3+kx][k-step][n-tile][lane][2]
 *         (mlp_pack.pack_conv3d_small); for the transposed layer tap k maps input i to output 2i - 1 + k.
 * Instantiated: 16 -> 32, 32 -> 32, 32 -> 64, 64 -> 64; transposed 64 -> 32.
 */
typedef struct bmv_conv3d_small_params {
  const void* x; int64_t x_n_stride, x_d_stride, x_y_stride, x_x_stride;
  int32_t N, D, H, W, Cin, Cout;
  int32_t stride, transposed, relu, out_half;
  const uint32_t* wfrag; const float* bias;
  const void* skip;
  void* out;
} bmv_conv3d_small_params;
BMV_API int bmv_conv3d_small(const bmv_conv3d_small_params* p, bmv_stream_t stream);
BMV_API int bmv_conv3d_small_weight_words(int Cin, int Cout, int transposed);

/* ------------------------------------------------------------------------------------------
 * Fused top-down step + 3x3 smoothing convolution of the feature pyramid:
 *     mid = up2x(prev) + conv1x1(lateral_in) + lat_bias   (32 channels; as bmv_fpn_topdown, exact fp32)
 *     out = conv3x3(mid, padding 1) + bias                 (Cout = 8 or 16)
 * (`_upsample_add` + `smooth0/smooth1`, reference lib/networks/enerf/feature_net.py:24-47.)
 * The 3x3 convolution uses fp16 operands / fp32 accumulation (TF32-class; same gating as bmv_conv3d_k3).
 * All tensors channels-last fp32; mid (N,H,W,32) is written only when non-NULL.
 * wfrag: bmv_fpn_topdown_smooth_weight_words(Cout) words, order [dy][dx*2+half][n-tile][lane][2]
 * (mlp_pack.pack_conv2d_k3_c32).
 */
typedef struct bmv_fpn_fused_params {
  const float* prev; const float* lateral_in; const float* lat_weight; const float* lat_bias;
  const uint32_t* wfrag; const float* bias;
  int32_t N, H, W, Cin, Cout;
  float* mid;                   /* (N,H,W,32) or NULL */
  float* out;                   /* (N,H,W,Cout), or NULL when only out16 is wanted */
  void* out16;                  /* optional fp16 version of out, (N,H,W,Cout) (for the cost-volume kernel's fp16 tap loads), or NULL */
  int32_t lat_half;             /* 1: lateral_in points to fp16 storage (N,H,W,Cin) */
  int32_t reserved0;
} bmv_fpn_fused_params;
BMV_API int bmv_fpn_topdown_smooth(const bmv_fpn_fused_params* p, bmv_stream_t stream);
BMV_API int bmv_fpn_topdown_smooth_weight_words(int Cout);

/* ------------------------------------------------------------------------------------------
 * 3x3 / pad-1 convolution (+bias, +ReLU) of the 2-D feature pyramid's middle layers on tensor cores (fp16 operands,
 * fp32 accumulation: TF32-class, same gating as bmv_conv3d_k3): conv1.x / conv2.x and, fused behind conv2.1, the 1x1 top
 * layer (reference lib/networks/enerf/feature_net.py:10-21,29-31; BN folded by the caller).
 *   x    channels-last input.  in_half = 1, s2d = 0: fp16 (N,H,W,Cin).  s2d = 1: fp32 or fp16 (N,2H,2W,Cin/4) read
 *        through space-to-depth(2) — conv channel (py*2 + px) * Cin/4 + c is source pixel (2y+py, 2x+px), channel c: a
 *        5x5 / stride-2 / pad-2 layer regrouped as a 3x3 one (weights zero-padded to 6x6, mlp_pack.pack_conv2d_k3).
 *   out  channels-last (N,H,W,Cout), fp32 or fp16 (out_half).
 *   wfrag: bmv_conv2d_k3_weight_words(Cin, Cout) words in B-fragment order [dy][k-step][n-tile][lane][2] with the output
 *        channels permuted across the n-tiles (mlp_pack.pack_conv2d_k3); bias (Cout) by channel, or NULL.
 *   wfrag1x1 / bias1x1 / C1x1_out: optional fused 1x1 convolution applied to relu(conv) (mlp_pack.pack_conv1x1_after);
 *        out is then (N,H,W,C1x1_out) fp32 and the 3x3 result is never stored.
 * Instantiated: (Cin 32 -> 16, s2d), (64 -> 32, s2d), (16 -> 16, fp16 dense), (32 -> 32, fp16 dense [+ 1x1 32 -> 32]).
 */
typedef struct bmv_conv2d_params {
  const void* x; int64_t x_n_stride, x_y_stride, x_x_stride;   /* elements of x's dtype */
  int32_t N, H, W, Cin, Cout;
  int32_t s2d, in_half, out_half, relu;
  int32_t C1x1_out;
  const uint32_t* wfrag; const float* bias;
  void* out; int64_t o_n_stride, o_y_stride, o_x_stride;
  const uint32_t* wfrag1x1; const float* bias1x1;
} bmv_conv2d_params;
BMV_API int bmv_conv2d_k3(const bmv_conv2d_params* p, bmv_stream_t stream);
BMV_API int bmv_conv2d_k3_weight_words(int Cin, int Cout);

/* ------------------------------------------------------------------------------------------
 * Fused stem of the feature pyramid: ConvBnReLU(3,8,3) -> ConvBnReLU(8,8,3) at full resolution
 * (reference lib/networks/enerf/feature_net.py:7-9,29; BN folded).  x: (N,3,H,W) fp32 via strides (any
 * layout); w0 (8,3,3,3) fp32 row-major + b0 (8); wfrag1: 384 words = the 8->8 weights in B-fragment
 * order [dy][k-step][lane][2] (mlp_pack.pack_conv2d_k3_c8) + b1 (8); out (N,H,W,8) channels-last fp32.
 * First layer fp32 on CUDA cores, second on tensor cores with fp16 operands (TF32-class gating).
 */
typedef struct bmv_fpn_stem_params {
  const float* x; int64_t x_n_stride, x_c_stride, x_y_stride, x_x_stride;
  const float* w0; const float* b0;
  const uint32_t* wfrag1; const float* b1;
  int32_t N, H, W;
  float* out;
  float* rgb4;                  /* optional by-product: x as (N,H,W,4) channels-last [r,g,b,0] (see rgb_*_stride of
                                   bmv_raygen_fetch_params), or NULL */
  float* out_s2d;               /* optional second copy of the output in space-to-depth(2) layout (N,H/2,W/2,32), channel
                                   (y&1)*16 + (x&1)*8 + c: the input of the regrouped 5x5/stride-2 conv1.0; H, W even; or NULL */
  int32_t out_half;             /* 1: out points to fp16 storage (N,H,W,8): its consumers (bmv_conv2d_k3, the lateral of
                                   bmv_fpn_topdown_smooth) round it to fp16 anyway; out_s2d must be NULL */
  int32_t reserved0;
} bmv_fpn_stem_params;
BMV_API int bmv_fpn_stem(const bmv_fpn_stem_params* p, bmv_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * K3+K5 for ALL K cost-volume chains of a frame in one persistent launch (csrc/render_multi.cu): the per-chain loop of
 * reference lib/networks/boost_enerf/network.py:212-222 (render_rays of chain k = 0..K-1) as one kernel.
 * g: the fields shared by the chains — rays / ray_gen, ray_begin, n_rays, H, W, hv, wv, depth_inv, t, S, the volume
 *    GEOMETRY (Cv, Dv, vol_*_stride), V, im_feat, rgb, cameras, render_scale; its depth / std / near_far / volume / view
 *    and output pointers are ignored.
 * Chain k reads depth + k*depth_k_stride (hv,wv), std likewise, near_far + k*nf_k_stride (2,hv,wv; stride 0 = shared),
 * volume + k*vol_k_stride, and views[3k..3k+2] — DEVICE memory when `views` is set (a captured graph then follows a
 * changed view selection by rewriting 3K ints), else views_host.  n_views = number of source views behind src_exts.
 * Outputs are K-stacked: raw (K,n_rays,S,4), z_vals / vis_mask / vis_count (K,n_rays,S) (the last three optional).
 * Requires Cv = Cf = 8, V = 3, dense channels-last volumes / feature maps, (N,Hf,Wf,4) colours, < 2^31 elements.
 * mlp_weights: mlp_pack.pack_nerf_weights_mma (bmv_render_rays_mma_weight_words words).
 */
typedef struct bmv_render_multi_params {
  bmv_raygen_fetch_params g;
  int32_t K, n_views;
  const float* depth; int64_t depth_k_stride;
  const float* std; int64_t std_k_stride;
  const float* near_far; int64_t nf_k_stride;
  const float* volume; int64_t vol_k_stride;
  const int32_t* views;                            /* DEVICE (K,3) or NULL */
  int32_t views_host[BMV_MAX_VOLUMES * 3];
  const uint32_t* mlp_weights;
  float* raw; float* z_vals; float* vis_mask; int32_t* vis_count;
  /* Row slabs (multi-GPU row tiles: a rank holds only the volume / map rows its rays touch): `volume` points at volume
   * row vol_row0 and `depth` / `std` / `near_far` at map row map_row0 (rows outside the slab must not be needed by
   * rays [ray_begin, ray_begin + n_rays)); g.vol_d_stride is then the slab's plane stride and nf_plane_stride the
   * distance between the two near_far planes (0: hv * wv).  All zero for whole tensors. */
  int32_t vol_row0, map_row0;
  int64_t nf_plane_stride;
} bmv_render_multi_params;
BMV_API int bmv_render_rays_multi(const bmv_render_multi_params* p, bmv_stream_t stream);
/* Same contract with the MLP on the 5th-generation tensor cores (csrc/render_multi_umma.cu: tcgen05.mma, accumulators in
 * tensor memory, a dedicated issuer warp, two threads per sample row); mlp_weights: mlp_pack.pack_nerf_weights_umma
 * (bmv_render_rays_umma_weight_words words).  z / visibility bit-identical to bmv_render_rays_multi, raw to ~1e-5. */
BMV_API int bmv_render_rays_multi_umma(const bmv_render_multi_params* p, bmv_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * f4  output sinks: what the reference's evaluator / visualiser consume, produced on the device.
 * bmv_frame_psnr_accumulate: reference lib/evaluators/enerf.py:45-71 — pred / gt (H*W,3) fp32 row-major, optional
 *   mask (H*W) uint8 (pixel counted when mask >= 1), optional centre crop (rows [crop_h, H-crop_h), columns
 *   [crop_w, W-crop_w); the reference uses int(0.1*h), int(0.1*w) under cfg.enerf.eval_center).  Adds the sum of
 *   squared differences (float64) to *sse and the number of compared ELEMENTS (3 per pixel) to *count; the caller
 *   zeroes them.  PSNR = 10 log10(1 / (sse / count)) (skimage.metrics.peak_signal_noise_ratio, data_range 1).
 * bmv_frame_to_u8: reference lib/visualizers/enerf.py:27-37 — rgb_u8 = (rgb * 255).astype(uint8);
 *   depth_u8 = ((depth - min) / (max - min) * 255).astype(uint8), min / max over the frame written to minmax[0..1]
 *   (optional).  minmax_ord: 2 words of device scratch.
 * bmv_frame_ssim: the SSIM the reference's evaluator takes from skimage, structural_similarity(gt, pred,
 *   channel_axis=-1, win_size, data_range) with uniform weights (scikit-image 0.19 / 0.20).  pred / gt (H*W,3) fp32
 *   row-major, optional centre crop as above (the metric then sees only the cropped image).  Per channel: box means
 *   ux, uy, uxx, uyy, uxy over the win_size x win_size window, v = w²/(w²-1) * (second moment - product of means),
 *   S = (2 ux uy + C1)(2 vxy + C2) / ((ux² + uy² + C1)(vx + vy + C2)), C1 = (0.01 R)², C2 = (0.03 R)², averaged over
 *   the pixels whose window lies inside the image; *ssim = mean of the three channel values.  All in float64.
 *   win_size odd, >= 3 and <= both cropped sides; data_range > 0.  The reference does not record its arguments:
 *   skimage's defaults for a float image are win_size 7 and data_range 2 (dtype range (-1, 1)).
 *   scratch: BMV_FRAME_SSIM_SCRATCH_WORDS doubles of device scratch (per-CTA partials, summed in a fixed order: two
 *   launches on the same inputs give the same bits).
 */
#define BMV_FRAME_SSIM_SCRATCH_WORDS 2048
typedef struct bmv_frame_psnr_params {
  const float* pred; const float* gt; const uint8_t* mask;   /* mask may be NULL */
  int32_t H, W, crop_h, crop_w;
  double* sse; unsigned long long* count;                    /* DEVICE accumulators */
} bmv_frame_psnr_params;
BMV_API int bmv_frame_psnr_accumulate(const bmv_frame_psnr_params* p, bmv_stream_t stream);

typedef struct bmv_frame_to_u8_params {
  int64_t R;
  const float* rgb; uint8_t* rgb_u8;        /* (R,3) each, or both NULL */
  const float* depth; uint8_t* depth_u8;    /* (R) each, or both NULL */
  uint32_t* minmax_ord; float* minmax;      /* scratch (2 words); optional output (2 floats) */
} bmv_frame_to_u8_params;
BMV_API int bmv_frame_to_u8(const bmv_frame_to_u8_params* p, bmv_stream_t stream);

typedef struct bmv_frame_ssim_params {
  const float* pred; const float* gt;
  int32_t H, W, crop_h, crop_w;
  int32_t win_size, reserved0;
  double data_range;
  double* scratch;                          /* DEVICE, BMV_FRAME_SSIM_SCRATCH_WORDS doubles */
  double* ssim;                             /* DEVICE, 1 double: the frame's SSIM */
} bmv_frame_ssim_params;
BMV_API int bmv_frame_ssim(const bmv_frame_ssim_params* p, bmv_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* BMV_H_ */
