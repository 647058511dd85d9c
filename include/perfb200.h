/*
 * perfb200.h -- C-ABI of libperfb200.so: the B200-native (sm_100a) implementation of PeRF's
 * per-ray hot path (equirect ray-gen -> fixed-S sampling -> hash-grid encode + 64-wide MLP ->
 * alpha composite, forward and backward, + fused Adam).
 *
 * Boundary rules (SURVEY.md section 8b):
 *   - extern "C", plain C types; no torch / pybind types cross this boundary.
 *   - Every pointer named d_* is a DEVICE pointer owned by the caller; h_* is a host pointer.
 *   - Every entry point enqueues work on `stream` (a cudaStream_t passed as void*) of the
 *     CURRENT device and returns without synchronising.  The library never allocates.
 *   - Return value: PERF_OK (0) or a negative PERF_E* code; perf_last_error() returns a
 *     thread-local human-readable message for the last failure.
 *   - Re-entrant across distinct streams / devices.
 *
 * Each function cites the reference interface it replaces (paths relative to the PeRF
 * repository, perf-project/PeRF @ 1431a35a).  The third-party modules the reference calls on
 * this path (tinycudann 1.7, nerfacc 0.5.3, torch_efficient_distloss 0.1.3) are not vendored;
 * the call sites are cited instead.
 */
#ifndef PERFB200_H
#define PERFB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PERF_ABI_VERSION 1

#define PERF_OK            0
#define PERF_EINVAL       -1   /* bad argument (null pointer, unsupported size, misaligned) */
#define PERF_EUNSUPPORTED -2   /* configuration outside what the kernels implement          */
#define PERF_ECUDA        -3   /* a CUDA runtime call failed (launch error, wrong arch ...)  */

#define PERF_MAX_LEVELS 16

/* encoding_config of tcnn.NetworkWithInputEncoding / tcnn.Encoding as the reference passes it
 * (modules/fields/ngp_nerf.py:99-106,119-126; modules/geo_predictors/pano_joint_predictor.py:30). */
typedef struct perf_grid_cfg {
    uint32_t n_levels;              /* <= PERF_MAX_LEVELS                       */
    uint32_t n_features_per_level;  /* must be 2                                */
    uint32_t log2_hashmap_size;
    uint32_t base_resolution;
    float    per_level_scale;
    uint32_t interpolation;         /* 0 = Linear, 1 = Smoothstep               */
} perf_grid_cfg;

typedef struct perf_level {
    float    scale;        /* exp2f(l*log2f(s))*base - 1                       */
    uint32_t resolution;   /* ceilf(scale) + 1                                 */
    uint32_t size;         /* entries in the level                             */
    uint32_t offset;       /* first entry of the level in the flat table       */
    uint32_t hashed;       /* 1: xor-prime hash, 0: dense x-fastest indexing   */
} perf_level;

/* network_config of tcnn FullyFusedMLP (ngp_nerf.py:107-113,127-133): bias-free, ReLU hidden. */
typedef struct perf_mlp_cfg {
    uint32_t n_in;               /* must be 32 (= 16 levels x 2 features)       */
    uint32_t n_out;              /* 1..16; last matrix is stored padded to 16 rows */
    uint32_t n_neurons;          /* must be 64                                  */
    uint32_t n_hidden_layers;    /* 1 or 2                                      */
    uint32_t output_activation;  /* 0 = None, 1 = Sigmoid                       */
} perf_mlp_cfg;

/* flags of the render / field entry points */
#define PERF_FLAG_TRAINING   1u   /* stratified jitter + training background rule        */
#define PERF_FLAG_SIMT_MLP   2u   /* debug only: MLP on CUDA cores instead of tcgen05     */
#define PERF_FLAG_GENERIC_ADDR 8u  /* render: disable the specialised (4 dense + hashed pow2) addressing path */
#define PERF_FLAG_L0_SMEM 16u      /* render_pano (measured variant, profiles/r02_render_variants.md): level 0 of the table staged into
                                      shared memory by one cp.async.bulk per CTA, 3 CTAs/SM instead of 4 */
#define PERF_FLAG_SCAN_KERNEL 4u   /* render: samples-along-lanes kernel (warp-shuffle scan composite) instead of ray marching */

int         perf_abi_version(void);
const char* perf_last_error(void);
/* compute capability of the current device as major*10+minor (100 on B200), or <0 */
int         perf_device_arch(void);

/* Level/offset table of a grid config (tcnn GridEncodingTemplated ctor; SURVEY.md Appendix A).
 * h_levels: n_levels entries (may be NULL); h_n_entries: total table entries (may be NULL). */
int perf_grid_describe(const perf_grid_cfg* cfg, perf_level* h_levels, uint64_t* h_n_entries);
/* Length of the flat `params` vector of a network (MLP matrices, then the grid). */
int perf_network_param_count(const perf_grid_cfg* grid, const perf_mlp_cfg* mlp, uint64_t* h_count);

/* fp32 master params -> fp16 shadow, n elements (replaces the per-forward `params.to(half)` of
 * the tcnn torch binding; ngp_nerf.py:142,158 call sites). */
int perf_params_to_half(const float* d_params, void* d_params_half, uint64_t n, void* stream);

/* Interleave the two fp16 grid tables into one {geo.f0,geo.f1,app.f0,app.f1} table so one
 * 8-byte gather serves both fields.  d_*_params_half: full fp16 params of each network.
 * Layout of d_packed (8-byte entries, 16-byte aligned buffer): entries [0, n_entries) in parameter order,
 * followed by a cell-major copy of the leading dense levels (up to four; for each, res^3 cells x the 8 corner
 * entries of the cell = one 64-byte record per cell) which the fused field kernels read with four 16-byte
 * loads per sample and level.  perf_packed_table_entries gives the total entry count to allocate. */
int perf_packed_table_entries(const perf_grid_cfg* cfg, uint64_t* h_entries);
int perf_pack_tables(const perf_grid_cfg* grid, const perf_mlp_cfg* geo_mlp, const perf_mlp_cfg* app_mlp,
                     const void* d_geo_params_half, const void* d_app_params_half,
                     void* d_packed /* perf_packed_table_entries() * 8 bytes */, void* stream);

/* Equirect rays for image rows [row0,row0+rows) of an H x W panorama; h_pose: row-major 4x4
 * camera-to-world.  d_rays_o/d_rays_d: [rows*W,3] fp32.
 * Replaces utils/camera_utils.py:229-234 gen_pano_rays (+ :113-155). */
int perf_raygen_pano(const float* h_pose, int H, int W, int row0, int rows,
                     float* d_rays_o, float* d_rays_d, void* stream);

/* Perspective (OpenCV-style) rays of an H x W camera with vertical field of view `fovy` (radians).
 * Replaces utils/camera_utils.py:237-241 gen_pers_rays (+ :60-80 cam_rays_cam_space), the
 * cam_type != 'pano' branch of render_dense (core_exp_runner.py:234-235). */
int perf_raygen_pers(const float* h_pose, float fovy, int H, int W, float* d_rays_o, float* d_rays_d, void* stream);

/* Hash-grid encode forward: d_x01 [N,3] fp32 in [0,1] -> d_feat [N, L*2] fp16.
 * d_table: fp16 [n_entries,2].  Replaces tcnn kernel_grid (Encoding.forward). */
int perf_hashgrid_fwd(const perf_grid_cfg* cfg, const void* d_table, const float* d_x01,
                      uint64_t N, void* d_feat, void* stream);
/* Hash-grid backward w.r.t. the table: d_dtable [n_entries,2] fp32 += scatter(w * dfeat)
 * (caller zeroes it).  d_dfeat [N, L*2] fp32.  Replaces tcnn kernel_grid_backward. */
int perf_hashgrid_bwd(const perf_grid_cfg* cfg, const float* d_x01, const float* d_dfeat,
                      uint64_t N, float* d_dtable, void* stream);

/* Hash-grid backward w.r.t. the INPUT positions: d_dx [N,3] fp32 = sum_f dfeat_f * d feat_f / d x01
 * (Linear and Smoothstep).  d_table_half: fp16 [n_entries,2]; d_dfeat [N, L*2] fp32.
 * Replaces tcnn kernel_grid_backward_input, reached by tcnn.Encoding when its input requires grad
 * (modules/geo_predictors/pano_joint_predictor.py:30-41,48-52; pano_geo_refiner.py:19). */
int perf_hashgrid_bwd_input(const perf_grid_cfg* cfg, const void* d_table_half, const float* d_x01,
                            const float* d_dfeat, uint64_t N, float* d_dx, void* stream);
/* Double backward of perf_hashgrid_bwd_input: with d_ddx [N,3] = d(loss)/d(d_dx), writes the gradient
 * w.r.t. dfeat (d_ddfeat [N, L*2] fp32, overwritten), accumulates the gradient w.r.t. the table
 * (d_dtable [n_entries,2] fp32 +=, caller zeroes) and w.r.t. x01 (d_dx2 [N,3] fp32 +=, caller zeroes).
 * Any of the three outputs may be NULL.  Replaces tcnn kernel_grid_backward_input_backward_dLdoutput /
 * _backward_grid / _backward_input, i.e. what torch.autograd.grad(distance, directions,
 * create_graph=True) followed by loss.backward() runs (pano_joint_predictor.py:58-64). */
int perf_hashgrid_bwd_bwd_input(const perf_grid_cfg* cfg, const void* d_table_half, const float* d_x01,
                                const float* d_dfeat, const float* d_ddx, uint64_t N,
                                float* d_ddfeat, float* d_dtable, float* d_dx2, void* stream);

/* MLP backward from the saved fp16 activations, one tcgen05 kernel (tcnn FullyFusedMLP backward for the two
 * PeRF networks, ngp_nerf.py:107-113,127-133).  d_feat [N,32], d_h1 [N,64], d_h2 [N,64] (two hidden layers,
 * else NULL): fp16 saves of perf_network_fwd / perf_train_forward; d_dz [N,n_out] fp32 = gradient w.r.t. the
 * output pre-activation (n_out <= 3).  d_dweights: fp32 gradient of the flat MLP params, ACCUMULATED (caller
 * zeroes); d_dfeat [N,32] fp32 overwritten.  flags: PERF_FLAG_SIMT_MLP selects the CUDA-core twin.
 * Validated on B200 in round 2; the training steps call it (no library GEMM is left on that path). */
int perf_mlp_bwd(const perf_mlp_cfg* mlp, const void* d_weights_half, const void* d_feat, const void* d_h1, const void* d_h2,
                 const float* d_dz, uint64_t N, const int64_t* d_n_dev /* nullable: live row count in device memory, <= N */,
                 float* d_dweights, float* d_dfeat, uint32_t flags, void* stream);

/* Network forward = encode + MLP fused (tcnn NetworkWithInputEncoding.forward;
 * ngp_nerf.py:142,158).  d_x01 [N,3] fp32; d_params_half: fp16 flat params (MLP | grid);
 * d_out [N, n_out] fp16.  Optional saves for the backward pass (NULL to skip):
 * d_feat [N,32] fp16, d_h1 [N,64] fp16, d_h2 [N,64] fp16 (2-hidden-layer nets only). */
int perf_network_fwd(const perf_grid_cfg* grid, const perf_mlp_cfg* mlp, const void* d_params_half,
                     const float* d_x01, uint64_t N, void* d_out,
                     void* d_feat, void* d_h1, void* d_h2, uint32_t flags, void* stream);

/* MLP forward alone on the tensor cores: d_in [N,32] fp16 -> d_out [N,n_out] fp16
 * (tcnn kernel_mlp_fused).  d_weights_half: the MLP part of the fp16 flat params. */
int perf_mlp_fwd(const perf_mlp_cfg* mlp, const void* d_weights_half, const void* d_in,
                 uint64_t N, void* d_out, void* d_h1, void* d_h2, uint32_t flags, void* stream);

/* Packed transmittance scan (nerfacc render_weight_from_density; nerf_renderer.py:170-171).
 * Samples sorted by ray; d_ray_indices int64 [N].  Outputs fp32 [N] (any may be NULL). */
int perf_weights_from_density(const float* d_t_starts, const float* d_t_ends, const float* d_sigmas,
                              const int64_t* d_ray_indices, uint64_t N, uint64_t n_rays,
                              float* d_weights, float* d_trans, float* d_alphas, void* stream);
/* Backward of the above w.r.t. sigmas given dL/dweights (and optional dL/dtrans). */
int perf_weights_from_density_bwd(const float* d_t_starts, const float* d_t_ends, const float* d_sigmas,
                                  const int64_t* d_ray_indices, uint64_t N, uint64_t n_rays,
                                  const float* d_weights, const float* d_trans,
                                  const float* d_grad_weights, const float* d_grad_trans /*nullable*/,
                                  float* d_grad_sigmas, void* stream);
/* out[r, :] = sum_{i in ray r} w_i * v_i[:]  (nerfacc accumulate_along_rays;
 * nerf_renderer.py:173,175,183).  d_values [N,D] fp32 or NULL (D=1, v=1).  d_out [n_rays,D]
 * is overwritten.  Deterministic (no atomics). */
int perf_accumulate_along_rays(const float* d_weights, const float* d_values, int D,
                               const int64_t* d_ray_indices, uint64_t N, uint64_t n_rays,
                               float* d_out, void* stream);

/* Arguments of the fused renderer (NeRFOCCRenderer.render, nerf_renderer.py:112-209, with the
 * fixed-S sampler; NeRFScene.render, nerf.py:74-99). */
typedef struct perf_render_args {
    perf_grid_cfg grid;           /* both fields use the same grid config (ngp_nerf.py:96-134) */
    const void*   d_packed_table; /* from perf_pack_tables (perf_packed_table_entries() * 8 bytes) */
    const void*   d_geo_mlp_half; /* fp16 MLP matrices of the density net (3072 values)         */
    const void*   d_app_mlp_half; /* fp16 MLP matrices of the colour net  (7168 values)         */
    float         aabb[6];        /* min xyz, max xyz (nerf.py:35)                              */
    uint32_t      n_samples;      /* S                                                          */
    float         near, far;      /* nerf.py:317-318: 1e-2, 1.0                                 */
    uint32_t      flags;          /* PERF_FLAG_*                                                */
    const float*  d_jitter;       /* [R] U[0,1) per-ray offset (training) or NULL               */
    const float*  d_bg_noise;     /* [R,4] training background rgb + distance noise or NULL     */
    float*        d_rgb;          /* [R,3]                                                      */
    float*        d_distance;     /* [R]                                                        */
    float*        d_opacity;      /* [R] or NULL                                                */
    uint32_t      image_width;    /* perf_render_rays only: >0 = the R rays are a row-major image of this
                                     width (locality hint: threads are tiled as 16x8 pixel patches); 0 = no structure */
} perf_render_args;

/* Render explicit rays: d_rays_o / d_rays_d [R,3] fp32. */
int perf_render_rays(const perf_render_args* args, const float* d_rays_o, const float* d_rays_d,
                     uint64_t R, void* stream);
/* Render rays whose samples are given as packed intervals sorted by ray (the output of an occupancy
 * estimator, nerf_renderer.py:145-155): ray r owns samples [d_offsets[r], d_offsets[r+1]) of
 * d_t_starts / d_t_ends.  args->n_samples / near / far are ignored; eval-mode background rule. */
int perf_render_packed(const perf_render_args* args, const float* d_rays_o, const float* d_rays_d, uint64_t R,
                       const int64_t* d_offsets, const float* d_t_starts, const float* d_t_ends, void* stream);
/* Render rows [row0,row0+rows) of an H x W equirect panorama with ray generation fused in
 * (core_exp_runner.py:229-238 render_dense inner loop).  Outputs are [rows*W, .]. */
int perf_render_pano(const perf_render_args* args, const float* h_pose, int H, int W,
                     int row0, int rows, void* stream);

/* ---- one-launch render with the occupancy-grid sampler (nerf_renderer.py:145-197 in eval mode) ----
 * Each ray walks the grid itself (the intervals of perf_occ_count / perf_occ_write with no jitter, bit for bit),
 * evaluates both fields at each interval it emits and composites it, and stops at its first interval whose exclusive
 * transmittance exp(-sum_{j<i} sigma_j dt_j) is below early_stop_eps (nerfacc render_visibility_from_density with
 * alpha_thre = 0).  Nothing per sample is written.  Of perf_render_args, n_samples / near / far / d_jitter / d_bg_noise
 * are ignored; PERF_FLAG_SIMT_MLP and PERF_FLAG_GENERIC_ADDR are honoured, PERF_FLAG_TRAINING / _SCAN_KERNEL / _L0_SMEM
 * return PERF_EUNSUPPORTED; eval-mode background rule. */
typedef struct perf_occ_render_args {
    const uint8_t* d_binaries;        /* [res0][res1][res2] bool/uint8, x slowest (OccGridEstimator.binaries[0])        */
    int            res[3];
    float          aabb[6];           /* the estimator's roi_aabb (independent of perf_render_args.aabb, the field's)    */
    float          near, far, step;   /* PeRF: 0, 1.5, 5e-4 (nerf_renderer.py:149-151)                                 */
    float          early_stop_eps;    /* PeRF: 1e-4 (nerfacc default); 0 = keep every interval; must be in [0, 1)       */
    uint32_t*      d_n_samples;       /* [R] intervals composited per ray, or NULL                                     */
} perf_occ_render_args;
/* Explicit rays d_rays_o / d_rays_d [R,3] fp32 (args->image_width as for perf_render_rays). */
int perf_render_rays_occ(const perf_render_args* args, const perf_occ_render_args* occ, const float* d_rays_o,
                         const float* d_rays_d, uint64_t R, void* stream);
/* Rows [row0,row0+rows) of an H x W equirect panorama, ray generation fused in (as perf_render_pano). */
int perf_render_pano_occ(const perf_render_args* args, const perf_occ_render_args* occ, const float* h_pose,
                         int H, int W, int row0, int rows, void* stream);

/* ---- fused training step (fixed-S sampler): forward with saves, composite backward, grid scatter ----
 * All per-sample buffers are SAMPLE-MAJOR: row = k * R + ray (k = sample index along the ray), so
 * that a warp of neighbouring rays reads/writes contiguous rows.  Replaces, for one optimisation
 * step, the call chain modules/scene/nerf.py:186-297 -> nerf_renderer.py:112-209 -> tcnn/nerfacc
 * forward + the autograd backward through them. */
#define PERF_PHASE_GEO 1   /* density net trained: nerf.py:186-257 (colour under no_grad)           */
#define PERF_PHASE_APP 2   /* colour net trained:  nerf.py:259-297 (density under no_grad)           */
typedef struct perf_train_buffers {
    float* d_sigma;      /* [S*R] density                                                   */
    float* d_weights;    /* [S*R] w = T * alpha                                             */
    float* d_trans;      /* [S*R] T                                                         */
    void*  d_rgb;        /* [S*R,4] fp16 sample colours (PHASE_APP only, 4th lane unused)   */
    void*  d_feat;       /* [S*R,32] fp16 features of the trained network                   */
    void*  d_h1;         /* [S*R,64] fp16 hidden 1                                          */
    void*  d_h2;         /* [S*R,64] fp16 hidden 2 (PHASE_APP only)                         */
    float* d_dist_acc;   /* [R] sum w*t_mid before the background rule                      */
    float* d_distloss;   /* [R] distortion-loss numerator per ray (flatten_eff_distloss * n_rays) */
    /* Ray splitting for small batches (optional, both NULL = off): the forward may cut every ray into
     * `segments` pieces handled by different threads; then d_weights / d_trans hold segment-LOCAL values
     * (T = 1 at the segment start) and d_seg_trans [PERF_MAX_SEGMENTS * R] the transmittance at each
     * segment start (row = segment * R + ray).  The forward writes the count it chose to *h_segments_out;
     * pass the same struct (and that count) to perf_train_backward_composite. */
    float*    d_seg_trans;
    uint32_t* h_segments_out;
} perf_train_buffers;
#define PERF_MAX_SEGMENTS 64

/* Forward of a training step: like perf_render_rays (PERF_FLAG_TRAINING semantics: jitter, training
 * background rule) and additionally fills `buf`. */
int perf_train_forward(const perf_render_args* args, const float* d_rays_o, const float* d_rays_d,
                       uint64_t R, int phase, const perf_train_buffers* buf, void* stream);

/* Backward through the composite given per-ray gradients of the renderer outputs.
 * PHASE_GEO: d_out [S*R]   = dL/d(raw density logit)   (trunc_exp backward included)
 * PHASE_APP: d_out [S*R,3] = dL/d(colour pre-sigmoid)  (weights are detached, nerf_renderer.py:183)
 * d_g_* may be NULL (zero gradient).  d_distance_out: the forward's distance output (ReLU mask). */
int perf_train_backward_composite(int phase, uint32_t n_samples, uint32_t segments, float near, float far, uint64_t R,
                                  const float* d_jitter, const float* d_bg_noise, const perf_train_buffers* buf,
                                  const float* d_g_rgb, const float* d_g_distance, const float* d_g_opacity,
                                  const float* d_g_distloss, const float* d_distance_out, const float* d_opacity_out,
                                  float* d_out, void* stream);

/* The scalar losses of one training step and their gradients w.r.t. the renderer outputs in ONE launch
 * (nerf.py:208-238: smooth-L1 depth, beta 1e-2, + w_distloss * ratio * flatten_eff_distloss; nerf.py:281-287: smooth-L1
 * colour, beta 5e-2; torch `reduction='mean'`).  d_pred / d_gt [n] (n = R distances or 3 R colours); d_distloss [R] =
 * per-ray numerators from the forward or NULL; d_ratio: device scalar (the ramp min(2 progress, 1)) or NULL = 1;
 * d_inv_n_rays: device scalar 1 / (ray_id.max() + 1) or NULL = 1 / R.  d_loss3 = {total, mean smooth-L1, distortion
 * term}; d_g_pred [n], d_g_distloss [R] = d total / d input (NOT multiplied by the 2^7 loss scale). */
int perf_train_loss(const float* d_pred, const float* d_gt, uint64_t n, uint64_t R, float beta, float w_main,
                    const float* d_distloss, const float* d_ratio, const float* d_inv_n_rays, float w_distloss,
                    float* d_loss3, float* d_g_pred, float* d_g_distloss, void* stream);

/* Grid gradient for sample-major rows whose positions are recomputed from the rays:
 * d_dfeat [S*R, 32] fp32.  Same-cell neighbours inside a warp are merged before the atomics. */
int perf_hashgrid_bwd_rays(const perf_grid_cfg* cfg, const float* aabb6, const float* d_rays_o, const float* d_rays_d,
                           const float* d_jitter, uint64_t R, uint32_t n_samples, float near, float far,
                           const float* d_dfeat, float* d_dtable, void* stream);

/* The fixed-S training step's MLP backward WITH the fine-level grid scatter in its epilogue: perf_mlp_bwd on the R x S
 * sample-major rows (row = k * R + ray) of perf_train_forward; the thread that owns a row issues the reductions of levels
 * [8, 16) into d_dtable itself (positions recomputed from the rays as in perf_hashgrid_bwd_rays) and writes only the coarse
 * half of the feature gradient into d_dfeat (capacity >= 16 N floats) as eight LEVEL-MAJOR planes, plane l = float2 [N]
 * (what the march kernel reads coalesced).  Follow with perf_hashgrid_bwd_rays_coarse for levels [0, 8).  Together they
 * replace perf_mlp_bwd + perf_hashgrid_bwd_rays; the fine half of dfeat never reaches HBM and the L2-reduction-bound
 * scatter overlaps the latency-bound MMA phases. */
int perf_mlp_bwd_scatter(const perf_mlp_cfg* mlp, const void* d_weights_half, const void* d_feat, const void* d_h1, const void* d_h2,
                         const float* d_dz, uint64_t N, float* d_dweights, float* d_dfeat,
                         const perf_grid_cfg* grid, const float* aabb6, const float* d_rays_o, const float* d_rays_d, const float* d_jitter,
                         uint64_t R, uint32_t n_samples, float near, float far, float* d_dtable, void* stream);
int perf_hashgrid_bwd_rays_coarse(const perf_grid_cfg* cfg, const float* aabb6, const float* d_rays_o, const float* d_rays_d,
                                  const float* d_jitter, uint64_t R, uint32_t n_samples, float near, float far,
                                  const float* d_dfeat, float* d_dtable, void* stream);

/* Occupancy-grid interval sampler (nerfacc OccGridEstimator.sampling, levels=1, cone_angle=0;
 * nerf_renderer.py:145-155; SURVEY.md 8f row 1).  d_binaries: bool/uint8 [rx*ry*rz] (x slowest).
 * Pass 1 writes the per-ray sample counts; the caller exclusive-scans them into d_offsets and
 * allocates the packed outputs; pass 2 writes (ray_indices int64, t_starts, t_ends), sorted by ray. */
int perf_occ_count(const uint8_t* d_binaries, const int* h_res3, const float* h_aabb6, const float* d_rays_o, const float* d_rays_d,
                   const float* d_jitter, uint64_t R, float near, float far, float step, uint32_t pieces, int32_t* d_counts,
                   uint32_t* d_masks /* nullable, see below */, void* stream);
int perf_occ_write(const uint8_t* d_binaries, const int* h_res3, const float* h_aabb6, const float* d_rays_o, const float* d_rays_d,
                   const float* d_jitter, uint64_t R, float near, float far, float step, uint32_t pieces, const int64_t* d_offsets, uint64_t capacity,
                   const uint32_t* d_masks /* nullable */, int64_t* d_ray_indices, float* d_t_starts, float* d_t_ends, void* stream);
/* d_masks [R * pieces * 4] uint32 (optional, the same buffer in both passes): the count pass records WHICH lattice points of
 * every piece are samples (one bit each) and the write pass only expands those bits -- the grid is marched once, not twice.
 * Usable when a piece holds at most 128 lattice points, i.e. (far - near) / step / pieces + 1 <= 128 (else PERF_EINVAL). */
/* `pieces` (>= 1, the same in both passes): every ray's lattice range is cut into that many consecutive parts marched by
 * different threads -- a ray is a serial walk of up to (far - near) / step lattice points, and 8192 rays alone leave the GPU
 * empty.  d_counts and d_offsets then have R * pieces entries indexed [ray * pieces + piece] (exclusive scan over all of
 * them); the packed output is the same, sorted by ray and t.  A ray's range is d_offsets[ray * pieces] .. [(ray+1) * pieces]. */

/* ---- fused training step for PACKED samples (the occupancy sampler PeRF trains with, configs/nerf.yaml:25;
 * nerf_renderer.py:145-183, nerf.py:186-297): perf_occ_count/write -> perf_fields_packed ->
 * perf_composite_packed_fwd -> losses -> perf_composite_packed_bwd -> perf_mlp_bwd -> perf_hashgrid_bwd_merged.
 * All per-sample buffers are indexed by the packed sample number n (sorted by ray). */

/* Both fields at N packed samples in one launch: position o + d (ts+te)/2, aabb normalisation and selector
 * (ngp_nerf.py:136-162), encode of both grids, both MLPs.  args: only grid / tables / weights / aabb / flags are read.
 * d_sigma [N] fp32, d_rgb_half4 [N,4] fp16 (4th lane unused), d_x01 [N,3] fp32 (normalised position; masked-out
 * samples get the in-box stand-in their features were taken at).  phase 0: no saves; PERF_PHASE_GEO / _APP: also
 * d_feat [N,32], d_h1 [N,64] (and d_h2 [N,64] for _APP) fp16 of the trained network. */
int perf_fields_packed(const perf_render_args* args, const float* d_rays_o, const float* d_rays_d, const int64_t* d_ray_indices,
                       const float* d_t_starts, const float* d_t_ends, uint64_t N, const int64_t* d_n_dev /* nullable, see below */,
                       int phase, float* d_sigma, void* d_rgb_half4, float* d_x01, void* d_feat, void* d_h1, void* d_h2, void* stream);

/* Composite of packed samples, one warp per ray: w, T (nerfacc render_weight_from_density), opacity / distance /
 * colour (accumulate_along_rays), background rule (PERF_FLAG_TRAINING in flags: nerf_renderer.py:192-194, else
 * :195-197), distortion-loss numerator per ray (flatten_eff_distloss * n_rays).  Samples whose transmittance is below
 * early_stop_eps get weight 0 and T = 0 -- identical to nerfacc dropping them inside OccGridEstimator.sampling.
 * d_offsets int64 [R+1]; d_weights / d_trans [N]; d_rgb_out [R,3]; the others [R]. */
int perf_composite_packed_fwd(const int64_t* d_offsets, const float* d_t_starts, const float* d_t_ends, const float* d_sigma,
                              const void* d_rgb_half4, uint64_t R, float early_stop_eps, uint32_t flags, const float* d_bg_noise,
                              float* d_weights, float* d_trans, float* d_rgb_out, float* d_distance_out, float* d_opacity_out,
                              float* d_dist_acc, float* d_distloss, void* stream);
/* Its backward: d_dz [N] = dL/d(raw density logit) (PERF_PHASE_GEO, trunc_exp backward included) or [N,3] =
 * dL/d(colour pre-sigmoid) (PERF_PHASE_APP).  d_g_* [R,.] may be NULL. */
int perf_composite_packed_bwd(int phase, const int64_t* d_offsets, const float* d_t_starts, const float* d_t_ends, const float* d_sigma,
                              const void* d_rgb_half4, uint64_t R, const float* d_bg_noise, const float* d_weights, const float* d_trans,
                              const float* d_distance_out, const float* d_opacity_out, const float* d_dist_acc,
                              const float* d_g_rgb, const float* d_g_distance, const float* d_g_opacity, const float* d_g_distloss,
                              float* d_dz, void* stream);
/* perf_hashgrid_bwd with the number of levels whose same-cell runs of consecutive samples are merged before the
 * atomics chosen by the caller (packed samples are 5e-4 apart: runs exist up to resolution ~1000). */
int perf_hashgrid_bwd_merged(const perf_grid_cfg* cfg, const float* d_x01, const float* d_dfeat, uint64_t N, const int64_t* d_n_dev,
                             float* d_dtable, uint32_t n_merge_levels, void* stream);
/* d_n_dev (perf_fields_packed, perf_mlp_bwd, perf_hashgrid_bwd_merged): the sample count of a step is only known on the device
 * (it is the last entry of the offsets scan).  Passing N = the CAPACITY of the buffers and d_n_dev = a device int64 holding the
 * live count makes the launch sequence independent of the count -- the whole occupancy-sampler step can be captured into a CUDA
 * graph and replayed without a host read.  perf_occ_write's `capacity` (0 = unlimited) drops samples that would not fit; the
 * caller clamps the offsets and the count to it. */

/* Batch draw (sup_info.py:253-259): dst_k[b, :] = src_k[idx[b], :] for up to 6 row-major fp32 arrays of row widths
 * h_width[k] in one launch.  h_src / h_dst: HOST arrays of device pointers. */
int perf_gather_rows(const int64_t* d_idx, uint64_t B, int n_arrays, const float* const* h_src, float* const* h_dst, const int* h_width, void* stream);

/* The whole batch draw in one launch: B SORTED uniform row indices in [0, M) from the running sums d_csum [B+1] (fp64) of i.i.d.
 * Exp(1) variates -- S_k / S_{B+1} are the order statistics of B uniforms, i.e. torch.randint followed by a sort, without the
 * sort -- and the gather of perf_gather_rows with them.  d_idx_out [B] int64 or NULL.  With the pool stored in Morton order
 * of its pixels a sorted batch is a spatially coherent one. */
int perf_draw_gather_rows(const double* d_csum, uint64_t B, uint64_t M, int64_t* d_idx_out, int n_arrays, const float* const* h_src,
                          float* const* h_dst, const int* h_width, void* stream);

/* Diagnostic (bench.py's train_roofline denominator): n_atomics reductions of `vec` (1, 2 or 4) floats at pseudo-random
 * vec-aligned slots of d_table [n_floats] -- the L2 atomic rate that bounds the grid-gradient scatter. */
int perf_debug_atomic_rate(float* d_table, uint64_t n_floats, uint64_t n_atomics, int vec, void* stream);

/* Occupancy-grid update (nerfacc OccGridEstimator.update_every_n_steps, levels = 1; nerf.py:159-168).
 * perf_occ_points: a uniformly jittered point inside each listed cell (d_cell_idx int64 [n], NULL = cells 0..n-1),
 * d_x [n,3]; the caller evaluates its occ_eval_fn there.  perf_occ_update: occs[c] = max(occs[c] * ema_decay, occ),
 * then binaries = occs > min(mean(occs), occ_thre) (deterministic two-stage mean).  d_workspace: 2 * PERF_OCC_PARTIALS doubles. */
#define PERF_OCC_PARTIALS 1024
int perf_occ_points(const int64_t* d_cell_idx, uint64_t n, const int* h_res3, const float* h_aabb6, uint64_t seed, float* d_x, void* stream);
int perf_occ_update(float* d_occs, uint64_t n_cells, const int64_t* d_cell_idx, const float* d_occ_new, uint64_t n, float ema_decay,
                    float occ_thre, uint8_t* d_binaries, double* d_workspace, void* stream);

/* MLP backward helpers on the saved fp16 activations (tcnn kernel_mlp_fused_backward pieces; the
 * matrix products themselves are plain GEMMs left to cuBLAS):
 *   perf_mlp_bwd_out: d_dh [N,64] fp16 = (d_dz [N,n_out] fp32 @ Wout[:n_out] fp16) * (d_h > 0)
 *   perf_relu_mask:   d_dh *= (d_h > 0), in place, n_values fp16 values each */
int perf_mlp_bwd_out(const float* d_dz, int n_out, const void* d_wout_half, const void* d_h, void* d_dh, uint64_t N, void* stream);
int perf_relu_mask(void* d_dh, const void* d_h, uint64_t n_values, void* stream);

/* Fused Adam on a flat fp32 parameter vector + refresh of its fp16 shadow
 * (torch.optim.Adam at nerf.py:171,180,253,293; betas/eps defaults).  grad_scale multiplies
 * the gradient first (the reference never unscales its 128x GradScaler; pass 1 to keep that). */
int perf_adam_step(float* d_params, const float* d_grads, float* d_exp_avg, float* d_exp_avg_sq,
                   void* d_params_half /*nullable*/, uint64_t n, float lr, float beta1, float beta2,
                   float eps, uint32_t step /*1-based*/, float grad_scale, void* stream);

/* d_dst[0..n) = h_values[0..n), n <= 8, stream-ordered; the values travel as kernel arguments, so the
 * host array may be reused immediately (feeds the device-side schedule of a replayed CUDA graph). */
int perf_set_scalars(float* d_dst, const float* h_values, int n, void* stream);

/* Same update with {lr, 1 - beta1^step, sqrt(1 - beta2^step)} read from DEVICE memory (d_hyper[3]) at
 * run time: the launch can live inside a captured CUDA graph and be replayed with a new schedule. */
int perf_adam_step_dev(float* d_params, const float* d_grads, float* d_exp_avg, float* d_exp_avg_sq,
                       void* d_params_half /*nullable*/, uint64_t n, const float* d_hyper, float beta1, float beta2,
                       float eps, float grad_scale, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PERFB200_H */
