// render.cu -- the fused per-ray megakernel: ray-gen -> fixed-S sampling -> hash-grid encode of
// BOTH fields (hashed levels: one 8-byte gather per corner from the interleaved table; dense levels:
// one 64-byte cell record) -> density MLP and colour MLP on tcgen05 -> alpha composite (a running
// sum per thread in render_march_kernel, warp-shuffle segmented scans in the legacy render_kernel).
// Nothing per-sample ever touches HBM: inputs are the pose (or [R,3] rays) and the tables,
// outputs are 16-20 B per ray.
//
// Replaces the whole inner stack of SURVEY.md section 3.1:
//   NeRFScene.render / render_once      modules/scene/nerf.py:74-123
//   NeRFOCCRenderer.render              modules/scene/nerf_renderer.py:112-209 (fixed-S sampler)
//   NGPNeRF.query_density / query_rgb   modules/fields/ngp_nerf.py:136-162
//   gen_pano_rays                       utils/camera_utils.py:229-234
// Arithmetic contract: oracle/render.py::render_rays(mixed=True).
#include "mlp_tc.cuh"
#include "occ_walk.cuh"

namespace perf {

struct RenderArgs {
    LevelTable    lt;
    const uint2*  table;        // {geo half2, app half2} per entry
    const uint4*  cells[PERF_CELL_LEVELS];   // cell-major copies of the dense levels inside the same buffer (common.cuh::PackedLayout)
    const __half* geo_w;        // W1 [64,32] | Wout [16,64]
    const __half* app_w;        // W1 [64,32] | W2 [64,64] | Wout [16,64]
    float         aabb_min[3], aabb_ext[3];
    uint32_t      S;            // samples per ray
    uint32_t      rays_per_unit, tiles_per_unit;
    float         near, far;
    uint32_t      training;
    uint32_t      tile_mul;     // image-shaped work: tile = (i * tile_mul) % n_tiles (a bijection, gcd(tile_mul, n_tiles) == 1); 0 / 1 = row-major
    uint32_t      div_generic;  // 1: an aabb extent whose significand is all ones -> div_uniform() falls back to the IEEE division
    const float*  jitter;       // [R] or null
    const float*  bg_noise;     // [R,4] or null
    float*        rgb;          // [R,3]
    float*        distance;     // [R]
    float*        opacity;      // [R] or null
    uint64_t      R;
    // ray source
    const float*  rays_o;       // [R,3]  (PANO == false)
    const float*  rays_d;
    float         pose_r[9], pose_t[3];
    int           H, W, row0;   // (PANO == true): ray r is pixel (row0 + r / W, r % W)
    // packed variable-length samples (perf_render_packed): ray r owns samples [pk_offsets[r], pk_offsets[r+1])
    const int64_t* pk_offsets;  // [R+1] or null (fixed-S lattice)
    const float*   pk_ts;       // [N]
    const float*   pk_te;       // [N]
    // training-forward saves (SAVE != 0), all sample-major: row = k * R + ray
    float*        s_sigma;      // [S*R]
    float*        s_w;          // [S*R]
    float*        s_trans;      // [S*R]
    __half*       s_rgb;        // [S*R, 4] (colour phase only; 4th lane unused)
    uint4*        s_feat;       // [S*R, 32] fp16 of the network being trained
    uint4*        s_h1;         // [S*R, 64] fp16
    uint4*        s_h2;         // [S*R, 64] fp16 (colour phase only)
    float*        s_dacc;       // [R] distance accumulate BEFORE the background rule
    float*        s_dl;         // [R] distortion-loss numerator of the ray
    // ray splitting (explicit rays, fixed S): every ray is cut into `seg` consecutive segments of
    // S/seg samples handled by `seg` different threads of the tile (tile = 128/seg rays); the segment
    // results are combined with the transmittance product rule.  Fills the GPU for small ray batches
    // (an 8192-ray training batch is only 64 tiles of 128 rays, but 512 tiles of 16 rays x 8 segments).
    uint32_t      seg;          // power of two, divides S and 128; 1 = off
    float*        s_toff;       // [seg * R] transmittance at the start of each segment (SAVE, seg > 1)
};

constexpr int RS_A     = 0;                         // 16 KB: A_geo | A_app, later H (K=64)
constexpr int RS_W1G   = RS_A + A64_BYTES;
constexpr int RS_W1A   = RS_W1G + W32_BYTES;
constexpr int RS_W2A   = RS_W1A + W32_BYTES;
constexpr int RS_WOUT  = RS_W2A + W64_BYTES;        // fp32: geo [64] then app [3][64]
constexpr int RS_TAILS = RS_WOUT + 4 * HID * 4;     // [2 scans][4 warps][8] floats
constexpr int RS_CARRY = RS_TAILS + 2 * 4 * 8 * 4;  // [2 parities][8] floats
constexpr int RS_BAR   = RS_CARRY + 2 * 8 * 4;
constexpr int RS_BARW  = RS_BAR + 16;               // mbarrier of the weight bulk copy
constexpr int RS_TOTAL = RS_BARW + 16;
// measurement hook (tools/ab_lib.py, profiles/r02_render_variants.md): extra, unused dynamic shared memory per CTA of the
// march kernels, i.e. what a second activation tile would cost in L1 capacity (4 CTAs/SM: 136 KB -> 200 KB of shared memory)
#ifndef PERF_RS_PAD
#define PERF_RS_PAD 0
#endif
constexpr int RS_LAUNCH = RS_TOTAL + PERF_RS_PAD;
constexpr int W_IMG_BYTES = W32_BYTES + W32_BYTES + W64_BYTES;       // 16 KB: W1 density | W1 colour | W2 colour
static_assert(RS_W1A == RS_W1G + W32_BYTES && RS_W2A == RS_W1A + W32_BYTES, "the three weight images are one contiguous block");
// experiment (PERF_FLAG_L0_SMEM): level 0 of the packed table (16^3 entries x 8 B = 32 KB) resident in shared memory,
// staged once per persistent CTA by ONE bulk copy (cp.async.bulk -> UBLKCP, completion on an mbarrier)
constexpr int RS_BAR2  = (RS_TOTAL + 127) / 128 * 128;
constexpr int RS_L0    = RS_BAR2 + 128;
constexpr int L0_BYTES = 4096 * 8;
constexpr int RS_TOTAL_L0 = RS_L0 + L0_BYTES;

// Output-layer weights of both networks as fp32 in the CONSTANT bank: [0,64) density row, [64,256) the three colour
// rows.  The 64 * n_out FMAs per sample of the output layers then take their weight operand straight from c[bank][imm]
// -- no load instruction.  (Round 1 kept them in shared memory: 64 broadcast LDS.128 per thread and sample, 1.2e9
// shared-load wavefronts per panorama on the L1 data pipe that bounds the kernel, profiles/r01_*.)  Filled from the fp16
// parameter vectors by weights_prepare_kernel, stream-ordered in front of every render launch (graph-capturable).
// One slot per device: renders of DIFFERENT fields on the same device must not overlap in time (different streams).
__constant__ float c_wout[4 * HID];
// The three hidden-layer matrices as ready-made UMMA operand images (no-swizzle K-major canonical layout, mlp_tc.cuh), 16 KB:
// every persistent CTA stages them with ONE bulk copy (cp.async.bulk -> UBLKCP, completion on an mbarrier) instead of 1024
// 16-byte LDG + STS per CTA.  Written by the same preparation kernel, same single-slot rule as c_wout.
__device__ uint4 g_wimg[W_IMG_BYTES / 16];

__global__ void __launch_bounds__(1024) weights_prepare_kernel(const __half* __restrict__ geo_w, const __half* __restrict__ app_w, float* __restrict__ c_dst)
{
    const int c = threadIdx.x;                       // 1024 threads = 1024 16-byte chunks of the images
    if (c < 4 * HID) c_dst[c] = __half2float(c < HID ? geo_w[HID * 32 + c] : app_w[HID * 32 + HID * HID + (c - HID)]);
    const __half* src; int K, cc;
    if (c < 256)      { src = geo_w;            K = 32; cc = c; }
    else if (c < 512) { src = app_w;            K = 32; cc = c - 256; }
    else              { src = app_w + HID * 32; K = 64; cc = c - 512; }
    const int n = cc % HID, kg = cc / HID;           // image chunk (kg * 64 + n) <- row n, columns [8 kg, 8 kg + 8)
    g_wimg[c] = *reinterpret_cast<const uint4*>(src + (size_t)n * K + kg * 8);
}

// all threads of the CTA: weight images global -> shared memory by one bulk copy; returns when they have landed
__device__ __forceinline__ void stage_weights_bulk(uint8_t* smem, int tid)
{
    uint64_t* barw = reinterpret_cast<uint64_t*>(smem + RS_BARW);
    if (tid == 0) {
        mbar_init(barw, 1); fence_mbar_init();
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(barw)), "r"(W_IMG_BYTES) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     :: "r"(smem_u32(smem + RS_W1G)), "l"(reinterpret_cast<const void*>(g_wimg)), "r"(W_IMG_BYTES), "r"(smem_u32(barw)) : "memory");
    }
    __syncthreads();                                 // the barrier is initialised before anyone polls it
    mbar_wait(barw, 0);
}

// acc[o] += h[32C + 2j, 32C + 2j + 1] * c_wout[BASE + 64 o + 32 C + 2j, ... + 1]: even / odd partial sums, one FFMA2 per
// packed pair of activations (mlp_tc.cuh::out_dots has the same order); C is a compile-time constant so that the
// weights come straight from the constant bank (LDCU.128 of four weights into uniform registers).
template <int NOUT, int BASE, int C>
__device__ __forceinline__ void out_dots_const(const uint32_t (&p)[16], float2 (&acc)[NOUT])
{
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const float2 f = unpack_half2(p[j]);
#pragma unroll
        for (int o = 0; o < NOUT; ++o)
            ffma2(acc[o], f, make_float2(c_wout[BASE + o * HID + 32 * C + 2 * j], c_wout[BASE + o * HID + 32 * C + 2 * j + 1]));
    }
}

__device__ __forceinline__ float linspace_val_r(int i, int n)
{
    const float start = (float)(0.5 / (double)n), end = (float)(1.0 - 0.5 / (double)n);
    if (n == 1) return start;
    const float step = (end - start) / (float)(n - 1);
    return (i < n / 2) ? __fadd_rn(start, __fmul_rn(step, (float)i)) : __fsub_rn(end, __fmul_rn(step, (float)(n - i - 1)));
}

// Inclusive scan of NV values along the ray across the whole CTA tile (and across the tiles of
// a unit through `carry`).  Lanes are consecutive samples; a ray may start anywhere.
//   k        : index of this sample inside its ray
//   k0_tile  : in-ray index of the tile's first sample (sample of thread 0)
// Deterministic: tree inside a warp, then warps in order, then tiles in order.
template <int NV>
__device__ __forceinline__ void ray_scan(float (&val)[NV], float (&excl)[NV], uint32_t k, uint32_t k0_tile, uint32_t S, int tid,
                                         float* tails /*[4][8]*/, const float* carry_in /*[8] or null*/, float* carry_out /*[8]*/)
{
    const int lane = tid & 31, warp = tid >> 5;
    const int seg_start = (k >= (uint32_t)lane) ? 0 : lane - (int)k;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
#pragma unroll
        for (int j = 0; j < NV; ++j) {
            const float t = __shfl_up_sync(0xffffffffu, val[j], off);
            if (lane - off >= seg_start) val[j] += t;
        }
    }
#pragma unroll
    for (int j = 0; j < NV; ++j) {               // exclusive prefix inside the warp (no inf - inf)
        const float t = __shfl_up_sync(0xffffffffu, val[j], 1);
        excl[j] = (lane - 1 >= seg_start) ? t : 0.f;
    }
    if (lane == 31) {
#pragma unroll
        for (int j = 0; j < NV; ++j) tails[warp * 8 + j] = val[j];
    }
    __syncthreads();
    // carry into the ray of lane 0 of warp w:  c[0] = carry_in;  c[w+1] = k0(w+1)==0 ? 0 : (one_seg(w) ? c[w] : 0) + tail[w]
    float c[NV];
#pragma unroll
    for (int j = 0; j < NV; ++j) c[j] = (carry_in != nullptr && k0_tile != 0) ? carry_in[j] : 0.f;
    const int upto = (carry_out != nullptr && tid == 0) ? 4 : warp;     // thread 0 also produces the tile's carry-out
    float cw[NV];
#pragma unroll
    for (int j = 0; j < NV; ++j) cw[j] = c[j];
#pragma unroll 1
    for (int w = 0; w < upto; ++w) {
        const uint32_t k0w = (k0_tile + 32u * w) % S;            // in-ray index of lane 0 of warp w
        const uint32_t k0n = (k0_tile + 32u * (w + 1)) % S;      // ... of lane 0 of warp w+1
        const bool one_seg = (k0w + 31u) < S;                    // warp w lies inside one ray
#pragma unroll
        for (int j = 0; j < NV; ++j) {
            const float prev = one_seg ? c[j] : 0.f;
            c[j] = (k0n == 0) ? 0.f : prev + tails[w * 8 + j];
        }
        if (w + 1 == warp) {
#pragma unroll
            for (int j = 0; j < NV; ++j) cw[j] = c[j];
        }
    }
    if (carry_out != nullptr && tid == 0) {
#pragma unroll
        for (int j = 0; j < NV; ++j) carry_out[j] = c[j];
    }
    if (k >= (uint32_t)lane) {               // same ray as lane 0 of my warp
#pragma unroll
        for (int j = 0; j < NV; ++j) { val[j] += cw[j]; excl[j] += cw[j]; }
    }
}

// Pixel-patch tiling of a 128-thread tile: a warp covers PATCH_WW x PATCH_WH pixels, the CTA's four
// warps are arranged PATCH_WX x PATCH_WY.
#ifndef PATCH_WW
#define PATCH_WW 8
#define PATCH_WH 4
#define PATCH_WX 2
#define PATCH_WY 2
#endif
constexpr int PATCH_W = PATCH_WW * PATCH_WX, PATCH_H = PATCH_WH * PATCH_WY;
static_assert(PATCH_WW * PATCH_WH == 32 && PATCH_WX * PATCH_WY == 4, "a warp is 32 pixels, a tile 4 warps");

struct RenderSmem {
    uint8_t *sA, *sAg, *sAa, *sW1g, *sW1a, *sW2a;
    float *sWoutG, *sWoutA;
    uint64_t* bar;
    const uint2* l0;        // level 0 of the packed table in shared memory, or null
};

// base + 8 * idx as ONE IMAD.WIDE.U32 (left to itself ptxas splits the 64-bit address into LEA + IADD3.X per corner)
__device__ __forceinline__ const uint2* entry_ptr(const uint2* base, uint32_t idx)
{
    uint64_t p;
    asm("mad.wide.u32 %0, %1, 8, %2;" : "=l"(p) : "r"(idx), "l"(reinterpret_cast<uint64_t>(base)));
    return reinterpret_cast<const uint2*>(p);
}

// L1 eviction hints of the table gathers.  The fine hashed levels stream through L1 (a ray leaves a fine cell with every
// step) while the dense / coarse levels are re-read from one sample to the next: 0 = default, 1 = L1::evict_first,
// 2 = L1::no_allocate, 3 = L1::evict_last.  (Measured: tools/ab_lib.py, profiles/r02_render_variants.md.)
#ifndef PERF_L1_HASHED
#define PERF_L1_HASHED 0
#endif
#ifndef PERF_L1_DENSE
#define PERF_L1_DENSE 0
#endif
template <int HINT>
__device__ __forceinline__ uint2 ldg_entry(const uint2* p)
{
    if constexpr (HINT == 0) return __ldg(p);
    uint2 v;
    if constexpr (HINT == 1) asm("ld.global.nc.L1::evict_first.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p));
    if constexpr (HINT == 2) asm("ld.global.nc.L1::no_allocate.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p));
    if constexpr (HINT == 3) asm("ld.global.nc.L1::evict_last.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p));
    return v;
}
template <int HINT>
__device__ __forceinline__ uint4 ldg_cell(const uint4* p)
{
    if constexpr (HINT == 0) return __ldg(p);
    uint4 v;
    if constexpr (HINT == 1) asm("ld.global.nc.L1::evict_first.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    if constexpr (HINT == 2) asm("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    if constexpr (HINT == 3) asm("ld.global.nc.L1::evict_last.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}

// Levels [4q, 4q+4) of both fields -> one 16-byte k-group of each feature tile.
// KIND 0: generic addressing, 1: dense (fast), 2: hashed power-of-two (fast).
template <int KIND, int SAVE, bool L0SMEM = false>
__device__ __forceinline__ void encode_group(const RenderArgs& a, const RenderSmem& sm, int q, float x, float y, float z, int tid, uint64_t srow)
{
    uint32_t pg[4], pa[4];
#pragma unroll
    for (int ll = 0; ll < 4; ++ll) {
        const int l = 4 * q + ll;
        uint2 v[8]; float w[8];
        if constexpr (KIND == 0) {
            Corner8 c; level_corners(a.lt, l, x, y, z, c);
#pragma unroll
            for (int kk = 0; kk < 8; ++kk) { v[kk] = __ldg(a.table + c.idx[kk]); w[kk] = c.w[kk]; }
        } else if constexpr (KIND == 1) {
            if (L0SMEM && l == 0) {                // measured variant: level 0 (entry-major, offset 0) resident in shared memory
                uint32_t idx[8];
                level_corners_rel<false>(a.lt, l, x, y, z, idx, w);
#pragma unroll
                for (int kk = 0; kk < 8; ++kk) v[kk] = sm.l0[idx[kk]];
            } else {
                // dense level: ONE 64-byte cell record (all 8 corners of both fields), 4 x LDG.128 from one address
                const uint32_t cell = level_cell_dense(a.lt, l, x, y, z, w);
                const uint4* const cp = a.cells[l] + 4ull * cell;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const uint4 c2 = ldg_cell<PERF_L1_DENSE>(cp + j);
                    v[2 * j] = make_uint2(c2.x, c2.y); v[2 * j + 1] = make_uint2(c2.z, c2.w);
                }
            }
        } else {
            // hashed level, level-local indices: the level offset goes into the pointer once, not into each of the 8 indices
            uint32_t idx[8];
            level_corners_rel<true>(a.lt, l, x, y, z, idx, w);
            const uint2* const tl = a.table + a.lt.offset[l];
#pragma unroll
            for (int kk = 0; kk < 8; ++kk) v[kk] = ldg_entry<PERF_L1_HASHED>(entry_ptr(tl, idx[kk]));
        }
        uint32_t vg[8], va[8];
#pragma unroll
        for (int kk = 0; kk < 8; ++kk) { vg[kk] = v[kk].x; va[kk] = v[kk].y; }
        pg[ll] = blend8_half(w, vg); pa[ll] = blend8_half(w, va);
    }
    *reinterpret_cast<uint4*>(sm.sAg + (q * TILE + tid) * 16) = make_uint4(pg[0], pg[1], pg[2], pg[3]);
    *reinterpret_cast<uint4*>(sm.sAa + (q * TILE + tid) * 16) = make_uint4(pa[0], pa[1], pa[2], pa[3]);
    if constexpr (SAVE == 1) { if (srow != ~0ull) a.s_feat[srow * 4 + q] = make_uint4(pg[0], pg[1], pg[2], pg[3]); }
    if constexpr (SAVE == 2) { if (srow != ~0ull) a.s_feat[srow * 4 + q] = make_uint4(pa[0], pa[1], pa[2], pa[3]); }
}

// Encode + both MLPs for the CTA's current 128 samples (thread t = sample t at normalised
// position (x,y,z)).  Contains 2 block-wide barriers + 2 mbarrier waits; all 128 threads call it.
// NDENSE >= 0: specialised addressing (level_corners_fast; first NDENSE levels dense, rest hashed
// power-of-two) -- branch-free and ~1/3 smaller code; NDENSE < 0: generic addressing.
// SAVE 1 / 2: also write the fp16 features and hidden activations of the density / colour network
// to row `srow` of the training buffers (srow == ~0: masked-out thread).
template <bool SIMT, int NDENSE, int SAVE = 0, bool L0SMEM = false>
__device__ __forceinline__ void eval_fields(const RenderArgs& a, const RenderSmem& sm, float x, float y, float z, bool selector,
                                            uint32_t tmem_base, uint32_t tmem_row, uint32_t& parity, int tid,
                                            float& sigma, float& cr, float& cg, float& cb, uint64_t srow = ~0ull)
{
    uint8_t* const sA = sm.sA; uint8_t* const sAg = sm.sAg; uint8_t* const sAa = sm.sAa;
    uint8_t* const sW1g = sm.sW1g; uint8_t* const sW1a = sm.sW1a; uint8_t* const sW2a = sm.sW2a;
    float* const sWoutG = sm.sWoutG; float* const sWoutA = sm.sWoutA; uint64_t* const bar = sm.bar;
    if (NDENSE >= 0 && !selector) { x = 0.5f; y = 0.5f; z = 0.5f; }   // masked sample: any in-box address will do
    // ---- encode both fields: 16 levels x 8 corners, one 8-byte gather per corner
    if constexpr (NDENSE == 4) {
        // dense group unrolled; the three hashed groups share ONE copy of the code (the fully
        // unrolled body was ~70 KB of SASS and stalled on instruction fetch)
        encode_group<1, SAVE, L0SMEM>(a, sm, 0, x, y, z, tid, srow);
#pragma unroll 1
        for (int q = 1; q < 4; ++q) encode_group<2, SAVE>(a, sm, q, x, y, z, tid, srow);
    } else {
#pragma unroll
        for (int q = 0; q < 4; ++q) encode_group<0, SAVE>(a, sm, q, x, y, z, tid, srow);
    }

    // ---- layer 1 of both nets
    if constexpr (!SIMT) {
        fence_proxy_async();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            issue_layer(tmem_base, smem_u32(sAg), smem_u32(sW1g), 32);
            issue_layer(tmem_base + 64, smem_u32(sAa), smem_u32(sW1a), 32);
            umma_commit(bar);
        }
        mbar_wait(bar, parity); parity ^= 1u;
        tc_fence_after();
    } else {
        __syncthreads();
    }

    // density: ReLU hidden -> 64-long dot -> fp16 logit -> exp     (ngp_nerf.py:141-150)
    float2 og[1] = {make_float2(0.f, 0.f)};
#pragma unroll
    for (int c = 0; c < 2; ++c) {                          // unrolled: the constant-bank offsets must be immediates
        float v[32]; uint32_t hp[16];
        acc_chunk<SIMT>(c, 32, tmem_row, sAg, sW1g, tid, v);
        relu_pack(v, hp);
        if constexpr (SAVE == 1) { if (srow != ~0ull) store_chunk_global(a.s_h1 + srow * 8, c, hp); }
        if (c == 0) out_dots_const<1, 0, 0>(hp, og); else out_dots_const<1, 0, 1>(hp, og);
    }
    sigma = selector ? expf(finish_output(out_sum(og[0]), 0)) : 0.f;

    // colour hidden 1 -> H tile (aliases the feature tiles: both layer-1 MMAs are complete)
#pragma unroll 1
    for (int c = 0; c < 2; ++c) {
        float v[32]; uint32_t hp[16];
        acc_chunk<SIMT>(c, 32, tmem_row + 64, sAa, sW1a, tid, v);
        relu_pack(v, hp);
        if constexpr (SAVE == 2) { if (srow != ~0ull) store_chunk_global(a.s_h1 + srow * 8, c, hp); }
        store_chunk_canonical(sA, tid, 4 * c, hp);
    }
    if constexpr (!SIMT) {
        fence_proxy_async();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            issue_layer(tmem_base + 64, smem_u32(sA), smem_u32(sW2a), 64);
            umma_commit(bar);
        }
        mbar_wait(bar, parity); parity ^= 1u;
        tc_fence_after();
    } else {
        __syncthreads();
    }
    float2 oa[3] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
#pragma unroll
    for (int c = 0; c < 2; ++c) {
        float v[32]; uint32_t hp[16];
        acc_chunk<SIMT>(c, 64, tmem_row + 64, sA, sW2a, tid, v);
        relu_pack(v, hp);
        if constexpr (SAVE == 2) { if (srow != ~0ull) store_chunk_global(a.s_h2 + srow * 8, c, hp); }
        if (c == 0) out_dots_const<3, HID, 0>(hp, oa); else out_dots_const<3, HID, 1>(hp, oa);
    }
    cr = selector ? finish_output(out_sum(oa[0]), 1) : 0.f;      // ngp_nerf.py:156-161
    cg = selector ? finish_output(out_sum(oa[1]), 1) : 0.f;
    cb = selector ? finish_output(out_sum(oa[2]), 1) : 0.f;
}

template <bool PANO, bool SIMT>
__global__ void __launch_bounds__(TILE, 4) render_kernel(const __grid_constant__ RenderArgs a)
{
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* sA   = smem + RS_A;
    uint8_t* sAg  = sA;                     // geo features, K=32
    uint8_t* sAa  = sA + A32_BYTES;         // app features, K=32
    uint8_t* sW1g = smem + RS_W1G;
    uint8_t* sW1a = smem + RS_W1A;
    uint8_t* sW2a = smem + RS_W2A;
    float*   sWoutG = reinterpret_cast<float*>(smem + RS_WOUT);
    float*   sWoutA = sWoutG + HID;
    float*   sTails = reinterpret_cast<float*>(smem + RS_TAILS);
    float*   sCarry = reinterpret_cast<float*>(smem + RS_CARRY);
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + RS_BAR);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + RS_BAR + 8);

    const int tid = threadIdx.x, warp = tid >> 5;
    const RenderSmem sm = {sA, sAg, sAa, sW1g, sW1a, sW2a, sWoutG, sWoutA, bar, nullptr};

    stage_weights_bulk(smem, tid);                   // W1 density | W1 colour | W2 colour operand images, one UBLKCP
    uint32_t tmem_base = 0;
    if (!SIMT) {
        if (tid == 0) { mbar_init(bar, 1); fence_mbar_init(); }
        __syncwarp();
        if (warp == 0) tmem_alloc<128>(tmem_slot);
        fence_proxy_async();
        tc_fence_before();
        __syncthreads();
        tc_fence_after();
        tmem_base = *tmem_slot;
    } else {
        __syncthreads();
    }
    const uint32_t tmem_row = tmem_base + ((uint32_t)(warp * 32) << 16);
    uint32_t parity = 0;

    const uint32_t S = a.S;
    const float step = __fdiv_rn(__fsub_rn(a.far, a.near), (float)S);
    const uint64_t n_units = (a.R + a.rays_per_unit - 1) / a.rays_per_unit;
    uint32_t tile_counter = 0;

    for (uint64_t unit = blockIdx.x; unit < n_units; unit += gridDim.x) {
        for (uint32_t t = 0; t < a.tiles_per_unit; ++t, ++tile_counter) {
            const uint32_t u = t * TILE + tid;                  // sample index inside the unit
            const uint32_t ray_in_unit = u / S;
            const uint32_t k = u - ray_in_unit * S;
            const uint32_t k0_tile = (t * TILE) % S;
            const uint64_t ray = unit * a.rays_per_unit + ray_in_unit;
            const bool valid = ray < a.R;

            // ---- ray + sample position (nerf_renderer.py:127, oracle/sampler.py)
            float ox = 0.f, oy = 0.f, oz = 0.f, dx = 1.f, dy = 0.f, dz = 0.f, jit = 0.f;
            if (valid) {
                if constexpr (PANO) {
                    const int row = a.row0 + (int)(ray / (uint64_t)a.W), col = (int)(ray % (uint64_t)a.W);
                    const float yy = linspace_val_r(row, a.H), xx = linspace_val_r(col, a.W);
                    const float beta = -(yy - 0.5f) * 3.14159274101257324f;
                    const float alpha = -(xx - 0.5f) * 6.28318548202514648f;
                    float sa, ca, sb, cb;
                    sincosf(alpha, &sa, &ca); sincosf(beta, &sb, &cb);
                    const float cx = ca * cb, cy = sa * cb, cz = sb;
                    dx = a.pose_r[0] * cx + a.pose_r[1] * cy + a.pose_r[2] * cz;
                    dy = a.pose_r[3] * cx + a.pose_r[4] * cy + a.pose_r[5] * cz;
                    dz = a.pose_r[6] * cx + a.pose_r[7] * cy + a.pose_r[8] * cz;
                    ox = a.pose_t[0]; oy = a.pose_t[1]; oz = a.pose_t[2];
                } else {
                    ox = a.rays_o[3 * ray]; oy = a.rays_o[3 * ray + 1]; oz = a.rays_o[3 * ray + 2];
                    dx = a.rays_d[3 * ray]; dy = a.rays_d[3 * ray + 1]; dz = a.rays_d[3 * ray + 2];
                }
                if (a.training && a.jitter) jit = a.jitter[ray];
            }
            const float ts = __fadd_rn(a.near, __fmul_rn(__fadd_rn((float)k, jit), step));
            const float te = __fadd_rn(a.near, __fmul_rn(__fadd_rn((float)(k + 1), jit), step));
            const float tsum = __fadd_rn(ts, te);
            const float px = __fadd_rn(ox, __fmul_rn(dx, tsum) * 0.5f);
            const float py = __fadd_rn(oy, __fmul_rn(dy, tsum) * 0.5f);
            const float pz = __fadd_rn(oz, __fmul_rn(dz, tsum) * 0.5f);
            // ngp_nerf.py:137-140
            const float x = __fdiv_rn(__fsub_rn(px, a.aabb_min[0]), a.aabb_ext[0]);
            const float y = __fdiv_rn(__fsub_rn(py, a.aabb_min[1]), a.aabb_ext[1]);
            const float z = __fdiv_rn(__fsub_rn(pz, a.aabb_min[2]), a.aabb_ext[2]);
            const bool selector = valid && x > 0.f && x < 1.f && y > 0.f && y < 1.f && z > 0.f && z < 1.f;

            float sigma, cr, cg, cb;
            eval_fields<SIMT, -1>(a, sm, x, y, z, selector, tmem_base, tmem_row, parity, tid, sigma, cr, cg, cb);

            // ---- composite (nerf_renderer.py:170-183; oracle/composite.py)
            const float dt = __fsub_rn(te, ts);
            const float sd = valid ? sigma * dt : 0.f;
            float* carry_prev = sCarry + (tile_counter & 1u) * 8;
            float* carry_next = sCarry + ((tile_counter + 1u) & 1u) * 8;
            const bool has_carry = (t > 0);
            float sc[1] = {sd}, sx[1];
            ray_scan<1>(sc, sx, k, k0_tile, S, tid, sTails, has_carry ? carry_prev : nullptr, carry_next);
            const float T = expf(-sx[0]);
            const float alpha = 1.f - expf(-sd);
            const float w = T * alpha;
            const float tmid = tsum * 0.5f;
            float q[5] = {w, w * tmid, w * cr, w * cg, w * cb}, qx[5];
            ray_scan<5>(q, qx, k, k0_tile, S, tid, sTails + 32, has_carry ? carry_prev + 1 : nullptr, carry_next + 1);

            if (valid && k == S - 1) {
                const float op = q[0], one_m = 1.f - op;
                float dist = q[1], r = q[2], g = q[3], b = q[4];
                if (a.training) {                                 // nerf_renderer.py:192-194
                    float n0 = 0.f, n1 = 0.f, n2 = 0.f, n3 = 0.f;
                    if (a.bg_noise) { n0 = a.bg_noise[4 * ray]; n1 = a.bg_noise[4 * ray + 1]; n2 = a.bg_noise[4 * ray + 2]; n3 = a.bg_noise[4 * ray + 3]; }
                    dist = fmaxf(dist + (n3 * 2.f - 1.f) * one_m, 0.f);
                    r += n0 * one_m; g += n1 * one_m; b += n2 * one_m;
                } else {                                          // nerf_renderer.py:195-197
                    dist += 5.f * one_m;
                    r += 0.5f * one_m; g += 0.5f * one_m; b += 0.5f * one_m;
                }
                a.rgb[3 * ray] = r; a.rgb[3 * ray + 1] = g; a.rgb[3 * ray + 2] = b;
                a.distance[ray] = dist;
                if (a.opacity) a.opacity[ray] = op;
            }
            // the feature tiles / TMEM are rewritten by the next tile; every read of this tile
            // (MMA via mbarrier, tcgen05.ld via wait::ld, smem rows in SIMT mode) is complete and
            // the barrier before the next MMA issue orders them.
            if constexpr (SIMT) __syncthreads();
        }
    }

    if (!SIMT) {
        tc_fence_before();
        __syncthreads();
        if (warp == 0) tmem_dealloc<128>(tmem_base);
    }
}


// The ray of thread `tid` in work tile `tile` of the ray-marching kernels: a PATCH_W x PATCH_H pixel patch of the panorama
// window (PANO) or of a row-major image of explicit rays (patch), otherwise `rpt` consecutive explicit rays.  The origin and
// direction are left as they are for a thread without a ray (valid == false).  render_march_kernel has the same selection
// written inline: routed through this function, ptxas allocates its registers differently, and the benchmarked kernel's
// code is kept as measured.
template <bool PANO>
__device__ __forceinline__ void march_tile_ray(const RenderArgs& a, uint64_t tile, bool patch, uint32_t tiles_x, int rows, uint32_t rpt, int tid,
                                               uint64_t& ray, bool& valid, float& ox, float& oy, float& oz, float& dx, float& dy, float& dz)
{
    const int warp = tid >> 5, lane = tid & 31;
    if constexpr (PANO) {
        const int ty = (int)(tile / tiles_x), tx = (int)(tile % tiles_x);
        const int prow = ty * PATCH_H + (warp / PATCH_WX) * PATCH_WH + lane / PATCH_WW;   // row inside the window
        const int pcol = tx * PATCH_W + (warp % PATCH_WX) * PATCH_WW + lane % PATCH_WW;
        valid = prow < rows && pcol < a.W;
        ray = (uint64_t)prow * (uint64_t)a.W + (uint64_t)pcol;
        if (valid) {
            const float yy = linspace_val_r(a.row0 + prow, a.H), xx = linspace_val_r(pcol, a.W);
            const float beta = -(yy - 0.5f) * 3.14159274101257324f;
            const float alpha = -(xx - 0.5f) * 6.28318548202514648f;
            float sa, ca, sb, cb;
            sincosf(alpha, &sa, &ca); sincosf(beta, &sb, &cb);
            const float cx = ca * cb, cy = sa * cb, cz = sb;
            dx = a.pose_r[0] * cx + a.pose_r[1] * cy + a.pose_r[2] * cz;
            dy = a.pose_r[3] * cx + a.pose_r[4] * cy + a.pose_r[5] * cz;
            dz = a.pose_r[6] * cx + a.pose_r[7] * cy + a.pose_r[8] * cz;
            ox = a.pose_t[0]; oy = a.pose_t[1]; oz = a.pose_t[2];
        }
    } else {
        if (patch) {
            const int ty = (int)(tile / tiles_x), tx = (int)(tile % tiles_x);
            const int prow = ty * PATCH_H + (warp / PATCH_WX) * PATCH_WH + lane / PATCH_WW;
            const int pcol = tx * PATCH_W + (warp % PATCH_WX) * PATCH_WW + lane % PATCH_WW;
            valid = prow < rows && pcol < a.W;
            ray = (uint64_t)prow * (uint64_t)a.W + (uint64_t)pcol;
        } else {
            ray = tile * rpt + (uint32_t)tid % rpt;
            valid = ray < a.R;
        }
        if (valid) {
            ox = a.rays_o[3 * ray]; oy = a.rays_o[3 * ray + 1]; oz = a.rays_o[3 * ray + 2];
            dx = a.rays_d[3 * ray]; dy = a.rays_d[3 * ray + 1]; dz = a.rays_d[3 * ray + 2];
        }
    }
}

// ------------------------------------------------------------------------------------------------
// render_march_kernel: thread = RAY, the 128 rows of an MMA tile are 128 neighbouring rays at the
// same sample index k.  For a panorama a warp is an 8x4 pixel patch and a CTA a 16x8 patch, so the
// 32 lanes of every gather instruction sit next to each other in space (few distinct cache lines
// per request at the coarse and middle levels) and a thread revisits the same cells from k to k+1
// (temporal L1 reuse).  The composite is a per-thread running sum: no shuffles, no carries.
// Transmittance uses the sequential exclusive sum, the order of the oracle's cumsum.
template <bool PANO, bool SIMT, int NDENSE, int SAVE = 0, bool L0SMEM = false>
__global__ void __launch_bounds__(TILE, L0SMEM ? 3 : 4) render_march_kernel(const __grid_constant__ RenderArgs a)
{
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* sA   = smem + RS_A;
    uint8_t* sW1g = smem + RS_W1G;
    uint8_t* sW1a = smem + RS_W1A;
    uint8_t* sW2a = smem + RS_W2A;
    float*   sWoutG = reinterpret_cast<float*>(smem + RS_WOUT);
    float*   sWoutA = sWoutG + HID;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + RS_BAR);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + RS_BAR + 8);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const RenderSmem sm = {sA, sA, sA + A32_BYTES, sW1g, sW1a, sW2a, sWoutG, sWoutA, bar,
                           L0SMEM ? reinterpret_cast<const uint2*>(smem + RS_L0) : nullptr};

    stage_weights_bulk(smem, tid);                   // W1 density | W1 colour | W2 colour operand images, one UBLKCP
    uint32_t tmem_base = 0;
    if (!SIMT) {
        if (tid == 0) { mbar_init(bar, 1); fence_mbar_init(); }
        __syncwarp();
        if (warp == 0) tmem_alloc<128>(tmem_slot);
        fence_proxy_async();
        tc_fence_before();
        __syncthreads();
        tc_fence_after();
        tmem_base = *tmem_slot;
    } else {
        __syncthreads();
    }
    const uint32_t tmem_row = tmem_base + ((uint32_t)(warp * 32) << 16);
    uint32_t parity = 0;
    if constexpr (L0SMEM) {
        uint64_t* bar2 = reinterpret_cast<uint64_t*>(smem + RS_BAR2);
        if (tid == 0) {
            mbar_init(bar2, 1); fence_mbar_init();
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar2)), "r"(L0_BYTES) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         :: "r"(smem_u32(smem + RS_L0)), "l"(a.table), "r"(L0_BYTES), "r"(smem_u32(bar2)) : "memory");
        }
        __syncthreads();                                   // the barrier is initialised before anyone polls it
        mbar_wait(bar2, 0);
    }

    const uint32_t S = a.S;
    const float step = __fdiv_rn(__fsub_rn(a.far, a.near), (float)S);
    const float rext0 = __frcp_rn(a.aabb_ext[0]), rext1 = __frcp_rn(a.aabb_ext[1]), rext2 = __frcp_rn(a.aabb_ext[2]);
    // PANO, or explicit rays that form a row-major image of width a.W (perf_render_args.image_width):
    // tiles are 16x8 pixel patches; otherwise 128 consecutive rays
    const bool patch = PANO || a.W > 0;
    const int rows = patch ? (int)(a.R / (uint64_t)a.W) : 0;
    const uint32_t tiles_x = patch ? (uint32_t)((a.W + PATCH_W - 1) / PATCH_W) : 0u;
    const uint32_t seg = (PANO || patch || a.pk_offsets != nullptr || a.seg == 0) ? 1u : a.seg;
    const uint32_t rpt = TILE / seg, kps = S / seg;                 // rays per tile, samples per segment
    const uint32_t my_seg = (uint32_t)tid / rpt;
    const uint64_t n_tiles = patch ? (uint64_t)tiles_x * (uint64_t)((rows + PATCH_H - 1) / PATCH_H) : (a.R + rpt - 1) / rpt;

    for (uint64_t work = blockIdx.x; work < n_tiles; work += gridDim.x) {
        // Image-shaped work is dealt out in a scattered order: the tiles in flight at any moment (4 per SM) are spread over
        // the whole image instead of forming one band of neighbouring tiles that all pull the same table lines through the
        // same L2 slices at the same time (measured: profiles/r02_render_variants.md).
        const uint64_t tile = (patch && a.tile_mul > 1u) ? (work * a.tile_mul) % n_tiles : work;
        // ---- this thread's ray
        uint64_t ray; bool valid;
        float ox = 0.f, oy = 0.f, oz = 0.f, dx = 1.f, dy = 0.f, dz = 0.f, jit = 0.f;
        if constexpr (PANO) {
            const int ty = (int)(tile / tiles_x), tx = (int)(tile % tiles_x);
            const int prow = ty * PATCH_H + (warp / PATCH_WX) * PATCH_WH + lane / PATCH_WW;   // row inside the window
            const int pcol = tx * PATCH_W + (warp % PATCH_WX) * PATCH_WW + lane % PATCH_WW;
            valid = prow < rows && pcol < a.W;
            ray = (uint64_t)prow * (uint64_t)a.W + (uint64_t)pcol;
            if (valid) {
                const float yy = linspace_val_r(a.row0 + prow, a.H), xx = linspace_val_r(pcol, a.W);
                const float beta = -(yy - 0.5f) * 3.14159274101257324f;
                const float alpha = -(xx - 0.5f) * 6.28318548202514648f;
                float sa, ca, sb, cb;
                sincosf(alpha, &sa, &ca); sincosf(beta, &sb, &cb);
                const float cx = ca * cb, cy = sa * cb, cz = sb;
                dx = a.pose_r[0] * cx + a.pose_r[1] * cy + a.pose_r[2] * cz;
                dy = a.pose_r[3] * cx + a.pose_r[4] * cy + a.pose_r[5] * cz;
                dz = a.pose_r[6] * cx + a.pose_r[7] * cy + a.pose_r[8] * cz;
                ox = a.pose_t[0]; oy = a.pose_t[1]; oz = a.pose_t[2];
            }
        } else {
            if (patch) {
                const int ty = (int)(tile / tiles_x), tx = (int)(tile % tiles_x);
                const int prow = ty * PATCH_H + (warp / PATCH_WX) * PATCH_WH + lane / PATCH_WW;
                const int pcol = tx * PATCH_W + (warp % PATCH_WX) * PATCH_WW + lane % PATCH_WW;
                valid = prow < rows && pcol < a.W;
                ray = (uint64_t)prow * (uint64_t)a.W + (uint64_t)pcol;
            } else {
                ray = tile * rpt + (uint32_t)tid % rpt;
                valid = ray < a.R;
            }
            if (valid) {
                ox = a.rays_o[3 * ray]; oy = a.rays_o[3 * ray + 1]; oz = a.rays_o[3 * ray + 2];
                dx = a.rays_d[3 * ray]; dy = a.rays_d[3 * ray + 1]; dz = a.rays_d[3 * ray + 2];
            }
        }
        if (valid && a.training && a.jitter) jit = a.jitter[ray];

        float sum_sd = 0.f;                                   // exclusive running sum of sigma*dt
        float acc_w = 0.f, acc_d = 0.f, acc_r = 0.f, acc_g = 0.f, acc_b = 0.f;
        float dl_uni = 0.f, dl_bi = 0.f;                      // distortion loss pieces (SAVE only)
        // packed mode: every thread walks ITS ray's samples; the tile iterates to the longest ray
        // (neighbouring rays cross the same occupied shells, so lengths inside a tile are similar)
        uint32_t n_iter = kps, my_count = S;
        int64_t pk_base = 0;
        if (!PANO && a.pk_offsets != nullptr) {
            my_count = 0;
            if (valid) { pk_base = a.pk_offsets[ray]; my_count = (uint32_t)(a.pk_offsets[ray + 1] - pk_base); }
            const uint32_t wmax = __reduce_max_sync(0xffffffffu, my_count);
            uint32_t* s_max = reinterpret_cast<uint32_t*>(smem + RS_TAILS);
            __syncthreads();                                  // previous tile's readers are done
            if (lane == 0) s_max[warp] = wmax;
            __syncthreads();
            n_iter = max(max(s_max[0], s_max[1]), max(s_max[2], s_max[3]));
        }
#pragma unroll 1
        for (uint32_t kk = 0; kk < n_iter; ++kk) {
            const uint32_t k = my_seg * kps + kk;                 // seg == 1: k == kk
            const bool live = valid && k < my_count;
            float ts, te;
            if (!PANO && a.pk_offsets != nullptr) {
                ts = live ? a.pk_ts[pk_base + k] : 0.f; te = live ? a.pk_te[pk_base + k] : 0.f;
            } else {
                ts = __fadd_rn(a.near, __fmul_rn(__fadd_rn((float)k, jit), step));
                te = __fadd_rn(a.near, __fmul_rn(__fadd_rn((float)(k + 1), jit), step));
            }
            const float tsum = __fadd_rn(ts, te);
            const float px = __fadd_rn(ox, __fmul_rn(dx, tsum) * 0.5f);
            const float py = __fadd_rn(oy, __fmul_rn(dy, tsum) * 0.5f);
            const float pz = __fadd_rn(oz, __fmul_rn(dz, tsum) * 0.5f);
            const float x = div_uniform(__fsub_rn(px, a.aabb_min[0]), a.aabb_ext[0], rext0, a.div_generic != 0u);
            const float y = div_uniform(__fsub_rn(py, a.aabb_min[1]), a.aabb_ext[1], rext1, a.div_generic != 0u);
            const float z = div_uniform(__fsub_rn(pz, a.aabb_min[2]), a.aabb_ext[2], rext2, a.div_generic != 0u);
            const bool selector = live && x > 0.f && x < 1.f && y > 0.f && y < 1.f && z > 0.f && z < 1.f;

            float sigma, cr, cg, cb;
            const uint64_t srow = (SAVE != 0 && valid) ? (uint64_t)k * a.R + ray : ~0ull;
            eval_fields<SIMT, NDENSE, SAVE, L0SMEM>(a, sm, x, y, z, selector, tmem_base, tmem_row, parity, tid, sigma, cr, cg, cb, srow);

            const float dt = __fsub_rn(te, ts);
            const float sd = sigma * dt;
            const float T = expf(-sum_sd);
            const float w = T * (1.f - expf(-sd));
            sum_sd += sd;
            if constexpr (SAVE != 0) {
                if (valid) {
                    a.s_sigma[srow] = sigma; a.s_w[srow] = w; a.s_trans[srow] = T;
                    if constexpr (SAVE == 2) {
                        const __half2 c01 = __floats2half2_rn(cr, cg), c2 = __floats2half2_rn(cb, 0.f);
                        *reinterpret_cast<uint2*>(a.s_rgb + srow * 4) = make_uint2(*reinterpret_cast<const uint32_t*>(&c01), *reinterpret_cast<const uint32_t*>(&c2));
                    }
                }
                // torch_efficient_distloss, per ray: sum iv w^2 / 3 + 2 sum w (m W_excl - WM_excl)
                const float m = tsum * 0.5f;
                dl_uni = fmaf(dt * w, w, dl_uni);
                dl_bi = fmaf(w, m * acc_w - acc_d, dl_bi);
            }
            acc_w += w; acc_d = fmaf(w, tsum * 0.5f, acc_d);
            acc_r = fmaf(w, cr, acc_r); acc_g = fmaf(w, cg, acc_g); acc_b = fmaf(w, cb, acc_b);
            if constexpr (SIMT) __syncthreads();
        }

        bool writer = valid;
        if (seg > 1) {
            // combine the `seg` partial composites of every ray (each computed as if T = 1 at the segment
            // start): w = Toff w', Wx = Wpre + Toff Wx', ... ; scratch = the (now idle) feature tiles
            float* part = reinterpret_cast<float*>(sA);
            __syncthreads();
            part[0 * TILE + tid] = sum_sd; part[1 * TILE + tid] = acc_w; part[2 * TILE + tid] = acc_d;
            part[3 * TILE + tid] = acc_r;  part[4 * TILE + tid] = acc_g; part[5 * TILE + tid] = acc_b;
            part[6 * TILE + tid] = dl_uni; part[7 * TILE + tid] = dl_bi;
            __syncthreads();
            writer = valid && my_seg == 0;
            if (writer) {
                float cum_sd = 0.f, W = 0.f, D = 0.f, cr = 0.f, cg = 0.f, cb = 0.f, du = 0.f, db = 0.f;
                for (uint32_t sgi = 0; sgi < seg; ++sgi) {
                    const int t = (int)(sgi * rpt) + tid;         // thread that handled segment sgi of my ray
                    const float toff = expf(-cum_sd);
                    if (SAVE != 0) a.s_toff[(uint64_t)sgi * a.R + ray] = toff;
                    const float pW = part[1 * TILE + t], pD = part[2 * TILE + t];
                    du = fmaf(toff * toff, part[6 * TILE + t], du);
                    db += toff * (W * pD - D * pW) + toff * toff * part[7 * TILE + t];
                    W = fmaf(toff, pW, W); D = fmaf(toff, pD, D);
                    cr = fmaf(toff, part[3 * TILE + t], cr); cg = fmaf(toff, part[4 * TILE + t], cg); cb = fmaf(toff, part[5 * TILE + t], cb);
                    cum_sd += part[0 * TILE + t];
                }
                acc_w = W; acc_d = D; acc_r = cr; acc_g = cg; acc_b = cb; dl_uni = du; dl_bi = db;
            }
            __syncthreads();                                      // scratch is rewritten by the next tile's features
        }
        if (writer) {
            const float one_m = 1.f - acc_w;
            float dist = acc_d, r = acc_r, g = acc_g, b = acc_b;
            if constexpr (SAVE != 0) { a.s_dacc[ray] = acc_d; a.s_dl[ray] = dl_uni * (1.f / 3.f) + 2.f * dl_bi; }
            if (a.training) {                                     // nerf_renderer.py:192-194
                float n0 = 0.f, n1 = 0.f, n2 = 0.f, n3 = 0.f;
                if (a.bg_noise) { n0 = a.bg_noise[4 * ray]; n1 = a.bg_noise[4 * ray + 1]; n2 = a.bg_noise[4 * ray + 2]; n3 = a.bg_noise[4 * ray + 3]; }
                dist = fmaxf(dist + (n3 * 2.f - 1.f) * one_m, 0.f);
                r += n0 * one_m; g += n1 * one_m; b += n2 * one_m;
            } else {                                              // nerf_renderer.py:195-197
                dist += 5.f * one_m;
                r += 0.5f * one_m; g += 0.5f * one_m; b += 0.5f * one_m;
            }
            a.rgb[3 * ray] = r; a.rgb[3 * ray + 1] = g; a.rgb[3 * ray + 2] = b;
            a.distance[ray] = dist;
            if (a.opacity) a.opacity[ray] = acc_w;
        }
    }

    if (!SIMT) {
        tc_fence_before();
        __syncthreads();
        if (warp == 0) tmem_dealloc<128>(tmem_base);
    }
}

// ------------------------------------------------------------------------------------------------
// render_occ_kernel: the eval render of the occupancy-grid sampler (nerf_renderer.py:145-197) in ONE launch.  Tiles, tile
// order, weight staging and eval_fields are render_march_kernel's; the samples of a ray are not a fixed lattice but the
// intervals its grid walk emits (occ_walk.cuh), produced one per tile iteration by the thread that owns the ray.  A ray
// stops at its first interval whose exclusive transmittance is below early_stop_eps (nerfacc's
// render_visibility_from_density with alpha_thre = 0: T never increases, so no later interval could pass), i.e. only
// the intervals that contribute are evaluated, and nothing per sample leaves the SM.  The tile iterates until its last
// ray has stopped; rows without an interval enter eval_fields masked out.
struct OccRenderArgs {
    OccGrid   grid;
    float     early_stop_eps;
    uint32_t* n_samples;        // [R] intervals composited per ray, or null
};

template <bool PANO, bool SIMT, int NDENSE>
__global__ void __launch_bounds__(TILE, 4) render_occ_kernel(const __grid_constant__ RenderArgs a, const __grid_constant__ OccRenderArgs g)
{
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* sA   = smem + RS_A;
    uint8_t* sW1g = smem + RS_W1G;
    uint8_t* sW1a = smem + RS_W1A;
    uint8_t* sW2a = smem + RS_W2A;
    float*   sWoutG = reinterpret_cast<float*>(smem + RS_WOUT);
    float*   sWoutA = sWoutG + HID;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + RS_BAR);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + RS_BAR + 8);

    const int tid = threadIdx.x, warp = tid >> 5;
    const RenderSmem sm = {sA, sA, sA + A32_BYTES, sW1g, sW1a, sW2a, sWoutG, sWoutA, bar, nullptr};

    stage_weights_bulk(smem, tid);                   // W1 density | W1 colour | W2 colour operand images, one UBLKCP
    uint32_t tmem_base = 0;
    if (!SIMT) {
        if (tid == 0) { mbar_init(bar, 1); fence_mbar_init(); }
        __syncwarp();
        if (warp == 0) tmem_alloc<128>(tmem_slot);
        fence_proxy_async();
        tc_fence_before();
        __syncthreads();
        tc_fence_after();
        tmem_base = *tmem_slot;
    } else {
        __syncthreads();
    }
    const uint32_t tmem_row = tmem_base + ((uint32_t)(warp * 32) << 16);
    uint32_t parity = 0;

    const float rext0 = __frcp_rn(a.aabb_ext[0]), rext1 = __frcp_rn(a.aabb_ext[1]), rext2 = __frcp_rn(a.aabb_ext[2]);
    const bool patch = PANO || a.W > 0;
    const int rows = patch ? (int)(a.R / (uint64_t)a.W) : 0;
    const uint32_t tiles_x = patch ? (uint32_t)((a.W + PATCH_W - 1) / PATCH_W) : 0u;
    const uint64_t n_tiles = patch ? (uint64_t)tiles_x * (uint64_t)((rows + PATCH_H - 1) / PATCH_H) : (a.R + TILE - 1) / TILE;

    for (uint64_t work = blockIdx.x; work < n_tiles; work += gridDim.x) {
        const uint64_t tile = (patch && a.tile_mul > 1u) ? (work * a.tile_mul) % n_tiles : work;
        uint64_t ray; bool valid;
        float o[3] = {0.f, 0.f, 0.f}, d[3] = {1.f, 0.f, 0.f};
        march_tile_ray<PANO>(a, tile, patch, tiles_x, rows, TILE, tid, ray, valid, o[0], o[1], o[2], d[0], d[1], d[2]);
        OccWalk walk = {0.f, 0.f, 0u, 0u};
        if (valid) occ_walk_begin(g.grid, o, d, walk);

        bool live = valid;
        uint32_t n = 0;
        float sum_sd = 0.f;                                   // exclusive running sum of sigma*dt
        float acc_w = 0.f, acc_d = 0.f, acc_r = 0.f, acc_g = 0.f, acc_b = 0.f;
#pragma unroll 1
        for (;;) {
            // the next interval of my ray, unless the ray is exhausted or its transmittance fell below the cut
            float ts = 0.f, te = 0.f;
            const float T = expf(-sum_sd);
            live = live && T >= g.early_stop_eps && occ_walk_next(g.grid, o, d, walk, ts, te);
            // also orders the previous iteration's reads of the feature / hidden tiles before this one's writes
            if (!__syncthreads_or(live)) break;
            const float tsum = __fadd_rn(ts, te);
            const float px = __fadd_rn(o[0], __fmul_rn(d[0], tsum) * 0.5f);
            const float py = __fadd_rn(o[1], __fmul_rn(d[1], tsum) * 0.5f);
            const float pz = __fadd_rn(o[2], __fmul_rn(d[2], tsum) * 0.5f);
            const float x = div_uniform(__fsub_rn(px, a.aabb_min[0]), a.aabb_ext[0], rext0, a.div_generic != 0u);
            const float y = div_uniform(__fsub_rn(py, a.aabb_min[1]), a.aabb_ext[1], rext1, a.div_generic != 0u);
            const float z = div_uniform(__fsub_rn(pz, a.aabb_min[2]), a.aabb_ext[2], rext2, a.div_generic != 0u);
            const bool selector = live && x > 0.f && x < 1.f && y > 0.f && y < 1.f && z > 0.f && z < 1.f;

            float sigma, cr, cg, cb;
            eval_fields<SIMT, NDENSE>(a, sm, x, y, z, selector, tmem_base, tmem_row, parity, tid, sigma, cr, cg, cb);

            if (live) {                                       // render_march_kernel's composite, same operations in the same order
                const float sd = sigma * __fsub_rn(te, ts);
                const float w = T * (1.f - expf(-sd));
                sum_sd += sd;
                acc_w += w; acc_d = fmaf(w, tsum * 0.5f, acc_d);
                acc_r = fmaf(w, cr, acc_r); acc_g = fmaf(w, cg, acc_g); acc_b = fmaf(w, cb, acc_b);
                ++n;
            }
        }

        if (valid) {                                          // eval background rule, nerf_renderer.py:195-197
            const float one_m = 1.f - acc_w;
            a.rgb[3 * ray] = acc_r + 0.5f * one_m; a.rgb[3 * ray + 1] = acc_g + 0.5f * one_m; a.rgb[3 * ray + 2] = acc_b + 0.5f * one_m;
            a.distance[ray] = acc_d + 5.f * one_m;
            if (a.opacity) a.opacity[ray] = acc_w;
            if (g.n_samples) g.n_samples[ray] = n;
        }
    }

    if (!SIMT) {
        tc_fence_before();
        __syncthreads();
        if (warp == 0) tmem_dealloc<128>(tmem_base);
    }
}

// ------------------------------------------------------------------------------------------------
// packed_fields_kernel: both fields at PACKED samples (the output of the occupancy sampler), thread = sample,
// a tile = 128 CONSECUTIVE packed samples.  Consecutive samples of a ray are 5e-4 apart (nerf_renderer.py:151):
// a warp's 32 lanes sit in one cell of every level up to resolution ~1000, the best gather locality there is.
// Used by the fused occupancy-sampler training step (perf_train_forward_packed): writes sigma, the fp16 colour and
// the normalised position of every sample and saves the trained network's features / hidden activations at row n.
struct PackedFieldArgs {
    const int64_t* ray_indices;   // [N]
    const float*   ts;            // [N]
    const float*   te;            // [N]
    uint64_t       N;
    const int64_t* n_dev;         // optional live sample count in device memory (<= N = capacity)
    float*         sigma;         // [N]
    __half*        rgb;           // [N,4] fp16
    float*         x01;           // [N,3]
};

template <int NDENSE, int SAVE>
__global__ void __launch_bounds__(TILE, 4) packed_fields_kernel(const __grid_constant__ RenderArgs a, const PackedFieldArgs p)
{
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* sA   = smem + RS_A;
    uint8_t* sW1g = smem + RS_W1G;
    uint8_t* sW1a = smem + RS_W1A;
    uint8_t* sW2a = smem + RS_W2A;
    float*   sWoutG = reinterpret_cast<float*>(smem + RS_WOUT);
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + RS_BAR);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + RS_BAR + 8);
    const int tid = threadIdx.x, warp = tid >> 5;
    const RenderSmem sm = {sA, sA, sA + A32_BYTES, sW1g, sW1a, sW2a, sWoutG, sWoutG + HID, bar, nullptr};
    stage_weights_bulk(smem, tid);                   // W1 density | W1 colour | W2 colour operand images, one UBLKCP
    if (tid == 0) { mbar_init(bar, 1); fence_mbar_init(); }
    __syncwarp();
    if (warp == 0) tmem_alloc<128>(tmem_slot);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t tmem_row = tmem_base + ((uint32_t)(warp * 32) << 16);
    uint32_t parity = 0;
    uint64_t N = p.N;
    if (p.n_dev) { const int64_t nd = *p.n_dev; N = nd < 0 ? 0 : ((uint64_t)nd < N ? (uint64_t)nd : N); }      // graph-replayable count
    const uint64_t n_tiles = (N + TILE - 1) / TILE;
    const float rext0 = __frcp_rn(a.aabb_ext[0]), rext1 = __frcp_rn(a.aabb_ext[1]), rext2 = __frcp_rn(a.aabb_ext[2]);
    for (uint64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const uint64_t n = tile * TILE + tid;
        const bool valid = n < N;
        float x = 0.5f, y = 0.5f, z = 0.5f;
        if (valid) {
            const int64_t ray = p.ray_indices[n];
            const float tsum = __fadd_rn(p.ts[n], p.te[n]);
            const float px = __fadd_rn(a.rays_o[3 * ray], __fmul_rn(a.rays_d[3 * ray], tsum) * 0.5f);
            const float py = __fadd_rn(a.rays_o[3 * ray + 1], __fmul_rn(a.rays_d[3 * ray + 1], tsum) * 0.5f);
            const float pz = __fadd_rn(a.rays_o[3 * ray + 2], __fmul_rn(a.rays_d[3 * ray + 2], tsum) * 0.5f);
            x = div_uniform(__fsub_rn(px, a.aabb_min[0]), a.aabb_ext[0], rext0, a.div_generic != 0u);
            y = div_uniform(__fsub_rn(py, a.aabb_min[1]), a.aabb_ext[1], rext1, a.div_generic != 0u);
            z = div_uniform(__fsub_rn(pz, a.aabb_min[2]), a.aabb_ext[2], rext2, a.div_generic != 0u);
        }
        const bool selector = valid && x > 0.f && x < 1.f && y > 0.f && y < 1.f && z > 0.f && z < 1.f;
        float sigma, cr, cg, cb;
        eval_fields<false, NDENSE, SAVE>(a, sm, x, y, z, selector, tmem_base, tmem_row, parity, tid, sigma, cr, cg, cb, valid ? n : ~0ull);
        if (valid) {
            p.sigma[n] = sigma;
            const __half2 c01 = __floats2half2_rn(cr, cg), c2 = __floats2half2_rn(cb, 0.f);
            *reinterpret_cast<uint2*>(p.rgb + n * 4) = make_uint2(*reinterpret_cast<const uint32_t*>(&c01), *reinterpret_cast<const uint32_t*>(&c2));
            // masked-out samples: the in-box stand-in position the features were taken at (their gradient is zero)
            p.x01[3 * n] = selector ? x : 0.5f; p.x01[3 * n + 1] = selector ? y : 0.5f; p.x01[3 * n + 2] = selector ? z : 0.5f;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc<128>(tmem_base);
}

static int prepare_weights(const RenderArgs& a, cudaStream_t stream)
{
    static thread_local int sym_dev = -1; static thread_local float* sym = nullptr;
    int dev_ = 0; PERF_CUDA(cudaGetDevice(&dev_));
    if (sym_dev != dev_) { PERF_CUDA(cudaGetSymbolAddress((void**)&sym, c_wout)); sym_dev = dev_; }
    weights_prepare_kernel<<<1, 1024, 0, stream>>>(a.geo_w, a.app_w, sym);
    PERF_LAUNCH_CHECK();
    return PERF_OK;
}

// div_uniform()'s precondition: no box extent with an all-ones significand (Markstein's exception) or out of the normal range
static void set_div_mode(RenderArgs& a)
{
    a.div_generic = 0u;
    for (int i = 0; i < 3; ++i) if (!div_uniform_ok(a.aabb_ext[i])) a.div_generic = 1u;
}

static uint32_t gcd_u32(uint32_t a, uint32_t b) { while (b) { uint32_t t = a % b; a = b; b = t; } return a; }

// Table, weights, field box, flags and outputs of a render launch: everything but the sampler.  No CUDA call.
static int fill_render_args(const perf_render_args* args, RenderArgs& a, PackedLayout& pl)
{
    PERF_CHECK_ARG((uintptr_t)args->d_packed_table % 16 == 0 && (uintptr_t)args->d_geo_mlp_half % 16 == 0 && (uintptr_t)args->d_app_mlp_half % 16 == 0, "misaligned table / weights");
    uint64_t n_entries = 0;
    int rc = build_level_table(&args->grid, &a.lt, &n_entries); if (rc) return rc;
    PERF_CHECK_SUP(args->grid.n_levels == 16, "fused renderer needs n_levels == 16 (got %u)", args->grid.n_levels);
    a.table = (const uint2*)args->d_packed_table;
    pl = packed_layout(a.lt, n_entries);
    for (uint32_t l = 0; l < pl.n_cell_levels; ++l) a.cells[l] = reinterpret_cast<const uint4*>(a.table + pl.cell_start[l]);
    a.geo_w = (const __half*)args->d_geo_mlp_half; a.app_w = (const __half*)args->d_app_mlp_half;
    for (int i = 0; i < 3; ++i) { a.aabb_min[i] = args->aabb[i]; a.aabb_ext[i] = args->aabb[3 + i] - args->aabb[i]; }
    set_div_mode(a);
    a.training = (args->flags & PERF_FLAG_TRAINING) ? 1u : 0u;
    a.jitter = args->d_jitter; a.bg_noise = args->d_bg_noise;
    a.rgb = args->d_rgb; a.distance = args->d_distance; a.opacity = args->d_opacity;
    return PERF_OK;
}

#ifndef PERF_TILE_SCATTER
#define PERF_TILE_SCATTER 1
#endif
// Persistent grid of a render launch (4 CTAs per SM, at most one per work tile); image-shaped work (`image`) also gets
// its scattered tile order in a.tile_mul
static unsigned schedule_tiles(RenderArgs& a, uint64_t n_work, bool image)
{
    const unsigned grid = (unsigned)(n_work < (uint64_t)num_sms() * 4 ? n_work : (uint64_t)num_sms() * 4);
    a.tile_mul = 0;
    if (PERF_TILE_SCATTER && image && n_work > grid && n_work < (1ull << 31)) {
        // golden-ratio stride, made coprime with the tile count: consecutive work items land far apart, evenly spread
        uint32_t m = (uint32_t)((double)n_work * 0.6180339887498949) | 1u;
        while (m > 1u && gcd_u32(m, (uint32_t)n_work) != 1u) m += 2u;
        a.tile_mul = m % (uint32_t)n_work;
    }
    return grid;
}

static int launch_render(const perf_render_args* args, RenderArgs& a, bool pano, cudaStream_t stream, int save = 0)
{
    PERF_CHECK_ARG(args->d_packed_table && args->d_geo_mlp_half && args->d_app_mlp_half, "NULL table / weights");
    PERF_CHECK_ARG(args->d_rgb && args->d_distance, "NULL output");
    PERF_CHECK_ARG(args->n_samples >= 1 && args->n_samples <= 4096, "n_samples=%u not in [1,4096]", args->n_samples);
    PERF_CHECK_ARG(args->far > args->near, "far <= near");
    PackedLayout pl;
    int rc = fill_render_args(args, a, pl); if (rc) return rc;
    a.S = args->n_samples; a.near = args->near; a.far = args->far;
    const uint32_t g = gcd_u32(a.S, TILE);
    a.rays_per_unit = TILE / g; a.tiles_per_unit = a.S / g;       // unit = lcm(S,128) samples
    if (a.R == 0) return PERF_OK;
    const bool simt = (args->flags & PERF_FLAG_SIMT_MLP) != 0;
    const bool scan = (args->flags & PERF_FLAG_SCAN_KERNEL) != 0;
    uint64_t n_work;
    if (scan) n_work = (a.R + a.rays_per_unit - 1) / a.rays_per_unit;
    else if (pano || a.W > 0) n_work = (uint64_t)((a.W + PATCH_W - 1) / PATCH_W) * (uint64_t)(((int)(a.R / (uint64_t)a.W) + PATCH_H - 1) / PATCH_H);
    else {
        const uint32_t rpt = TILE / (a.seg ? a.seg : 1u);
        n_work = (a.R + rpt - 1) / rpt;
    }
    const unsigned grid = schedule_tiles(a, n_work, !scan && (pano || a.W > 0));
    rc = prepare_weights(a, stream); if (rc) return rc;     // constant-bank output weights + operand images (c_wout, g_wimg)
#define PERF_RENDER_LAUNCH(...) do { \
        auto k = __VA_ARGS__; \
        static thread_local int attr_dev = -1; int dev_ = 0; PERF_CUDA(cudaGetDevice(&dev_)); \
        if (attr_dev != dev_) { PERF_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, RS_LAUNCH)); \
            attr_dev = dev_; } \
        k<<<grid, TILE, RS_LAUNCH, stream>>>(a); } while (0)
    const bool fast = fast_addressing_ok(a.lt, 4) && pl.n_cell_levels == 4 && (args->flags & PERF_FLAG_GENERIC_ADDR) == 0;   // PeRF's grid: 4 dense + 12 hashed levels
    if (save != 0) {
        PERF_CHECK_SUP(!pano && !simt && !scan, "training forward runs on the ray-marching tensor-core kernel only");
        if (fast) { if (save == 1) PERF_RENDER_LAUNCH(render_march_kernel<false, false, 4, 1>); else PERF_RENDER_LAUNCH(render_march_kernel<false, false, 4, 2>); }
        else      { if (save == 1) PERF_RENDER_LAUNCH(render_march_kernel<false, false, -1, 1>); else PERF_RENDER_LAUNCH(render_march_kernel<false, false, -1, 2>); }
    } else if (scan) {
        if (pano) { if (simt) PERF_RENDER_LAUNCH(render_kernel<true, true>); else PERF_RENDER_LAUNCH(render_kernel<true, false>); }
        else      { if (simt) PERF_RENDER_LAUNCH(render_kernel<false, true>); else PERF_RENDER_LAUNCH(render_kernel<false, false>); }
    } else if (simt) {
        if (pano) PERF_RENDER_LAUNCH(render_march_kernel<true, true, -1>); else PERF_RENDER_LAUNCH(render_march_kernel<false, true, -1>);
    } else if (fast && pano && (args->flags & PERF_FLAG_L0_SMEM)) {
        auto k = render_march_kernel<true, false, 4, 0, true>;           // experiment: level 0 in shared memory, 3 CTAs/SM
        static thread_local int attr_dev0 = -1; int dev_ = 0; PERF_CUDA(cudaGetDevice(&dev_));
        if (attr_dev0 != dev_) { PERF_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, RS_TOTAL_L0)); attr_dev0 = dev_; }
        const unsigned grid3 = (unsigned)(n_work < (uint64_t)num_sms() * 3 ? n_work : (uint64_t)num_sms() * 3);
        k<<<grid3, TILE, RS_TOTAL_L0, stream>>>(a);
    } else if (fast) {
        if (pano) PERF_RENDER_LAUNCH(render_march_kernel<true, false, 4>); else PERF_RENDER_LAUNCH(render_march_kernel<false, false, 4>);
    } else {
        if (pano) PERF_RENDER_LAUNCH(render_march_kernel<true, false, -1>); else PERF_RENDER_LAUNCH(render_march_kernel<false, false, -1>);
    }
#undef PERF_RENDER_LAUNCH
    PERF_LAUNCH_CHECK();
    return PERF_OK;
}

// render_occ_kernel: every argument is checked before the first CUDA call
static int launch_render_occ(const perf_render_args* args, const perf_occ_render_args* occ, RenderArgs& a, bool pano, cudaStream_t stream)
{
    PERF_CHECK_ARG(args->d_packed_table && args->d_geo_mlp_half && args->d_app_mlp_half, "NULL table / weights");
    PERF_CHECK_ARG(args->d_rgb && args->d_distance, "NULL output");
    PERF_CHECK_SUP((args->flags & (PERF_FLAG_TRAINING | PERF_FLAG_SCAN_KERNEL | PERF_FLAG_L0_SMEM)) == 0,
                   "occupancy-grid rendering is eval mode on the ray-marching kernel (no TRAINING / SCAN_KERNEL / L0_SMEM flag)");
    PERF_CHECK_ARG(occ->d_binaries, "NULL occupancy grid");
    PERF_CHECK_ARG(occ->res[0] > 0 && occ->res[1] > 0 && occ->res[2] > 0, "occupancy grid resolution %d x %d x %d", occ->res[0], occ->res[1], occ->res[2]);
    PERF_CHECK_ARG(occ->aabb[3] > occ->aabb[0] && occ->aabb[4] > occ->aabb[1] && occ->aabb[5] > occ->aabb[2], "empty occupancy grid box");
    PERF_CHECK_ARG(occ->step > 0.f && occ->far > occ->near, "bad occupancy lattice near=%g far=%g step=%g", occ->near, occ->far, occ->step);
    PERF_CHECK_ARG(occ->early_stop_eps >= 0.f && occ->early_stop_eps < 1.f, "early_stop_eps=%g not in [0,1)", occ->early_stop_eps);
    PackedLayout pl;
    int rc = fill_render_args(args, a, pl); if (rc) return rc;
    OccRenderArgs g; memset(&g, 0, sizeof(g));
    g.grid.binaries = occ->d_binaries;
    for (int i = 0; i < 3; ++i) {
        g.grid.res[i] = occ->res[i];
        g.grid.amin[i] = occ->aabb[i]; g.grid.amax[i] = occ->aabb[3 + i]; g.grid.aext[i] = occ->aabb[3 + i] - occ->aabb[i];
    }
    g.grid.near = occ->near; g.grid.far = occ->far; g.grid.step = occ->step;
    g.early_stop_eps = occ->early_stop_eps; g.n_samples = occ->d_n_samples;
    if (a.R == 0) return PERF_OK;
    const bool image = pano || a.W > 0;
    const uint64_t n_work = image ? (uint64_t)((a.W + PATCH_W - 1) / PATCH_W) * (uint64_t)(((int)(a.R / (uint64_t)a.W) + PATCH_H - 1) / PATCH_H)
                                  : (a.R + TILE - 1) / TILE;
    const unsigned grid = schedule_tiles(a, n_work, image);
    rc = prepare_weights(a, stream); if (rc) return rc;
#define PERF_OCC_LAUNCH(...) do { \
        auto k = __VA_ARGS__; \
        static thread_local int attr_dev = -1; int dev_ = 0; PERF_CUDA(cudaGetDevice(&dev_)); \
        if (attr_dev != dev_) { PERF_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, RS_LAUNCH)); \
            attr_dev = dev_; } \
        k<<<grid, TILE, RS_LAUNCH, stream>>>(a, g); } while (0)
    const bool simt = (args->flags & PERF_FLAG_SIMT_MLP) != 0;
    const bool fast = fast_addressing_ok(a.lt, 4) && pl.n_cell_levels == 4 && (args->flags & PERF_FLAG_GENERIC_ADDR) == 0;
    if (pano) {
        if (simt) { if (fast) PERF_OCC_LAUNCH(render_occ_kernel<true, true, 4>);  else PERF_OCC_LAUNCH(render_occ_kernel<true, true, -1>); }
        else      { if (fast) PERF_OCC_LAUNCH(render_occ_kernel<true, false, 4>); else PERF_OCC_LAUNCH(render_occ_kernel<true, false, -1>); }
    } else {
        if (simt) { if (fast) PERF_OCC_LAUNCH(render_occ_kernel<false, true, 4>);  else PERF_OCC_LAUNCH(render_occ_kernel<false, true, -1>); }
        else      { if (fast) PERF_OCC_LAUNCH(render_occ_kernel<false, false, 4>); else PERF_OCC_LAUNCH(render_occ_kernel<false, false, -1>); }
    }
#undef PERF_OCC_LAUNCH
    PERF_LAUNCH_CHECK();
    return PERF_OK;
}

}  // namespace perf

using namespace perf;

extern "C" {
#pragma GCC visibility push(default)

int perf_render_rays(const perf_render_args* args, const float* d_rays_o, const float* d_rays_d, uint64_t R, void* stream)
{
    PERF_CHECK_ARG(args && d_rays_o && d_rays_d, "NULL pointer");
    RenderArgs a; memset(&a, 0, sizeof(a));
    a.rays_o = d_rays_o; a.rays_d = d_rays_d; a.R = R;
    if (args->image_width > 0 && (args->flags & PERF_FLAG_SCAN_KERNEL) == 0) {
        PERF_CHECK_ARG(R % args->image_width == 0, "image_width=%u does not divide the %llu rays", args->image_width, (unsigned long long)R);
        a.W = (int)args->image_width;
    }
    return launch_render(args, a, false, (cudaStream_t)stream);
}

int perf_render_packed(const perf_render_args* args, const float* d_rays_o, const float* d_rays_d, uint64_t R,
                       const int64_t* d_offsets, const float* d_t_starts, const float* d_t_ends, void* stream)
{
    PERF_CHECK_ARG(args && d_rays_o && d_rays_d && d_offsets, "NULL pointer");
    PERF_CHECK_SUP((args->flags & (PERF_FLAG_SCAN_KERNEL | PERF_FLAG_TRAINING)) == 0, "packed rendering: eval mode on the ray-marching kernel only");
    RenderArgs a; memset(&a, 0, sizeof(a));
    a.rays_o = d_rays_o; a.rays_d = d_rays_d; a.R = R;
    a.pk_offsets = d_offsets; a.pk_ts = d_t_starts; a.pk_te = d_t_ends;
    perf_render_args t = *args; t.n_samples = 1; if (!(t.far > t.near)) { t.near = 0.f; t.far = 1.f; }
    return launch_render(&t, a, false, (cudaStream_t)stream);
}

int perf_train_forward(const perf_render_args* args, const float* d_rays_o, const float* d_rays_d, uint64_t R, int phase,
                       const perf_train_buffers* buf, void* stream)
{
    PERF_CHECK_ARG(args && d_rays_o && d_rays_d && buf, "NULL pointer");
    PERF_CHECK_ARG(phase == PERF_PHASE_GEO || phase == PERF_PHASE_APP, "phase must be PERF_PHASE_GEO or PERF_PHASE_APP");
    PERF_CHECK_ARG(buf->d_sigma && buf->d_weights && buf->d_trans && buf->d_feat && buf->d_h1 && buf->d_dist_acc && buf->d_distloss, "NULL training buffer");
    PERF_CHECK_ARG(phase == PERF_PHASE_GEO || (buf->d_rgb && buf->d_h2), "colour phase needs d_rgb and d_h2");
    PERF_CHECK_ARG(((uintptr_t)buf->d_feat | (uintptr_t)buf->d_h1 | (uintptr_t)buf->d_h2) % 16 == 0 && (uintptr_t)buf->d_rgb % 8 == 0, "misaligned training buffer");
    RenderArgs a; memset(&a, 0, sizeof(a));
    a.rays_o = d_rays_o; a.rays_d = d_rays_d; a.R = R;
    a.s_sigma = buf->d_sigma; a.s_w = buf->d_weights; a.s_trans = buf->d_trans; a.s_rgb = (__half*)buf->d_rgb;
    a.s_feat = (uint4*)buf->d_feat; a.s_h1 = (uint4*)buf->d_h1; a.s_h2 = (uint4*)buf->d_h2;
    a.s_dacc = buf->d_dist_acc; a.s_dl = buf->d_distloss;
    // split rays into segments until the tiles fill the machine (4 CTAs / SM), if the caller gave room
    a.seg = 1; a.s_toff = buf->d_seg_trans;
    if (buf->d_seg_trans != nullptr) {
        const uint64_t slots = (uint64_t)num_sms() * 4;
        while (a.seg < PERF_MAX_SEGMENTS && args->n_samples % (a.seg * 2) == 0 && (R * a.seg + TILE - 1) / TILE < slots) a.seg *= 2;
    }
    PERF_CHECK_ARG(buf->h_segments_out != nullptr || a.seg == 1, "d_seg_trans given without h_segments_out");
    if (buf->h_segments_out) *buf->h_segments_out = a.seg;
    perf_render_args t = *args; t.flags |= PERF_FLAG_TRAINING;
    return launch_render(&t, a, false, (cudaStream_t)stream, phase);
}

int perf_fields_packed(const perf_render_args* args, const float* d_rays_o, const float* d_rays_d, const int64_t* d_ray_indices,
                       const float* d_t_starts, const float* d_t_ends, uint64_t N, const int64_t* d_n_dev, int phase, float* d_sigma, void* d_rgb_half4,
                       float* d_x01, void* d_feat, void* d_h1, void* d_h2, void* stream)
{
    PERF_CHECK_ARG(args && d_rays_o && d_rays_d && d_ray_indices && d_t_starts && d_t_ends && d_sigma && d_rgb_half4 && d_x01, "NULL pointer");
    PERF_CHECK_ARG(phase == 0 || phase == PERF_PHASE_GEO || phase == PERF_PHASE_APP, "phase must be 0, PERF_PHASE_GEO or PERF_PHASE_APP");
    PERF_CHECK_ARG(phase == 0 || (d_feat && d_h1 && (phase == PERF_PHASE_GEO || d_h2)), "NULL save buffer");
    PERF_CHECK_ARG(args->d_packed_table && args->d_geo_mlp_half && args->d_app_mlp_half, "NULL table / weights");
    PERF_CHECK_ARG(((uintptr_t)d_feat | (uintptr_t)d_h1 | (uintptr_t)d_h2) % 16 == 0 && (uintptr_t)d_rgb_half4 % 8 == 0, "misaligned buffer");
    RenderArgs a; memset(&a, 0, sizeof(a));
    uint64_t n_entries = 0;
    int rc = build_level_table(&args->grid, &a.lt, &n_entries); if (rc) return rc;
    PERF_CHECK_SUP(args->grid.n_levels == 16, "fused field kernel needs n_levels == 16 (got %u)", args->grid.n_levels);
    a.table = (const uint2*)args->d_packed_table;
    PERF_CHECK_ARG((uintptr_t)args->d_packed_table % 16 == 0, "misaligned table");
    const PackedLayout pl = packed_layout(a.lt, n_entries);
    for (uint32_t l = 0; l < pl.n_cell_levels; ++l) a.cells[l] = reinterpret_cast<const uint4*>(a.table + pl.cell_start[l]);
    a.geo_w = (const __half*)args->d_geo_mlp_half; a.app_w = (const __half*)args->d_app_mlp_half;
    for (int i = 0; i < 3; ++i) { a.aabb_min[i] = args->aabb[i]; a.aabb_ext[i] = args->aabb[3 + i] - args->aabb[i]; }
    set_div_mode(a);
    a.rays_o = d_rays_o; a.rays_d = d_rays_d;
    a.s_feat = (uint4*)d_feat; a.s_h1 = (uint4*)d_h1; a.s_h2 = (uint4*)d_h2;
    if (N == 0) return PERF_OK;
    PackedFieldArgs p = {d_ray_indices, d_t_starts, d_t_ends, N, d_n_dev, d_sigma, (__half*)d_rgb_half4, d_x01};
    cudaStream_t st = (cudaStream_t)stream;
    rc = prepare_weights(a, st); if (rc) return rc;
    const uint64_t n_tiles = (N + TILE - 1) / TILE;
    const unsigned grid = (unsigned)(n_tiles < (uint64_t)num_sms() * 4 ? n_tiles : (uint64_t)num_sms() * 4);
    const bool fast = fast_addressing_ok(a.lt, 4) && pl.n_cell_levels == 4 && (args->flags & PERF_FLAG_GENERIC_ADDR) == 0;
#define PERF_PACKED_LAUNCH(...) do { \
        auto k = __VA_ARGS__; \
        static thread_local int attr_dev = -1; int dev_ = 0; PERF_CUDA(cudaGetDevice(&dev_)); \
        if (attr_dev != dev_) { PERF_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, RS_TOTAL)); attr_dev = dev_; } \
        k<<<grid, TILE, RS_TOTAL, st>>>(a, p); } while (0)
    if (fast) {
        if (phase == 0) PERF_PACKED_LAUNCH(packed_fields_kernel<4, 0>);
        else if (phase == PERF_PHASE_GEO) PERF_PACKED_LAUNCH(packed_fields_kernel<4, 1>);
        else PERF_PACKED_LAUNCH(packed_fields_kernel<4, 2>);
    } else {
        if (phase == 0) PERF_PACKED_LAUNCH(packed_fields_kernel<-1, 0>);
        else if (phase == PERF_PHASE_GEO) PERF_PACKED_LAUNCH(packed_fields_kernel<-1, 1>);
        else PERF_PACKED_LAUNCH(packed_fields_kernel<-1, 2>);
    }
#undef PERF_PACKED_LAUNCH
    PERF_LAUNCH_CHECK();
    return PERF_OK;
}

int perf_render_pano(const perf_render_args* args, const float* h_pose, int H, int W, int row0, int rows, void* stream)
{
    PERF_CHECK_ARG(args && h_pose, "NULL pointer");
    PERF_CHECK_ARG(H > 0 && W > 0 && row0 >= 0 && rows >= 0 && row0 + rows <= H, "bad panorama window H=%d W=%d row0=%d rows=%d", H, W, row0, rows);
    RenderArgs a; memset(&a, 0, sizeof(a));
    for (int r = 0; r < 3; ++r) { for (int c = 0; c < 3; ++c) a.pose_r[3 * r + c] = h_pose[4 * r + c]; a.pose_t[r] = h_pose[4 * r + 3]; }
    a.H = H; a.W = W; a.row0 = row0; a.R = (uint64_t)rows * W;
    return launch_render(args, a, true, (cudaStream_t)stream);
}

int perf_render_rays_occ(const perf_render_args* args, const perf_occ_render_args* occ, const float* d_rays_o, const float* d_rays_d,
                         uint64_t R, void* stream)
{
    PERF_CHECK_ARG(args && occ && d_rays_o && d_rays_d, "NULL pointer");
    RenderArgs a; memset(&a, 0, sizeof(a));
    a.rays_o = d_rays_o; a.rays_d = d_rays_d; a.R = R;
    if (args->image_width > 0) {
        PERF_CHECK_ARG(R % args->image_width == 0, "image_width=%u does not divide the %llu rays", args->image_width, (unsigned long long)R);
        a.W = (int)args->image_width;
    }
    return launch_render_occ(args, occ, a, false, (cudaStream_t)stream);
}

int perf_render_pano_occ(const perf_render_args* args, const perf_occ_render_args* occ, const float* h_pose, int H, int W, int row0, int rows,
                         void* stream)
{
    PERF_CHECK_ARG(args && occ && h_pose, "NULL pointer");
    PERF_CHECK_ARG(H > 0 && W > 0 && row0 >= 0 && rows >= 0 && row0 + rows <= H, "bad panorama window H=%d W=%d row0=%d rows=%d", H, W, row0, rows);
    RenderArgs a; memset(&a, 0, sizeof(a));
    for (int r = 0; r < 3; ++r) { for (int c = 0; c < 3; ++c) a.pose_r[3 * r + c] = h_pose[4 * r + c]; a.pose_t[r] = h_pose[4 * r + 3]; }
    a.H = H; a.W = W; a.row0 = row0; a.R = (uint64_t)rows * W;
    return launch_render_occ(args, occ, a, true, (cudaStream_t)stream);
}

#pragma GCC visibility pop
}  // extern "C"
