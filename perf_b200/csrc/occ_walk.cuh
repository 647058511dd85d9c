// occ_walk.cuh -- the occupancy-grid walk of ONE ray as a resumable generator: every call of occ_walk_next() yields the
// ray's next emitted interval [t_start, t_end).  The expressions are those of occ.cu::occ_march_ray with u = 0 (eval
// mode: no jitter) -- slab clip, midpoint test, cell index, empty-cell jump with its 3-step margin, PERF_OCC_MAX_STEPS
// bound -- so the intervals are bit-identical to that sampler's (tests/test_occ_walk_host.py).  Used by render.cu's
// render_occ_kernel, which marches, evaluates and composites a ray one interval at a time; __host__ __device__ so that
// tests/occ_walk_harness.cu runs the same body on the CPU.
#pragma once
#include "common.cuh"

namespace perf {

constexpr uint32_t OCC_WALK_MAX_STEPS = 1u << 22;      // == occ.cu's PERF_OCC_MAX_STEPS: lattice points one ray may visit

// launch-uniform grid and lattice (a kernel parameter: lives in the constant bank, costs no registers)
struct OccGrid {
    const uint8_t* binaries;     // [res0][res1][res2], x slowest
    int            res[3];
    float          amin[3], aext[3], amax[3];
    float          near, far, step;
};

// per-ray state between calls: the ray/box overlap and the next lattice index to test
struct OccWalk {
    float    tn, tf;
    uint32_t k, k_end;           // k == k_end: the ray is exhausted
};

__host__ __device__ __forceinline__ void occ_walk_begin(const OccGrid& g, const float (&o)[3], const float (&d)[3], OccWalk& w)
{
    float tn = -INFINITY, tf = INFINITY;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const float inv = PERF_FDIV_RN(1.0f, fabsf(d[i]) < 1e-12f ? 1e-12f : d[i]);
        const float t0 = PERF_FMUL_RN(PERF_FSUB_RN(g.amin[i], o[i]), inv), t1 = PERF_FMUL_RN(PERF_FSUB_RN(g.amax[i], o[i]), inv);
        tn = fmaxf(tn, fminf(t0, t1)); tf = fminf(tf, fmaxf(t0, t1));
    }
    tn = fmaxf(tn, g.near); tf = fminf(tf, g.far);
    w.tn = tn; w.tf = tf; w.k = 0u; w.k_end = 0u;
    if (tf >= tn) {
        const float kf = floorf((tn - g.near) / g.step - 0.5f) - 2.0f;
        w.k = kf > 0.f ? (uint32_t)kf : 0u;
        const float span = (tf - tn) / g.step;
        w.k_end = span < (float)OCC_WALK_MAX_STEPS ? w.k + (uint32_t)span + 8u : w.k;
    }
}

// Advances the ray to its next emitted interval: true and (ts, te), or false once the ray has none left.
__host__ __device__ __forceinline__ bool occ_walk_next(const OccGrid& g, const float (&o)[3], const float (&d)[3], OccWalk& w,
                                                       float& ts, float& te)
{
    const float half_step = PERF_FMUL_RN(0.5f, g.step);
    for (; w.k < w.k_end; ++w.k) {
        const float t = PERF_FADD_RN(g.near, PERF_FMUL_RN((float)w.k, g.step));
        const float mid = PERF_FADD_RN(t, half_step);
        if (mid > w.tf) { w.k_end = w.k; break; }
        if (mid < w.tn) continue;
        int c[3]; float pnt[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const float p = PERF_FADD_RN(o[i], PERF_FMUL_RN(d[i], mid));
            pnt[i] = p;
            const int ci = (int)floorf(PERF_FMUL_RN(PERF_FDIV_RN(PERF_FSUB_RN(p, g.amin[i]), g.aext[i]), (float)g.res[i]));
            c[i] = ci < 0 ? 0 : (ci > g.res[i] - 1 ? g.res[i] - 1 : ci);
        }
        if (g.binaries[((int64_t)c[0] * g.res[1] + c[1]) * g.res[2] + c[2]]) {
            ts = t; te = PERF_FADD_RN(t, g.step);
            ++w.k;
            return true;
        }
        // empty cell: jump to 3 lattice steps before its exit (occ_march_ray explains the margin)
        float t_exit = INFINITY;
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const float cell = g.aext[i] / (float)g.res[i];
            if (d[i] > 1e-9f)       t_exit = fminf(t_exit, mid + (g.amin[i] + (float)(c[i] + 1) * cell - pnt[i]) / d[i]);
            else if (d[i] < -1e-9f) t_exit = fminf(t_exit, mid + (g.amin[i] + (float)c[i] * cell - pnt[i]) / d[i]);
        }
        if (t_exit < INFINITY) {
            const float kf2 = floorf((t_exit - g.near) / g.step - 0.5f) - 3.0f;
            if (kf2 > (float)w.k && kf2 < (float)w.k_end) w.k = (uint32_t)kf2;          // the loop's ++k follows
        }
    }
    return false;
}

}  // namespace perf
