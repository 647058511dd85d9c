// TEST HARNESS (compiled only by tests/test_occ_walk_host.py into tests/_build/, never into libperfb200.so): a host entry
// point that runs the __host__ __device__ occupancy-grid walker of perf_b200/csrc/occ_walk.cuh over host arrays, so the
// CPU test-suite can compare its intervals with the two-pass sampler (occ.cu::occ_march_ray) and the oracle.
#include "../perf_b200/csrc/occ_walk.cuh"

using namespace perf;

extern "C" {
#pragma GCC visibility push(default)

// occ_walk_begin / occ_walk_next over R host rays, each walked to its end: the emitted intervals in ray order (at most
// `capacity` are written) and their total in *n_total -- the packed output of occ_march_ray with no jitter
int perf_host_occ_walk(const uint8_t* h_binaries, const int* h_res3, const float* h_aabb6, const float* h_rays_o, const float* h_rays_d,
                       uint64_t R, float near, float far, float step, uint64_t capacity, int64_t* ray_indices, float* t_starts,
                       float* t_ends, uint64_t* n_total)
{
    if (!h_binaries || !h_res3 || !h_aabb6 || !h_rays_o || !h_rays_d || !n_total) return PERF_EINVAL;
    OccGrid g;
    g.binaries = h_binaries;
    for (int i = 0; i < 3; ++i) {
        g.res[i] = h_res3[i]; g.amin[i] = h_aabb6[i]; g.amax[i] = h_aabb6[3 + i]; g.aext[i] = h_aabb6[3 + i] - h_aabb6[i];
    }
    g.near = near; g.far = far; g.step = step;
    uint64_t n = 0;
    for (uint64_t r = 0; r < R; ++r) {
        const float o[3] = {h_rays_o[3 * r], h_rays_o[3 * r + 1], h_rays_o[3 * r + 2]};
        const float d[3] = {h_rays_d[3 * r], h_rays_d[3 * r + 1], h_rays_d[3 * r + 2]};
        OccWalk w; occ_walk_begin(g, o, d, w);
        float ts, te;
        while (occ_walk_next(g, o, d, w, ts, te)) {
            if (n < capacity) { ray_indices[n] = (int64_t)r; t_starts[n] = ts; t_ends[n] = te; }
            ++n;
        }
    }
    *n_total = n;
    return PERF_OK;
}

#pragma GCC visibility pop
}
