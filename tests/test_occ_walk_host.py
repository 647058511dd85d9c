"""The resumable occupancy-grid walker of the one-launch grid renderer (perf_b200/csrc/occ_walk.cuh, compiled for the
host from tests/occ_walk_harness.cu) against the two-pass sampler occ.cu::occ_march_ray (tests/host_harness.py) and
oracle/occ_sampler.py: the intervals it yields must be bit-identical.  Also the argument checks of perf_render_rays_occ /
perf_render_pano_occ, which all run before the first CUDA call (no device needed)."""
import ctypes as C
import hashlib
import os
import subprocess

import numpy as np
import pytest
import torch
from hypothesis import given, settings, strategies as st

import host_harness as hh
from oracle.occ_sampler import occ_sample

AABB = [-1.0, -1.0, -1.0, 1.0, 1.0, 1.0]
HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(os.path.dirname(HERE), "perf_b200", "csrc")
_WALK_LIB = None


def walk_lib():
    """tests/occ_walk_harness.cu compiled for the host (as host_harness.py compiles its sources: round-to-nearest intrinsics
    become plain IEEE operations, no contraction) into tests/_build/, one object per content of its sources."""
    global _WALK_LIB
    if _WALK_LIB is None:
        from perf_b200.build import _nvcc
        srcs = [os.path.join(HERE, "occ_walk_harness.cu"), os.path.join(CSRC, "occ_walk.cuh"), os.path.join(CSRC, "common.cuh"),
                os.path.join(os.path.dirname(HERE), "include", "perfb200.h")]
        h = hashlib.sha256(b"".join(open(f, "rb").read() for f in srcs)).hexdigest()[:16]
        out = os.path.join(HERE, "_build", f"libocc_walk_harness-{h}.so")
        if not os.path.exists(out):
            os.makedirs(os.path.dirname(out), exist_ok=True)
            tmp = f"{out}.{os.getpid()}.tmp"
            cmd = [_nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-O2", "-std=c++17", "--shared", "-Xcompiler", "-fPIC",
                   "-Xcompiler", "-fvisibility=hidden", "-Xcompiler", "-ffp-contract=off", srcs[0], "-o", tmp]
            proc = subprocess.run(cmd, capture_output=True, text=True)
            if proc.returncode != 0:
                raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + proc.stdout + proc.stderr)
            os.replace(tmp, out)
        _WALK_LIB = C.CDLL(out)
        _WALK_LIB.perf_host_occ_walk.restype = C.c_int
    return _WALK_LIB


def occ_walk(binaries: np.ndarray, aabb, rays_o: np.ndarray, rays_d: np.ndarray, near: float, far: float, step: float):
    """occ_walk_begin / occ_walk_next of every ray to its end -> (ray_indices, t_starts, t_ends), packed in ray order."""
    f = walk_lib().perf_host_occ_walk
    bins = np.ascontiguousarray(binaries, np.uint8)
    o, d = np.ascontiguousarray(rays_o, np.float32), np.ascontiguousarray(rays_d, np.float32)
    res3 = (C.c_int * 3)(*binaries.shape)
    a6 = (C.c_float * 6)(*[float(v) for v in aabb])
    R, n = o.shape[0], C.c_uint64(0)
    args = (hh._p(bins), res3, a6, hh._p(o), hh._p(d), C.c_uint64(R), C.c_float(near), C.c_float(far), C.c_float(step))
    assert f(*args, C.c_uint64(0), None, None, None, C.byref(n)) == 0
    cap = max(int(n.value), 1)
    ri, ts, te = np.zeros(cap, np.int64), np.zeros(cap, np.float32), np.zeros(cap, np.float32)
    assert f(*args, C.c_uint64(cap), hh._p(ri), hh._p(ts), hh._p(te), C.byref(n)) == 0
    k = int(n.value)
    return ri[:k], ts[:k], te[:k]


def _assert_same(got, want, what):
    for name, g, w in zip(("ray_indices", "t_starts", "t_ends"), got, want):
        w = w.numpy() if torch.is_tensor(w) else w
        assert np.array_equal(g, w), f"{what}: {name}"
        if name != "ray_indices":
            assert g.view(np.uint32).tolist() == np.asarray(w, np.float32).view(np.uint32).tolist(), f"{what}: {name} bits"


def _rays(g, n):
    o = (torch.rand(n, 3, generator=g) * 2 - 1) * 1.3                 # some origins outside [-1,1]^3
    d = torch.nn.functional.normalize(torch.randn(n, 3, generator=g), dim=-1)
    d[0] = torch.tensor([1.0, 0.0, 0.0])                                # axis-parallel: two zero components
    d[1] = torch.tensor([0.0, 0.0, -1.0])
    d[2] = torch.tensor([0.0, 1.0, 0.0]); o[2] = torch.tensor([0.3, -1.5, 0.2])     # enters through a face, from outside
    o[3] = torch.tensor([3.0, 3.0, 3.0]); d[3] = torch.tensor([1.0, 0.0, 0.0])      # never enters the box
    o[4] = torch.tensor([1.6, 0.1, -0.2]); d[4] = torch.tensor([-1.0, 0.0, 0.0])    # outside, pointing at the box
    o[5] = torch.zeros(3)
    return o, d


@settings(max_examples=80, deadline=None)
@given(seed=st.integers(0, 2 ** 20), rx=st.integers(1, 24), ry=st.integers(1, 24), rz=st.integers(1, 24),
       step=st.sampled_from([5e-4, 3e-3, 1e-2, 0.0625, 0.3]), near=st.sampled_from([0.0, 1e-2, 0.2]),
       far=st.sampled_from([0.5, 1.5, 4.0]), occupancy=st.sampled_from([0.0, 0.05, 0.3, 0.6, 1.0]))
def test_walker_matches_two_pass_sampler_and_oracle(seed, rx, ry, rz, step, near, far, occupancy):
    g = torch.Generator().manual_seed(seed)
    binaries = torch.rand(rx, ry, rz, generator=g) < occupancy
    n_rays = 24 if step < 1e-3 else 64
    o, d = _rays(g, n_rays)
    got = occ_walk(binaries.numpy(), AABB, o.numpy(), d.numpy(), near, far, step)
    _assert_same(got, hh.occ_sample(binaries.numpy(), AABB, o.numpy(), d.numpy(), near, far, step), "occ_march_ray")
    _assert_same(got, occ_sample(binaries, torch.tensor(AABB), o, d, near, far, step), "oracle")
    assert np.all(np.diff(got[0]) >= 0), "packed in ray order"
    if occupancy == 0.0:
        assert got[0].size == 0


def test_non_unit_box_and_axis_parallel_rays():
    g = torch.Generator().manual_seed(11)
    aabb = [-0.5, -1.0, -0.25, 1.5, 0.5, 0.75]
    binaries = torch.rand(7, 5, 3, generator=g) < 0.5
    o, d = _rays(g, 48)
    for i, axis in enumerate(torch.eye(3)):                             # rays along +-x, +-y, +-z through the box centre
        o[6 + 2 * i], d[6 + 2 * i] = torch.tensor([0.5, -0.25, 0.25]), axis
        o[7 + 2 * i], d[7 + 2 * i] = torch.tensor([0.5, -0.25, 0.25]), -axis
    got = occ_walk(binaries.numpy(), aabb, o.numpy(), d.numpy(), 0.0, 4.0, 0.01)
    _assert_same(got, hh.occ_sample(binaries.numpy(), aabb, o.numpy(), d.numpy(), 0.0, 4.0, 0.01), "occ_march_ray")
    _assert_same(got, occ_sample(binaries, torch.tensor(aabb), o, d, 0.0, 4.0, 0.01), "oracle")
    assert all((got[0] == r).any() for r in range(6, 12)), "every axis-parallel ray through the centre emits"


def test_one_cell_grid_lattice():
    """A single occupied cell in the middle: the walker emits exactly the global-lattice intervals whose midpoint is
    inside the cell, starting on a lattice point, not at the cell entry."""
    res, step = 5, 0.03
    binaries = torch.zeros(res, res, res, dtype=torch.bool)
    binaries[2, 2, 2] = True                                            # cell [-0.2, 0.2]^3
    o = torch.tensor([[-0.96, 0.01, -0.02]])
    d = torch.tensor([[1.0, 0.0, 0.0]])
    ri, ts, te = occ_walk(binaries.numpy(), AABB, o.numpy(), d.numpy(), 0.0, 1.5, step)
    _assert_same((ri, ts, te), occ_sample(binaries, torch.tensor(AABB), o, d, 0.0, 1.5, step), "oracle")
    k = ts / step
    assert np.allclose(k, np.round(k), atol=1e-3)
    mids = ts + 0.5 * step
    assert mids.min() >= 0.76 and mids.max() <= 1.16 and mids.min() - step < 0.76 and mids.max() + step > 1.16
    assert abs(ts[0] - 0.76) > 1e-3


def test_perf_lattice_on_sparse_256_shell():
    """PeRF's sampler (near 0, far 1.5, step 5e-4: up to 3000 lattice points per ray) on a 256^3 grid whose occupied
    cells form a thin spherical shell -- the empty-cell jumps of the walk are exercised thousands of times per ray."""
    n = 256
    c = (np.arange(n) + 0.5) / n * 2 - 1
    r = np.sqrt(c[:, None, None] ** 2 + c[None, :, None] ** 2 + c[None, None, :] ** 2)
    binaries = (np.abs(r - 0.8) < 0.02)
    assert 0.001 < binaries.mean() < 0.05
    g = torch.Generator().manual_seed(3)
    o = (torch.rand(64, 3, generator=g) - 0.5) * 0.4
    d = torch.nn.functional.normalize(torch.randn(64, 3, generator=g), dim=-1)
    d[0] = torch.tensor([0.0, 0.0, 1.0])
    got = occ_walk(binaries, AABB, o.numpy(), d.numpy(), 0.0, 1.5, 5e-4)
    _assert_same(got, hh.occ_sample(binaries, AABB, o.numpy(), d.numpy(), 0.0, 1.5, 5e-4), "occ_march_ray")
    _assert_same(got, occ_sample(torch.from_numpy(binaries), torch.tensor(AABB), o, d, 0.0, 1.5, 5e-4), "oracle")
    counts = np.bincount(got[0], minlength=64)
    assert counts.min() > 0, "every ray from inside crosses the shell"


# ---------------------------------------------------------------- argument checks of the C entry points
@pytest.fixture(scope="module")
def lib():
    from perf_b200 import _lib
    return _lib.load()


def _args(flags=0):
    from perf_b200 import _lib
    from perf_b200.config import PERF_GRID
    a = _lib.RenderArgs()
    a.grid = PERF_GRID.c()
    a.d_packed_table = a.d_geo_mlp_half = a.d_app_mlp_half = 0x10000          # never dereferenced: the checks fail first
    a.aabb = (C.c_float * 6)(*AABB)
    a.flags = flags
    a.d_rgb = a.d_distance = 0x20000
    g = _lib.OccRenderArgs()
    g.d_binaries = 0x30000
    g.res = (C.c_int * 3)(16, 16, 16)
    g.aabb = (C.c_float * 6)(*AABB)
    g.near, g.far, g.step, g.early_stop_eps = 0.0, 1.5, 5e-4, 1e-4
    return a, g


def _both(lib, a, g):
    rays = 0x40000
    pose = (C.c_float * 16)(*np.eye(4, dtype=np.float32).ravel().tolist())
    return (lib.perf_render_rays_occ(C.byref(a), C.byref(g), rays, rays, 128, None),
            lib.perf_render_pano_occ(C.byref(a), C.byref(g), pose, 8, 16, 0, 8, None))


@pytest.mark.parametrize("field,value", [("d_binaries", None), ("res", (0, 16, 16)), ("res", (16, -1, 16)), ("step", 0.0),
                                         ("step", -5e-4), ("far", 0.0), ("far", float("nan")), ("early_stop_eps", -1e-4),
                                         ("early_stop_eps", 1.0), ("early_stop_eps", float("nan")), ("aabb", (1., -1., -1., -1., 1., 1.))])
def test_bad_occupancy_arguments(lib, field, value):
    a, g = _args()
    setattr(g, field, (C.c_int * 3)(*value) if field == "res" else (C.c_float * 6)(*value) if field == "aabb" else value)
    assert _both(lib, a, g) == (-1, -1), lib.perf_last_error()


def test_bad_render_arguments(lib):
    a, g = _args()
    assert lib.perf_render_rays_occ(C.byref(a), None, 0x40000, 0x40000, 128, None) == -1
    assert lib.perf_render_rays_occ(C.byref(a), C.byref(g), None, 0x40000, 128, None) == -1
    a.image_width = 100                                                    # does not divide the 128 rays
    assert lib.perf_render_rays_occ(C.byref(a), C.byref(g), 0x40000, 0x40000, 128, None) == -1
    pose = (C.c_float * 16)(*np.eye(4, dtype=np.float32).ravel().tolist())
    a, g = _args()
    assert lib.perf_render_pano_occ(C.byref(a), C.byref(g), pose, 8, 16, 4, 8, None) == -1      # rows past the panorama
    assert lib.perf_render_pano_occ(C.byref(a), C.byref(g), None, 8, 16, 0, 8, None) == -1
    a.d_rgb = None
    assert _both(lib, a, g) == (-1, -1)
    a, g = _args()
    a.d_packed_table = None
    assert _both(lib, a, g) == (-1, -1)
    a, g = _args()
    a.d_packed_table = 0x10008                                             # not 16-byte aligned
    assert _both(lib, a, g) == (-1, -1)


@pytest.mark.parametrize("flag", ["PERF_FLAG_TRAINING", "PERF_FLAG_SCAN_KERNEL", "PERF_FLAG_L0_SMEM"])
def test_unsupported_flags(lib, flag):
    from perf_b200 import _lib
    a, g = _args(getattr(_lib, flag))
    assert _both(lib, a, g) == (-2, -2)
    assert b"eval mode" in lib.perf_last_error()
