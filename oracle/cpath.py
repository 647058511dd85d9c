"""ctypes wrapper of oracle/cpath.c (the plain-C / OpenMP restatement of the eval render path).

TEST INFRASTRUCTURE ONLY.  Compiled lazily with gcc for the CPU it runs on (`-march=native`), one
shared object per CPU-flag set under oracle/_build/ (git-ignored), so the object built in the
build container is never executed on a different host CPU."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def _cpu_tag() -> str:
    try:
        flags = next(l for l in open("/proc/cpuinfo") if l.startswith("flags"))
    except Exception:
        flags = "unknown"
    return hashlib.sha1(flags.encode()).hexdigest()[:10]


def build() -> str:
    """Up-to-date object under oracle/_build/, compiled there when the tree is writable, else in a temporary directory."""
    src = os.path.join(HERE, "cpath.c")
    name = f"liboracle_c_{_cpu_tag()}.so"
    out_dir = os.path.join(HERE, "_build")
    out = os.path.join(out_dir, name)
    if os.path.exists(out) and os.path.getmtime(src) <= os.path.getmtime(out):
        return out
    try:
        os.makedirs(out_dir, exist_ok=True)
    except OSError:
        pass
    if not os.access(out_dir, os.W_OK):
        out_dir = os.path.join(tempfile.gettempdir(), f"perf_b200_oracle_{os.getuid()}")
        os.makedirs(out_dir, exist_ok=True)
        out = os.path.join(out_dir, name)
    if not os.path.exists(out) or os.path.getmtime(src) > os.path.getmtime(out):
        tmp = f"{out}.{os.getpid()}.tmp"
        cmd = ["gcc", "-O3", "-march=native", "-fopenmp", "-shared", "-fPIC", "-o", tmp, src, "-lm"]
        proc = subprocess.run(cmd, capture_output=True, text=True)
        if proc.returncode != 0:
            raise RuntimeError("gcc failed: " + " ".join(cmd) + "\n" + proc.stderr)
        os.replace(tmp, out)
    return out


def lib() -> C.CDLL:
    global _LIB
    if _LIB is None:
        _LIB = C.CDLL(build())
        fp = C.POINTER(C.c_float)
        _LIB.oracle_render_rays.restype = C.c_int
        _LIB.oracle_render_rays.argtypes = [fp, fp, fp, fp, C.c_long, C.c_int, C.c_float, C.c_float, fp, fp, fp, C.c_int]
        _LIB.oracle_c_max_threads.restype = C.c_int
    return _LIB


def max_threads() -> int:
    return int(lib().oracle_c_max_threads())


def render_rays(field, rays_o: torch.Tensor, rays_d: torch.Tensor, n_samples: int, near: float = 1e-2, far: float = 1.0,
                n_threads: int = 0):
    """Eval-mode render (mixed precision) of [R,3] rays -> dict(rgb [R,3], distance [R,1], opacities [R,1])."""
    as_f = lambda t: np.ascontiguousarray(t.detach().cpu().numpy(), dtype=np.float32)
    g, a, o, d = as_f(field.geo_params), as_f(field.app_params), as_f(rays_o.reshape(-1, 3)), as_f(rays_d.reshape(-1, 3))
    R = o.shape[0]
    rgb, dist, op = np.empty((R, 3), np.float32), np.empty((R, 1), np.float32), np.empty((R, 1), np.float32)
    p = lambda x: x.ctypes.data_as(C.POINTER(C.c_float))
    rc = lib().oracle_render_rays(p(g), p(a), p(o), p(d), R, int(n_samples), float(near), float(far), p(rgb), p(dist), p(op), int(n_threads))
    if rc != 0:
        raise MemoryError("oracle_render_rays failed")
    return {"rgb": torch.from_numpy(rgb), "distance": torch.from_numpy(dist), "opacities": torch.from_numpy(op)}
