"""torch-facing wrappers over the C-ABI of libperfb200.so + the autograd Functions built on them.

PyTorch is plumbing here: it owns device memory and the current stream; every op below hands raw
pointers to the library, which enqueues hand-written sm_100a kernels on that stream.  There is no
CPU path: a non-CUDA tensor raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

from . import _lib
from .config import APP_MLP, GEO_MLP, PERF_GRID, GridConfig, MLPConfig

_L = _lib.load


def _stream() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t: Optional[torch.Tensor]) -> Optional[C.c_void_p]:
    return None if t is None else C.c_void_p(t.data_ptr())


def _chk(t: torch.Tensor, dtype, name: str) -> torch.Tensor:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError(f"perf_b200: `{name}` must be a CUDA tensor (there is no CPU path)")
    if t.dtype != dtype:
        raise TypeError(f"perf_b200: `{name}` must be {dtype}, got {t.dtype}")
    return t.contiguous()


def launch_count() -> int:
    """Number of libperfb200 kernel launches issued through this module (bench.py reports it)."""
    return _LAUNCHES[0]


_LAUNCHES = [0]


_NVTX = os.environ.get("PERF_B200_NVTX") == "1"     # NVTX range per C-ABI call (SURVEY 5: ranges around K1-K7), for nsys / ncu --nvtx


def _call(fn, *args, launches: int = 1):
    if _NVTX:
        torch.cuda.nvtx.range_push(getattr(fn, "__name__", None) or getattr(fn, "_name", "perf"))
        try:
            _lib.check(fn(*args))
        finally:
            torch.cuda.nvtx.range_pop()
    else:
        _lib.check(fn(*args))
    _LAUNCHES[0] += launches


# ------------------------------------------------------------------ parameters / tables
def params_to_half(params: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    params = _chk(params, torch.float32, "params")
    if out is None:
        out = torch.empty_like(params, dtype=torch.float16)
    with torch.cuda.device(params.device):
        _call(_L().perf_params_to_half, _p(params), _p(out), params.numel(), _stream())
    return out


_PACKED_ROWS = {}


def packed_table_entries(grid: GridConfig = PERF_GRID) -> int:
    """Rows of the packed gather table of a grid (entries + cell-major dense levels): perf_packed_table_entries."""
    key = (grid.n_levels, grid.n_features_per_level, grid.log2_hashmap_size, grid.base_resolution, grid.per_level_scale, grid.interpolation)
    n = _PACKED_ROWS.get(key)
    if n is None:
        v = C.c_uint64(0)
        _call(_L().perf_packed_table_entries, grid.c(), C.byref(v))
        n = _PACKED_ROWS[key] = int(v.value)
    return n


def pack_tables(geo_half: torch.Tensor, app_half: torch.Tensor, grid: GridConfig = PERF_GRID,
                geo_mlp: MLPConfig = GEO_MLP, app_mlp: MLPConfig = APP_MLP,
                out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Interleaved {geo.f0, geo.f1, app.f0, app.f1} fp16 table [packed_table_entries(grid), 4]: the first n_entries rows in
    parameter order, then the cell-major copy of the dense levels (include/perfb200.h::perf_pack_tables)."""
    geo_half, app_half = _chk(geo_half, torch.float16, "geo_half"), _chk(app_half, torch.float16, "app_half")
    n_rows = packed_table_entries(grid)
    if out is None:
        out = torch.empty(n_rows, 4, dtype=torch.float16, device=geo_half.device)
    if out.shape[0] != n_rows or out.dtype != torch.float16 or not out.is_contiguous():
        raise ValueError(f"pack_tables: out must be a contiguous fp16 [{n_rows}, 4] tensor, got {tuple(out.shape)} {out.dtype}")
    with torch.cuda.device(geo_half.device):
        _call(_L().perf_pack_tables, grid.c(), geo_mlp.c(), app_mlp.c(), _p(geo_half), _p(app_half), _p(out), _stream())
    return out


# ------------------------------------------------------------------ ray generation
_POSE_CACHE = {}


def _pose_array(pose) -> "C.Array":
    """The 4x4 pose by value (a kernel parameter).  A pose that lives on the GPU -- the reference makes CUDA the default
    tensor type, `core_exp_runner.py:266` -- costs a device-to-host read: cached per (storage, version), so a pose rendered
    again (row tiles, repeated frames) is read once."""
    key = None
    if torch.is_tensor(pose) and pose.is_cuda:
        key = (pose.data_ptr(), pose._version, tuple(pose.shape))
        hit = _POSE_CACHE.get(key)
        if hit is not None:
            return hit
    flat = [float(v) for v in torch.as_tensor(pose, dtype=torch.float32).cpu().reshape(-1).tolist()]
    assert len(flat) == 16, "pose must be 4x4"
    arr = (C.c_float * 16)(*flat)
    if key is not None:
        if len(_POSE_CACHE) > 64:
            _POSE_CACHE.clear()
        _POSE_CACHE[key] = arr
    return arr


def raygen_pano(pose, H: int, W: int, row0: int = 0, rows: Optional[int] = None, device="cuda"):
    """(rays_o, rays_d) [rows, W, 3]; `utils/camera_utils.py:229-234` gen_pano_rays."""
    rows = H - row0 if rows is None else rows
    dev = torch.device(device)
    o = torch.empty(rows, W, 3, dtype=torch.float32, device=dev)
    d = torch.empty(rows, W, 3, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _call(_L().perf_raygen_pano, _pose_array(pose), H, W, row0, rows, _p(o), _p(d), _stream())
    return o, d


def raygen_pers(pose, fov: float, res: int, width: Optional[int] = None, device="cuda"):
    """(rays_o, rays_d) [res, width, 3]; `utils/camera_utils.py:237-241` gen_pers_rays (width defaults to res)."""
    width = res if width is None else width
    dev = torch.device(device)
    o = torch.empty(res, width, 3, dtype=torch.float32, device=dev)
    d = torch.empty(res, width, 3, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _call(_L().perf_raygen_pers, _pose_array(pose), float(fov), res, width, _p(o), _p(d), _stream())
    return o, d


# ------------------------------------------------------------------ hash grid
def hashgrid_fwd(table_half: torch.Tensor, x01: torch.Tensor, grid: GridConfig = PERF_GRID) -> torch.Tensor:
    table_half, x01 = _chk(table_half, torch.float16, "table"), _chk(x01, torch.float32, "x01")
    N = x01.shape[0]
    feat = torch.empty(N, grid.n_features, dtype=torch.float16, device=x01.device)
    with torch.cuda.device(x01.device):
        _call(_L().perf_hashgrid_fwd, grid.c(), _p(table_half), _p(x01), N, _p(feat), _stream())
    return feat


def hashgrid_bwd(x01: torch.Tensor, dfeat: torch.Tensor, grid: GridConfig = PERF_GRID,
                 out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """d(table) [n_entries, 2] fp32 (+= into ``out`` when given)."""
    x01, dfeat = _chk(x01, torch.float32, "x01"), _chk(dfeat, torch.float32, "dfeat")
    if out is None:
        out = torch.zeros(grid.n_entries, 2, dtype=torch.float32, device=x01.device)
    with torch.cuda.device(x01.device):
        _call(_L().perf_hashgrid_bwd, grid.c(), _p(x01), _p(dfeat), x01.shape[0], _p(out), _stream())
    return out


def hashgrid_bwd_input(table_half: torch.Tensor, x01: torch.Tensor, dfeat: torch.Tensor, grid: GridConfig = PERF_GRID) -> torch.Tensor:
    """d(loss)/d(x01) [N,3] fp32 of the encode (Linear or Smoothstep); ``dfeat`` [N, L*2] fp32."""
    table_half, x01, dfeat = _chk(table_half, torch.float16, "table"), _chk(x01, torch.float32, "x01"), _chk(dfeat, torch.float32, "dfeat")
    dx = torch.empty_like(x01)
    if x01.shape[0] == 0:
        return dx
    with torch.cuda.device(x01.device):
        _call(_L().perf_hashgrid_bwd_input, grid.c(), _p(table_half), _p(x01), _p(dfeat), x01.shape[0], _p(dx), _stream())
    return dx


def hashgrid_bwd_bwd_input(table_half: torch.Tensor, x01: torch.Tensor, dfeat: torch.Tensor, ddx: torch.Tensor,
                           grid: GridConfig = PERF_GRID, want=(True, True, True)):
    """Double backward of :func:`hashgrid_bwd_input`.  ``ddx`` [N,3] = d(loss)/d(dx).  Returns
    ``(d_dfeat [N, L*2], d_table [n_entries, 2], d_x01 [N,3])`` fp32, ``None`` where ``want`` is False."""
    table_half, x01 = _chk(table_half, torch.float16, "table"), _chk(x01, torch.float32, "x01")
    dfeat, ddx = _chk(dfeat, torch.float32, "dfeat"), _chk(ddx, torch.float32, "ddx")
    N, dev = x01.shape[0], x01.device
    ddfeat = torch.empty(N, grid.n_features, dtype=torch.float32, device=dev) if want[0] else None
    dtable = torch.zeros(grid.n_entries, 2, dtype=torch.float32, device=dev) if want[1] else None
    dx2 = torch.zeros(N, 3, dtype=torch.float32, device=dev) if want[2] else None
    if N and any(want):
        with torch.cuda.device(dev):
            _call(_L().perf_hashgrid_bwd_bwd_input, grid.c(), _p(table_half), _p(x01), _p(dfeat), _p(ddx), N,
                  _p(ddfeat), _p(dtable), _p(dx2), _stream())
    return ddfeat, dtable, dx2


def hashgrid_bwd_rays(rays_o, rays_d, jitter, n_samples: int, near: float, far: float, dfeat: torch.Tensor,
                      aabb=(-1., -1., -1., 1., 1., 1.), grid: GridConfig = PERF_GRID, out: Optional[torch.Tensor] = None):
    """d(table) from sample-major rows (row = k * R + ray) whose positions are recomputed from the
    rays (fixed-S sampler); coarse levels are accumulated per cell along each ray before the atomics."""
    rays_o, rays_d, dfeat = _chk(rays_o, torch.float32, "rays_o"), _chk(rays_d, torch.float32, "rays_d"), _chk(dfeat, torch.float32, "dfeat")
    jitter = None if jitter is None else _chk(jitter, torch.float32, "jitter")
    if out is None:
        out = torch.zeros(grid.n_entries, 2, dtype=torch.float32, device=rays_o.device)
    a6 = (C.c_float * 6)(*[float(v) for v in aabb])
    with torch.cuda.device(rays_o.device):
        _call(_L().perf_hashgrid_bwd_rays, grid.c(), a6, _p(rays_o), _p(rays_d), _p(jitter), rays_o.shape[0], n_samples,
              near, far, _p(dfeat), _p(out), _stream(), launches=2)
    return out


# ------------------------------------------------------------------ network (encode + MLP)
def network_fwd(params_half: torch.Tensor, x01: torch.Tensor, grid: GridConfig, mlp: MLPConfig,
                save: bool = False, simt: bool = False):
    """tcnn NetworkWithInputEncoding.forward.  Returns out [N, n_out] fp16, or
    (out, feat, h1, h2) when ``save`` (h2 is None for 1-hidden-layer nets)."""
    params_half, x01 = _chk(params_half, torch.float16, "params_half"), _chk(x01, torch.float32, "x01")
    N, dev = x01.shape[0], x01.device
    out = torch.empty(N, mlp.n_out, dtype=torch.float16, device=dev)
    feat = h1 = h2 = None
    if save:
        feat = torch.empty(N, 32, dtype=torch.float16, device=dev)
        h1 = torch.empty(N, 64, dtype=torch.float16, device=dev)
        if mlp.n_hidden_layers == 2:
            h2 = torch.empty(N, 64, dtype=torch.float16, device=dev)
    with torch.cuda.device(dev):
        _call(_L().perf_network_fwd, grid.c(), mlp.c(), _p(params_half), _p(x01), N, _p(out),
              _p(feat), _p(h1), _p(h2), _lib.PERF_FLAG_SIMT_MLP if simt else 0, _stream())
    return (out, feat, h1, h2) if save else out


def mlp_fwd(weights_half: torch.Tensor, feat: torch.Tensor, mlp: MLPConfig, save: bool = False, simt: bool = False):
    weights_half, feat = _chk(weights_half, torch.float16, "weights_half"), _chk(feat, torch.float16, "feat")
    N, dev = feat.shape[0], feat.device
    out = torch.empty(N, mlp.n_out, dtype=torch.float16, device=dev)
    h1 = torch.empty(N, 64, dtype=torch.float16, device=dev) if save else None
    h2 = torch.empty(N, 64, dtype=torch.float16, device=dev) if save and mlp.n_hidden_layers == 2 else None
    with torch.cuda.device(dev):
        _call(_L().perf_mlp_fwd, mlp.c(), _p(weights_half), _p(feat), N, _p(out), _p(h1), _p(h2),
              _lib.PERF_FLAG_SIMT_MLP if simt else 0, _stream())
    return (out, h1, h2) if save else out


def mlp_backward(mlp: MLPConfig, weights_half: torch.Tensor, feat, h1, h2, out, dout: torch.Tensor):
    """Backward of the bias-free MLP from the saved fp16 activations.  Returns
    (d_weights_flat fp32 [mlp.n_params], dfeat fp32 [N,32]).

    The three weight-gradient products and the two activation-gradient products are plain GEMMs
    (cuBLAS through torch.matmul, fp32); the ReLU / sigmoid masks are elementwise."""
    W = weights_half.float()
    w1 = W[:64 * 32].view(64, 32)
    p = 64 * 32
    w2 = None
    if mlp.n_hidden_layers == 2:
        w2 = W[p:p + 64 * 64].view(64, 64); p += 64 * 64
    wout = W[p:p + mlp.padded_out * 64].view(mlp.padded_out, 64)[:mlp.n_out]
    dz = dout.float()
    if mlp.output_activation == "Sigmoid":
        y = out.float()
        dz = dz * y * (1.0 - y)
    h_last = (h2 if w2 is not None else h1).float()
    d_wout = torch.zeros(mlp.padded_out, 64, dtype=torch.float32, device=dz.device)
    d_wout[:mlp.n_out] = dz.t() @ h_last
    dh = (dz @ wout) * (h_last > 0)
    grads = []
    if w2 is not None:
        h1f = h1.float()
        d_w2 = dh.t() @ h1f
        dh = (dh @ w2) * (h1f > 0)
        grads.append(d_w2.reshape(-1))
    d_w1 = dh.t() @ feat.float()
    dfeat = dh @ w1
    return torch.cat([d_w1.reshape(-1)] + grads + [d_wout.reshape(-1)]), dfeat.contiguous()


class _NetworkFunction(torch.autograd.Function):
    """out = MLP(encode(x01; params[grid]); params[mlp]), differentiable w.r.t. ``params``."""

    @staticmethod
    def forward(ctx, params, x01, grid, mlp, params_half):
        need_grad = ctx.needs_input_grad[0]
        if params_half is None:
            params_half = params_to_half(params.detach())
        x01 = x01.detach().float().contiguous()
        if need_grad:
            out, feat, h1, h2 = network_fwd(params_half, x01, grid, mlp, save=True)
            ctx.save_for_backward(x01, params_half, feat, h1, h2 if h2 is not None else h1, out)
        else:
            out = network_fwd(params_half, x01, grid, mlp)
        ctx.grid, ctx.mlp = grid, mlp
        return out

    @staticmethod
    def backward(ctx, dout):
        x01, params_half, feat, h1, h2, out = ctx.saved_tensors
        grid, mlp = ctx.grid, ctx.mlp
        dz = dout.float()
        if mlp.output_activation == "Sigmoid":
            y = out.float()
            dz = dz * y * (1.0 - y)
        # one flat gradient in the parameter layout [MLP | grid]; fp16 tensor-core GEMMs for the MLP part
        grad = torch.zeros(mlp.n_params + 2 * grid.n_entries, dtype=torch.float32, device=dz.device)
        _, dfeat = mlp_backward_half(mlp, params_half[:mlp.n_params], feat, h1, h2 if mlp.n_hidden_layers == 2 else None,
                                     dz.contiguous(), grad_out=grad[:mlp.n_params])
        hashgrid_bwd(x01, dfeat, grid, out=grad[mlp.n_params:].view(-1, 2))
        return grad, None, None, None, None


def network_apply(params: torch.Tensor, x01: torch.Tensor, grid: GridConfig, mlp: MLPConfig,
                  params_half: Optional[torch.Tensor] = None) -> torch.Tensor:
    return _NetworkFunction.apply(params, x01, grid, mlp, params_half)


class _EncodingFunction(torch.autograd.Function):
    """tcnn.Encoding: feat = encode(x01; params), differentiable w.r.t. ``params`` and -- when the
    positions require grad -- w.r.t. ``x01``, once more differentiable through that input gradient
    (tcnn's ``_module_function`` / ``_module_function_backward`` pair; what
    `pano_joint_predictor.py:58-64` needs for ``autograd.grad(distance, directions, create_graph=True)``)."""

    @staticmethod
    def forward(ctx, params, x01, grid):
        xd = x01.detach().float().contiguous()
        half = params_to_half(params.detach()).view(-1, 2)
        feat = hashgrid_fwd(half, xd, grid)
        ctx.save_for_backward(params, x01)
        ctx.grid, ctx.half = grid, half
        return feat

    @staticmethod
    def backward(ctx, dfeat):
        params, x01 = ctx.saved_tensors
        if not ctx.needs_input_grad[1]:
            dparams = hashgrid_bwd(x01.detach().float().contiguous(), dfeat.float().contiguous(), ctx.grid).reshape(-1) \
                if ctx.needs_input_grad[0] else None
            return dparams, None, None
        dparams, dx = _EncodingBackward.apply(params, x01, dfeat, ctx.half, ctx.grid, ctx.needs_input_grad[0])
        return (dparams if ctx.needs_input_grad[0] else None), dx.to(x01.dtype), None


class _EncodingBackward(torch.autograd.Function):
    """(d_params, d_x01) of the encode as a differentiable node: its own backward is the double
    backward w.r.t. the INPUT gradient only (as in tcnn, gradients flowing into ``d_params`` are
    not propagated)."""

    @staticmethod
    def forward(ctx, params, x01, dfeat, half, grid, want_params):
        xd, g = x01.detach().float().contiguous(), dfeat.detach().float().contiguous()
        dx = hashgrid_bwd_input(half, xd, g, grid)
        dparams = hashgrid_bwd(xd, g, grid).reshape(-1) if want_params else torch.zeros((), device=xd.device)
        ctx.save_for_backward(xd, g)
        ctx.grid, ctx.half, ctx.x_dtype, ctx.g_dtype = grid, half, x01.dtype, dfeat.dtype
        ctx.set_materialize_grads(False)
        ctx.mark_non_differentiable(dparams)
        return dparams, dx

    @staticmethod
    def backward(ctx, _unused, ddx):
        if ddx is None:
            return None, None, None, None, None, None
        xd, g = ctx.saved_tensors
        want = (ctx.needs_input_grad[2], ctx.needs_input_grad[0], ctx.needs_input_grad[1])
        ddfeat, dtable, dx2 = hashgrid_bwd_bwd_input(ctx.half, xd, g, ddx.float().contiguous(), ctx.grid, want)
        return (None if dtable is None else dtable.reshape(-1),
                None if dx2 is None else dx2.to(ctx.x_dtype),
                None if ddfeat is None else ddfeat.to(ctx.g_dtype),
                None, None, None)


def encoding_apply(params: torch.Tensor, x01: torch.Tensor, grid: GridConfig) -> torch.Tensor:
    return _EncodingFunction.apply(params, x01, grid)


# ------------------------------------------------------------------ packed composite (nerfacc semantics)
def weights_from_density(t_starts, t_ends, sigmas, ray_indices, n_rays: int):
    t_starts, t_ends = _chk(t_starts, torch.float32, "t_starts"), _chk(t_ends, torch.float32, "t_ends")
    sigmas, ray_indices = _chk(sigmas, torch.float32, "sigmas"), _chk(ray_indices, torch.int64, "ray_indices")
    N = sigmas.numel()
    w, T, a = torch.empty_like(sigmas), torch.empty_like(sigmas), torch.empty_like(sigmas)
    with torch.cuda.device(sigmas.device):
        _call(_L().perf_weights_from_density, _p(t_starts), _p(t_ends), _p(sigmas), _p(ray_indices), N, n_rays,
              _p(w), _p(T), _p(a), _stream())
    return w, T, a


def weights_from_density_bwd(t_starts, t_ends, sigmas, ray_indices, n_rays, weights, trans, grad_w, grad_T=None):
    gs = torch.empty_like(sigmas)
    grad_w = _chk(grad_w, torch.float32, "grad_weights")
    grad_T = None if grad_T is None else _chk(grad_T, torch.float32, "grad_trans")
    with torch.cuda.device(sigmas.device):
        _call(_L().perf_weights_from_density_bwd, _p(t_starts), _p(t_ends), _p(sigmas), _p(ray_indices),
              sigmas.numel(), n_rays, _p(weights), _p(trans), _p(grad_w), _p(grad_T), _p(gs), _stream())
    return gs


def accumulate_along_rays(weights, values, ray_indices, n_rays: int) -> torch.Tensor:
    weights, ray_indices = _chk(weights, torch.float32, "weights"), _chk(ray_indices, torch.int64, "ray_indices")
    D = 1 if values is None else values.shape[-1]
    values = None if values is None else _chk(values, torch.float32, "values")
    out = torch.empty(n_rays, D, dtype=torch.float32, device=weights.device)
    with torch.cuda.device(weights.device):
        _call(_L().perf_accumulate_along_rays, _p(weights), _p(values), D, _p(ray_indices), weights.numel(), n_rays,
              _p(out), _stream())
    return out


# ------------------------------------------------------------------ occupancy-grid sampler
def _occ_pieces(R: int) -> int:
    """Parts every ray's lattice walk is cut into so that ~256 k threads march (a ray alone is a serial walk of up to
    (far - near) / step = 3000 lattice points; 8192 ray-threads left the GPU empty: 1.08 ms per pass, profiles/r02)."""
    p = 1
    while p < 64 and R * p * 2 <= 262144:
        p *= 2
    return p


def _occ_masks_ok(near: float, far: float, step: float, pieces: int) -> bool:
    """The single-march form (sample bits recorded by the count pass, expanded by the write pass) needs <= 128 lattice points per piece."""
    return ((far - near) / step + 16.0) / pieces + 1.0 <= 126.0


def occ_sample(binaries: torch.Tensor, aabb, rays_o, rays_d, near: float, far: float, step: float, jitter=None, pieces: Optional[int] = None):
    """Packed (ray_indices, t_starts, t_ends) of the lattice samples whose midpoint is inside the aabb
    in an occupied cell (two kernels around one cumsum; one host sync for the total, as nerfacc)."""
    rays_o, rays_d = _chk(rays_o, torch.float32, "rays_o"), _chk(rays_d, torch.float32, "rays_d")
    jitter = None if jitter is None else _chk(jitter, torch.float32, "jitter")
    if not binaries.is_cuda or binaries.dim() != 3:
        raise RuntimeError("perf_b200.occ_sample: `binaries` must be a CUDA bool tensor [rx, ry, rz]")
    bins = binaries.contiguous().view(torch.uint8) if binaries.dtype == torch.bool else _chk(binaries, torch.uint8, "binaries")
    R, dev = rays_o.shape[0], rays_o.device
    P = _occ_pieces(R) if pieces is None else int(pieces)
    res3 = (C.c_int * 3)(*[int(v) for v in binaries.shape])
    a6 = (C.c_float * 6)(*[float(v) for v in aabb])
    counts = torch.empty(R * P, dtype=torch.int32, device=dev)
    masks = torch.empty(R * P * 4, dtype=torch.int32, device=dev) if _occ_masks_ok(near, far, step, P) else None
    with torch.cuda.device(dev):
        _call(_L().perf_occ_count, _p(bins), res3, a6, _p(rays_o), _p(rays_d), _p(jitter), R, near, far, step, P, _p(counts), _p(masks), _stream())
    incl = torch.cumsum(counts, 0, dtype=torch.int64)
    total = int(incl[-1].item()) if R else 0
    offsets = (incl - counts).contiguous()                                  # [R * P], exclusive
    # per-ray ranges [R + 1]: the first piece's offset of every ray, then the total
    occ_sample.last_offsets = torch.cat([offsets[::P], incl[-1:]]) if R else torch.zeros(1, dtype=torch.int64, device=dev)
    ri = torch.empty(total, dtype=torch.int64, device=dev)
    ts, te = torch.empty(total, dtype=torch.float32, device=dev), torch.empty(total, dtype=torch.float32, device=dev)
    if total:
        with torch.cuda.device(dev):
            _call(_L().perf_occ_write, _p(bins), res3, a6, _p(rays_o), _p(rays_d), _p(jitter), R, near, far, step, P, _p(offsets), 0,
                  _p(masks), _p(ri), _p(ts), _p(te), _stream())
    return ri, ts, te


class OccStaticBuffers:
    """Fixed-capacity buffers of :func:`occ_sample_static` (one set per (R, capacity, device); reused every step)."""

    def __init__(self, R: int, capacity: int, dev, pieces: Optional[int] = None):
        self.R, self.capacity, self.pieces = R, capacity, (_occ_pieces(R) if pieces is None else int(pieces))
        P = self.pieces
        self.counts = torch.empty(R * P, dtype=torch.int32, device=dev)
        self.offsets_all = torch.zeros(R * P + 1, dtype=torch.int64, device=dev)  # exclusive scan over (ray, piece); [0] stays 0
        self.offsets = torch.zeros(R + 1, dtype=torch.int64, device=dev)         # per-ray ranges, clamped to the capacity
        self.raw_total = torch.zeros(1, dtype=torch.int64, device=dev)           # un-clamped sample count of the last call
        self.n = torch.zeros(1, dtype=torch.int64, device=dev)                   # live count = min(raw_total, capacity)
        self.ri = torch.zeros(capacity, dtype=torch.int64, device=dev)
        self.ts = torch.zeros(capacity, dtype=torch.float32, device=dev)
        self.te = torch.zeros(capacity, dtype=torch.float32, device=dev)
        self.overflowed = torch.zeros(1, dtype=torch.int64, device=dev)          # running max of raw_total (host reads it rarely)
        self.masks = torch.zeros(R * P * 4, dtype=torch.int32, device=dev)        # sample bits per (ray, piece), when usable


def occ_sample_static(binaries: torch.Tensor, aabb, rays_o, rays_d, near: float, far: float, step: float, jitter, buf: OccStaticBuffers):
    """:func:`occ_sample` without the host read of the sample count: the packed intervals go into ``buf`` (capacity-sized),
    ``buf.n`` holds the live count ON THE DEVICE and ``buf.offsets`` the per-ray ranges, both clamped to the capacity
    (samples that do not fit are dropped from the END of the batch; ``buf.overflowed`` remembers the largest request).
    Everything is stream-ordered device work with shapes that do not depend on the count: capturable into a CUDA graph."""
    rays_o, rays_d = _chk(rays_o, torch.float32, "rays_o"), _chk(rays_d, torch.float32, "rays_d")
    jitter = None if jitter is None else _chk(jitter, torch.float32, "jitter")
    bins = binaries.contiguous().view(torch.uint8) if binaries.dtype == torch.bool else _chk(binaries, torch.uint8, "binaries")
    R, P = rays_o.shape[0], buf.pieces
    assert R == buf.R
    res3 = (C.c_int * 3)(*[int(v) for v in binaries.shape])
    a6 = (C.c_float * 6)(*[float(v) for v in aabb])
    masks = buf.masks if _occ_masks_ok(near, far, step, P) else None
    with torch.cuda.device(rays_o.device):
        _call(_L().perf_occ_count, _p(bins), res3, a6, _p(rays_o), _p(rays_d), _p(jitter), R, near, far, step, P, _p(buf.counts), _p(masks), _stream())
        torch.cumsum(buf.counts, 0, dtype=torch.int64, out=buf.offsets_all[1:])
        buf.raw_total.copy_(buf.offsets_all[R * P:])
        torch.maximum(buf.overflowed, buf.raw_total, out=buf.overflowed)
        _call(_L().perf_occ_write, _p(bins), res3, a6, _p(rays_o), _p(rays_d), _p(jitter), R, near, far, step, P, _p(buf.offsets_all), buf.capacity,
              _p(masks), _p(buf.ri), _p(buf.ts), _p(buf.te), _stream())
        torch.clamp(buf.offsets_all[::P], max=buf.capacity, out=buf.offsets)        # [R + 1]: (R * P) % P == 0, so the total is included
        buf.n.copy_(buf.offsets[R:])
    return buf.ri, buf.ts, buf.te, buf.offsets, buf.n


# ------------------------------------------------------------------ fused renderer
def _render_args(packed_table, geo_mlp_half, app_mlp_half, aabb, n_samples, near, far, training, simt,
                 jitter, bg_noise, rgb, distance, opacity, grid: GridConfig, kernel: str = "march") -> "_lib.RenderArgs":
    a = _lib.RenderArgs()
    a.grid = grid.c()
    a.d_packed_table, a.d_geo_mlp_half, a.d_app_mlp_half = packed_table.data_ptr(), geo_mlp_half.data_ptr(), app_mlp_half.data_ptr()
    a.aabb = (C.c_float * 6)(*[float(v) for v in aabb])
    a.n_samples, a.near, a.far = int(n_samples), float(near), float(far)
    if kernel not in ("march", "march_generic", "march_l0smem", "scan"):
        raise ValueError(f"unknown render kernel {kernel!r}")
    a.flags = ((_lib.PERF_FLAG_TRAINING if training else 0) | (_lib.PERF_FLAG_SIMT_MLP if simt else 0)
               | (_lib.PERF_FLAG_SCAN_KERNEL if kernel == "scan" else 0)
               | (_lib.PERF_FLAG_GENERIC_ADDR if kernel == "march_generic" else 0)
               | (_lib.PERF_FLAG_L0_SMEM if kernel == "march_l0smem" else 0))
    a.d_jitter = None if jitter is None else jitter.data_ptr()
    a.d_bg_noise = None if bg_noise is None else bg_noise.data_ptr()
    a.d_rgb, a.d_distance = rgb.data_ptr(), distance.data_ptr()
    a.d_opacity = None if opacity is None else opacity.data_ptr()
    return a


def render_rays(packed_table, geo_mlp_half, app_mlp_half, rays_o, rays_d, n_samples: int, near=1e-2, far=1.0,
                aabb=(-1., -1., -1., 1., 1., 1.), training=False, jitter=None, bg_noise=None,
                grid: GridConfig = PERF_GRID, simt=False, kernel="march", image_width: int = 0):
    """Fused render of explicit rays [R,3] -> (rgb [R,3], distance [R,1], opacity [R,1]).
    ``image_width`` > 0 declares the rays a row-major image of that width (pixel-patch tiling)."""
    rays_o, rays_d = _chk(rays_o, torch.float32, "rays_o"), _chk(rays_d, torch.float32, "rays_d")
    R, dev = rays_o.shape[0], rays_o.device
    rgb = torch.empty(R, 3, dtype=torch.float32, device=dev)
    dist = torch.empty(R, 1, dtype=torch.float32, device=dev)
    op = torch.empty(R, 1, dtype=torch.float32, device=dev)
    if R == 0:
        return rgb, dist, op
    jitter = None if jitter is None else _chk(jitter, torch.float32, "jitter")
    bg_noise = None if bg_noise is None else _chk(bg_noise, torch.float32, "bg_noise")
    a = _render_args(packed_table, geo_mlp_half, app_mlp_half, aabb, n_samples, near, far, training, simt,
                     jitter, bg_noise, rgb, dist, op, grid, kernel)
    a.image_width = int(image_width) if image_width and R % int(image_width) == 0 else 0
    with torch.cuda.device(dev):
        _call(_L().perf_render_rays, C.byref(a), _p(rays_o), _p(rays_d), R, _stream())
    return rgb, dist, op


def render_packed(packed_table, geo_mlp_half, app_mlp_half, rays_o, rays_d, ray_indices, t_starts, t_ends,
                  aabb=(-1., -1., -1., 1., 1., 1.), grid: GridConfig = PERF_GRID, simt=False, offsets: Optional[torch.Tensor] = None):
    """Fused eval render of packed variable-length samples (sorted by ray, as an occupancy estimator
    returns them) -> (rgb [R,3], distance [R,1], opacity [R,1])."""
    rays_o, rays_d = _chk(rays_o, torch.float32, "rays_o"), _chk(rays_d, torch.float32, "rays_d")
    ray_indices = _chk(ray_indices, torch.int64, "ray_indices")
    t_starts, t_ends = _chk(t_starts, torch.float32, "t_starts"), _chk(t_ends, torch.float32, "t_ends")
    R, dev = rays_o.shape[0], rays_o.device
    rgb = torch.empty(R, 3, dtype=torch.float32, device=dev)
    dist = torch.empty(R, 1, dtype=torch.float32, device=dev)
    op = torch.empty(R, 1, dtype=torch.float32, device=dev)
    if R == 0:
        return rgb, dist, op
    if offsets is None:                                   # callers that sampled with occ_sample pass occ_sample.last_offsets
        offsets = torch.zeros(R + 1, dtype=torch.int64, device=dev)
        offsets[1:] = torch.cumsum(torch.bincount(ray_indices, minlength=R), 0)
    else:
        offsets = _chk(offsets, torch.int64, "offsets")
    a = _render_args(packed_table, geo_mlp_half, app_mlp_half, aabb, 1, 0.0, 1.0, False, simt, None, None, rgb, dist, op, grid)
    with torch.cuda.device(dev):
        _call(_L().perf_render_packed, C.byref(a), _p(rays_o), _p(rays_d), R, _p(offsets), _p(t_starts), _p(t_ends), _stream())
    return rgb, dist, op


def render_occ(packed_table, geo_mlp_half, app_mlp_half, rays_o, rays_d, offsets, ray_indices, t_starts, t_ends,
               early_stop_eps: float = 1e-4, aabb=(-1., -1., -1., 1., 1., 1.), grid: GridConfig = PERF_GRID):
    """Eval render of packed intervals: perf_fields_packed (no saves) + perf_composite_packed_fwd (eval background)."""
    rays_o, rays_d = _chk(rays_o, torch.float32, "rays_o"), _chk(rays_d, torch.float32, "rays_d")
    offsets, ray_indices = _chk(offsets, torch.int64, "offsets"), _chk(ray_indices, torch.int64, "ray_indices")
    t_starts, t_ends = _chk(t_starts, torch.float32, "t_starts"), _chk(t_ends, torch.float32, "t_ends")
    R, N, dev = rays_o.shape[0], t_starts.shape[0], rays_o.device
    f32 = lambda *sh: torch.empty(*sh, dtype=torch.float32, device=dev)
    rgb, dist, op = f32(R, 3), f32(R, 1), f32(R, 1)
    if R == 0:
        return rgb, dist, op
    sigma, c16, x01 = f32(N), torch.empty(N, 4, dtype=torch.float16, device=dev), f32(N, 3)
    w, T, dacc, dl = f32(N), f32(N), f32(R), f32(R)
    a = _render_args(packed_table, geo_mlp_half, app_mlp_half, aabb, 1, 0.0, 1.0, False, False, None, None, rgb, dist, op, grid)
    with torch.cuda.device(dev):
        _call(_L().perf_fields_packed, C.byref(a), _p(rays_o), _p(rays_d), _p(ray_indices), _p(t_starts), _p(t_ends), N, None, 0,
              _p(sigma), _p(c16), _p(x01), None, None, None, _stream(), launches=2)
        _call(_L().perf_composite_packed_fwd, _p(offsets), _p(t_starts), _p(t_ends), _p(sigma), _p(c16), R, float(early_stop_eps), 0, None,
              _p(w), _p(T), _p(rgb), _p(dist), _p(op), _p(dacc), _p(dl), _stream())
    return rgb, dist, op


def render_pano(packed_table, geo_mlp_half, app_mlp_half, pose, H: int, W: int, n_samples: int, near=1e-2, far=1.0,
                row0: int = 0, rows: Optional[int] = None, aabb=(-1., -1., -1., 1., 1., 1.),
                grid: GridConfig = PERF_GRID, simt=False, out=None, kernel="march"):
    """Fused render of rows [row0,row0+rows) of an HxW equirect panorama (ray-gen inside the kernel).
    Returns (rgb [rows,W,3], distance [rows,W,1], opacity [rows,W,1])."""
    rows = H - row0 if rows is None else rows
    dev = packed_table.device
    if out is None:
        rgb = torch.empty(rows, W, 3, dtype=torch.float32, device=dev)
        dist = torch.empty(rows, W, 1, dtype=torch.float32, device=dev)
        op = torch.empty(rows, W, 1, dtype=torch.float32, device=dev)
    else:
        rgb, dist, op = out
    a = _render_args(packed_table, geo_mlp_half, app_mlp_half, aabb, n_samples, near, far, False, simt,
                     None, None, rgb, dist, op, grid, kernel)
    with torch.cuda.device(dev):
        _call(_L().perf_render_pano, C.byref(a), _pose_array(pose), H, W, row0, rows, _stream())
    return rgb, dist, op


def _occ_render_args(binaries: torch.Tensor, grid_aabb, near: float, far: float, step: float, early_stop_eps: float,
                     n_samples: Optional[torch.Tensor]) -> "_lib.OccRenderArgs":
    if not isinstance(binaries, torch.Tensor) or not binaries.is_cuda or binaries.dim() != 3:
        raise RuntimeError("perf_b200: `binaries` must be a CUDA bool / uint8 tensor [rx, ry, rz]")
    if not binaries.is_contiguous():
        raise ValueError("perf_b200: `binaries` must be contiguous")
    bins = binaries.view(torch.uint8) if binaries.dtype == torch.bool else _chk(binaries, torch.uint8, "binaries")
    g = _lib.OccRenderArgs()
    g.d_binaries = bins.data_ptr()
    g.res = (C.c_int * 3)(*[int(v) for v in binaries.shape])
    g.aabb = (C.c_float * 6)(*[float(v) for v in grid_aabb])
    g.near, g.far, g.step, g.early_stop_eps = float(near), float(far), float(step), float(early_stop_eps)
    g.d_n_samples = None if n_samples is None else n_samples.data_ptr()
    return g


def render_rays_occ(packed_table, geo_mlp_half, app_mlp_half, rays_o, rays_d, binaries, grid_aabb, near=0.0, far=1.5, step=5e-4,
                    early_stop_eps=1e-4, aabb=(-1., -1., -1., 1., 1., 1.), grid: GridConfig = PERF_GRID, simt=False,
                    image_width: int = 0, want_n_samples: bool = False, kernel: str = "march"):
    """One-launch eval render of explicit rays [R,3] with the occupancy-grid sampler inside the kernel (grid walk, both
    fields, composite with the ``early_stop_eps`` transmittance cut) -> (rgb [R,3], distance [R,1], opacity [R,1]) and, with
    ``want_n_samples``, the intervals composited per ray [R] int32 as a fourth element.  ``binaries`` [rx,ry,rz] and
    ``grid_aabb`` are the estimator's grid and roi; ``aabb`` is the field's box.  No host read, no allocation besides
    the outputs (capturable into a CUDA graph)."""
    rays_o, rays_d = _chk(rays_o, torch.float32, "rays_o"), _chk(rays_d, torch.float32, "rays_d")
    R, dev = rays_o.shape[0], rays_o.device
    rgb = torch.empty(R, 3, dtype=torch.float32, device=dev)
    dist = torch.empty(R, 1, dtype=torch.float32, device=dev)
    op = torch.empty(R, 1, dtype=torch.float32, device=dev)
    n = torch.empty(R, dtype=torch.int32, device=dev) if want_n_samples else None
    if R == 0:
        return (rgb, dist, op, n) if want_n_samples else (rgb, dist, op)
    a = _render_args(packed_table, geo_mlp_half, app_mlp_half, aabb, 1, 0.0, 1.0, False, simt, None, None, rgb, dist, op, grid, kernel)
    a.image_width = int(image_width) if image_width and R % int(image_width) == 0 else 0
    g = _occ_render_args(binaries, grid_aabb, near, far, step, early_stop_eps, n)
    with torch.cuda.device(dev):
        _call(_L().perf_render_rays_occ, C.byref(a), C.byref(g), _p(rays_o), _p(rays_d), R, _stream())
    return (rgb, dist, op, n) if want_n_samples else (rgb, dist, op)


def render_pano_occ(packed_table, geo_mlp_half, app_mlp_half, pose, H: int, W: int, binaries, grid_aabb, near=0.0, far=1.5, step=5e-4,
                    early_stop_eps=1e-4, row0: int = 0, rows: Optional[int] = None, aabb=(-1., -1., -1., 1., 1., 1.),
                    grid: GridConfig = PERF_GRID, simt=False, out=None, want_n_samples: bool = False, kernel: str = "march"):
    """:func:`render_rays_occ` for rows [row0,row0+rows) of an HxW equirect panorama, ray generation fused in.
    Returns (rgb [rows,W,3], distance [rows,W,1], opacity [rows,W,1]) (+ n_samples [rows,W] int32)."""
    rows = H - row0 if rows is None else rows
    dev = packed_table.device
    if out is None:
        rgb = torch.empty(rows, W, 3, dtype=torch.float32, device=dev)
        dist = torch.empty(rows, W, 1, dtype=torch.float32, device=dev)
        op = torch.empty(rows, W, 1, dtype=torch.float32, device=dev)
    else:
        rgb, dist, op = out
    n = torch.empty(rows, W, dtype=torch.int32, device=dev) if want_n_samples else None
    a = _render_args(packed_table, geo_mlp_half, app_mlp_half, aabb, 1, 0.0, 1.0, False, simt, None, None, rgb, dist, op, grid, kernel)
    g = _occ_render_args(binaries, grid_aabb, near, far, step, early_stop_eps, n)
    with torch.cuda.device(dev):
        _call(_L().perf_render_pano_occ, C.byref(a), C.byref(g), _pose_array(pose), H, W, row0, rows, _stream())
    return (rgb, dist, op, n) if want_n_samples else (rgb, dist, op)


# ------------------------------------------------------------------ fused training step
class FusedTrainContext:
    """Everything one fused training step needs besides the rays: the fp16 shadows / gather table,
    sampler constants, and the per-sample buffers (cached per (R, S, phase); sample-major rows)."""

    def __init__(self, grid: GridConfig = PERF_GRID, aabb=(-1., -1., -1., 1., 1., 1.), n_samples=128, near=1e-2, far=1.0):
        self.grid, self.aabb, self.n_samples, self.near, self.far = grid, tuple(float(v) for v in aabb), n_samples, near, far
        self.packed = self.geo_half = self.app_half = None
        self._bufs = {}
        self.generation = 0          # bumped by every forward; backward refuses stale per-sample buffers

    def buffers(self, R: int, phase: int, dev):
        key = (R, self.n_samples, phase, str(dev))
        if key not in self._bufs:
            N = R * self.n_samples
            f32 = lambda *s: torch.empty(*s, dtype=torch.float32, device=dev)
            f16 = lambda *s: torch.empty(*s, dtype=torch.float16, device=dev)
            b = {"sigma": f32(N), "w": f32(N), "T": f32(N), "feat": f16(N, 32), "h1": f16(N, 64),
                 "dacc": f32(R), "dl": f32(R), "rgb": None, "h2": None,
                 "toff": f32(_lib.PERF_MAX_SEGMENTS * R), "segments": C.c_uint32(1)}
            if phase == _lib.PERF_PHASE_APP:
                b["rgb"], b["h2"] = f16(N, 4), f16(N, 64)
            # keep the latest TWO shapes: dropping the previous shape's buffers while a not-yet-run backward still
            # references them would leave that graph pointing at freed (re-usable) memory; the generation check in
            # _FusedTrainStep.backward turns any remaining misuse into an error
            last = list(self._bufs.items())[-1:]
            self._bufs = dict(last + [(key, b)])
        return self._bufs[key]

    def packed_buffers(self, R: int, N: int, phase: int, dev):
        """Per-sample buffers of the packed (occupancy) step, cached per (R, N, phase): with capacity-sized sample tensors N
        never changes, so a captured step always sees the same storage."""
        key = ("packed", R, N, phase, str(dev))
        if key not in self._bufs:
            geo = phase == _lib.PERF_PHASE_GEO
            f32 = lambda *s: torch.empty(*s, dtype=torch.float32, device=dev)
            f16 = lambda *s: torch.empty(*s, dtype=torch.float16, device=dev)
            b = {"sigma": f32(N), "rgb": f16(N, 4), "x01": f32(N, 3), "feat": f16(N, 32), "h1": f16(N, 64), "h2": None if geo else f16(N, 64),
                 "w": f32(N), "T": f32(N), "dacc": f32(R), "dl": f32(R), "dz": f32(N, 1 if geo else 3)}
            last = list(self._bufs.items())[-1:]
            self._bufs = dict(last + [(key, b)])
        return self._bufs[key]

    @staticmethod
    def c_buffers(b) -> "_lib.TrainBuffers":
        ptr = lambda t: None if t is None else t.data_ptr()
        return _lib.TrainBuffers(ptr(b["sigma"]), ptr(b["w"]), ptr(b["T"]), ptr(b["rgb"]), ptr(b["feat"]), ptr(b["h1"]),
                                 ptr(b["h2"]), ptr(b["dacc"]), ptr(b["dl"]), ptr(b["toff"]), C.pointer(b["segments"]))


def mlp_backward_half(mlp: MLPConfig, weights_half: torch.Tensor, feat, h1, h2, dz: torch.Tensor,
                      grad_out: Optional[torch.Tensor] = None, n_dev: Optional[torch.Tensor] = None):
    """MLP backward from saved fp16 activations (tcnn ``FullyFusedMLP::backward_impl``, reached from
    `ngp_nerf.py:142,158` under autograd): ONE tcgen05 kernel, :func:`mlp_backward_fused` (csrc/mlp_bwd.cu).
    ``dz`` [N, n_out] fp32: gradient w.r.t. the output layer's pre-activation.
    Returns (d_weights_flat fp32 [mlp.n_params] -- written into ``grad_out`` when given --, dfeat fp32 [N,32]).
    ``PERF_B200_GEMM_MLP_BWD=1`` selects :func:`mlp_backward_gemm` (library GEMMs; the A/B reference of round 1)."""
    if os.environ.get("PERF_B200_GEMM_MLP_BWD") == "1" and n_dev is None:
        return mlp_backward_gemm(mlp, weights_half, feat, h1, h2, dz, grad_out)
    return mlp_backward_fused(mlp, weights_half, feat, h1, h2, dz, grad_out, n_dev=n_dev)


def mlp_backward_gemm(mlp: MLPConfig, weights_half: torch.Tensor, feat, h1, h2, dz: torch.Tensor,
                      grad_out: Optional[torch.Tensor] = None):
    """Round-1 path, kept as the A/B reference of the tests and tools/ab_mlp_bwd.py only: the five matrix products as
    fp16 cuBLAS GEMMs (fp32 out) around perf_mlp_bwd_out / perf_relu_mask.  NOT on any default path."""
    N, dev = dz.shape[0], dz.device
    W = weights_half
    w1 = W[:64 * 32].view(64, 32)
    p = 64 * 32
    w2 = None
    if mlp.n_hidden_layers == 2:
        w2 = W[p:p + 64 * 64].view(64, 64); p += 64 * 64
    wout = W[p:p + mlp.padded_out * 64].view(mlp.padded_out, 64)[:mlp.n_out].contiguous()
    h_last = h2 if w2 is not None else h1
    if grad_out is None:
        grad_out = torch.zeros(mlp.n_params, dtype=torch.float32, device=dev)
    g_w1 = grad_out[:2048].view(64, 32)
    g_w2 = grad_out[2048:2048 + 4096].view(64, 64) if w2 is not None else None
    g_wout = grad_out[p:p + mlp.padded_out * 64].view(mlp.padded_out, 64)
    dz = dz.contiguous()
    g_wout[:mlp.n_out] = torch.mm(dz.half().t(), h_last, out_dtype=torch.float32)
    dh = torch.empty(N, 64, dtype=torch.float16, device=dev)
    with torch.cuda.device(dev):
        _call(_L().perf_mlp_bwd_out, _p(dz), mlp.n_out, _p(wout), _p(h_last), _p(dh), N, _stream())
    if w2 is not None:
        g_w2.copy_(torch.mm(dh.t(), h1, out_dtype=torch.float32))
        dh = dh @ w2
        with torch.cuda.device(dev):
            _call(_L().perf_relu_mask, _p(dh), _p(h1), N * 64, _stream())
    g_w1.copy_(torch.mm(dh.t(), feat, out_dtype=torch.float32))
    dfeat = torch.mm(dh, w1, out_dtype=torch.float32)
    return grad_out, dfeat


def mlp_backward_fused(mlp: MLPConfig, weights_half: torch.Tensor, feat, h1, h2, dz: torch.Tensor,
                       grad_out: Optional[torch.Tensor] = None, simt: bool = False, dbg: int = 0, n_dev: Optional[torch.Tensor] = None):
    """The whole MLP backward as ONE tcgen05 kernel (perf_mlp_bwd, csrc/mlp_bwd.cu): output-layer backward on CUDA
    cores, data gradients dh W as MMAs against the forward weight images read MN-major, weight gradients
    [dh]^T [h] accumulated in TMEM over the CTA's tiles and flushed once.  Validated on B200 in round 2 against a
    torch fp32 reference (tools/diag_mlp_bwd.py: rel. err <= 2e-5) and the GEMM path (tests/test_gpu_train.py)."""
    N, dev = dz.shape[0], dz.device
    if grad_out is None:
        grad_out = torch.zeros(mlp.n_params, dtype=torch.float32, device=dev)
    else:
        grad_out[:mlp.n_params].zero_()
    dfeat = torch.empty(N, 32, dtype=torch.float32, device=dev)
    dz = _chk(dz.reshape(N, mlp.n_out), torch.float32, "dz")
    with torch.cuda.device(dev):
        _call(_L().perf_mlp_bwd, mlp.c(), _p(_chk(weights_half, torch.float16, "weights")), _p(_chk(feat, torch.float16, "feat")),
              _p(_chk(h1, torch.float16, "h1")), _p(None if h2 is None else _chk(h2, torch.float16, "h2")), _p(dz), N, _p(n_dev),
              _p(grad_out), _p(dfeat), (_lib.PERF_FLAG_SIMT_MLP if simt else 0) | (dbg << 8), _stream(), launches=2)
    return grad_out, dfeat


class _FusedTrainStep(torch.autograd.Function):
    """(rgb, distance, opacity, distloss_numerator_per_ray) of a training-mode render, differentiable
    w.r.t. the flat params of the network selected by ``phase``.  Forward = ONE kernel
    (perf_train_forward), backward = composite-backward kernel, ONE tcgen05 MLP-backward kernel, grid scatter."""

    @staticmethod
    def forward(ctx, params, rays_o, rays_d, jitter, bg_noise, tc: FusedTrainContext, phase: int):
        R, dev = rays_o.shape[0], rays_o.device
        b = tc.buffers(R, phase, dev)
        rgb = torch.empty(R, 3, dtype=torch.float32, device=dev)
        dist = torch.empty(R, 1, dtype=torch.float32, device=dev)
        op = torch.empty(R, 1, dtype=torch.float32, device=dev)
        a = _render_args(tc.packed, tc.geo_half, tc.app_half, tc.aabb, tc.n_samples, tc.near, tc.far, True, False,
                         jitter, bg_noise, rgb, dist, op, tc.grid)
        cb = FusedTrainContext.c_buffers(b)
        with torch.cuda.device(dev):
            _call(_L().perf_train_forward, C.byref(a), _p(rays_o), _p(rays_d), R, phase, C.byref(cb), _stream())
        tc.generation += 1
        ctx.tc, ctx.phase, ctx.b, ctx.generation = tc, phase, b, tc.generation
        ctx.save_for_backward(rays_o, rays_d, jitter, bg_noise, dist, op)
        return rgb, dist, op, b["dl"].clone()

    @staticmethod
    def backward(ctx, g_rgb, g_dist, g_op, g_dl):
        rays_o, rays_d, jitter, bg_noise, dist, op = ctx.saved_tensors
        tc, phase, b = ctx.tc, ctx.phase, ctx.b
        if ctx.generation != tc.generation:
            raise RuntimeError("perf_b200 fused training step: backward() after a newer forward() on the same context -- the "
                               "per-sample buffers are reused between steps; call backward before the next forward")
        R, S, dev = rays_o.shape[0], tc.n_samples, rays_o.device
        N = R * S
        geo = phase == _lib.PERF_PHASE_GEO
        mlp = GEO_MLP if geo else APP_MLP
        dz = torch.empty(N, mlp.n_out, dtype=torch.float32, device=dev)
        c = lambda t: None if t is None else t.contiguous().float()
        g_rgb, g_dist, g_op, g_dl = c(g_rgb), c(g_dist), c(g_op), c(g_dl)
        cb = FusedTrainContext.c_buffers(b)
        with torch.cuda.device(dev):
            _call(_L().perf_train_backward_composite, phase, S, int(b["segments"].value), tc.near, tc.far, R, _p(jitter), _p(bg_noise), C.byref(cb),
                  _p(g_rgb), _p(g_dist), _p(g_op), _p(g_dl), _p(dist), _p(op), _p(dz), _stream())
        half = tc.geo_half if geo else tc.app_half
        # ONE flat gradient in the parameter layout [MLP | grid]: the MLP backward and the scatter write into it
        grad = torch.zeros(mlp.n_params + 2 * tc.grid.n_entries, dtype=torch.float32, device=dev)
        d_table = grad[mlp.n_params:]
        aabb = (C.c_float * 6)(*tc.aabb)
        fuse = (os.environ.get("PERF_B200_FUSE_SCATTER", "1") != "0" and os.environ.get("PERF_B200_GEMM_MLP_BWD") != "1"
                and tc.grid.n_levels == 16 and d_table.data_ptr() % 16 == 0)
        if fuse:
            # MLP backward with the fine levels' reductions issued from its epilogue, then the coarse levels' march kernel
            dfeat = torch.empty(N, 32, dtype=torch.float32, device=dev)
            with torch.cuda.device(dev):
                _call(_L().perf_mlp_bwd_scatter, mlp.c(), _p(half[:mlp.n_params]), _p(b["feat"]), _p(b["h1"]), _p(b["h2"]), _p(dz.reshape(N, mlp.n_out)), N,
                      _p(grad[:mlp.n_params]), _p(dfeat), tc.grid.c(), aabb, _p(rays_o), _p(rays_d), _p(jitter), R, S, tc.near, tc.far, _p(d_table),
                      _stream(), launches=2)
                _call(_L().perf_hashgrid_bwd_rays_coarse, tc.grid.c(), aabb, _p(rays_o), _p(rays_d), _p(jitter), R, S, tc.near, tc.far,
                      _p(dfeat), _p(d_table), _stream())
            return grad, None, None, None, None, None, None
        _, dfeat = mlp_backward_half(mlp, half[:mlp.n_params], b["feat"], b["h1"], b["h2"], dz, grad_out=grad[:mlp.n_params])
        with torch.cuda.device(dev):
            _call(_L().perf_hashgrid_bwd_rays, tc.grid.c(), aabb, _p(rays_o), _p(rays_d), _p(jitter), R, S, tc.near, tc.far,
                  _p(dfeat), _p(d_table), _stream(), launches=2)
        return grad, None, None, None, None, None, None


class _FusedPackedTrainStep(torch.autograd.Function):
    """(rgb, distance, opacity, distloss_numerator_per_ray) of a training-mode render of PACKED samples (the
    occupancy sampler's output, all of them -- the 1e-4 transmittance cut of ``OccGridEstimator.sampling`` is applied
    inside the composite), differentiable w.r.t. the flat params of the network selected by ``phase``
    (`nerf_renderer.py:145-209` under `nerf.py:186-297`).  Forward: perf_fields_packed + perf_composite_packed_fwd;
    backward: perf_composite_packed_bwd + perf_mlp_bwd + perf_hashgrid_bwd_merged.  No torch glue on per-sample data.
    ``n_dev`` (device int64 [1]): the live sample count when the sample tensors are capacity-sized (graph capture)."""

    MERGE_LEVELS = 13          # same-cell runs of consecutive 5e-4 samples exist up to resolution ~1350 (level 12)

    @staticmethod
    def forward(ctx, params, rays_o, rays_d, offsets, ray_indices, t_starts, t_ends, bg_noise, tc: FusedTrainContext, phase: int,
                early_stop_eps: float, n_dev):
        R, N, dev = rays_o.shape[0], t_starts.shape[0], rays_o.device
        geo = phase == _lib.PERF_PHASE_GEO
        b = tc.packed_buffers(R, N, phase, dev)
        f32 = lambda *sh: torch.empty(*sh, dtype=torch.float32, device=dev)
        rgb, dist, op = f32(R, 3), f32(R, 1), f32(R, 1)
        a = _render_args(tc.packed, tc.geo_half, tc.app_half, tc.aabb, 1, 0.0, 1.0, True, False, None, bg_noise, rgb, dist, op, tc.grid)
        with torch.cuda.device(dev):
            _call(_L().perf_fields_packed, C.byref(a), _p(rays_o), _p(rays_d), _p(ray_indices), _p(t_starts), _p(t_ends), N, _p(n_dev), phase,
                  _p(b["sigma"]), _p(b["rgb"]), _p(b["x01"]), _p(b["feat"]), _p(b["h1"]), _p(b["h2"]), _stream(), launches=2)
            _call(_L().perf_composite_packed_fwd, _p(offsets), _p(t_starts), _p(t_ends), _p(b["sigma"]), _p(b["rgb"]), R, float(early_stop_eps),
                  _lib.PERF_FLAG_TRAINING, _p(bg_noise), _p(b["w"]), _p(b["T"]), _p(rgb), _p(dist), _p(op), _p(b["dacc"]), _p(b["dl"]), _stream())
        ctx.tc, ctx.phase, ctx.b, ctx.n_dev = tc, phase, b, n_dev
        ctx.save_for_backward(offsets, t_starts, t_ends, bg_noise, dist, op)
        return rgb, dist, op, b["dl"].clone()

    @staticmethod
    def backward(ctx, g_rgb, g_dist, g_op, g_dl):
        offsets, t_starts, t_ends, bg_noise, dist, op = ctx.saved_tensors
        tc, phase, b, n_dev = ctx.tc, ctx.phase, ctx.b, ctx.n_dev
        R, N, dev = op.shape[0], t_starts.shape[0], op.device
        geo = phase == _lib.PERF_PHASE_GEO
        mlp = GEO_MLP if geo else APP_MLP
        dz = b["dz"]
        c = lambda t: None if t is None else t.contiguous().float()
        g_rgb, g_dist, g_op, g_dl = c(g_rgb), c(g_dist), c(g_op), c(g_dl)
        with torch.cuda.device(dev):
            _call(_L().perf_composite_packed_bwd, phase, _p(offsets), _p(t_starts), _p(t_ends), _p(b["sigma"]), _p(b["rgb"]), R, _p(bg_noise),
                  _p(b["w"]), _p(b["T"]), _p(dist), _p(op), _p(b["dacc"]), _p(g_rgb), _p(g_dist), _p(g_op), _p(g_dl), _p(dz), _stream())
        half = tc.geo_half if geo else tc.app_half
        grad = torch.zeros(mlp.n_params + 2 * tc.grid.n_entries, dtype=torch.float32, device=dev)
        _, dfeat = mlp_backward_half(mlp, half[:mlp.n_params], b["feat"], b["h1"], b["h2"], dz, grad_out=grad[:mlp.n_params], n_dev=n_dev)
        with torch.cuda.device(dev):
            _call(_L().perf_hashgrid_bwd_merged, tc.grid.c(), _p(b["x01"]), _p(dfeat), N, _p(n_dev), _p(grad[mlp.n_params:]),
                  _FusedPackedTrainStep.MERGE_LEVELS, _stream(), launches=2)
        return (grad,) + (None,) * 11


def fused_packed_train_step(params, rays_o, rays_d, offsets, ray_indices, t_starts, t_ends, bg_noise, tc: FusedTrainContext, phase: int,
                            early_stop_eps: float = 1e-4, n_dev: Optional[torch.Tensor] = None):
    rays_o, rays_d = _chk(rays_o, torch.float32, "rays_o"), _chk(rays_d, torch.float32, "rays_d")
    offsets, ray_indices = _chk(offsets, torch.int64, "offsets"), _chk(ray_indices, torch.int64, "ray_indices")
    t_starts, t_ends = _chk(t_starts, torch.float32, "t_starts"), _chk(t_ends, torch.float32, "t_ends")
    bg_noise = _chk(bg_noise, torch.float32, "bg_noise")
    if offsets.numel() != rays_o.shape[0] + 1:
        raise RuntimeError("perf_b200.fused_packed_train_step: offsets must have R + 1 entries")
    if n_dev is not None:
        n_dev = _chk(n_dev, torch.int64, "n_dev")
    return _FusedPackedTrainStep.apply(params, rays_o, rays_d, offsets, ray_indices, t_starts, t_ends, bg_noise, tc, phase, early_stop_eps, n_dev)


def gather_rows(idx: torch.Tensor, *arrays: torch.Tensor):
    """``tuple(a[idx] for a in arrays)`` for row-major fp32 CUDA arrays [M, w_k] in ONE launch (the batch draw of a step)."""
    idx = _chk(idx, torch.int64, "idx")
    B, dev = idx.shape[0], idx.device
    srcs = [_chk(a.reshape(a.shape[0], -1), torch.float32, "array") for a in arrays]
    outs = [torch.empty((B,) + tuple(a.shape[1:]), dtype=torch.float32, device=dev) for a in arrays]
    n = len(srcs)
    sp = (C.c_void_p * n)(*[s.data_ptr() for s in srcs])
    dp = (C.c_void_p * n)(*[o.data_ptr() for o in outs])
    wd = (C.c_int * n)(*[int(s.shape[1]) for s in srcs])
    with torch.cuda.device(dev):
        _call(_L().perf_gather_rows, _p(idx), B, n, sp, dp, wd, _stream())
    return tuple(outs)


def draw_gather_rows(csum: torch.Tensor, M: int, *arrays: torch.Tensor, want_idx: bool = False):
    """Sorted uniform batch draw + gather in ONE launch: ``csum`` [B+1] fp64 = cumsum of i.i.d. Exp(1); row index of draw b =
    floor(csum[b] / csum[B] * M).  Returns the gathered arrays (and the indices when ``want_idx``)."""
    csum = _chk(csum, torch.float64, "csum")
    B, dev = csum.shape[0] - 1, csum.device
    srcs = [_chk(a.reshape(a.shape[0], -1), torch.float32, "array") for a in arrays]
    outs = [torch.empty((B,) + tuple(a.shape[1:]), dtype=torch.float32, device=dev) for a in arrays]
    idx = torch.empty(B, dtype=torch.int64, device=dev) if want_idx else None
    n = len(srcs)
    sp = (C.c_void_p * n)(*[s_.data_ptr() for s_ in srcs])
    dp = (C.c_void_p * n)(*[o.data_ptr() for o in outs])
    wd = (C.c_int * n)(*[int(s_.shape[1]) for s_ in srcs])
    with torch.cuda.device(dev):
        _call(_L().perf_draw_gather_rows, _p(csum), B, int(M), _p(idx), n, sp, dp, wd, _stream())
    return tuple(outs) + ((idx,) if want_idx else ())


class _FusedLoss(torch.autograd.Function):
    """total = w_main * smooth_l1(pred, gt, beta).mean() + w_dl * ratio * dl.sum() * inv_n  as ONE kernel that also
    produces the gradients (`nerf.py:208-238,281-287`); backward only scales them by the incoming gradient."""

    @staticmethod
    def forward(ctx, pred, gt, dl, ratio, inv_n, beta, w_main, w_dl):
        dev, n, R = pred.device, pred.numel(), pred.shape[0]
        loss3 = torch.empty(3, dtype=torch.float32, device=dev)
        g_pred = torch.empty_like(pred, dtype=torch.float32)
        g_dl = None if dl is None else torch.empty(R, dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            _call(_L().perf_train_loss, _p(_chk(pred.detach(), torch.float32, "pred")), _p(_chk(gt, torch.float32, "gt")), n, R, float(beta), float(w_main),
                  _p(None if dl is None else _chk(dl.detach(), torch.float32, "dl")), _p(ratio), _p(inv_n), float(w_dl), _p(loss3), _p(g_pred), _p(g_dl), _stream())
        ctx.save_for_backward(g_pred, g_dl)
        ctx.terms = loss3
        return loss3[0], loss3[1].detach(), loss3[2].detach()

    @staticmethod
    def backward(ctx, go, _g1, _g2):
        g_pred, g_dl = ctx.saved_tensors
        return g_pred * go, None, (None if g_dl is None else g_dl * go), None, None, None, None, None


def fused_loss(pred, gt, beta: float, w_main: float, dl=None, ratio=None, inv_n=None, w_dl: float = 0.0):
    """(total, main term, distortion term); see :class:`_FusedLoss`.  ``ratio`` / ``inv_n``: device scalars or None."""
    for t in (ratio, inv_n):
        if t is not None and not (torch.is_tensor(t) and t.is_cuda and t.dtype == torch.float32):
            raise RuntimeError("perf_b200.fused_loss: ratio / inv_n must be fp32 CUDA tensors")
    return _FusedLoss.apply(pred, gt.reshape(pred.shape), dl, None if ratio is None else ratio.reshape(-1).contiguous(),
                            None if inv_n is None else inv_n.reshape(-1).contiguous(), beta, w_main, w_dl)


def atomic_rate(n_floats: int = 2 * 8 * 262144, n_atomics: int = 1 << 26, vec: int = 4, device="cuda", iters: int = 5) -> float:
    """Measured L2 reduction rate (atomics / s) for random vec-wide fp32 atomics into a table the size of the eight fine
    levels' gradient (default): the physical bound of the grid-gradient scatter (bench.py `train_roofline`)."""
    table = torch.zeros(n_floats, dtype=torch.float32, device=device)
    fn = lambda: _call(_L().perf_debug_atomic_rate, _p(table), n_floats, n_atomics, vec, _stream())
    with torch.cuda.device(table.device):
        fn(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record(); torch.cuda.synchronize()
    return n_atomics * iters / (e0.elapsed_time(e1) * 1e-3)


def occ_points(cell_idx: Optional[torch.Tensor], n: int, res3, aabb, seed: int, device) -> torch.Tensor:
    """A uniformly jittered point in each listed occupancy cell (``cell_idx`` int64 [n]; None = cells 0..n-1) -> [n,3]."""
    x = torch.empty(n, 3, dtype=torch.float32, device=device)
    r3, a6 = (C.c_int * 3)(*[int(v) for v in res3]), (C.c_float * 6)(*[float(v) for v in aabb])
    with torch.cuda.device(x.device):
        _call(_L().perf_occ_points, _p(None if cell_idx is None else _chk(cell_idx, torch.int64, "cell_idx")), n, r3, a6, int(seed) & (2 ** 63 - 1),
              _p(x), _stream())
    return x


def occ_update(occs: torch.Tensor, cell_idx: Optional[torch.Tensor], occ_new: torch.Tensor, ema_decay: float, occ_thre: float,
               binaries_u8: torch.Tensor, workspace: torch.Tensor) -> None:
    """occs[c] = max(occs[c] * ema_decay, occ_new) on the listed cells, then binaries = occs > min(mean(occs), occ_thre)."""
    occs, occ_new = _chk(occs, torch.float32, "occs"), _chk(occ_new.reshape(-1), torch.float32, "occ_new")
    with torch.cuda.device(occs.device):
        _call(_L().perf_occ_update, _p(occs), occs.numel(), _p(None if cell_idx is None else _chk(cell_idx, torch.int64, "cell_idx")),
              _p(occ_new), occ_new.numel(), float(ema_decay), float(occ_thre), _p(binaries_u8), _p(workspace), _stream(), launches=3)


def fused_train_step(params, rays_o, rays_d, jitter, bg_noise, tc: FusedTrainContext, phase: int):
    rays_o, rays_d = _chk(rays_o, torch.float32, "rays_o"), _chk(rays_d, torch.float32, "rays_d")
    jitter, bg_noise = _chk(jitter, torch.float32, "jitter"), _chk(bg_noise, torch.float32, "bg_noise")
    return _FusedTrainStep.apply(params, rays_o, rays_d, jitter, bg_noise, tc, phase)


# ------------------------------------------------------------------ optimiser
def adam_step(params, grads, exp_avg, exp_avg_sq, step: int, lr: float, params_half=None,
              beta1=0.9, beta2=0.999, eps=1e-8, grad_scale=1.0):
    """In-place fused Adam (torch.optim.Adam semantics) + optional fp16 shadow refresh."""
    for t, n in ((params, "params"), (grads, "grads"), (exp_avg, "exp_avg"), (exp_avg_sq, "exp_avg_sq")):
        if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
            raise RuntimeError(f"perf_b200.adam_step: `{n}` must be a contiguous fp32 CUDA tensor")
    with torch.cuda.device(params.device):
        _call(_L().perf_adam_step, _p(params), _p(grads), _p(exp_avg), _p(exp_avg_sq), _p(params_half),
              params.numel(), lr, beta1, beta2, eps, step, grad_scale, _stream())


def adam_step_dev(params, grads, exp_avg, exp_avg_sq, hyper: torch.Tensor, params_half=None,
                  beta1=0.9, beta2=0.999, eps=1e-8, grad_scale=1.0):
    """``adam_step`` with {lr, 1-beta1^t, sqrt(1-beta2^t)} in the device tensor ``hyper`` [3] (graph-replayable)."""
    with torch.cuda.device(params.device):
        _call(_L().perf_adam_step_dev, _p(params), _p(grads), _p(exp_avg), _p(exp_avg_sq), _p(params_half),
              params.numel(), _p(hyper), beta1, beta2, eps, grad_scale, _stream())


def set_scalars(dst: torch.Tensor, values) -> None:
    """dst[:len(values)] = values (<= 8 floats), stream-ordered, race-free w.r.t. the host (by-value kernel args)."""
    vals = [float(v) for v in values]
    arr = (C.c_float * len(vals))(*vals)
    with torch.cuda.device(dst.device):
        _call(_L().perf_set_scalars, _p(dst), arr, len(vals), _stream())
