"""FusedPanoRenderer -- the fast path behind ``NeRFScene.render`` / ``render_dense``.

Mirrors the reference's renderer interface for the fixed-S sampler:
``NeRFScene.render(rays, query_keys)`` (`/root/reference/modules/scene/nerf.py:74-99`) and the
inner loop of ``CoreRunner.render_dense`` (`/root/reference/core_exp_runner.py:229-238`), but as
ONE kernel launch per call (no 32768-ray chunk loop, no per-sample tensors in HBM).
"""
from __future__ import annotations

from typing import Optional, Sequence

import torch

from . import ops
from .config import APP_MLP, GEO_MLP, PERF_GRID, GridConfig


class FusedPanoRenderer:
    """Holds the fp16 shadow of both field networks (the flat tcnn ``params`` vectors stored in
    PeRF checkpoints under ``nerf.geo_mlp.params`` / ``nerf.app_mlp.params``) in kernel layout."""

    def __init__(self, grid: GridConfig = PERF_GRID, aabb: Sequence[float] = (-1., -1., -1., 1., 1., 1.),
                 near: float = 1e-2, far: float = 1.0, kernel: str = "march"):
        self.grid, self.aabb, self.near, self.far = grid, tuple(float(v) for v in aabb), near, far
        self.kernel = kernel          # "march": thread = ray (default); "scan": lanes = samples of one ray
        self.geo_half = self.app_half = self.packed = None
        self.occ = None               # set_occupancy(): grid + lattice of render_rays_occ / render_pano_occ

    @classmethod
    def from_params(cls, geo_params: torch.Tensor, app_params: torch.Tensor, **kw) -> "FusedPanoRenderer":
        r = cls(**kw)
        r.set_params(geo_params, app_params)
        return r

    @classmethod
    def from_state_dict(cls, nerf_state: dict, estimator_state: Optional[dict] = None, device="cuda", **kw) -> "FusedPanoRenderer":
        """``nerf_state`` = ``checkpoint['scene']['nerf']`` of a PeRF ``ckpt.pth``
        (`modules/scene/nerf.py:374-380`): keys ``aabb``, ``geo_mlp.params``, ``app_mlp.params``.
        ``estimator_state`` = ``checkpoint['scene']['estimator']`` (an ``OccGridEstimator``'s buffers): its ``binaries`` and
        ``aabbs`` become the occupancy grid of :meth:`render_rays_occ` / :meth:`render_pano_occ` (PeRF's lattice defaults)."""
        kw.setdefault("aabb", nerf_state["aabb"].tolist())
        r = cls.from_params(nerf_state["geo_mlp.params"].to(device), nerf_state["app_mlp.params"].to(device), **kw)
        if estimator_state is not None:
            binaries, aabbs = estimator_state["binaries"], estimator_state["aabbs"]
            if binaries.dim() != 4 or binaries.shape[0] != 1 or aabbs.shape[0] != 1:
                raise NotImplementedError(f"occupancy grid with {binaries.shape[0]} levels: only levels=1 is implemented (PeRF uses 1)")
            r.set_occupancy(binaries[0].to(device), aabbs[0].tolist())
        return r

    def set_occupancy(self, binaries: torch.Tensor, roi_aabb: Sequence[float], near: float = 0., far: float = 1.5, step: float = 5e-4,
                      early_stop_eps: float = 1e-4) -> None:
        """The occupancy grid of the one-launch grid renderer: ``binaries`` [rx,ry,rz] bool (``OccGridEstimator.binaries[0]``,
        x slowest), its ``roi_aabb`` and the sampling lattice (PeRF: ``nerf_renderer.py:145-155``).  The tensor is used
        as it is, not copied: an estimator update that rewrites it in place is seen by the next render."""
        if binaries.dim() != 3 or not binaries.is_cuda:
            raise ValueError(f"binaries must be a CUDA tensor [rx, ry, rz], got {tuple(binaries.shape)} on {binaries.device}")
        self.occ = {"binaries": binaries.contiguous(), "grid_aabb": tuple(float(v) for v in roi_aabb), "near": float(near),
                    "far": float(far), "step": float(step), "early_stop_eps": float(early_stop_eps)}

    def set_params(self, geo_params: torch.Tensor, app_params: torch.Tensor) -> None:
        """fp32 master params -> fp16 shadows + interleaved gather table (3 small kernels).
        Call again after every optimiser step that changed them."""
        n_g = GEO_MLP.n_params + 2 * self.grid.n_entries
        n_a = APP_MLP.n_params + 2 * self.grid.n_entries
        if geo_params.numel() != n_g or app_params.numel() != n_a:
            raise ValueError(f"params have {geo_params.numel()}/{app_params.numel()} values, expected {n_g}/{n_a}")
        self.geo_half = ops.params_to_half(geo_params.detach().float(), out=self.geo_half)
        self.app_half = ops.params_to_half(app_params.detach().float(), out=self.app_half)
        self.packed = ops.pack_tables(self.geo_half, self.app_half, self.grid, out=self.packed)

    def set_halves(self, geo_half: torch.Tensor, app_half: torch.Tensor) -> None:
        """Adopt already-cast fp16 shadows (e.g. the ones the fused Adam kernel maintains) and
        rebuild the interleaved gather table (one kernel)."""
        self.geo_half, self.app_half = geo_half, app_half
        self.packed = ops.pack_tables(geo_half, app_half, self.grid, out=self.packed)

    def _ready(self):
        if self.packed is None:
            raise RuntimeError("FusedPanoRenderer: call set_params() first")

    def render_rays(self, rays_o: torch.Tensor, rays_d: torch.Tensor, n_samples: int, near: Optional[float] = None,
                    far: Optional[float] = None, training: bool = False, jitter: Optional[torch.Tensor] = None,
                    bg_noise: Optional[torch.Tensor] = None, simt: bool = False) -> dict:
        self._ready()
        # [H, W, 3] ray images are tiled as pixel patches (same locality as render_pano)
        image_width = rays_o.shape[-2] if rays_o.dim() == 3 else 0
        rgb, dist, op = ops.render_rays(self.packed, self.geo_half, self.app_half, rays_o.reshape(-1, 3), rays_d.reshape(-1, 3),
                                        n_samples, self.near if near is None else near, self.far if far is None else far,
                                        self.aabb, training, jitter, bg_noise, self.grid, simt, self.kernel, image_width)
        return {"rgb": rgb, "distance": dist, "opacities": op, "is_valid": True}

    def render_packed(self, rays_o: torch.Tensor, rays_d: torch.Tensor, ray_indices: torch.Tensor, t_starts: torch.Tensor,
                      t_ends: torch.Tensor, simt: bool = False) -> dict:
        """Eval render of packed per-ray intervals (``OccGridEstimator.sampling`` output) in one launch:
        the body of ``NeRFOCCRenderer.render`` after the sampling call (`nerf_renderer.py:164-197`)."""
        self._ready()
        rgb, dist, op = ops.render_packed(self.packed, self.geo_half, self.app_half, rays_o.reshape(-1, 3), rays_d.reshape(-1, 3),
                                          ray_indices, t_starts, t_ends, self.aabb, self.grid, simt)
        return {"rgb": rgb, "distance": dist, "opacities": op, "is_valid": True}

    def render_occ(self, rays_o: torch.Tensor, rays_d: torch.Tensor, offsets: torch.Tensor, ray_indices: torch.Tensor,
                   t_starts: torch.Tensor, t_ends: torch.Tensor, early_stop_eps: float = 1e-4) -> dict:
        """Eval render of ALL intervals an occupancy sampler emitted (no visibility pre-pass): both fields at every
        interval in one launch (perf_fields_packed), then the per-ray composite with nerfacc's transmittance cut applied
        inside (perf_composite_packed_fwd) -- `nerf_renderer.py:145-197` without the second density evaluation."""
        self._ready()
        rgb, dist, op = ops.render_occ(self.packed, self.geo_half, self.app_half, rays_o.reshape(-1, 3), rays_d.reshape(-1, 3),
                                       offsets, ray_indices, t_starts, t_ends, early_stop_eps, self.aabb, self.grid)
        return {"rgb": rgb, "distance": dist, "opacities": op, "is_valid": True}

    def _occ_ready(self, overrides: dict) -> dict:
        self._ready()
        if self.occ is None:
            raise RuntimeError("FusedPanoRenderer: call set_occupancy() (or from_state_dict with estimator_state) first")
        return {**self.occ, **{k: v for k, v in overrides.items() if v is not None}}

    def render_rays_occ(self, rays_o: torch.Tensor, rays_d: torch.Tensor, early_stop_eps: Optional[float] = None, simt: bool = False,
                        want_n_samples: bool = False) -> dict:
        """Eval render of explicit rays with the occupancy grid of :meth:`set_occupancy` in ONE launch: the grid walk, both
        fields and the composite with the transmittance cut per ray (`nerf_renderer.py:145-197`).  [H, W, 3] ray images are
        tiled as pixel patches.  ``want_n_samples`` adds ``n_samples`` (intervals composited per ray, int32)."""
        occ = self._occ_ready({"early_stop_eps": early_stop_eps})
        image_width = rays_o.shape[-2] if rays_o.dim() == 3 else 0
        res = ops.render_rays_occ(self.packed, self.geo_half, self.app_half, rays_o.reshape(-1, 3), rays_d.reshape(-1, 3), occ["binaries"],
                                  occ["grid_aabb"], occ["near"], occ["far"], occ["step"], occ["early_stop_eps"], self.aabb, self.grid, simt,
                                  image_width, want_n_samples, self.kernel)
        out = {"rgb": res[0], "distance": res[1], "opacities": res[2], "is_valid": True}
        if want_n_samples:
            out["n_samples"] = res[3]
        return out

    def render_pano_occ(self, pose, H: int, W: int, row0: int = 0, rows: Optional[int] = None, early_stop_eps: Optional[float] = None,
                        simt: bool = False, out=None, want_n_samples: bool = False) -> dict:
        """Rows [row0,row0+rows) of an HxW equirect panorama with the occupancy grid, ray generation fused in (one launch)."""
        occ = self._occ_ready({"early_stop_eps": early_stop_eps})
        res = ops.render_pano_occ(self.packed, self.geo_half, self.app_half, pose, H, W, occ["binaries"], occ["grid_aabb"], occ["near"],
                                  occ["far"], occ["step"], occ["early_stop_eps"], row0, rows, self.aabb, self.grid, simt, out,
                                  want_n_samples, self.kernel)
        ret = {"rgb": res[0], "distance": res[1], "opacities": res[2], "is_valid": True}
        if want_n_samples:
            ret["n_samples"] = res[3]
        return ret

    def render_pano(self, pose, H: int, W: int, n_samples: int, row0: int = 0, rows: Optional[int] = None,
                    near: Optional[float] = None, far: Optional[float] = None, simt: bool = False, out=None) -> dict:
        self._ready()
        rgb, dist, op = ops.render_pano(self.packed, self.geo_half, self.app_half, pose, H, W, n_samples,
                                        self.near if near is None else near, self.far if far is None else far,
                                        row0, rows, self.aabb, self.grid, simt, out, self.kernel)
        return {"rgb": rgb, "distance": dist, "opacities": op, "is_valid": True}

    @torch.no_grad()
    def render(self, rays, query_keys=("rgb",), n_samples: int = 128) -> dict:
        """Drop-in for ``NeRFScene.render(rays, query_keys)``: ``rays`` has ``.o`` / ``.d`` of shape
        [..., 3]; returns ``{key: tensor[..., C]}`` (eval-mode background rule)."""
        pre_shape = list(rays.o.shape[:-1])
        o, d = rays.o.float(), rays.d.float()
        if o.dim() != 3:
            o, d = o.reshape(-1, 3), d.reshape(-1, 3)
        out = self.render_rays(o, d, n_samples)
        return {k: out[k].reshape(pre_shape + [-1]) for k in query_keys}
