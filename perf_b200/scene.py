"""Host-side mirror of PeRF's scene layer for the fixed-S sampler, on libperfb200.

Mirrors (same method names, argument meaning, dict keys, error behaviour):
  ``NeRFScene``            `/root/reference/modules/scene/nerf.py:28-396`
  ``NeRFOCCRenderer``      `/root/reference/modules/scene/nerf_renderer.py:105-209`
  ``SupInfoPool.rand_ray_color_data``  `/root/reference/modules/dataset/sup_info.py:236-259`
What differs by design: ``render`` (eval, no grad) is ONE fused-kernel launch instead of a
32768-ray chunk loop; the optimiser is the fused Adam kernel; with WORLD_SIZE > 1 the ray batch is
sharded over ranks and the flat gradient is all-reduced once per step.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional

import numpy as np
import torch
import torch.nn.functional as F

from . import ops, parallel
from .config import Conf
from .field import NGPNeRF
from .renderer import FusedPanoRenderer
from .shims import nerfacc
from .shims.torch_efficient_distloss import flatten_eff_distloss


@dataclass
class Rays:                                   # utils/camera_utils.py:9-20
    o: torch.Tensor
    d: torch.Tensor

    def __len__(self):
        return len(self.o)

    def __getitem__(self, idx):
        return Rays(self.o[idx], self.d[idx])

    def collapse(self):
        return self.o, self.d


def gen_pano_rays(pose, height=512, width=1024, device="cuda") -> Rays:
    """`utils/camera_utils.py:229-234` on the GPU (perf_raygen_pano)."""
    o, d = ops.raygen_pano(pose, height, width, device=device)
    return Rays(o, d)


def gen_pers_rays(pose, fov, res, device="cuda") -> Rays:
    """`utils/camera_utils.py:237-241` on the GPU (perf_raygen_pers)."""
    o, d = ops.raygen_pers(pose, fov, res, device=device)
    return Rays(o, d)


@dataclass
class BoundedRays:                            # utils/camera_utils.py:22-35
    o: torch.Tensor
    d: torch.Tensor
    near: torch.Tensor
    far: torch.Tensor

    def __len__(self):
        return len(self.o)

    def __getitem__(self, idx):
        return BoundedRays(self.o[idx], self.d[idx], self.near[idx], self.far[idx])

    def collapse(self):
        return self.o, self.d, self.near, self.far


class FixedSampleEstimator(torch.nn.Module):
    """Stands where ``OccGridEstimator`` stands in the renderer: the benchmark's fixed-S sampler
    (SURVEY.md 8 a7'): ``t_s[k] = near + (k + u_r) * step``, one jitter ``u_r`` per ray when
    stratified.  Returns packed (ray_indices, t_starts, t_ends) like nerfacc."""

    def __init__(self, n_samples: int = 128, near: float = 1e-2, far: float = 1.0):
        super().__init__()
        self.n_samples, self.near, self.far = n_samples, near, far
        self._ri = None

    @torch.no_grad()
    def sampling(self, rays_o, rays_d, sigma_fn=None, stratified=False, jitter=None, **_):
        R, S, dev = rays_o.shape[0], self.n_samples, rays_o.device
        near, far = torch.tensor(self.near, device=dev), torch.tensor(self.far, device=dev)
        step = (far - near) / float(S)
        k = torch.arange(S + 1, device=dev, dtype=torch.float32)[None, :]
        if jitter is None:
            jitter = torch.rand(R, device=dev) if stratified else torch.zeros(R, device=dev)
        edges = near + (k + jitter.reshape(R, 1)) * step
        if self._ri is None or self._ri.numel() != R * S or self._ri.device != dev:
            self._ri = torch.arange(R, device=dev).repeat_interleave(S)
        return self._ri, edges[:, :-1].reshape(-1), edges[:, 1:].reshape(-1)


class NeRFOCCRenderer(torch.nn.Module):
    """Differentiable (training) render path = the reference's renderer line by line on the plugin
    functions; `nerf_renderer.py:112-209`."""

    def __init__(self, max_radius=2, bg_color="rand_noise"):
        super().__init__()
        assert bg_color in ["rand_noise", "black", "white"]
        self.max_radius, self.bg_color = max_radius, bg_color

    def render(self, nerf: NGPNeRF, estimator, rays_o, rays_d, near=None, far=None, geo_inference=False, app_inference=False):
        n_rays, dev = rays_o.shape[0], rays_o.device

        def positions(t_starts, t_ends, ray_indices):
            return rays_o[ray_indices] + rays_d[ray_indices] * (t_starts + t_ends)[:, None] / 2.0

        def sigma_fn(t_starts, t_ends, ray_indices):
            return nerf.query_density(positions(t_starts, t_ends, ray_indices)).squeeze(-1)

        ray_indices, t_starts, t_ends = estimator.sampling(rays_o, rays_d, sigma_fn=sigma_fn, near_plane=0., far_plane=1.5,
                                                           render_step_size=5e-4, stratified=nerf.training,
                                                           cone_angle=0., alpha_thre=0.)
        if ray_indices.numel() <= 0:
            return {"is_valid": False, "rgb": torch.zeros(n_rays, 3, device=dev), "distance": torch.zeros(n_rays, 1, device=dev),
                    "opacities": torch.zeros(n_rays, 1, device=dev)}
        pos = positions(t_starts, t_ends, ray_indices)
        with torch.set_grad_enabled(torch.is_grad_enabled() and not geo_inference):
            sigmas = nerf.query_density(pos).squeeze(-1)
        weights, trans, alphas = nerfacc.render_weight_from_density(t_starts, t_ends, sigmas, ray_indices=ray_indices, n_rays=n_rays)
        opacities = nerfacc.accumulate_along_rays(weights, values=None, ray_indices=ray_indices, n_rays=n_rays)
        sampled_distances = ((t_starts + t_ends) / 2.0)[..., None]
        distances = nerfacc.accumulate_along_rays(weights, sampled_distances, ray_indices=ray_indices, n_rays=n_rays)
        with torch.set_grad_enabled(torch.is_grad_enabled() and not app_inference):
            rgbs = nerf.query_rgb(pos)
        colors = nerfacc.accumulate_along_rays(weights.detach(), values=rgbs, ray_indices=ray_indices, n_rays=n_rays)
        if self.bg_color == "rand_noise":
            bg_color = torch.rand(n_rays, 3, device=dev)
        elif self.bg_color == "white":
            bg_color = torch.ones(n_rays, 3, device=dev)
        else:
            bg_color = torch.zeros(n_rays, 3, device=dev)
        if nerf.training:
            distances = torch.relu(distances + (torch.rand_like(distances) * 2. - 1.) * (1. - opacities))
            colors = colors + bg_color * (1. - opacities).detach()
        else:
            distances = distances + 5. * (1. - opacities).detach()
            colors = colors + .5 * (1. - opacities).detach()
        return {"is_valid": True, "rgb": colors, "distance": distances, "weights": weights, "opacities": opacities,
                "trans": trans, "t_starts": t_starts, "t_ends": t_ends, "ray_indices": ray_indices}


class RaySupervision:
    """Flat pool of supervised rays = what ``SupInfoPool`` exposes to the trainer
    (`sup_info.py:236-259`: ``all_sup_rays / all_sup_colors / all_sup_distances``)."""

    def __init__(self, rays: Rays, colors: torch.Tensor, distances: torch.Tensor, normals: Optional[torch.Tensor] = None, seed: int = 0):
        self.all_sup_rays, self.all_sup_colors = rays, colors
        self.all_sup_distances = distances.reshape(-1, 1)
        self.all_sup_normals = torch.zeros_like(colors) if normals is None else normals
        self.generator = torch.Generator(device=colors.device).manual_seed(seed + parallel.rank())
        self.locality_key = None      # optional int64 key per ray; batches are ordered by it
        self.morton_sorted = False    # from_panorama stores the pool in Morton order and draws sorted batches without a sort
        self.use_default_generator = False

    @staticmethod
    def from_panorama(pose, rgb: torch.Tensor, distance: torch.Tensor, seed: int = 0) -> "RaySupervision":
        h, w = distance.shape[:2]
        rays = gen_pano_rays(pose, h, w, device=rgb.device)
        pool = RaySupervision(Rays(rays.o.reshape(-1, 3), rays.d.reshape(-1, 3)), rgb.reshape(-1, 3).float(), distance.reshape(-1, 1).float(), seed=seed)
        # Morton (Z-order) code of the pixel: a batch sorted by it puts rays that are neighbours on the
        # sphere into the same warp, so their hash-grid gathers share cache lines at the coarse levels.
        # The batch is the same multiset of rays torch.randint drew (sup_info.py:253-257); only its order changes.
        yy, xx = torch.meshgrid(torch.arange(h, device=rgb.device), torch.arange(w, device=rgb.device), indexing="ij")
        key = torch.zeros(h, w, dtype=torch.int32, device=rgb.device)   # int32: half the radix-sort passes of int64
        xx, yy = xx.to(torch.int32), yy.to(torch.int32)
        for b in range(15):                                              # panoramas up to 32768 x 32768
            key |= ((xx >> b) & 1) << (2 * b)
            key |= ((yy >> b) & 1) << (2 * b + 1)
        # Store the pool IN Morton order: a batch of SORTED row indices is then spatially coherent by itself, and sorted
        # uniform indices can be drawn directly (order statistics from exponential spacings) -- no radix sort, no key gather,
        # no index permutation per step (13 launches -> 3).  The batch is still B i.i.d. uniform draws with replacement
        # (sup_info.py:253-257) up to its order.
        perm = torch.argsort(key.reshape(-1))
        pool.all_sup_rays = Rays(pool.all_sup_rays.o[perm].contiguous(), pool.all_sup_rays.d[perm].contiguous())
        pool.all_sup_colors, pool.all_sup_distances = pool.all_sup_colors[perm].contiguous(), pool.all_sup_distances[perm].contiguous()
        pool.all_sup_normals = pool.all_sup_normals[perm].contiguous()
        pool.morton_sorted = True
        return pool

    def gen_occ_grid(self, res: int):
        """`sup_info.py:304-330`: voxels within +-1 cell of every un-projected RGB-D point ->
        (uint8 grid [res^3] with x slowest, centres of the occupied voxels)."""
        rays_o, rays_d = self.all_sup_rays.collapse()
        pts = rays_o + rays_d * self.all_sup_distances.squeeze()[..., None]
        occ_grid = torch.zeros(res * res * res, dtype=torch.uint8, device=pts.device)
        shift = 1. / res
        lin = torch.linspace(-shift, shift, 3, device=pts.device)
        shifts = torch.stack(torch.meshgrid(lin, lin, lin, indexing="ij"), -1).reshape(-1, 3)
        for shift_xyz in shifts:
            shifted = ((shift_xyz[None, :] + pts).clip(-0.999, 0.999) * .5 + .5) * res
            shifted = shifted.to(torch.int64)
            occ_grid[shifted[..., 0] * res * res + shifted[..., 1] * res + shifted[..., 2]] = 1
        valid_idx = torch.where(occ_grid > 0)[0]
        valid_pts = torch.stack([valid_idx // (res * res), (valid_idx // res) % res, valid_idx % res], -1)
        return occ_grid, (valid_pts / float(res) - .5) * 2.

    @staticmethod
    def sorted_uniform_csum(batch_size: int, device, generator=None) -> torch.Tensor:
        """Running sums S_1..S_{B+1} (fp64) of i.i.d. Exp(1): S_k / S_{B+1} are the order statistics of B i.i.d. U(0,1)."""
        e = torch.empty(batch_size + 1, dtype=torch.float64, device=device).exponential_(generator=generator)
        return torch.cumsum(e, 0)

    def rand_ray_color_data(self, batch_size, rand_mode="by_all_pixels"):
        gen = None if self.use_default_generator else self.generator     # default generator: CUDA-graph safe
        if getattr(self, "morton_sorted", False):
            M = len(self.all_sup_colors)
            csum = self.sorted_uniform_csum(batch_size, self.all_sup_colors.device, gen)
            if self.all_sup_colors.is_cuda:
                o, d, c, dist, nrm = ops.draw_gather_rows(csum, M, self.all_sup_rays.o, self.all_sup_rays.d, self.all_sup_colors,
                                                          self.all_sup_distances, self.all_sup_normals)
                return Rays(o, d), c, dist, nrm
            idx = (csum[:-1] / csum[-1] * M).to(torch.int64).clamp_(0, M - 1)
            return self.all_sup_rays[idx], self.all_sup_colors[idx], self.all_sup_distances[idx], self.all_sup_normals[idx]
        idx = torch.randint(0, len(self.all_sup_colors), (batch_size,), device=self.all_sup_colors.device, generator=gen)
        if self.locality_key is not None:
            idx = idx[torch.argsort(self.locality_key[idx])]
        if self.all_sup_colors.is_cuda and self.all_sup_colors.dtype == torch.float32:
            # one gather launch for the five arrays (sup_info.py:253-259 indexes each of them separately)
            o, d, c, dist, nrm = ops.gather_rows(idx, self.all_sup_rays.o, self.all_sup_rays.d, self.all_sup_colors,
                                                 self.all_sup_distances, self.all_sup_normals)
            return Rays(o, d), c, dist, nrm
        return self.all_sup_rays[idx], self.all_sup_colors[idx], self.all_sup_distances[idx], self.all_sup_normals[idx]


class _Lazy:
    """A renderer output that costs launches to form (the scalar distortion loss): evaluated only when a caller asks for it."""

    def __init__(self, fn):
        self.fn = fn

    def __call__(self):
        return self.fn()


class FusedAdam:
    """``torch.optim.Adam(params, lr)`` semantics (defaults betas=(.9,.999), eps=1e-8) on one flat
    fp32 parameter through perf_adam_step; exposes ``param_groups`` so ``update_lr`` reads as in
    `nerf.py:300-311`.

    Distributed (world > 1), default ``parallel.dp_mode() == 'sharded'``: the local gradients are reduce-scattered
    (sum; the 1/world of the mean is the Adam kernel's ``grad_scale``), this rank updates ITS contiguous 1/world shard
    of the parameters -- the moments exist only for that shard -- and the fp16 shadow every kernel reads is
    all-gathered.  The fp32 master vector is therefore current only inside the rank's shard until
    :meth:`sync_master` all-gathers it (called at the end of a phase and by ``NeRFScene.state_dict``)."""

    def __init__(self, param: torch.nn.Parameter, lr: float = 0.0, betas=(0.9, 0.999), eps: float = 1e-8, module=None):
        self.param, self.betas, self.eps = param, betas, eps
        self.module = module        # tinycudann shim module owning `param`: its fp16 shadow is refreshed by the Adam kernel
        self.param_groups = [{"lr": lr}]
        self.world, self.rank = parallel.world_size(), parallel.rank()
        self.sharded = self.world > 1 and parallel.dp_mode() == "sharded" and module is not None
        n = param.numel()
        if self.sharded:
            self.shard = parallel.shard_len(n, self.world)
            self.lo = min(n, self.rank * self.shard)
            self.hi = min(n, self.lo + self.shard)
            self.padded = self.world * self.shard
            z = lambda: torch.zeros(self.hi - self.lo, dtype=torch.float32, device=param.device)
            self.exp_avg, self.exp_avg_sq = z(), z()
            # scratch with room for the padding tail when numel is not a multiple of world * 8 (never for PeRF's nets at 2/4/8)
            self._grad_pad = torch.zeros(self.padded, dtype=torch.float32, device=param.device) if self.padded != n else None
            self._half_pad = torch.zeros(self.padded, dtype=torch.float16, device=param.device) if self.padded != n else None
            self._master_pad = None
        else:
            self.exp_avg, self.exp_avg_sq = torch.zeros_like(param.data), torch.zeros_like(param.data)
        self.master_stale = False
        self.step_count = 0
        # graph mode: lr / bias corrections live in a device tensor refreshed from pinned memory before each replay
        self.hyper = None

    def enable_graph_mode(self):
        self.hyper = torch.zeros(3, dtype=torch.float32, device=self.param.device)

    def push_hyper(self):
        """(graph mode) advance the step count and upload {lr, 1-b1^t, sqrt(1-b2^t)}; call before replay."""
        self.step_count += 1
        t = self.step_count
        ops.set_scalars(self.hyper, [self.param_groups[0]["lr"], 1.0 - self.betas[0] ** t, (1.0 - self.betas[1] ** t) ** 0.5])

    def zero_grad(self):
        self.param.grad = None

    def _adam(self, p, g, m, v, half, grad_scale):
        if self.hyper is not None:                           # graph mode: schedule comes from device memory
            ops.adam_step_dev(p, g, m, v, self.hyper, params_half=half, beta1=self.betas[0], beta2=self.betas[1], eps=self.eps,
                              grad_scale=grad_scale)
        else:
            self.step_count += 1
            ops.adam_step(p, g, m, v, self.step_count, self.param_groups[0]["lr"], params_half=half,
                          beta1=self.betas[0], beta2=self.betas[1], eps=self.eps, grad_scale=grad_scale)

    def step(self, valid: bool = True):
        """One optimiser step = exchange -> Adam -> gather (see the three stage methods; `GraphedTrainStep(split=True)`
        captures them separately to time them).  ``valid=False`` (this rank produced no samples, `nerf.py:204-206`):
        the rank still takes part in the exchange with a zero gradient so that the other ranks do not block."""
        if getattr(self, "deferred", False):                 # split capture: the stages are replayed on their own
            self._valid = valid
            return
        if not self.stage_exchange(valid):
            return
        self.stage_adam()
        if getattr(self, "skip_gather", False):              # the gather is captured at the start of the NEXT step
            self._mark_updated()
        else:
            self.stage_gather()

    def stage_exchange(self, valid: bool = True) -> bool:
        """Gradient exchange: reduce-scatter (sharded) or all-reduce + mean.  False = nothing to do."""
        g = self.param.grad
        if g is None:
            if self.world == 1 or valid:
                return False
            g = torch.zeros_like(self.param.data)
        g = g.contiguous()
        n = self.param.numel()
        if self.sharded:
            if self._grad_pad is not None:
                self._grad_pad[:n].copy_(g); g = self._grad_pad
            self._g = parallel.reduce_scatter_sum_(g, self.shard)[: self.hi - self.lo]
        else:
            self._g = parallel.allreduce_mean_(g)
        return True

    def stage_adam(self):
        half = self.module._half() if self.module is not None else None     # allocate / reuse the module's fp16 shadow buffer
        if self.sharded:
            self._hbuf = half if self._half_pad is None else self._half_pad
            self._adam(self.param.data[self.lo:self.hi], self._g, self.exp_avg, self.exp_avg_sq, self._hbuf[self.lo:self.hi], 1.0 / self.world)
        else:
            self._adam(self.param.data, self._g, self.exp_avg, self.exp_avg_sq, half, 1.0)
        self._g = None

    def stage_gather(self):
        if self.sharded:
            parallel.all_gather_(self._hbuf, self.shard)
            if self._half_pad is not None:
                self.module._half().copy_(self._hbuf[:self.param.numel()])
            self.master_stale = True
        self._mark_updated()

    def _mark_updated(self):
        # the kernel wrote through .data: bump autograd's version counter so version-keyed caches notice
        torch._C._increment_version([self.param])   # takes an ITERABLE of tensors
        if self.module is not None:                          # the shadow is already current for the new version
            self.module._half_key = (self.param._version, self.param.data_ptr())

    def sync_master(self):
        """(sharded mode) all-gather the fp32 master parameters so that every rank holds the full current vector."""
        if not (self.sharded and self.master_stale):
            return
        n = self.param.numel()
        if self.padded != n:
            if self._master_pad is None:
                self._master_pad = torch.zeros(self.padded, dtype=torch.float32, device=self.param.device)
            self._master_pad[self.lo:self.hi].copy_(self.param.data[self.lo:self.hi])
            parallel.all_gather_(self._master_pad, self.shard)
            self.param.data.copy_(self._master_pad[:n])
        else:
            parallel.all_gather_(self.param.data, self.shard)
        self.master_stale = False
        torch._C._increment_version([self.param])
        if self.module is not None:
            self.module._half_key = (self.param._version, self.param.data_ptr())


DEFAULT_TRAIN_CONF = Conf.wrap({
    "raw_phase_iter_geo": 3000, "raw_phase_iter_app": 1500,
    "geo_optimizer": {"init_lr": 0.0, "peak_lr": 1e-2, "peak_at": 0.2, "lr_alpha": 1e-2},
    "app_optimizer": {"init_lr": 0.0, "peak_lr": 1e-2, "peak_at": 0.2, "lr_alpha": 1e-2},
    "color_loss_weight": 1., "depth_loss_weight": 1., "distortion_loss_weight": 0.1, "density_loss_weight": 0.,
    "pixel_loss_batch_size": 8192})                                   # configs/nerf.yaml:28-66


class NeRFScene:
    """`nerf.py:28-396` for ``sampler: fixed``.  ``train_conf`` takes the reference's YAML node."""

    LOSS_SCALE = 2 ** 7                                               # GradScaler(2**7), never unscaled (nerf.py:139,249-253)
    OCC_STEP = 5e-4                                                   # render_step_size (nerf_renderer.py:151)

    def __init__(self, base_exp_dir=".", train_conf=None, estimator_type="fixed", renderer_conf=None,
                 n_samples: int = 128, near: float = 1e-2, far: float = 1.0, device="cuda", writer=None, fused_train: bool = True,
                 occ_resolution: int = 256, graph_train: bool = False):
        if estimator_type not in ("fixed", "occ"):
            raise NotImplementedError(f"perf_b200 NeRFScene: estimator_type={estimator_type!r} (the reference's 'prop' renderer is "
                                      "broken upstream, nerf_renderer.py:73, and not implemented)")
        self.estimator_type, self.occ_resolution = estimator_type, occ_resolution
        self.device = torch.device(device)
        self.aabb = torch.tensor([-1.0, -1.0, -1.0, 1.0, 1.0, 1.0], device=self.device)        # nerf.py:35
        self.base_exp_dir, self.writer = base_exp_dir, writer
        self.train_conf = DEFAULT_TRAIN_CONF if train_conf is None else Conf.wrap(train_conf)
        self.nerf = NGPNeRF(aabb=self.aabb).to(self.device)
        if estimator_type == "occ":                                    # nerf.py:68
            from .shims.nerfacc.estimators.occ_grid import OccGridEstimator
            self.estimator = OccGridEstimator(roi_aabb=self.aabb, resolution=occ_resolution, levels=1).to(self.device)
        else:
            self.estimator = FixedSampleEstimator(n_samples, near, far)
        self.renderer = NeRFOCCRenderer(**(renderer_conf or {"max_radius": 2, "bg_color": "rand_noise"}))
        self.fused = FusedPanoRenderer(aabb=self.aabb.tolist(), near=near, far=far)
        self._fused_key = None
        # fused training step (one forward kernel + composite-backward kernel); False = the modular
        # path through the plugin functions, op for op like the reference
        self.fused_train = fused_train
        self.graph_train = graph_train and fused_train    # capture each phase's step into a CUDA graph (GraphedTrainStep)
        self.train_ctx = ops.FusedTrainContext(aabb=self.aabb.tolist(), n_samples=n_samples, near=near, far=far)
        self.global_iter_step_geo = self.global_iter_step_app = 0

    # ---- inference ---------------------------------------------------------------------------
    def _sync_fused(self):
        # (sharded data parallelism with the shadow all-gather moved to the START of the next step, GraphedTrainStep)
        join, pend = getattr(self, "_join_gather", None), getattr(self, "_pending_gather", None)
        if join is not None:                                # capture of a step: the side-stream all-gather joins here, before the pack
            join(); self._join_gather = None
        elif pend is not None and not torch.cuda.is_current_stream_capturing():
            pend.stage_gather(); self._pending_gather = None            # eager use between replays: complete the shadow first
            self._fused_key = None
        g, a = self.nerf.geo_mlp.params, self.nerf.app_mlp.params
        key = (g._version, a._version, g.data_ptr(), a.data_ptr())
        if key != self._fused_key:
            # the plugin modules keep version-tracked fp16 shadows (refreshed in place by the Adam kernel)
            self.fused.set_halves(self.nerf.geo_mlp._half(), self.nerf.app_mlp._half())
            self._fused_key = key

    def _sync_occupancy(self):
        """The estimator's current grid (a view: in-place updates are seen) as the fused renderer's occupancy grid."""
        est = self.estimator
        self.fused.set_occupancy(est.binaries[0], est._aabb_list(), near=0.0, far=1.5, step=self.OCC_STEP, early_stop_eps=1e-4)

    @torch.no_grad()
    def render(self, rays: Rays, query_keys=("rgb",), sampling_requires_grad=False):
        """`nerf.py:74-99`: eval-mode render of arbitrarily shaped rays -> {key: [..., C]}."""
        self._sync_fused()
        rays_o, rays_d = rays.collapse()
        pre_shape = list(rays_o.shape[:-1])
        image = rays_o.dim() == 3                      # [H, W, 3] image of rays: keep the shape as a locality hint
        rays_o_img, rays_d_img = rays_o.float(), rays_d.float()
        rays_o, rays_d = rays_o.reshape(-1, 3).float(), rays_d.reshape(-1, 3).float()
        if self.estimator_type == "occ":
            # nerf_renderer.py:145-197 in one launch: each ray walks the occupancy grid, evaluates both fields at the
            # intervals it emits and stops at nerfacc's 1e-4 transmittance cut (csrc/render.cu::render_occ_kernel)
            self._sync_occupancy()
            out = self.fused.render_rays_occ(rays_o_img if image else rays_o, rays_d_img if image else rays_d)
        else:
            out = self.fused.render_rays(rays_o_img if image else rays_o, rays_d_img if image else rays_d, self.estimator.n_samples)
        return {k: out[k].reshape(pre_shape + [-1]) for k in query_keys}

    @torch.no_grad()
    def render_pano(self, pose, height, width, row0=0, rows=None):
        """render_dense inner loop (`core_exp_runner.py:229-238`) with ray generation fused in."""
        self._sync_fused()
        if self.estimator_type == "occ":
            self._sync_occupancy()
            return self.fused.render_pano_occ(pose, height, width, row0=row0, rows=rows)
        return self.fused.render_pano(pose, height, width, self.estimator.n_samples, row0=row0, rows=rows)

    @torch.no_grad()
    def get_pano_visibility_mask(self, sup_pool, rays: Rays):
        """`nerf.py:320-358`: render the distance of ``rays`` [H,W,3], un-project, and ask every registered
        panorama whether it sees that surface point (1 visible, 0 invisible; ``SupInfoPool.pano_visibility_mask``)."""
        distance = self.render(rays, query_keys=["distance"])["distance"].squeeze()
        return sup_pool.pano_visibility_mask(rays, distance)

    def _render_once_fused(self, rays: Rays, geo_inference: bool, app_inference: bool):
        """Training-mode render as ONE forward kernel; gradients reach the network that is not in
        inference mode.  Same outputs as the modular path except the per-sample tensors: instead of
        `weights/t_starts/t_ends/ray_indices` it returns `dist_loss` (= flatten_eff_distloss)."""
        from . import _lib
        rays_o, rays_d = rays.collapse()
        R, dev = rays_o.shape[0], rays_o.device
        self._sync_fused()
        tc = self.train_ctx
        tc.packed, tc.geo_half, tc.app_half = self.fused.packed, self.fused.geo_half, self.fused.app_half
        jitter = torch.rand(R, device=dev) if self.nerf.training else torch.zeros(R, device=dev)
        if self.nerf.training and self.renderer.bg_color == "rand_noise":
            bg = torch.rand(R, 3, device=dev)
        else:
            bg = torch.full((R, 3), 1.0 if self.renderer.bg_color == "white" else 0.0, device=dev)
        noise = torch.cat([bg, torch.rand(R, 1, device=dev)], 1)
        phase = _lib.PERF_PHASE_APP if geo_inference else _lib.PERF_PHASE_GEO
        param = self.nerf.app_mlp.params if geo_inference else self.nerf.geo_mlp.params
        if self.estimator_type == "occ":
            # the sampler PeRF trains with (nerf_renderer.py:145-155): packed intervals, one offset per ray when training
            est = self.estimator
            static = getattr(self, "_occ_static", None)
            if static is not None and static.R == R:
                # capacity-sized buffers, sample count stays on the device: no host read, graph-capturable (GraphedTrainStep);
                # a batch without samples is a no-op step here instead of the reference's early return (nerf_renderer.py:156-162)
                ri, ts, te, offsets, n_dev = ops.occ_sample_static(est.binaries[0], est._aabb_list(), rays_o.float().contiguous(),
                                                                   rays_d.float().contiguous(), 0.0, 1.5, self.OCC_STEP,
                                                                   jitter if self.nerf.training else None, static)
                rgb, dist, op, dl = ops.fused_packed_train_step(param, rays_o.float(), rays_d.float(), offsets, ri, ts, te, noise, tc, phase, 1e-4, n_dev=n_dev)
                n_rays = (ri[(n_dev - 1).clamp(min=0)] + 1).float().reshape(())       # flatten_eff_distloss: ray_id.max() + 1
                return {"is_valid": True, "rgb": rgb, "distance": dist, "opacities": op, "dist_loss": _Lazy(lambda: dl.sum() / n_rays),
                        "dist_loss_rays": dl, "dist_loss_inv_n": 1.0 / n_rays}
            ri, ts, te = ops.occ_sample(est.binaries[0], est._aabb_list(), rays_o.float().contiguous(), rays_d.float().contiguous(),
                                        0.0, 1.5, self.OCC_STEP, jitter if self.nerf.training else None)
            if ri.numel() <= 0:                                              # nerf_renderer.py:156-162
                z = lambda c: torch.zeros(R, c, device=dev)
                return {"is_valid": False, "rgb": z(3), "distance": z(1), "opacities": z(1), "dist_loss": torch.zeros((), device=dev)}
            rgb, dist, op, dl = ops.fused_packed_train_step(param, rays_o.float(), rays_d.float(), ops.occ_sample.last_offsets, ri, ts, te,
                                                            noise, tc, phase, 1e-4)
            n_rays = (ri[-1] + 1).float()                                    # flatten_eff_distloss: ray_id.max() + 1
            return {"is_valid": True, "rgb": rgb, "distance": dist, "opacities": op, "dist_loss": _Lazy(lambda: dl.sum() / n_rays),
                    "dist_loss_rays": dl, "dist_loss_inv_n": 1.0 / n_rays, "n_samples": int(ri.numel())}
        rgb, dist, op, dl = ops.fused_train_step(param, rays_o, rays_d, jitter, noise, tc, phase)
        return {"is_valid": True, "rgb": rgb, "distance": dist, "opacities": op, "dist_loss": _Lazy(lambda: dl.sum() / R),
                "dist_loss_rays": dl, "dist_loss_inv_n": None}

    def render_once(self, rays: Rays, query_keys=("rgb",), sampling_requires_grad=False, geo_inference=False, app_inference=False):
        """`nerf.py:101-123` (differentiable path used by the train steps)."""
        rays_o, rays_d = rays.collapse()
        assert len(rays_o.shape) == 2
        if self.fused_train and self.nerf.training and (geo_inference != app_inference) and "weights" not in query_keys:
            res = self._render_once_fused(rays, geo_inference, app_inference)
            return {k: (res[k]() if isinstance(res[k], _Lazy) else res[k]) for k in list(query_keys) + ["is_valid"] if k in res}
        res = self.renderer.render(self.nerf, self.estimator, rays_o, rays_d, geo_inference=geo_inference, app_inference=app_inference)
        if (res is None) or (not res["is_valid"]):
            return res
        return {k: res[k] for k in list(query_keys) + ["is_valid"]}

    # ---- training ----------------------------------------------------------------------------
    def fit(self, sup_pool):
        self.train_one_episode(sup_pool, self.train_conf.raw_phase_iter_geo, self.train_conf.raw_phase_iter_app, "by_all_pixels")

    def train_one_episode(self, sup_pool, geo_res_iters, app_res_iters, pixel_sup_rand_mode="by_all_pixels"):
        """`nerf.py:137-184`: (occupancy grid from the supervision,) fresh density net, geo phase then app phase."""
        self.set_train()
        if self.estimator_type == "occ":
            self.build_occupancy(sup_pool)
        self.nerf.reset_geo()
        geo_optimizer = FusedAdam(self.nerf.geo_mlp.params, lr=self.train_conf.geo_optimizer.init_lr, module=self.nerf.geo_mlp)
        geo_step = GraphedTrainStep(self, "geo", sup_pool, geo_optimizer) if self.graph_train and geo_res_iters > 0 else None
        for iter_i in range(geo_res_iters):
            self.update_lr(geo_optimizer, self.train_conf.geo_optimizer, iter_i / geo_res_iters)
            # NB the reference divides by app_res_iters here (nerf.py:178); kept
            progress = iter_i / max(app_res_iters, 1)
            if geo_step is not None:
                geo_step(progress)
            else:
                self.train_one_step_geo(geo_optimizer, sup_pool, pixel_sup_rand_mode, progress=progress)
        if geo_step is not None:
            geo_step.finish()
        geo_optimizer.sync_master()
        app_optimizer = FusedAdam(self.nerf.app_mlp.params, lr=self.train_conf.app_optimizer.init_lr, module=self.nerf.app_mlp)
        app_step = GraphedTrainStep(self, "app", sup_pool, app_optimizer) if self.graph_train and app_res_iters > 0 else None
        for iter_i in range(app_res_iters):
            self.update_lr(app_optimizer, self.train_conf.app_optimizer, iter_i / app_res_iters)
            if app_step is not None:
                app_step(iter_i / app_res_iters)
            else:
                self.train_one_step_app(app_optimizer, sup_pool, pixel_sup_rand_mode, progress=iter_i / app_res_iters)
        if app_step is not None:
            app_step.finish()
        app_optimizer.sync_master()

    def build_occupancy(self, sup_pool, n_updates: int = 256):
        """`nerf.py:143-168`: a fresh estimator whose grid is the surface shell of the supervision (voxels within one cell of
        an un-projected RGB-D point, ``sup_pool.gen_occ_grid``), entered through 256 warm-up updates exactly as the reference
        does (each one: perf_occ_points -> the lookup below -> perf_occ_update)."""
        from .shims.nerfacc.estimators.occ_grid import OccGridEstimator
        occ_res = self.occ_resolution
        self.estimator = OccGridEstimator(roi_aabb=self.aabb, resolution=occ_res, levels=1).to(self.device)
        self.estimator.train()
        pre_grid, _ = sup_pool.gen_occ_grid(res=occ_res)

        def occ_eval_fn(x):
            x = ((x.clip(-0.999, 0.999) * .5 + .5) * occ_res).to(torch.int64)
            return pre_grid[x[..., 0] * occ_res * occ_res + x[..., 1] * occ_res + x[..., 2]].float()
        for i in range(n_updates):
            self.estimator.update_every_n_steps(step=i, occ_eval_fn=occ_eval_fn, occ_thre=1e-2, ema_decay=0.1, warmup_steps=256, n=1)

    def _local_batch(self):
        return max(1, int(self.train_conf.pixel_loss_batch_size) // parallel.world_size())

    def _log(self, tag, value, step):
        if self.writer is not None:
            self.writer.add_scalar(tag, value, step)

    def train_one_step_geo(self, optimizer, sup_pool, pixel_sup_rand_mode="by_all_pixels", progress=0.0):
        """`nerf.py:186-257`: depth smooth-L1 + ramped distortion loss; colour under no_grad."""
        conf, eps, loss = self.train_conf, 1e-7, 0.
        optimizer.zero_grad()
        rays, gt_colors, gt_depths, _ = sup_pool.rand_ray_color_data(self._local_batch(), rand_mode=pixel_sup_rand_mode)
        one_kernel_loss = self.fused_train and conf.density_loss_weight <= eps
        keys = (["rgb", "distance", "dist_loss_rays", "dist_loss_inv_n"] if one_kernel_loss else ["rgb", "distance", "dist_loss"]) if self.fused_train \
            else ["rgb", "distance", "weights", "t_starts", "t_ends", "trans", "ray_indices"]
        res = self.render_once(rays, keys, app_inference=True)
        if (res is None) or (not res["is_valid"]):
            optimizer.step(valid=False)            # no samples on this rank (nerf.py:204-206): still join the exchange
            self.global_iter_step_geo += 1
            return None
        if one_kernel_loss:
            # nerf.py:208-238 as one launch (+ its gradients): depth smooth-L1 and the ramped distortion loss
            use_dl = conf.distortion_loss_weight > eps
            ratio = progress if torch.is_tensor(progress) else torch.tensor([float(np.min([progress * 2., 1]))], device=self.device)
            loss, depth_loss, dist_loss = ops.fused_loss(res["distance"], gt_depths, 1e-2,
                                                         conf.depth_loss_weight if conf.depth_loss_weight > eps else 0.0,
                                                         dl=res["dist_loss_rays"] if use_dl else None, ratio=ratio if use_dl else None,
                                                         inv_n=res["dist_loss_inv_n"] if use_dl else None,
                                                         w_dl=conf.distortion_loss_weight if use_dl else 0.0)
            self._log("nerf_loss/depth_loss", depth_loss, self.global_iter_step_geo)
            self._log("nerf_loss/dist_loss", dist_loss, self.global_iter_step_geo)
            (loss * self.LOSS_SCALE).backward()
            optimizer.step()
            self.global_iter_step_geo += 1
            return loss.detach()
        if conf.depth_loss_weight > eps:
            depth_loss = F.smooth_l1_loss(res["distance"], gt_depths, beta=1e-2, reduction="mean")
            loss = loss + depth_loss * conf.depth_loss_weight
            self._log("nerf_loss/depth_loss", depth_loss, self.global_iter_step_geo)
        if conf.distortion_loss_weight > eps:
            if self.fused_train:
                dist_loss = res["dist_loss"]
            else:
                mid_dis = (res["t_ends"] + res["t_starts"]) * .5
                sec_lens = res["t_ends"] - res["t_starts"]
                dist_loss = flatten_eff_distloss(res["weights"], mid_dis, sec_lens, res["ray_indices"])
            ratio = progress if torch.is_tensor(progress) else float(np.min([progress * 2., 1]))   # tensor: pre-computed ramp (graph mode)
            loss = loss + dist_loss * conf.distortion_loss_weight * ratio
            self._log("nerf_loss/dist_loss", dist_loss, self.global_iter_step_geo)
        if conf.density_loss_weight > eps:
            rand_pts = (torch.rand(8192, 3, device=self.device) * 2. - 1.) * 0.99
            loss = loss + self.nerf.query_density(rand_pts).mean() * conf.density_loss_weight
        (loss * self.LOSS_SCALE).backward()
        optimizer.step()
        self.global_iter_step_geo += 1
        return loss.detach()

    def train_one_step_app(self, optimizer, sup_pool, pixel_sup_rand_mode="by_all_pixels", progress=0.0):
        """`nerf.py:259-297`: colour smooth-L1; density under no_grad."""
        conf, eps, loss = self.train_conf, 1e-7, 0.
        optimizer.zero_grad()
        rays, gt_colors, _, _ = sup_pool.rand_ray_color_data(self._local_batch(), rand_mode=pixel_sup_rand_mode)
        keys = ["rgb", "distance"] if self.fused_train else ["rgb", "distance", "weights", "t_starts", "t_ends", "trans", "ray_indices"]
        res = self.render_once(rays, keys, geo_inference=True)
        if (res is None) or (not res["is_valid"]):
            optimizer.step(valid=False)            # no samples on this rank (nerf.py:204-206): still join the exchange
            self.global_iter_step_app += 1
            return None
        if self.fused_train and conf.color_loss_weight > eps:          # nerf.py:281-287 as one launch (+ its gradient)
            loss, color_loss, _ = ops.fused_loss(res["rgb"], gt_colors, 5e-2, conf.color_loss_weight)
            self._log("nerf_loss/color_loss", color_loss, self.global_iter_step_app)
        elif conf.color_loss_weight > eps:
            color_loss = F.smooth_l1_loss(res["rgb"], gt_colors, beta=5e-2, reduction="mean")
            loss = loss + color_loss * conf.color_loss_weight
            self._log("nerf_loss/color_loss", color_loss, self.global_iter_step_app)
        (loss * self.LOSS_SCALE).backward()
        optimizer.step()
        self.global_iter_step_app += 1
        return loss.detach()

    def update_lr(self, optimizer, optim_conf, progress):
        """`nerf.py:300-311`: linear warm-up to peak_lr at peak_at, cosine to lr_alpha * peak_lr."""
        if progress < optim_conf.peak_at:
            local = progress / optim_conf.peak_at
            lr = optim_conf.peak_lr * local + optim_conf.init_lr * (1. - local)
        else:
            local = (progress - optim_conf.peak_at) / (1. - optim_conf.peak_at)
            lr = optim_conf.peak_lr * ((np.cos(local * np.pi) + 1.) * .5 * (1. - optim_conf.lr_alpha) + optim_conf.lr_alpha)
        for p in optimizer.param_groups:
            p["lr"] = float(lr)

    def to_bounded_rays(self, rays: Rays) -> BoundedRays:
        """`nerf.py:313-319` (near 1e-2 / far 1 tensors; like the reference's OCC renderer, the
        native renderer takes its range from the estimator, not from these)."""
        n = len(rays.o)
        return BoundedRays(rays.o, rays.d, 1e-2 * torch.ones(n, 1, device=rays.o.device), torch.ones(n, 1, device=rays.o.device))

    # ---- state -------------------------------------------------------------------------------
    def state_dict(self):
        """`nerf.py:374-380` keys."""
        return {"render": self.renderer.state_dict(), "nerf": self.nerf.state_dict(), "estimator": self.estimator.state_dict()}

    def load_state_dict(self, state_dict):
        """`nerf.py:368-372`.  A checkpoint written with another sampler (e.g. the reference's occupancy grid loaded
        into a fixed-S scene) restores the field and skips the estimator buffers that do not apply."""
        if "render" in state_dict:
            self.renderer.load_state_dict(state_dict["render"])
        self.nerf.load_state_dict(state_dict["nerf"])
        est = state_dict.get("estimator", {})
        if est and set(est) == set(self.estimator.state_dict()):
            self.estimator.load_state_dict(est)
        self._fused_key = None

    def set_train(self):
        self.nerf.train(); self.estimator.train(); self.renderer.train()

    def set_eval(self):
        self.nerf.eval(); self.estimator.eval(); self.renderer.eval()


class GraphedTrainStep:
    """One optimisation step (batch draw -> fused forward -> losses -> backward -> all-reduce -> Adam)
    captured ONCE into a CUDA graph and replayed: ~50 launches + Python bookkeeping become a single
    graph launch.  The learning rate / Adam bias corrections and the distortion-loss ramp are device
    scalars refreshed before every replay, so the reference's schedule (`nerf.py:173-184,300-311`)
    is followed exactly.  Usage::

        step = GraphedTrainStep(scene, "geo", sup_pool, optimizer)
        for i in range(iters):
            scene.update_lr(optimizer, conf.geo_optimizer, i / iters)
            loss = step(progress=i / app_iters)
    """

    def __init__(self, scene: NeRFScene, phase: str, sup_pool: RaySupervision, optimizer: FusedAdam, warmup: int = 3, split: bool = False,
                 occ_capacity: int = 0):
        """``split=True``: four graphs instead of one -- [batch draw + forward + losses + backward], [gradient exchange],
        [Adam], [shadow all-gather] -- replayed back to back with CUDA events in between (``self.stage_ms`` after each
        call): the timeline of a step (VERDICT r1 next #2).  Slightly slower than the single graph (three more launches)."""
        assert phase in ("geo", "app") and scene.fused_train
        self.scene, self.phase, self.pool, self.opt, self.split = scene, phase, sup_pool, optimizer, split
        dev = scene.device
        if scene.estimator_type == "occ":
            # Occupancy sampler: the sample count of a batch is data dependent.  Probe it once (eager, one host read), give the
            # step capacity-sized buffers with head-room and keep the live count on the device from then on
            # (ops.occ_sample_static): the replayed launch sequence does not depend on the count.  `occ_overflow()` reports
            # whether any replayed batch asked for more than the capacity (its last samples were then dropped).
            R = scene._local_batch()
            rays, _, _, _ = sup_pool.rand_ray_color_data(R)
            ro, rd = rays.collapse()
            est = scene.estimator
            probe = ops.occ_sample(est.binaries[0], est._aabb_list(), ro.float().contiguous(), rd.float().contiguous(), 0.0, 1.5,
                                   scene.OCC_STEP, torch.rand(R, device=dev))[0].numel()
            cap = occ_capacity or int(max(probe * 1.5, R * 16)) // 128 * 128 + 128
            scene._occ_static = ops.OccStaticBuffers(R, cap, dev)
        self.ratio = torch.zeros(1, device=dev)
        self.net = scene.nerf.geo_mlp if phase == "geo" else scene.nerf.app_mlp
        sup_pool.use_default_generator = True                 # graph-safe RNG; decorrelate the ranks' batches
        torch.cuda.manual_seed(int(sup_pool.generator.initial_seed()) + 7919 * parallel.rank())
        optimizer.enable_graph_mode()
        scene.set_train()
        # warm-up and capture run REAL optimiser steps: snapshot the parameters and put them back afterwards, so the
        # graphed fit starts from the same weights as the eager one for any init_lr (ADVICE r1)
        p0 = self.net.params.data.clone()
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):                         # eager warm-up on a side stream (NCCL, allocator)
            for _ in range(warmup):
                self._prepare(0.5)
                self._body()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self._prepare(0.5)
        # Sharded DP: the all-gather of the fp16 shadow depends only on the PREVIOUS step's Adam, the batch draw on nothing:
        # capture the gather at the START of the step on a side stream, concurrent with the draw, joined before the table
        # pack (hides ~60 us of NCCL at 8 GPUs behind ~50 us of small kernels).  The shard a step's Adam writes is then
        # gathered by the next replay -- or by finish() / the next eager _sync_fused().  PERF_B200_AG_OVERLAP=0: off.
        import os as _os
        self.overlap_gather = (not split) and optimizer.sharded and _os.environ.get("PERF_B200_AG_OVERLAP", "1") != "0"
        if not split:
            self.graph = torch.cuda.CUDAGraph()
            side_ag = torch.cuda.Stream(device=dev) if self.overlap_gather else None
            with torch.cuda.graph(self.graph):
                if self.overlap_gather:
                    main = torch.cuda.current_stream(dev)
                    side_ag.wait_stream(main)
                    with torch.cuda.stream(side_ag):
                        optimizer._hbuf = self.net._half() if optimizer._half_pad is None else optimizer._half_pad
                        optimizer.stage_gather()
                    scene._join_gather = lambda: main.wait_stream(side_ag)
                    scene._pending_gather = None
                    optimizer.skip_gather = True
                self.loss = self._body()
                if self.overlap_gather and scene._join_gather is not None:       # body never reached _sync_fused: join here
                    scene._join_gather(); scene._join_gather = None
            optimizer.skip_gather = False                      # (capture records, it does not execute: nothing to complete here)
            self.graphs = [self.graph]
        else:
            pool = torch.cuda.graph_pool_handle()
            self.graphs = [torch.cuda.CUDAGraph() for _ in range(4)]
            optimizer.deferred = True
            with torch.cuda.graph(self.graphs[0], pool=pool):
                self.loss = self._body()
            optimizer.deferred = False
            with torch.cuda.graph(self.graphs[1], pool=pool):
                optimizer.stage_exchange(getattr(optimizer, "_valid", True))
            with torch.cuda.graph(self.graphs[2], pool=pool):
                optimizer.stage_adam()
            with torch.cuda.graph(self.graphs[3], pool=pool):
                optimizer.stage_gather()
            self.events = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
            self.stage_ms = None
        optimizer.step_count = 0                               # warm-up / capture steps do not count
        optimizer.exp_avg.zero_(); optimizer.exp_avg_sq.zero_()
        self.net.params.data.copy_(p0)
        optimizer.master_stale = False
        ops.params_to_half(self.net.params.detach(), out=self.net._half())     # same buffer the captured kernels read
        torch._C._increment_version([self.net.params])
        self.net._half_key = (self.net.params._version, self.net.params.data_ptr())
        scene._fused_key = None

    def _prepare(self, progress: float):
        ops.set_scalars(self.ratio, [min(progress * 2.0, 1.0)])
        self.opt.push_hyper()

    def _body(self):
        sc = self.scene
        sc._fused_key = None                                   # always re-pack inside the step (captured)
        if self.phase == "geo":
            return sc.train_one_step_geo(self.opt, self.pool, progress=self.ratio[0])
        return sc.train_one_step_app(self.opt, self.pool, progress=self.ratio[0])

    STAGES = ("draw+forward+loss+backward", "gradient exchange", "adam", "shadow all-gather")

    def __call__(self, progress: float = 0.0):
        self._prepare(progress)
        if not self.split:
            self.graph.replay()
        else:
            self.events[0].record()
            for g, e in zip(self.graphs, self.events[1:]):
                g.replay(); e.record()
            self.opt.master_stale = self.opt.sharded
        # the replayed Adam kernel wrote params + fp16 shadow: tell the version-keyed caches
        p = self.net.params
        torch._C._increment_version([p])
        self.net._half_key = (p._version, p.data_ptr())
        self.scene._fused_key = None
        self.opt.master_stale = self.opt.sharded
        if self.overlap_gather:
            self.scene._pending_gather = self.opt             # this step's shard is gathered by the next replay / eager use
        return self.loss

    def occ_overflow(self) -> int:
        """(occupancy scenes) samples the largest replayed batch asked for beyond the capacity (0 = every batch fitted)."""
        st = getattr(self.scene, "_occ_static", None)
        return 0 if st is None else max(0, int(st.overflowed) - st.capacity)

    def finish(self):
        """Complete the state after the last replay: gather the last step's shadow shard (overlap mode) and the fp32 master."""
        if self.overlap_gather and getattr(self.scene, "_pending_gather", None) is self.opt:
            self.opt.stage_gather(); self.scene._pending_gather = None
            self.scene._fused_key = None
        self.opt.sync_master()

    def last_stage_ms(self):
        """(split mode) device time of the four stages of the last call, after a synchronize."""
        return [a.elapsed_time(b) for a, b in zip(self.events[:-1], self.events[1:])]
