"""``render_dense`` entry point on the fused renderer: the inner loop of
``CoreRunner.render_dense`` (`/root/reference/core_exp_runner.py:223-246`) for a PeRF checkpoint and
the reference's unchanged Hydra YAML, with the panorama row-tiled over the ranks of a torchrun job.

    python -m perf_b200.render_dense --config-dir /path/to/PeRF/configs --ckpt exp/checkpoints/ckpt.pth \\
        --poses poses.npy --out out_dir [--height 512 --width 1024] [--sampler fixed --n-samples 128 | --sampler occ] [key=value ...]

``--poses``: [n,4,4] camera-to-world matrices (the reference builds them with its
DenseTravelPoseSampler from the dataset's distance map, which is outside the hot path); without it
a small circle of 8 poses around the origin is rendered.  Frames are written as PNG by rank 0.

``--sampler fixed`` (the default) renders ``--n-samples`` evenly spaced samples on [1e-2, 1].  ``--sampler occ`` renders
with the occupancy grid the checkpoint stores under ``scene.estimator``, as PeRF itself does (``estimator_type: occ``,
``configs/nerf.yaml:25``; intervals of 5e-4 on [0, 1.5] inside occupied cells, cut at transmittance 1e-4).
"""
from __future__ import annotations

import argparse
import os

import numpy as np
import torch

from . import parallel
from .config import load_config
from .renderer import FusedPanoRenderer


def default_poses(n: int = 8, radius: float = 0.1) -> np.ndarray:
    poses = np.tile(np.eye(4, dtype=np.float32), (n, 1, 1))
    ang = np.linspace(0, 2 * np.pi, n, endpoint=False)
    poses[:, 0, 3], poses[:, 1, 3] = radius * np.cos(ang), radius * np.sin(ang)
    return poses


def render_frames(renderer: FusedPanoRenderer, poses, height: int, width: int, n_samples: int, sampler: str = "fixed"):
    """Yields (rgb [H,W,3], distance [H,W,1]) per pose; every rank renders its row tile and rank 0
    receives the full frame (one gather per frame, off the kernel's critical path).  ``sampler="occ"``: the
    renderer's occupancy grid (``n_samples`` does not apply)."""
    rank, world = parallel.rank(), parallel.world_size()
    sl = parallel.shard_slice(height, rank, world)
    for pose in poses:
        pose = torch.as_tensor(pose, dtype=torch.float32).clone()
        pose[:3, :3] = torch.eye(3)                                  # core_exp_runner.py:232
        if sampler == "occ":
            out = renderer.render_pano_occ(pose, height, width, row0=sl.start, rows=sl.stop - sl.start)
        else:
            out = renderer.render_pano(pose, height, width, n_samples, row0=sl.start, rows=sl.stop - sl.start)
        tile = parallel.gather_row_tiles(torch.cat([out["rgb"], out["distance"]], -1), height)
        if tile is None:
            continue
        yield tile[..., :3], tile[..., 3:]


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--config-dir", default=None)
    ap.add_argument("--config-name", default="nerf")
    ap.add_argument("--ckpt", required=True)
    ap.add_argument("--poses", default=None)
    ap.add_argument("--out", default="dense_images_new_pano")
    ap.add_argument("--height", type=int, default=512)
    ap.add_argument("--width", type=int, default=1024)
    ap.add_argument("--sampler", choices=("fixed", "occ"), default="fixed",
                    help="fixed: --n-samples evenly spaced samples; occ: the checkpoint's occupancy grid (scene.estimator)")
    ap.add_argument("--n-samples", type=int, default=128, help="samples per ray of --sampler fixed")
    ap.add_argument("overrides", nargs="*")
    args = ap.parse_args(argv)
    rank, world, local = parallel.init()
    torch.cuda.set_device(local)
    if args.config_dir:
        conf = load_config(args.config_dir, args.config_name, args.overrides)
        assert conf.scene_class_name == "NeRFScene", conf.scene_class_name
    ckpt = torch.load(args.ckpt, map_location="cpu")
    est = None
    if args.sampler == "occ":
        est = ckpt["scene"].get("estimator") or {}
        if "binaries" not in est or "aabbs" not in est:
            raise SystemExit(f"render_dense --sampler occ: {args.ckpt} has no occupancy grid (scene.estimator.binaries / aabbs); "
                             "it was not trained with estimator_type=occ -- render it with --sampler fixed")
    renderer = FusedPanoRenderer.from_state_dict(ckpt["scene"]["nerf"], est, device=torch.device("cuda", local))
    poses = np.load(args.poses) if args.poses else default_poses()
    if rank == 0:
        os.makedirs(args.out, exist_ok=True)
    import cv2
    for i, (rgb, dist) in enumerate(render_frames(renderer, poses, args.height, args.width, args.n_samples, args.sampler)):
        img = (rgb.clamp(0, 1) * 255).byte().cpu().numpy()[..., ::-1]
        cv2.imwrite(os.path.join(args.out, f"image_{i}.png"), img)
        inv = 1.0 / dist.clamp(min=1e-6)
        inv = (inv / inv.max() * 255).byte().cpu().numpy()
        cv2.imwrite(os.path.join(args.out, f"distance_{i}.png"), inv)
    if world > 1:
        import torch.distributed as dist_
        dist_.barrier()
        dist_.destroy_process_group()


if __name__ == "__main__":
    main()
