"""Eval render with the occupancy-grid sampler: the packed chain against the one-launch kernel.

    python tools/bench_render_occ.py [--steps 20 --warmup 3 --geo-iters 3000 --app-iters 1500]

Fits the synthetic box room with the occupancy sampler (as `examples/fit_and_render.py --sampler occ`: a random field has
no surface, so its rays would not stop the way they do on a real scene), then renders three workloads with PeRF's lattice
(near 0, far 1.5, step 5e-4, transmittance cut 1e-4) two ways:

  (a) packed: ops.raygen_pano -> ops.occ_sample (count kernel, cumsum, host read of the total, write kernel) ->
      ops.render_occ (perf_fields_packed at every emitted interval + perf_composite_packed_fwd); the grid render of
      NeRFScene.render before the one-launch kernel
  (b) one launch: ops.render_pano_occ / ops.render_rays_occ (csrc/render.cu::render_occ_kernel)

Workloads: a 512 x 1024 panorama (the reference's render_dense size), a 1024 x 2048 panorama, and one 32768-ray batch of
explicit rays (the reference's chunk: 32 consecutive rows of a 512 x 1024 panorama).  Time per frame from CUDA events
around each step, the L2 overwritten (256 MiB) between timed steps, as bench.py does; (a) includes its host read.  Prints
one JSON line with the card's name and power limit, read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from perf_b200 import ops, synthetic
from perf_b200.scene import NeRFScene, RaySupervision

NEAR, FAR, EPS = 0.0, 1.5, 1e-4


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader,nounits"], capture_output=True, text=True)
    name, power, clock = ([v.strip() for v in q.stdout.strip().split(",")] + ["?", "?", "?"])[:3]
    return {"name": torch.cuda.get_device_name(), "nvidia_smi_name": name, "power_limit_w": power, "max_sm_clock_mhz": clock}


def timed(fn, steps, warmup, flush):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for e0, e1 in evs:
        flush.fill_(1)
        e0.record()
        fn()
        e1.record()
    torch.cuda.synchronize()
    ms = sorted(e0.elapsed_time(e1) for e0, e1 in evs)
    return {"mean_ms": sum(ms) / len(ms), "median_ms": ms[len(ms) // 2], "min_ms": ms[0], "max_ms": ms[-1]}


def peak_bytes(fn):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    out = fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base, out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--geo-iters", type=int, default=3000)
    ap.add_argument("--app-iters", type=int, default=1500)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_render_occ needs a GPU")
    dev = "cuda"
    h, w = 512, 1024
    rgb, dist = synthetic.smooth_rgb(h, w, seed=0, device=dev), synthetic.box_room_distance(h, w, device=dev)
    conf = dict(NeRFScene(n_samples=8).train_conf)
    conf.update(raw_phase_iter_geo=args.geo_iters, raw_phase_iter_app=args.app_iters)
    torch.manual_seed(0)
    sc = NeRFScene(train_conf=conf, estimator_type="occ", graph_train=True)
    t0 = time.perf_counter()
    sc.fit(RaySupervision.from_panorama(torch.eye(4), rgb, dist, seed=0))
    torch.cuda.synchronize()
    t_fit = time.perf_counter() - t0
    sc.set_eval()
    sc._sync_fused()
    r, est = sc.fused, sc.estimator
    bins, roi = est.binaries[0], est._aabb_list()
    step = sc.OCC_STEP
    pose = torch.eye(4); pose[:3, 3] = torch.tensor([0.15, -0.1, 0.05])             # a novel view inside the room
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def packed(o, d):
        o, d = o.reshape(-1, 3).contiguous(), d.reshape(-1, 3).contiguous()
        ri, ts, te = ops.occ_sample(bins, roi, o, d, NEAR, FAR, step, None)
        out = ops.render_occ(r.packed, r.geo_half, r.app_half, o, d, ops.occ_sample.last_offsets, ri, ts, te, EPS, r.aabb, r.grid)
        return out, ri.numel()

    o_half, d_half = ops.raygen_pano(pose, h, w)
    chunk = (o_half[240:272].reshape(-1, 3).contiguous(), d_half[240:272].reshape(-1, 3).contiguous())      # 32768 rays
    workloads = {
        "pano_512x1024": (lambda: packed(*ops.raygen_pano(pose, 512, 1024)),
                          lambda: ops.render_pano_occ(r.packed, r.geo_half, r.app_half, pose, 512, 1024, bins, roi, NEAR, FAR, step, EPS,
                                                      aabb=r.aabb, grid=r.grid, want_n_samples=True), 512 * 1024),
        "pano_1024x2048": (lambda: packed(*ops.raygen_pano(pose, 1024, 2048)),
                           lambda: ops.render_pano_occ(r.packed, r.geo_half, r.app_half, pose, 1024, 2048, bins, roi, NEAR, FAR, step, EPS,
                                                       aabb=r.aabb, grid=r.grid, want_n_samples=True), 1024 * 2048),
        "rays_32768": (lambda: packed(*chunk),
                       lambda: ops.render_rays_occ(r.packed, r.geo_half, r.app_half, chunk[0], chunk[1], bins, roi, NEAR, FAR, step, EPS,
                                                   aabb=r.aabb, grid=r.grid, want_n_samples=True), 32768),
    }
    res = {}
    for name, (fa, fb, R) in workloads.items():
        fa(); fb()                                                                  # first calls: module load, kernel attributes
        mem_a, (out_a, n_emitted) = peak_bytes(fa)
        mem_b, out_b = peak_bytes(fb)
        n_comp = int(out_b[3].long().sum())
        diff = {k: float((a.reshape(-1) - b.reshape(-1)).abs().max()) for k, a, b in zip(("rgb", "distance", "opacity"), out_a, out_b[:3])}
        ta = timed(fa, args.steps, args.warmup, flush)
        tb = timed(fb, args.steps, args.warmup, flush)
        res[name] = {
            "rays": R,
            "a_packed": {**ta, "intervals_emitted_per_ray": n_emitted / R, "intervals_evaluated_per_ray": n_emitted / R,
                         "evaluated_msamples_per_s": n_emitted / (ta["mean_ms"] * 1e3), "peak_alloc_mib": mem_a / 2 ** 20},
            "b_one_launch": {**tb, "intervals_composited_per_ray": n_comp / R, "composited_msamples_per_s": n_comp / (tb["mean_ms"] * 1e3),
                             "peak_alloc_mib": mem_b / 2 ** 20},
            "speedup_a_over_b": ta["mean_ms"] / tb["mean_ms"],
            "max_abs_diff_a_b": diff,
        }
    line = {"metric": "occ_eval_render", "gpu": gpu_info(), "torch": torch.__version__,
            "fit": {"sampler": "occ", "geo_iters": args.geo_iters, "app_iters": args.app_iters, "seconds": t_fit,
                    "occupied_cells": float(bins.float().mean())},
            "lattice": {"near": NEAR, "far": FAR, "step": step, "early_stop_eps": EPS}, "pose_t": pose[:3, 3].tolist(),
            "timing": f"CUDA events per step, mean of {args.steps} after {args.warmup} warm-up, L2 overwritten (256 MiB) before each step",
            "workloads": res}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
