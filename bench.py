#!/usr/bin/env python
"""bench.py -- the driver's benchmark contract for the PeRF per-ray hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one synthetic batch: rendering ONE 1024x2048
equirectangular panorama at 128 samples/ray (BASELINE.json configs[1]/[2] field: L=16 hash
grid x2, 64-wide density/colour MLPs) = 268 435 456 samples.  With N GPUs the panorama is
row-tiled across the ranks (SURVEY.md section 8e, `render_dense`): total work is fixed ->
"scaling": "strong"; no data-path collective.  `value` = samples of the whole panorama / the
slowest rank's device time.

JSON keys beyond the base contract:
  roofline      dominant kernel (render_march_kernel): ALGORITHMIC bytes = 1024 B/sample (16 levels x 8
                corners x 2 features x 2 B x 2 fields, SURVEY.md section 8d) / CUDA-event time, against the
                measured HBM copy bandwidth in MEASURED_PEAKS.json.
  cpu_baseline  the oracle's plain-C / OpenMP port (oracle/cpath.c) on all host threads on a bounded
                sample of the same rays; the PyTorch port (oracle/render.py) is reported beside it.
  e2e           same metric through the public API with a host pose in and host images out.

--dump-outputs DIR writes what the last timed step rendered -- the whole panorama as a caller of
render_pano receives it -- to DIR/rgb.npy [H,W,3], DIR/distance.npy [H,W,1] and DIR/opacities.npy
[H,W,1], float32 (42 MB in all).  The field and the pose are seeded, so two builds run with the same
arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True                    # the benchmark leaves the source tree as it found it

H, W, S = 1024, 2048, 128
ALG_BYTES_PER_SAMPLE = 16 * 8 * 2 * 2 * 2        # levels x corners x features x sizeof(fp16) x fields
SEED = 0


def workload_config(n_gpus):
    return {"workload": f"render_dense tile: {H}x{W} equirect panorama, {S} samples/ray, L=16 T=2^18 F=2 hash grid x2 "
                        f"(density 32-64-1, colour 32-64-64-3), fixed-S sampler",
            "H": H, "W": W, "samples_per_ray": S, "rays": H * W, "samples_per_step": H * W * S,
            "parallelism": f"rows tiled over {n_gpus} GPU(s), no collective",
            "l2": "flushed between timed steps (256 MiB write); the packed gather table (37.8 MB) is re-fetched every step",
            # the numerics contract both arms compute in (the CPU port emulates the fp16 roundings; DESIGN.md section 4)
            "precision": "fp16 tables/operands (tcnn semantics), fp32 MLP accumulate, fp32 composite"}


def make_field(device):
    """Seeded random-init field of the reference architecture (there are no checkpoints)."""
    import torch
    from perf_b200.config import APP_MLP, GEO_MLP, PERF_GRID
    g = torch.Generator().manual_seed(SEED)
    n_e = PERF_GRID.n_entries

    def net(mlp):
        w = (torch.rand(mlp.n_params, generator=g) * 2 - 1) * 0.3
        t = (torch.rand(2 * n_e, generator=g) * 2 - 1) * 0.5
        return torch.cat([w, t])
    return net(GEO_MLP).to(device), net(APP_MLP).to(device)


def bench_pose():
    import torch
    pose = torch.eye(4)
    pose[:3, 3] = torch.tensor([0.05, -0.03, 0.02])
    return pose


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()

    def run(self):
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop_evt.wait(0.1)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=6)
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        smax = max((float(r[1]) for r in self.rows if r and r[1].replace(".", "").isdigit()), default=None)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "samples": len(sm), "reasons": sorted(reasons)}


def measured_peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------------
def cpu_oracle_sample(n_rays, threads=None):
    """Time the oracle (the reference's pure-PyTorch CPU field restatement + reference glue) on the
    first `n_rays` rays of the benchmark panorama.  Returns (Msamples/s, seconds, cores)."""
    import torch
    import oracle
    torch.set_num_threads(threads or min(16, os.cpu_count() or 1))
    g = torch.Generator().manual_seed(SEED)
    n_e = oracle.hashgrid.n_table_entries(oracle.field.PERF_GRID)

    def net(mlp):
        w = (torch.rand(oracle.mlp.flat_param_count(mlp), generator=g) * 2 - 1) * 0.3
        t = (torch.rand(2 * n_e, generator=g) * 2 - 1) * 0.5
        return torch.cat([w, t])
    field = oracle.Field(net(oracle.field.GEO_MLP), net(oracle.field.APP_MLP))
    o, d = oracle.gen_pano_rays(bench_pose(), H, W)
    # rays from the middle rows (the poles are degenerate)
    rows_needed = (n_rays + W - 1) // W
    o, d = o[H // 2:H // 2 + rows_needed].reshape(-1, 3)[:n_rays], d[H // 2:H // 2 + rows_needed].reshape(-1, 3)[:n_rays]
    n_rays = o.shape[0]
    t0 = time.perf_counter()
    with torch.no_grad():
        out = oracle.render_rays(field, o, d, S, mixed=True, accum=torch.float32)
    dt = time.perf_counter() - t0
    cpu_oracle_sample.last = {"rays_o": o, "rays_d": d, "rgb": out["rgb"], "distance": out["distance"]}
    return n_rays * S / dt / 1e6, dt, torch.get_num_threads()


_C_PORT = {}


def cpu_c_port_sample(n_rays):
    """The plain-C / OpenMP restatement (oracle/cpath.c) on ALL host threads visible to the process, on `n_rays`
    rays of the benchmark panorama (middle rows).  Returns (Msamples/s, seconds, threads)."""
    import torch
    import oracle
    from oracle import cpath
    if "field" not in _C_PORT:
        g = torch.Generator().manual_seed(SEED)
        n_e = oracle.hashgrid.n_table_entries(oracle.field.PERF_GRID)

        def net(mlp):
            w = (torch.rand(oracle.mlp.flat_param_count(mlp), generator=g) * 2 - 1) * 0.3
            t = (torch.rand(2 * n_e, generator=g) * 2 - 1) * 0.5
            return torch.cat([w, t])
        _C_PORT["field"] = oracle.Field(net(oracle.field.GEO_MLP), net(oracle.field.APP_MLP))
        _C_PORT["rays"] = oracle.gen_pano_rays(bench_pose(), H, W)
    field, (o, d) = _C_PORT["field"], _C_PORT["rays"]
    rows_needed = (n_rays + W - 1) // W
    r0 = (H - rows_needed) // 2
    o, d = o[r0:r0 + rows_needed].reshape(-1, 3)[:n_rays], d[r0:r0 + rows_needed].reshape(-1, 3)[:n_rays]
    if "threads" not in _C_PORT:
        # ONE stated thread count: every CPU visible to the process (explicit: torchrun exports OMP_NUM_THREADS=1).
        # Round 1 picked the fastest of {all, 1/2, 1/4, 1/8} on a short probe; on the shared GPU hosts that pick --
        # and with it the baseline -- swung 4x between runs (VERDICT r1 weak #6).
        _C_PORT["threads"] = len(os.sched_getaffinity(0))
        cpath.render_rays(field, o[:256], d[:256], S, n_threads=_C_PORT["threads"])       # build + warm up
    n_thr = _C_PORT["threads"]
    t0 = time.perf_counter()
    cpath.render_rays(field, o, d, S, n_threads=n_thr)
    dt = time.perf_counter() - t0
    return o.shape[0] * S / dt / 1e6, dt, n_thr


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path = the oracle port (the
    reference's third-party CUDA deps cannot be installed here and have no CPU path), host cores,
    bounded sample per step."""
    if rank != 0:
        return
    n_rays, sample_fn, which = 65536, cpu_c_port_sample, "oracle/cpath.c, OpenMP"    # 8.4 M samples per step, host threads
    try:
        cpu_c_port_sample(256)
    except Exception as e:                             # no gcc / OpenMP on this host: the PyTorch port, smaller sample
        print(f"C port unavailable ({type(e).__name__}: {e}); timing the PyTorch port", file=sys.stderr)
        n_rays, sample_fn, which = 4096, cpu_oracle_sample, "oracle/render.py, PyTorch"
    for _ in range(args.warmup):
        sample_fn(n_rays)
    ts = []
    cores = 1
    for _ in range(args.steps):
        v, dt, cores = sample_fn(n_rays)
        ts.append(dt)
    ms = 1e3 * sum(ts) / len(ts)
    value = n_rays * S / (ms / 1e3) / 1e6
    cfg = workload_config(args.gpus)
    line = {"impl": "reference", "metric": "Msamples/sec (rays x samples)", "value": value, "unit": "Msamples/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": value, "unit": "Msamples/s", "cores": cores, "kind": "port",
                             "sample": f"{n_rays} rays x {S} samples of the benchmark panorama per step ({which})"},
            "e2e": {"value": value, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def _dp_check(sc, dev, rank, world):
    """Hardware check of the data-parallel step (VERDICT r1 weak #1e), density network:
    (1) after the timed steps every rank holds bit-identical fp32 parameters and fp16 shadows;
    (2) the rank-averaged gradient of a fixed 8192-ray batch cut into `world` slices equals the gradient of the
        whole batch computed on one GPU (cosine, max relative error; the reference's losses are batch means)."""
    import torch
    import torch.distributed as dist
    import torch.nn.functional as F
    from perf_b200 import _lib, ops
    from perf_b200.scene import gen_pano_rays
    res = {}
    for name, t in (("params_fp32", sc.nerf.geo_mlp.params.data), ("shadow_fp16", sc.nerf.geo_mlp._half().float())):
        mx, mn = t.clone(), t.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX); dist.all_reduce(mn, op=dist.ReduceOp.MIN)
        res[f"{name}_identical_across_ranks"] = bool(torch.equal(mx, mn))
    g = torch.Generator(device="cpu").manual_seed(99)
    B = 8192
    rays = gen_pano_rays(torch.eye(4), 64, 128, device=dev)
    o, d = rays.o.reshape(-1, 3), rays.d.reshape(-1, 3)
    jitter, noise, gt = torch.rand(B, generator=g).to(dev), torch.rand(B, 4, generator=g).to(dev), (torch.rand(B, 1, generator=g) * 0.8).to(dev)
    sc._sync_fused()
    tc = sc.train_ctx
    tc.packed, tc.geo_half, tc.app_half = sc.fused.packed, sc.fused.geo_half, sc.fused.app_half
    p = sc.nerf.geo_mlp.params

    def grad_of(sl):
        p.grad = None
        rgb, dist_, op, dl = ops.fused_train_step(p, o[sl].contiguous(), d[sl].contiguous(), jitter[sl].contiguous(), noise[sl].contiguous(), tc, _lib.PERF_PHASE_GEO)
        loss = F.smooth_l1_loss(dist_, gt[sl], beta=1e-2) + 0.1 * dl.sum() / dist_.shape[0]
        (loss * 128).backward()
        return p.grad.detach().clone()
    per = B // world
    g_dp = grad_of(slice(rank * per, (rank + 1) * per))
    dist.all_reduce(g_dp, op=dist.ReduceOp.SUM); g_dp /= world
    g_full = grad_of(slice(0, per * world))
    p.grad = None
    res["dp_vs_single_gpu_gradient_cosine"] = float(F.cosine_similarity(g_dp, g_full, dim=0))
    res["dp_vs_single_gpu_gradient_max_rel_err"] = float((g_dp - g_full).abs().max() / g_full.abs().max())
    return res


def bench_train(dev, rank, world, steps=20, warmup=5):
    """Secondary measurement (not `value`): the optimisation step of configs[1]/[2] -- forward + backward + gradient
    exchange + fused Adam on a synthetic box-room RGB-D panorama, the whole step one CUDA graph.  Two batch rules:
    `fixed_global` = the reference's 8192-ray GLOBAL batch (configs/nerf.yaml pixel_loss_batch_size) cut over the ranks
    (strong scaling), `weak` = 8192 rays PER GPU.  Then the same step as four graphs with CUDA events in between
    (`timeline_us`) and, when world > 1, the hardware data-parallel check (`dp_check`)."""
    import torch
    import torch.distributed as dist
    from perf_b200 import parallel, synthetic
    from perf_b200.scene import FusedAdam, GraphedTrainStep, NeRFScene, RaySupervision
    h, w = 512, 1024
    rgb, distance = synthetic.smooth_rgb(h, w, device=dev), synthetic.box_room_distance(h, w, device=dev)
    sc = NeRFScene(n_samples=S, device=dev)
    sc.set_train()
    pool = RaySupervision.from_panorama(torch.eye(4), rgb, distance)
    out = {"rays_per_step_global": 8192, "samples_per_ray": S, "world": world, "dp_mode": parallel.dp_mode() if world > 1 else "single",
           "note": "forward+backward+gradient exchange+Adam per step captured in one CUDA graph; top-level *_ms_per_step = strong scaling of "
                   "the reference's 8192-ray global batch, `weak` = 8192 rays per GPU; random-init field, synthetic RGB-D"}

    def timed(step_fn, n):
        for _ in range(warmup):
            step_fn()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            step_fn()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / n], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    rules = [("fixed_global", 8192)] + ([("weak", 8192 * world)] if world > 1 else [])
    for rule, batch in rules:
        sc.train_conf["pixel_loss_batch_size"] = batch
        dst = out if rule == "fixed_global" else out.setdefault("weak", {"rays_per_step_global": batch, "rays_per_gpu": 8192})
        for phase in ("geo", "app"):
            net = sc.nerf.geo_mlp if phase == "geo" else sc.nerf.app_mlp
            opt = FusedAdam(net.params, lr=1e-3, module=net)
            graphed = GraphedTrainStep(sc, phase, pool, opt)       # the whole step = one CUDA-graph launch
            ms = timed(lambda: graphed(0.5), steps)
            graphed.finish()                                       # last step's shadow shard + fp32 master on every rank
            dst[f"{phase}_ms_per_step"] = ms
            dst[f"{phase}_msamples_per_s"] = batch * S / ms / 1e3
            if rule == "fixed_global":
                # the same step as four graphs: where the time goes (max over ranks per stage)
                split = GraphedTrainStep(sc, phase, pool, opt, split=True)
                for _ in range(warmup):
                    split(0.5)
                acc = torch.zeros(4, dtype=torch.float64, device=dev)
                for _ in range(steps):
                    if world > 1:
                        dist.barrier()
                    split(0.5)
                    torch.cuda.synchronize()
                    acc += torch.tensor(split.last_stage_ms(), dtype=torch.float64, device=dev)
                acc /= steps
                if world > 1:
                    dist.all_reduce(acc, op=dist.ReduceOp.MAX)
                out.setdefault("timeline_us", {})[phase] = {k: round(1e3 * float(v), 1) for k, v in zip(GraphedTrainStep.STAGES, acc.tolist())}
            opt.sync_master()
    sc.train_conf["pixel_loss_batch_size"] = 8192
    if world > 1:
        out["dp_check"] = _dp_check(sc, dev, rank, world)
    else:
        out["roofline"] = bench_train_roofline(dev)
        occ = bench_train_occ(dev)
        for phase in ("geo", "app"):                          # VERDICT r1 next #5: per-sample cost against the fixed-S step
            fixed_ns = 1e6 * out[f"{phase}_ms_per_step"] / (8192 * S)
            occ[f"{phase}_ns_per_sample_vs_fixed_s"] = (1e6 * occ[f"{phase}_ms_per_step"] / occ[f"{phase}_samples_per_step"]) / fixed_ns
            eqs = occ["equal_samples"]
            eqs[f"{phase}_ns_per_sample_vs_fixed_s"] = (1e6 * eqs[f"{phase}_ms_per_step"] / eqs[f"{phase}_samples_per_step"]) / fixed_ns
        out["occ"] = occ
    return out


def bench_train_roofline(dev):
    """Physical rooflines of the two training kernels that are NOT gather-bound (N = 1 only, VERDICT r1 next #3):
    the grid-gradient scatter against the measured L2 reduction rate, the Adam pass against the measured HBM bandwidth."""
    import torch
    from perf_b200 import ops
    g = torch.Generator().manual_seed(0)
    R = 8192
    o = ((torch.rand(R, 3, generator=g) - 0.5) * 0.2).to(dev)
    d = torch.nn.functional.normalize(torch.randn(R, 3, generator=g), dim=-1).to(dev)
    jit = torch.rand(R, generator=g).to(dev)
    dfeat = torch.randn(R * S, 32, generator=g).to(dev)
    table = torch.zeros(ops.PERF_GRID.n_entries, 2, device=dev)

    def timed(fn, iters=10):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters
    ms_scatter = timed(lambda: ops.hashgrid_bwd_rays(o, d, jit, S, 1e-2, 1.0, dfeat, out=table))
    rate4 = ops.atomic_rate(vec=4, device=dev)
    # fine levels (8..15): per sample and level 4 x-neighbour pairs, one 16-byte reduction when the pair shares a slot
    # (cell x even: half of the time), else two 8-byte ones -> 6 on average; coarse levels flush once per cell run
    fine_atomics = R * S * 8 * 6
    n = 6644288
    p, gr, m, v = (torch.randn(n, generator=g).to(dev) for _ in range(4))
    v.abs_()
    half = torch.empty(n, dtype=torch.float16, device=dev)
    ms_adam = timed(lambda: ops.adam_step(p, gr, m, v, 3, 1e-3, params_half=half))
    peak, peak_src = measured_peak_hbm()
    adam_gbs = n * 30 / (ms_adam * 1e-3) / 1e9
    return {"scatter": {"kernels": "hashgrid_bwd_both_kernel (8192 x 128 samples; coarse march blocks interleaved with fine-level blocks in one launch)",
                        "ms": ms_scatter, "fine_level_reductions_per_step": fine_atomics,
                        "achieved_g_reductions_per_s": fine_atomics / (ms_scatter * 1e-3) / 1e9,
                        "peak_g_reductions_per_s": rate4 / 1e9, "frac": fine_atomics / (ms_scatter * 1e-3) / rate4,
                        "peak_source": "measured in this run: perf_debug_atomic_rate, random 16-byte fp32 reductions into a 16.8 MB table",
                        "note": "achieved counts only the fine levels' reductions over the time of the whole launch (which also does the coarse levels), so frac is a lower bound"},
            "adam": {"kernel": "adam_kernel", "ms": ms_adam, "bytes_per_param": 30, "achieved": adam_gbs, "peak": peak, "unit": "GB/s",
                     "frac": adam_gbs / peak, "peak_source": peak_src}}


def bench_train_occ(dev, steps=20, warmup=5):
    """The optimisation step on the sampler PeRF really trains with (`estimator_type: occ`, configs/nerf.yaml:25): occupancy
    grid = surface shell of the synthetic box room at 256^3, intervals of 5e-4, 8192 rays per step, fused packed path
    (perf_occ_count/write, perf_fields_packed, perf_composite_packed_fwd/bwd, perf_mlp_bwd, perf_hashgrid_bwd_merged).
    Eager (one host read of the sample count per step, as nerfacc has).  N = 1 only."""
    import torch
    from perf_b200 import ops, synthetic
    from perf_b200.scene import FusedAdam, NeRFScene, RaySupervision
    h, w = 512, 1024
    rgb, distance = synthetic.smooth_rgb(h, w, device=dev), synthetic.box_room_distance(h, w, device=dev)
    sc = NeRFScene(estimator_type="occ", occ_resolution=256, device=dev)
    pool = RaySupervision.from_panorama(torch.eye(4), rgb, distance)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    sc.build_occupancy(pool)
    e1.record()
    torch.cuda.synchronize()
    out = {"rays_per_step": 8192, "render_step_size": sc.OCC_STEP, "occ_resolution": 256,
           "occupancy_build_ms_256_updates": e0.elapsed_time(e1), "occupied_cell_fraction": float(sc.estimator.binaries.float().mean())}
    sc.set_train()
    from perf_b200.scene import GraphedTrainStep
    for phase in ("geo", "app"):
        net = sc.nerf.geo_mlp if phase == "geo" else sc.nerf.app_mlp
        opt = FusedAdam(net.params, lr=1e-3, module=net)
        # (a) eager, as the reference's loop is: one host read of the sample count per step
        step = sc.train_one_step_geo if phase == "geo" else sc.train_one_step_app
        sc._occ_static = None
        for _ in range(warmup):
            step(opt, pool, progress=0.5)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(steps):
            step(opt, pool, progress=0.5)
        e1.record()
        torch.cuda.synchronize()
        out[f"{phase}_eager_ms_per_step"] = e0.elapsed_time(e1) / steps
        # (b) the same step as ONE CUDA graph: capacity-sized buffers, sample count kept on the device
        graphed = GraphedTrainStep(sc, phase, pool, opt)
        for _ in range(warmup):
            graphed(0.5)
        torch.cuda.synchronize()
        n_samples = 0
        acc = torch.zeros(1, dtype=torch.int64, device=dev)
        e0.record()
        for _ in range(steps):
            graphed(0.5)
            acc += sc._occ_static.n                                     # device-side add: no host read inside the timed region
        e1.record()
        torch.cuda.synchronize()
        n_samples = int(acc)
        graphed.finish()
        ms = e0.elapsed_time(e1) / steps
        out[f"{phase}_ms_per_step"] = ms
        out[f"{phase}_samples_per_step"] = n_samples / steps
        out[f"{phase}_samples_per_ray"] = n_samples / steps / 8192
        out[f"{phase}_msamples_per_s"] = n_samples / steps / ms / 1e3
        out[f"{phase}_capacity"] = sc._occ_static.capacity
        out[f"{phase}_overflow_samples"] = graphed.occ_overflow()
    out["note"] = "*_ms_per_step: whole step replayed as one CUDA graph (no host read); *_eager_ms_per_step: eager with the sample-count read, launch-bound"
    # The same step at the SAMPLE count of the fixed-S step (8192 x 128): 38.5 samples per ray make the reference's 8192-ray batch
    # 3.3x smaller than the fixed-S one, so its fixed costs (batch draw, Adam over 6.6 M parameters, table pack, the marcher's
    # empty space) weigh 3.3x more per sample; with as many rays as give 1.05 M samples the two steps do the same amount of field work.
    r2 = int(8192 * (8192 * S) / max(out["geo_samples_per_step"], 1.0)) // 128 * 128
    sc.train_conf["pixel_loss_batch_size"] = r2
    eq = {"rays_per_step": r2}
    for phase in ("geo", "app"):
        net = sc.nerf.geo_mlp if phase == "geo" else sc.nerf.app_mlp
        opt = FusedAdam(net.params, lr=1e-3, module=net)
        graphed = GraphedTrainStep(sc, phase, pool, opt)
        for _ in range(warmup):
            graphed(0.5)
        torch.cuda.synchronize()
        acc = torch.zeros(1, dtype=torch.int64, device=dev)
        e0.record()
        for _ in range(steps):
            graphed(0.5)
            acc += sc._occ_static.n
        e1.record()
        torch.cuda.synchronize()
        graphed.finish()
        ms, n = e0.elapsed_time(e1) / steps, int(acc) / steps
        eq[f"{phase}_ms_per_step"], eq[f"{phase}_samples_per_step"], eq[f"{phase}_msamples_per_s"] = ms, n, n / ms / 1e3
        eq[f"{phase}_overflow_samples"] = graphed.occ_overflow()
    out["equal_samples"] = eq
    sc.train_conf["pixel_loss_batch_size"] = 8192
    return out


def bench_extra_configs(renderer, dev, rank, world, steps=2):
    """BASELINE configs[3] and [4] as extra keys (VERDICT r1 missing #4), same field, same kernel:
    `render_c4` = render_dense 2048 x 4096, 256 samples/ray, row-tiled over the ranks, WITH the tile gather to rank 0 (the only
    collective of that path, timed separately); `render_c5` = 4096 x 8192, 192 samples/ray (the render half of the sweep;
    its training half is the 8192-ray step of `train`, whose cost does not depend on the panorama size)."""
    import torch
    import torch.distributed as dist
    from perf_b200 import parallel
    out = {}
    pose = bench_pose()
    for key, (h, w, s, gather) in (("render_c4", (2048, 4096, 256, True)), ("render_c5", (4096, 8192, 192, False))):
        sl = parallel.shard_slice(h, rank, world)
        bufs = tuple(torch.empty(sl.stop - sl.start, w, c, dtype=torch.float32, device=dev) for c in (3, 1, 1))
        run = lambda: renderer.render_pano(pose, h, w, s, row0=sl.start, rows=sl.stop - sl.start, out=bufs)
        r = run()
        if gather:                                          # untimed: NCCL sets up its point-to-point channels on first use
            parallel.gather_row_tiles(torch.cat([r["rgb"], r["distance"]], -1), h)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        t_render = t_total = 0.0
        for _ in range(steps):
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            ev[0].record()
            r = run()
            ev[1].record()
            if gather:
                parallel.gather_row_tiles(torch.cat([r["rgb"], r["distance"]], -1), h)
            ev[2].record()
            torch.cuda.synchronize()
            t_render += ev[0].elapsed_time(ev[1]); t_total += ev[0].elapsed_time(ev[2])
        t = torch.tensor([t_render / steps, t_total / steps], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_r, ms_t = (float(v) for v in t.tolist())
        n = h * w * s
        out[key] = {"H": h, "W": w, "samples_per_ray": s, "render_ms": ms_r, "msamples_per_s": n / ms_r / 1e3,
                    "rays_per_s": h * w / (ms_r / 1e3)}
        if gather:
            # both maxima over ranks from a common barrier: the frame is done when rank 0 holds every tile; the exposed
            # gather time is what that adds to the slowest rank's render (rank 0 renders the cheap pole rows and waits)
            out[key].update({"frame_ms_incl_gather": ms_t, "tile_gather_exposed_ms": ms_t - ms_r, "tile_bytes_per_gpu": (sl.stop - sl.start) * w * 16,
                             "msamples_per_s_incl_gather": n / ms_t / 1e3,
                             "note": "gather = torch.cat of rgb+distance into [rows,W,4] fp32 + NCCL gather to rank 0" if world > 1 else "single GPU: no gather"})
        del bufs
    return out


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from perf_b200 import ops
    from perf_b200.renderer import FusedPanoRenderer
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    geo, app = make_field(dev)
    renderer = FusedPanoRenderer.from_params(geo, app)
    pose = bench_pose()
    rows_per = (H + world - 1) // world
    row0 = rank * rows_per
    rows = max(0, min(rows_per, H - row0))
    out = tuple(torch.empty(rows, W, c, dtype=torch.float32, device=dev) for c in (3, 1, 1))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    host_rgb = torch.empty(rows, W, 3, dtype=torch.float32).pin_memory()
    host_dist = torch.empty(rows, W, 1, dtype=torch.float32).pin_memory()
    pose_pinned = pose.clone().pin_memory()

    def step():
        renderer.render_pano(pose, H, W, S, row0=row0, rows=rows, out=out)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()

    # ---- kernel-resident timing: CUDA events around each step, L2 flushed in between
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = ops.launch_count()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for e0, e1 in evs:
        flush.fill_(1)
        e0.record()
        step()
        e1.record()
    barrier()
    launches = ops.launch_count() - launches0
    total_ms = sum(e0.elapsed_time(e1) for e0, e1 in evs)
    # the last timed step's panorama, before the end-to-end loop below renders into the same buffers
    dumped = gather_panorama(out, rows_per, world) if args.dump_outputs else None

    # ---- end to end through the public API: host pose in, host images out, every step
    barrier()
    t_e2e = [torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)]
    t_e2e[0].record()
    for _ in range(args.steps):
        r = renderer.render_pano(pose_pinned, H, W, S, row0=row0, rows=rows, out=out)
        host_rgb.copy_(r["rgb"], non_blocking=True)
        host_dist.copy_(r["distance"], non_blocking=True)
        torch.cuda.current_stream().synchronize()
    t_e2e[1].record()
    barrier()
    e2e_ms = t_e2e[0].elapsed_time(t_e2e[1])
    clocks = sampler.stop()

    train = bench_train(dev, rank, world) if not args.no_train else None
    extra = bench_extra_configs(renderer, dev, rank, world) if not args.no_train else None

    t = torch.tensor([total_ms, e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, e2e_ms = (float(v) for v in t.tolist())
    if rank != 0:
        return
    if dumped is not None:
        write_outputs(args.dump_outputs, dumped)
    ms_per_step = total_ms / args.steps
    samples = H * W * S
    value = samples / (ms_per_step / 1e3) / 1e6
    e2e_value = samples / (e2e_ms / args.steps / 1e3) / 1e6
    peak, peak_src = measured_peak_hbm()
    achieved = ALG_BYTES_PER_SAMPLE * samples / world / (ms_per_step / 1e3) / 1e9     # per-GPU kernel
    traffic, physical = None, {}
    try:                                              # counters of this very launch from the committed ncu capture (profiles/)
        t = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        traffic = (t["dram_bytes_read"] + t["dram_bytes_write"]) if world == 1 else None
        # the PHYSICAL limiter: the tables are L2-resident, so `frac` (algorithmic bytes / HBM peak) is not a utilisation;
        # the unit that is busiest is the L1TEX pipe of the gathers, then instruction issue
        physical = {"frac_physical": t["l1tex_throughput_pct"] / 100.0, "physical_unit": "L1TEX throughput (ncu l1tex__throughput.avg.pct_of_peak_sustained_elapsed)",
                    "issue_active_frac": t["issue_active_pct"] / 100.0, "l2_throughput_frac": t["lts_throughput_pct"] / 100.0,
                    "tensor_pipe_frac": t["tensor_pipe_pct"] / 100.0,
                    "physical_source": "profiles/r02_traffic.json: one ncu --set full capture of the same launch, not measured in this run"}
    except Exception:
        pass
    cpu_v, cpu_s, cores = cpu_oracle_sample(4096) if world == 1 else (None, None, None)     # PyTorch port (+ parity reference)
    c_err = None
    try:
        c_v, c_s, c_cores = cpu_c_port_sample(65536) if world == 1 else (None, None, None)      # C / OpenMP port, host threads
    except Exception as e:                             # no gcc / OpenMP on this host: fall back to the PyTorch port's figure
        c_v, c_s, c_cores, c_err = cpu_v, cpu_s, cores, f"{type(e).__name__}: {e}"[:200]
    line = {"metric": "Msamples/sec (rays x samples)", "value": value, "unit": "Msamples/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f16", "data": "synthetic (seeded random-init field, no checkpoints exist)",
            "config": workload_config(world), "rays_per_sec": H * W / (ms_per_step / 1e3),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "Msamples/s", "h2d_bytes_per_step": 64,
                    "d2h_bytes_per_step": rows * W * 16 * world, "note": "input is a 4x4 pose; output rgb+distance images to pinned host memory"},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "kernel": "perf::render_march_kernel<PANO=true,SIMT=false,NDENSE=4>", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_sample": ALG_BYTES_PER_SAMPLE, **physical,
                         "note": "the packed table (37.8 MB fp16: 26.6 MB of entries + 11.2 MB cell-major dense levels) is L2-resident: DRAM traffic is far below algorithmic bytes, see profiles/"}}
    if cpu_v is not None:
        # parity of THIS run's kernel against the CPU restatement on the very rays the baseline timed
        # (the metric's second half: "PSNR delta vs reference")
        ref = cpu_oracle_sample.last
        got = renderer.render_rays(ref["rays_o"].to(dev), ref["rays_d"].to(dev), S)
        d_rgb = (got["rgb"].cpu() - ref["rgb"]).abs()
        d_dist = (got["distance"].cpu() - ref["distance"]).abs()
        mse = float((d_rgb ** 2).mean())
        import math
        line["parity"] = {"rays": int(ref["rays_o"].shape[0]), "samples_per_ray": S, "max_abs_rgb": float(d_rgb.max()),
                          "max_abs_distance": float(d_dist.max()),
                          "psnr_kernel_vs_cpu_oracle_db": 99.0 if mse == 0 else -10.0 * math.log10(mse),
                          "note": "same seeded field, same rays; trained-field PSNR delta (0.001 dB) is asserted in tests/test_gpu_train.py"}
    if train is not None:
        line["train"] = train
    if extra is not None:
        line.update(extra)
    if cpu_v is not None:
        line["cpu_baseline"] = {"value": c_v, "unit": "Msamples/s", "cores": c_cores, "kind": "port",
                                "sample": f"65536 rays x {S} samples (middle rows of the panorama), oracle/cpath.c = plain-C / OpenMP restatement, "
                                          f"{c_cores} threads = all {len(os.sched_getaffinity(0))} visible CPUs, {c_s:.1f} s",
                                **({"c_port_error": c_err} if c_err else {}),
                                "pytorch_port": {"value": cpu_v, "cores": cores, "sample": f"4096 rays x {S} samples, oracle/render.py, {cpu_s:.1f} s; threads "
                                                 f"capped at 16 of {os.cpu_count()} (many small torch ops: slower beyond that)"}}
    emit(line)


def gather_panorama(out, rows_per, world):
    """rgb / distance / opacities row tiles of every rank -> {name: [H, W, C] float32 on the host} on rank 0
    (None elsewhere).  Tiles are padded to `rows_per` rows for the gather and cropped to H after it."""
    import torch
    import torch.distributed as dist
    tile = torch.cat(out, -1)
    if world > 1:
        send = torch.zeros(rows_per, W, tile.shape[-1], dtype=tile.dtype, device=tile.device)
        send[:tile.shape[0]] = tile
        recv = [torch.empty_like(send) for _ in range(world)] if dist.get_rank() == 0 else None
        dist.gather(send, recv, dst=0)
        if recv is None:
            return None
        tile = torch.cat(recv)[:H]
    tile = tile.cpu()
    return {"rgb": tile[..., 0:3], "distance": tile[..., 3:4], "opacities": tile[..., 4:5]}


def write_outputs(dirname, arrays):
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(dirname, f"{name}.npy"), np.ascontiguousarray(t.numpy(), dtype=np.float32))


_REAL_STDOUT = None


def quiet_stdout():
    """Send everything libraries print to fd 1 (NCCL's version banner, ...) to stderr until emit()."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def emit(line: dict):
    """The ONE JSON line of the contract, on the real stdout."""
    sys.stdout.flush()
    if _REAL_STDOUT is not None:
        os.dup2(_REAL_STDOUT, 1)
    print(json.dumps(line), flush=True)


def main():
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-train", action="store_true", help="skip the secondary training-step measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's rgb / distance / opacities to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    rank, world, local_rank = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    import torch.distributed as dist
    if world > 1:
        import torch
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")      # keep stdout = the one JSON line
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
