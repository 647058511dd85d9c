"""GPU tests of the one-launch occupancy-grid renderer (perf_render_rays_occ / perf_render_pano_occ,
csrc/render.cu::render_occ_kernel): bit-identical to the packed renderer on the intervals it composites, equal to the
cull-then-render order of nerf_renderer.py:145-197, the same numbers for every tiling, the eval background for rays
without samples, no memory beyond its outputs, CUDA-graph capture, and the checkpoint path of render_dense."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import oracle

pytestmark = pytest.mark.gpu

AABB = torch.tensor([-1., -1., -1., 1., 1., 1.])
STEP = 4.0e-3                                # coarser than PeRF's 5e-4: the oracle evaluates every interval


@pytest.fixture(scope="module")
def dense_field(golden_field):
    """The golden field with the density row x30: rays saturate, so the 1e-4 transmittance cut bites."""
    geo = golden_field.geo_params.clone()
    geo[2048:2048 + 64] *= 30.0                                 # Wout row 0 of the density net (32-64-1: W1 2048 | Wout 16x64)
    return oracle.Field(geo, golden_field.app_params)


@pytest.fixture(scope="module")
def renderer(dense_field):
    from perf_b200.renderer import FusedPanoRenderer
    return FusedPanoRenderer.from_params(dense_field.geo_params.cuda(), dense_field.app_params.cuda())


def _case(seed, R, res=16, occupancy=0.6):
    g = torch.Generator().manual_seed(seed)
    binaries = torch.rand(res, res, res, generator=g) < occupancy
    o = (torch.rand(R, 3, generator=g) - .5) * .4
    d = F.normalize(torch.randn(R, 3, generator=g), dim=-1)
    o[:3] = 4.0                                                  # rays that miss the box: zero samples
    d[3] = torch.tensor([0.0, 1.0, 0.0])                         # axis-parallel
    return binaries, o, d


def _occ(r, binaries, aabb=AABB, step=STEP, eps=1e-4):
    r.set_occupancy(binaries.cuda(), aabb.tolist(), near=0.0, far=1.5, step=step, early_stop_eps=eps)


SIMT = pytest.mark.parametrize("simt", [True, False], ids=["simt", "tcgen05"])


@SIMT
@pytest.mark.parametrize("eps", [1e-4, 0.0])
def test_bit_identical_to_render_packed_on_composited_intervals(renderer, simt, eps):
    """The kernel composites each ray's first n_samples[r] intervals of the two-pass sampler, with the same arithmetic as
    perf_render_packed: rendering exactly those intervals with it gives the same bits."""
    from perf_b200 import ops
    binaries, o, d = _case(71, 300)
    _occ(renderer, binaries, eps=eps)
    out = renderer.render_rays_occ(o.cuda(), d.cuda(), simt=simt, want_n_samples=True)
    n = out["n_samples"].long()
    ri, ts, te = ops.occ_sample(binaries.cuda(), AABB.tolist(), o.cuda(), d.cuda(), 0.0, 1.5, STEP, None)
    off = ops.occ_sample.last_offsets
    counts = off[1:] - off[:-1]
    assert torch.all(n <= counts) and int(n[:3].sum()) == 0
    if eps == 0.0:
        assert torch.equal(n, counts)
    else:
        assert int((n < counts).sum()) > 30, "the cut must end a good share of the rays early"
    keep = (torch.arange(ri.numel(), device=ri.device) - off[ri]) < n[ri]
    want = renderer.render_packed(o.cuda(), d.cuda(), ri[keep], ts[keep], te[keep], simt=simt)
    for k in ("rgb", "distance", "opacities"):
        assert torch.equal(out[k], want[k]), k


@SIMT
def test_equals_cull_then_render_oracle(renderer, dense_field, simt):
    """nerf_renderer.py:145-197's order: evaluate the density at every interval, DROP those with T < 1e-4, render the rest."""
    from perf_b200 import ops
    R = 200
    binaries, o, d = _case(61, R)
    from oracle.occ_sampler import occ_sample
    ri, ts, te = occ_sample(binaries, AABB, o, d, 0.0, 1.5, STEP)
    pos = o[ri] + d[ri] * (ts + te)[:, None] / 2.0
    sig = oracle.query_density(dense_field, pos, mixed=True).squeeze(-1)
    _, T_all, _ = oracle.render_weight_from_density(ts, te, sig, ri)
    keep = T_all >= 1e-4
    assert 0.02 < float((~keep).float().mean()) < 0.9, float((~keep).float().mean())
    ri2, ts2, te2, sig2 = ri[keep], ts[keep], te[keep], sig[keep]
    rgbs = oracle.query_rgb(dense_field, pos[keep], mixed=True)
    w, _, _ = oracle.render_weight_from_density(ts2, te2, sig2, ri2)
    op = oracle.accumulate_along_rays(w, None, ri2, R)
    dist = oracle.accumulate_along_rays(w, ((ts2 + te2) / 2.0)[:, None], ri2, R) + 5.0 * (1 - op)
    col = oracle.accumulate_along_rays(w, rgbs, ri2, R) + 0.5 * (1 - op)
    _occ(renderer, binaries)
    out = renderer.render_rays_occ(o.cuda(), d.cuda(), simt=simt, want_n_samples=True)
    assert torch.equal(out["n_samples"].long().cpu(), torch.bincount(ri2, minlength=R))
    np.testing.assert_allclose(out["opacities"].cpu().numpy(), op.numpy(), atol=4e-3, rtol=0)
    np.testing.assert_allclose(out["rgb"].cpu().numpy(), col.numpy(), atol=4e-3, rtol=0)
    np.testing.assert_allclose(out["distance"].cpu().numpy(), dist.numpy(), atol=4e-3, rtol=0)
    # and the packed two-launch grid render (perf_fields_packed + perf_composite_packed_fwd)
    rk, tsk, tek = ops.occ_sample(binaries.cuda(), AABB.tolist(), o.cuda(), d.cuda(), 0.0, 1.5, STEP, None)
    old = renderer.render_occ(o.cuda(), d.cuda(), ops.occ_sample.last_offsets, rk, tsk, tek)
    for k in ("rgb", "distance", "opacities"):
        assert (old[k] - out[k]).abs().max() <= 2e-4, k


@SIMT
@pytest.mark.parametrize("H,W,split", [(37, 90, 17), (512, 1024, 200)])
def test_pano_equals_explicit_rays_and_row_tiling(renderer, simt, H, W, split):
    """Ray generation inside the kernel == rays from ops.raygen_pano, explicit rays with or without the image-shaped
    tiling == the panorama, and a frame rendered in two row windows == the whole frame: all bit for bit.  37 x 90 leaves
    partial 16 x 8 tiles on both edges."""
    from perf_b200 import ops
    g = torch.Generator().manual_seed(5)
    binaries = torch.rand(32, 32, 32, generator=g) < 0.3
    _occ(renderer, binaries, step=5e-4)
    pose = torch.eye(4); pose[:3, 3] = torch.tensor([0.1, 0.0, -0.05])
    full = renderer.render_pano_occ(pose, H, W, simt=simt)
    o, d = ops.raygen_pano(pose, H, W)
    flat = renderer.render_rays_occ(o.reshape(-1, 3), d.reshape(-1, 3), simt=simt)
    img = renderer.render_rays_occ(o, d, simt=simt)
    top = renderer.render_pano_occ(pose, H, W, row0=0, rows=split, simt=simt)
    bot = renderer.render_pano_occ(pose, H, W, row0=split, rows=H - split, simt=simt)
    for k, c in (("rgb", 3), ("distance", 1), ("opacities", 1)):
        assert full[k].shape == (H, W, c)
        assert torch.equal(full[k].reshape(-1, c), flat[k]), k
        assert torch.equal(img[k], flat[k]), k
        assert torch.equal(torch.cat([top[k], bot[k]]), full[k]), k


@SIMT
def test_rays_without_samples_get_the_background(renderer, simt):
    from perf_b200 import ops
    binaries, o, d = _case(3, 100)
    _occ(renderer, torch.zeros(8, 8, 8, dtype=torch.bool))                    # empty grid
    for out in (renderer.render_rays_occ(o.cuda(), d.cuda(), simt=simt, want_n_samples=True),
                renderer.render_pano_occ(torch.eye(4), 8, 16, simt=simt, want_n_samples=True)):
        assert torch.all(out["rgb"] == 0.5) and torch.all(out["distance"] == 5.0) and torch.all(out["opacities"] == 0.0)
        assert torch.all(out["n_samples"] == 0)
    _occ(renderer, binaries)                                                   # rays that miss the box
    out = renderer.render_rays_occ(o.cuda(), d.cuda(), simt=simt, want_n_samples=True)
    assert torch.equal(out["rgb"][:3].cpu(), torch.full((3, 3), 0.5)) and torch.equal(out["distance"][:3].cpu(), torch.full((3, 1), 5.0))
    assert torch.equal(out["opacities"][:3].cpu(), torch.zeros(3, 1)) and int(out["n_samples"][:3].abs().sum()) == 0
    rgb, dist, op = ops.render_rays_occ(renderer.packed, renderer.geo_half, renderer.app_half, o[:0].cuda(), d[:0].cuda(),
                                        binaries.cuda(), AABB.tolist())
    assert rgb.shape == (0, 3) and dist.shape == (0, 1)


@SIMT
def test_full_grid_and_non_unit_grid_box(renderer, dense_field, simt):
    """A full grid emits every lattice interval inside the box; a grid box that differs from the field's box (here the
    estimator's roi is smaller and off-centre) clips the walk to it.  Both bit-identical to render_packed on the intervals
    of the two-pass sampler, kept up to the kernel's counts."""
    from perf_b200 import ops
    _, o, d = _case(17, 256)
    for binaries, aabb in ((torch.ones(12, 12, 12, dtype=torch.bool), AABB),
                           (torch.rand(9, 5, 7, generator=torch.Generator().manual_seed(2)) < 0.5, torch.tensor([-0.5, -1.0, -0.25, 0.9, 0.5, 0.75]))):
        _occ(renderer, binaries, aabb=aabb, eps=0.0)
        out = renderer.render_rays_occ(o.cuda(), d.cuda(), simt=simt, want_n_samples=True)
        ri, ts, te = ops.occ_sample(binaries.cuda(), aabb.tolist(), o.cuda(), d.cuda(), 0.0, 1.5, STEP, None)
        off = ops.occ_sample.last_offsets
        assert torch.equal(out["n_samples"].long(), off[1:] - off[:-1])
        want = renderer.render_packed(o.cuda(), d.cuda(), ri, ts, te, simt=simt)
        for k in ("rgb", "distance", "opacities"):
            assert torch.equal(out[k], want[k]), k


def test_full_panorama_memory_and_cuda_graph(renderer):
    """1024 x 2048 with PeRF's lattice: no memory beyond the outputs (+ 1 MiB), and the launch replays from a CUDA graph
    with the same bits as the eager call."""
    H, W = 1024, 2048
    c = (torch.arange(64) + 0.5) / 64 * 2 - 1
    r = (c[:, None, None] ** 2 + c[None, :, None] ** 2 + c[None, None, :] ** 2).sqrt()
    _occ(renderer, (r - 0.7).abs() < 0.06, step=5e-4)                        # a spherical shell around the camera
    pose = torch.eye(4); pose[:3, 3] = torch.tensor([0.05, -0.02, 0.01])
    renderer.render_pano_occ(pose, 8, 16)                                     # first call: kernel attributes, weights symbol
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    eager = renderer.render_pano_occ(pose, H, W, want_n_samples=True)
    torch.cuda.synchronize()
    outputs = sum(t.numel() * t.element_size() for t in (eager["rgb"], eager["distance"], eager["opacities"], eager["n_samples"]))
    assert torch.cuda.max_memory_allocated() - base <= outputs + (1 << 20)
    assert int(eager["n_samples"].min()) > 0, "every ray crosses the shell"
    out = tuple(torch.full_like(eager[k], -1.0) for k in ("rgb", "distance", "opacities"))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        renderer.render_pano_occ(pose, H, W, out=out)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        renderer.render_pano_occ(pose, H, W, out=out)
    for t in out:
        t.fill_(-1.0)
    graph.replay()
    torch.cuda.synchronize()
    for k, t in zip(("rgb", "distance", "opacities"), out):
        assert torch.equal(t, eager[k]), k


def test_checkpoint_round_trip_and_render_dense(golden_field, tmp_path):
    """FusedPanoRenderer.from_state_dict(nerf, estimator) of a NeRFScene.state_dict() renders what the scene renders, and
    `python -m perf_b200.render_dense --sampler occ` on the checkpoint writes exactly its frames."""
    import cv2
    from perf_b200 import render_dense
    from perf_b200.renderer import FusedPanoRenderer
    from perf_b200.scene import NeRFScene
    sc = NeRFScene(estimator_type="occ", occ_resolution=32)
    g = torch.Generator().manual_seed(9)
    with torch.no_grad():
        sc.nerf.geo_mlp.params.copy_(golden_field.geo_params.half().float())
        sc.nerf.app_mlp.params.copy_(golden_field.app_params.half().float())
        sc.estimator.binaries.copy_((torch.rand(1, 32, 32, 32, generator=g) < 0.4).cuda())
    sc.set_eval()
    sd = sc.state_dict()
    r = FusedPanoRenderer.from_state_dict(sd["nerf"], sd["estimator"])
    assert r.occ["step"] == sc.OCC_STEP and (r.occ["near"], r.occ["far"], r.occ["early_stop_eps"]) == (0.0, 1.5, 1e-4)
    pose = torch.eye(4); pose[:3, 3] = torch.tensor([0.1, 0.05, 0.0])
    H, W = 32, 64
    want = sc.render_pano(pose, H, W)
    got = r.render_pano_occ(pose, H, W)
    for k in ("rgb", "distance", "opacities"):
        assert torch.equal(got[k], want[k]), k
    with pytest.raises(NotImplementedError, match="levels"):
        FusedPanoRenderer.from_state_dict(sd["nerf"], {**sd["estimator"], "binaries": sd["estimator"]["binaries"].expand(2, -1, -1, -1)})
    # render_dense on the checkpoint
    ckpt, poses, out_dir = tmp_path / "ckpt.pth", tmp_path / "poses.npy", tmp_path / "frames"
    torch.save({"scene": {k: v for k, v in sd.items()}}, ckpt)
    np.save(poses, pose[None].numpy())
    render_dense.main(["--ckpt", str(ckpt), "--poses", str(poses), "--out", str(out_dir), "--height", str(H), "--width", str(W),
                       "--sampler", "occ"])
    png = cv2.imread(str(out_dir / "image_0.png"))[..., ::-1]
    assert np.array_equal(png, (got["rgb"].clamp(0, 1) * 255).byte().cpu().numpy())
    # a checkpoint without a grid is refused with a message, not rendered with another sampler
    torch.save({"scene": {"nerf": sd["nerf"]}}, ckpt)
    with pytest.raises(SystemExit, match="occupancy grid"):
        render_dense.main(["--ckpt", str(ckpt), "--out", str(out_dir), "--sampler", "occ"])
