"""CPU tests: perf_b200's plugin shims provide the API surface the reference's OWN hot-path files use
(names, constructor arguments, parameter layout, state-dict keys).  What those files asked of the plugins
and built on the shims -- the tinycudann constructor calls of `ngp_nerf.py`, the names imported from
each plugin package, the state-dict of ``NGPNeRF``, the LR schedule and occupancy pre-grid -- was
recorded by running them unmodified on the shims (tests/golden/make_golden.py) into
``tests/golden/reference_api.json`` / ``reference_host.npz``.  No kernels run (no GPU here); forward on
CPU tensors must fail loudly."""
import importlib
import json
import os

import numpy as np
import pytest
import torch
import yaml

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def reference_api():
    return json.load(open(os.path.join(GOLDEN, "reference_api.json")))


def write_reference_configs(config_dir, api):
    """The reference's configs/ tree (nerf.yaml and the defaults it selects) from the parsed fixture."""
    for name, doc in api["configs"].items():
        path = os.path.join(str(config_dir), name)
        os.makedirs(os.path.dirname(path), exist_ok=True)
        with open(path, "w") as f:
            yaml.safe_dump(doc, f, sort_keys=False)
    return str(config_dir)


def test_reference_field_builds_on_shim(reference_api):
    from perf_b200 import shims
    from perf_b200 import field as F
    shims.install()
    import tinycudann
    assert getattr(tinycudann, "__perf_b200_shim__", False)
    calls = reference_api["tcnn_calls"]
    # the reference's constructor calls (ngp_nerf.py:96-134) build on the shim, with the parameter counts of the
    # state-dict it saw; perf_b200.field.NGPNeRF makes the same calls
    geo_kw, app_kw = calls["NGPNeRF"]
    assert [geo_kw, app_kw] == [{"n_input_dims": 3, "n_output_dims": n, "encoding_config": F.ENCODING_CONFIG, "network_config": net}
                                for n, net in ((1, F.GEO_NETWORK_CONFIG), (3, F.APP_NETWORK_CONFIG))]
    assert calls["NGPNeRF.reset_geo"] == [geo_kw]
    sd_ref = reference_api["nerf_state_dict"]
    assert tinycudann.NetworkWithInputEncoding(**geo_kw).params.shape == tuple(sd_ref["geo_mlp.params"]["shape"])
    assert tinycudann.NetworkWithInputEncoding(**app_kw).params.shape == tuple(sd_ref["app_mlp.params"]["shape"])
    f = F.NGPNeRF(aabb=[-1.0, -1.0, -1.0, 1.0, 1.0, 1.0])
    sd = f.state_dict()
    assert {k: {"shape": list(v.shape), "dtype": str(v.dtype)} for k, v in sd.items()} == sd_ref
    assert set(sd) == {"aabb", "geo_mlp.params", "app_mlp.params"}          # checkpoint keys, nerf.py:374-380
    assert sd["geo_mlp.params"].shape == (6644288,) and sd["app_mlp.params"].shape == (6648384,)
    assert sd["geo_mlp.params"].dtype == torch.float32
    grid = sd["geo_mlp.params"][3072:]
    assert float(grid.abs().max()) <= 1e-4 and float(grid.abs().max()) > 5e-5   # U(-1e-4, 1e-4)
    f.reset_geo()                                                               # ngp_nerf.py:178-197
    assert f.geo_mlp.params.shape == (6644288,)
    with pytest.raises(RuntimeError, match="CUDA"):                             # no CPU path
        f.query_density(torch.rand(4, 3))
    # the proposal field (L5 grid -> 10-wide MLP input) belongs to the reference's broken/unused
    # `estimator_type: prop` path: unsupported configurations fail at CONSTRUCTION, not silently
    from perf_b200._lib import PerfError
    (density_kw,) = calls["NGPDensityField"]
    assert density_kw["encoding_config"]["n_levels"] == 5
    with pytest.raises(PerfError, match="n_in=10"):
        tinycudann.NetworkWithInputEncoding(**density_kw)
    f.load_state_dict(sd)


def test_reference_renderer_and_scene_symbols(reference_api):
    from perf_b200 import shims
    from perf_b200 import scene as ours
    shims.install()
    # every name the reference's files import from (or read off) a plugin package exists on the shim
    for module, names in reference_api["shim_names"].items():
        m = importlib.import_module(module)
        assert getattr(importlib.import_module(module.split(".")[0]), "__perf_b200_shim__", False), module
        for name in names:
            assert hasattr(m, name), f"{module}.{name}"
    r = ours.NeRFOCCRenderer(max_radius=2, bg_color="rand_noise")
    assert sorted(r.state_dict()) == reference_api["renderer_state_dict_keys"] == []
    import inspect
    from nerfacc.estimators.occ_grid import OccGridEstimator
    est = OccGridEstimator(roi_aabb=torch.tensor([-1.0, -1.0, -1.0, 1.0, 1.0, 1.0]), resolution=16, levels=1)
    assert set(est.state_dict()) == {"resolution", "aabbs", "occs", "binaries"}
    # the keyword arguments the reference passes (nerf_renderer.py:145-155, nerf.py:161-168)
    sig = inspect.signature(est.sampling).parameters
    for k in ("sigma_fn", "near_plane", "far_plane", "render_step_size", "stratified", "cone_angle", "alpha_thre"):
        assert k in sig
    sig = inspect.signature(est.update_every_n_steps).parameters
    for k in ("step", "occ_eval_fn", "occ_thre", "ema_decay", "warmup_steps", "n"):
        assert k in sig
    from torch_efficient_distloss import flatten_eff_distloss
    assert hasattr(ours, "NeRFScene") and callable(flatten_eff_distloss)


def test_distloss_shim_matches_oracle():
    import oracle
    from perf_b200.shims import torch_efficient_distloss as dl
    g = torch.Generator().manual_seed(3)
    R, S = 6, 20
    w = (torch.rand(R * S, generator=g) / S).requires_grad_(True)
    ts, te = oracle.fixed_samples(R, S, 0.0, 1.0)
    m, iv = ((ts + te) / 2).reshape(-1), (te - ts).reshape(-1)
    ri = torch.arange(R).repeat_interleave(S)
    a = dl.flatten_eff_distloss(w, m, iv, ri)
    b = oracle.flatten_eff_distloss(w, m, iv, ri)
    assert torch.allclose(a, b, atol=1e-7)
    c = dl.eff_distloss(w.view(R, S), m.view(R, S), iv.view(R, S))
    assert torch.allclose(c, b, atol=1e-6)
    a.backward()
    assert torch.isfinite(w.grad).all()


class _Opt:
    def __init__(self):
        self.param_groups = [{"lr": 0.0}]


def test_lr_schedule_matches_reference(reference_api, tmp_path):
    """`NeRFScene.update_lr` (nerf.py:300-311) of the reference vs ours over the whole schedule,
    with the optimiser settings of configs/nerf.yaml read by our hydra-less loader."""
    from perf_b200.config import load_config
    from perf_b200.scene import NeRFScene as Ours
    conf = load_config(write_reference_configs(tmp_path, reference_api), "nerf")
    oc = conf.scene.train_conf.geo_optimizer
    assert (oc.init_lr, oc.peak_lr, oc.peak_at, oc.lr_alpha) == (0.0, 1e-2, 0.2, 1e-2)
    assert conf.scene.estimator_type == "occ" and conf.scene.train_conf.pixel_loss_batch_size == 8192
    assert conf.device.base_exp_dir == "."
    sched = reference_api["lr_schedule"]
    assert len(sched["progress"]) == len(range(0, 3000, 37))
    b = _Opt()
    for progress, want in zip(sched["progress"], sched["geo_optimizer_lr"]):
        Ours.update_lr(None, b, oc, progress)
        assert abs(want - b.param_groups[0]["lr"]) < 1e-12


def test_gen_occ_grid_and_batch_sampler_match_reference():
    """`SupInfoPool.gen_occ_grid` (sup_info.py:304-330) and the to_bounded_rays constants
    (nerf.py:313-319): the reference's functions ran on a stand-in `self` with these rays vs our RaySupervision."""
    from perf_b200.scene import RaySupervision, Rays, NeRFScene as Ours
    ref = np.load(os.path.join(GOLDEN, "reference_host.npz"))
    g = torch.Generator().manual_seed(0)
    n = 5000
    o = (torch.rand(n, 3, generator=g) - .5) * .2
    d = torch.nn.functional.normalize(torch.randn(n, 3, generator=g), dim=-1)
    dist = torch.rand(n, 1, generator=g) * .8 + .05
    pool = RaySupervision(Rays(o, d), torch.rand(n, 3, generator=g), dist)
    grid, pts = pool.gen_occ_grid(32)
    ref_grid, ref_pts = torch.from_numpy(ref["occ32_grid"]), torch.from_numpy(ref["occ32_pts"])
    assert grid.dtype == ref_grid.dtype and torch.equal(grid, ref_grid) and torch.equal(pts, ref_pts)
    br = Ours.to_bounded_rays(None, Rays(o, d))
    assert torch.equal(br.near, torch.from_numpy(ref["bounded_near"])) and torch.equal(br.far, torch.from_numpy(ref["bounded_far"]))
