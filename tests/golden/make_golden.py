"""Generate the golden fixtures in this directory from a checkout of the original PeRF project
(the reference): it imports the reference's own files, so the tests never need that checkout.

    python tests/golden/make_golden.py <path to the PeRF checkout>

What is the reference's own code and what is restated:

* ``raygen.npz``   -- `utils/camera_utils.py` (``gen_pano_rays``, imported unmodified; only
  ``trimesh.creation.icosphere`` is stubbed because trimesh is not installed and the
  symbol is unused on this path).
* ``field.npz``    -- `modules/fields/ngp_nerf.py` ``NGPNeRF.query_density/query_rgb``
  imported unmodified, running on a CPU stand-in for the un-vendored ``tinycudann``
  module whose arithmetic is ``oracle.network_forward`` (SURVEY.md Appendix A).
* ``render.npz``   -- `modules/scene/nerf_renderer.py` ``NeRFOCCRenderer.render`` imported
  unmodified, on CPU stand-ins for ``nerfacc`` (``oracle.composite``) and an estimator
  whose ``sampling`` returns the fixed-S intervals of ``oracle.sampler``.

* ``reference_host.npz`` / ``reference_api.json`` -- the host-side files the CPU tests compare
  with: `modules/pose_sampler/`, `modules/dataset/sup_info.py` (``kornia`` bound to the
  restatements in perf_b200/sup_info.py), ``NeRFScene.update_lr`` / ``gen_occ_grid`` /
  ``to_bounded_rays``, the tinycudann constructor calls of `modules/fields/ngp_nerf.py` and
  the names the reference imports from its three plugin packages, all run on the
  perf_b200 shims; plus the parsed YAML of `configs/nerf.yaml` and the defaults it selects.
* ``sup_info.npz`` -- a summary of the ``SupInfoPool`` of tests/test_sup_info.py.

So the glue (aabb normalise, selector, trunc_exp, sample-position rule, weights.detach,
background rules, dtype promotions) is pinned by the reference itself; the third-party
arithmetic is pinned only to our restatement ("parity unpinned", see oracle/__init__.py).
The field itself is NOT stored (2 x 6.6 M params): it is regenerated from
``oracle.Field.random(seed, grid_scale)`` -- torch's CPU generator is stable.
"""
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = None                                   # the PeRF checkout, from the command line
sys.path.insert(0, ROOT)

import oracle  # noqa: E402
from oracle.field import APP_MLP, GEO_MLP, PERF_GRID  # noqa: E402
from oracle.hashgrid import GridConfig  # noqa: E402
from oracle.mlp import MLPConfig  # noqa: E402

FIELD_SEED, FIELD_GRID_SCALE = 1337, 0.5


def install_stand_ins(mixed: bool):
    """CPU stand-ins for the reference's absent third-party imports."""
    trimesh = types.ModuleType("trimesh"); creation = types.ModuleType("trimesh.creation")
    creation.icosphere = lambda *a, **k: None
    trimesh.creation = creation
    sys.modules.update({"trimesh": trimesh, "trimesh.creation": creation})

    tcnn = types.ModuleType("tinycudann")

    class NetworkWithInputEncoding(torch.nn.Module):
        def __init__(self, n_input_dims, n_output_dims, encoding_config, network_config, seed=1337):
            super().__init__()
            self.grid = GridConfig.from_dict(encoding_config)
            self.mlp = MLPConfig.from_dict(network_config, self.grid.n_levels * self.grid.n_features_per_level,
                                           n_output_dims)
            n = oracle.field.network_param_count(self.grid, self.mlp)
            self.params = torch.nn.Parameter(torch.zeros(n))
            self.n_input_dims, self.n_output_dims = n_input_dims, n_output_dims

        def forward(self, x):
            y = oracle.field.network_forward(x, self.params, self.grid, self.mlp, mixed=mixed)
            return y.half() if mixed else y

    tcnn.NetworkWithInputEncoding = NetworkWithInputEncoding
    sys.modules["tinycudann"] = tcnn

    nerfacc = types.ModuleType("nerfacc")
    nerfacc.accumulate_along_rays = oracle.composite.accumulate_along_rays
    nerfacc.render_weight_from_density = oracle.composite.render_weight_from_density
    nerfacc.render_transmittance_from_alpha = lambda *a, **k: (_ for _ in ()).throw(NotImplementedError())
    est = types.ModuleType("nerfacc.estimators")
    prop = types.ModuleType("nerfacc.estimators.prop_net"); prop.PropNetEstimator = type("PropNetEstimator", (), {})
    occ = types.ModuleType("nerfacc.estimators.occ_grid"); occ.OccGridEstimator = type("OccGridEstimator", (), {})
    sys.modules.update({"nerfacc": nerfacc, "nerfacc.estimators": est,
                        "nerfacc.estimators.prop_net": prop, "nerfacc.estimators.occ_grid": occ})
    for m in [k for k in sys.modules if k.startswith("modules.") or k == "modules"]:
        del sys.modules[m]
    if REF not in sys.path:
        sys.path.insert(1, REF)


class FixedEstimator:
    """Stands where ``OccGridEstimator`` stands in ``NeRFOCCRenderer.render``; returns the
    packed fixed-S intervals."""
    def __init__(self, n_samples, near, far, jitter):
        self.S, self.near, self.far, self.jitter = n_samples, near, far, jitter

    def sampling(self, rays_o, rays_d, sigma_fn=None, stratified=False, **kw):
        R = rays_o.shape[0]
        ts, te = oracle.fixed_samples(R, self.S, self.near, self.far, self.jitter if stratified else None)
        ray_indices = torch.arange(R).repeat_interleave(self.S)
        return ray_indices, ts.reshape(-1), te.reshape(-1)


def rand_pose(g):
    q, _ = torch.linalg.qr(torch.randn(3, 3, generator=g))
    if torch.det(q) < 0:
        q[:, 0] = -q[:, 0]
    pose = torch.eye(4); pose[:3, :3] = q; pose[:3, 3] = (torch.rand(3, generator=g) - .5) * .4
    return pose


def make_raygen():
    install_stand_ins(True)
    from utils.camera_utils import gen_pano_rays
    g = torch.Generator().manual_seed(0)
    out = {}
    for name, (pose, h, w, rows) in {
        "eye_8x16": (torch.eye(4), 8, 16, None),
        "rot_6x10": (rand_pose(g), 6, 10, None),
        "rot_128x256": (rand_pose(g), 128, 256, [0, 1, 63, 64, 127]),
        "rot_1024x2048": (rand_pose(g), 1024, 2048, [0, 511, 1023]),
    }.items():
        rays = gen_pano_rays(pose, h, w)
        rows = list(range(h)) if rows is None else rows
        out[name + "_pose"] = pose.numpy(); out[name + "_hw"] = np.array([h, w])
        out[name + "_rows"] = np.array(rows)
        out[name + "_o"] = rays.o[rows].numpy(); out[name + "_d"] = rays.d[rows].numpy()
    from utils.camera_utils import gen_pers_rays
    for name, (pose, fov, res) in {"pers75_64": (rand_pose(g), float(np.deg2rad(75.)), 64), "pers90_33": (rand_pose(g), float(np.deg2rad(90.)), 33)}.items():
        rays = gen_pers_rays(pose, fov=fov, res=res)
        out[name + "_pose"], out[name + "_fov"], out[name + "_res"] = pose.numpy(), np.array(fov), np.array(res)
        out[name + "_o"], out[name + "_d"] = rays.o.numpy(), rays.d.numpy()
    np.savez_compressed(os.path.join(HERE, "raygen.npz"), **out)


def field_points(g, n):
    x = (torch.rand(n, 3, generator=g) * 2 - 1) * 1.1          # some outside the aabb
    x[:8] = torch.tensor([[0., 0., 0.], [1., 0., 0.], [-1., 0.5, 0.5], [0.999999, 0.2, -0.3],
                          [0.5, 0.5, 0.5], [-0.5, 0.25, 0.125], [1.0, 1.0, 1.0], [-1., -1., -1.]])
    return x


def make_field_and_render():
    out_f, out_r = {}, {}
    g = torch.Generator().manual_seed(1)
    x = field_points(g, 2048)
    R, S = 48, 32
    rays_o = (torch.rand(R, 3, generator=g) - .5) * .3
    rays_d = torch.nn.functional.normalize(torch.randn(R, 3, generator=g), dim=-1)
    jitter = torch.rand(R, generator=g)
    out_f["x"] = x.numpy()
    out_r.update(rays_o=rays_o.numpy(), rays_d=rays_d.numpy(), jitter=jitter.numpy(),
                 n_samples=np.array(S), near=np.array(1e-2), far=np.array(1.0))
    fld = oracle.Field.random(FIELD_SEED, FIELD_GRID_SCALE)
    for mixed in (True, False):
        tag = "mixed" if mixed else "fp32"
        install_stand_ins(mixed)
        from modules.fields.ngp_nerf import NGPNeRF
        from modules.scene.nerf_renderer import NeRFOCCRenderer
        nerf = NGPNeRF(aabb=torch.tensor([-1.0, -1.0, -1.0, 1.0, 1.0, 1.0]))
        with torch.no_grad():
            nerf.geo_mlp.params.copy_(fld.geo_params); nerf.app_mlp.params.copy_(fld.app_params)
            out_f[f"sigma_{tag}"] = nerf.query_density(x).numpy()
            out_f[f"rgb_{tag}"] = nerf.query_rgb(x).float().numpy()
            renderer = NeRFOCCRenderer(max_radius=2, bg_color="rand_noise")
            est = FixedEstimator(S, 1e-2, 1.0, jitter)
            near = 1e-2 * torch.ones(R, 1); far = torch.ones(R, 1)
            for mode in ("eval", "train"):
                nerf.train(mode == "train")
                torch.manual_seed(7)
                res = renderer.render(nerf, est, rays_o, rays_d, near, far)
                for k in ("rgb", "distance", "opacities", "weights", "trans"):
                    out_r[f"{mode}_{tag}_{k}"] = res[k].float().numpy()
            # the random numbers the training branch drew (nerf_renderer.py:185-192)
            torch.manual_seed(7)
            bg = torch.rand(R, 3); dn = torch.rand(R, 1)
            out_r["bg_noise"] = torch.cat([bg, dn], 1).numpy()
    out_f["seed"] = np.array(FIELD_SEED); out_f["grid_scale"] = np.array(FIELD_GRID_SCALE)
    np.savez_compressed(os.path.join(HERE, "field.npz"), **out_f)
    np.savez_compressed(os.path.join(HERE, "render.npz"), **out_r)


def install_host_stand_ins():
    """The perf_b200 plugin shims, ``kornia`` bound to perf_b200's restatements, and empty modules for the
    reference's third-party imports that the host-side files do not use on these paths."""
    from perf_b200 import shims
    from perf_b200 import sup_info as S
    for m in [k for k in sys.modules if k.split(".")[0] in ("modules", "utils", "tinycudann", "nerfacc")]:
        del sys.modules[m]
    shims.install()
    kornia = types.ModuleType("kornia"); filters = types.ModuleType("kornia.filters"); morph = types.ModuleType("kornia.morphology")
    filters.laplacian = lambda x, kernel_size: S.laplacian3(x) if kernel_size == 3 else None
    morph.erosion = lambda x, kernel: S.erosion(x, kernel)
    morph.dilation = lambda x, kernel: S.dilation(x, kernel)
    kornia.filters, kornia.morphology = filters, morph
    trimesh = types.ModuleType("trimesh"); creation = types.ModuleType("trimesh.creation")
    creation.icosphere = lambda *a, **k: None
    trimesh.creation = creation
    icecream = types.ModuleType("icecream"); icecream.ic = print
    sys.modules.update({"kornia": kornia, "kornia.filters": filters, "kornia.morphology": morph, "trimesh": trimesh,
                        "trimesh.creation": creation, "icecream": icecream})
    sys.modules.setdefault("imageio", types.ModuleType("imageio"))
    if REF not in sys.path:
        sys.path.insert(1, REF)


def shim_names_used():
    """{plugin package: sorted names} the reference's files import from it or read off it (``tcnn.X``)."""
    import ast
    out = {}
    for dirpath, _, files in os.walk(os.path.join(REF, "modules")):
        for f in files:
            if not f.endswith(".py"):
                continue
            tree = ast.parse(open(os.path.join(dirpath, f)).read())
            aliases = {}
            for node in ast.walk(tree):
                if isinstance(node, ast.ImportFrom) and node.module and node.module.split(".")[0] in ("nerfacc", "torch_efficient_distloss", "tinycudann"):
                    out.setdefault(node.module, set()).update(a.name for a in node.names)
                elif isinstance(node, ast.Import):
                    for a in node.names:
                        if a.name == "tinycudann":
                            aliases[a.asname or a.name] = a.name
            for node in ast.walk(tree):
                if isinstance(node, ast.Attribute) and isinstance(node.value, ast.Name) and node.value.id in aliases:
                    out.setdefault(aliases[node.value.id], set()).add(node.attr)
    return {k: sorted(v) for k, v in sorted(out.items())}


def make_reference_host():
    import hashlib
    import json
    import yaml
    from types import SimpleNamespace
    sys.path.insert(1, os.path.dirname(HERE))                        # tests/: the inputs the tests build
    import test_runner_host
    import test_sup_info as T
    install_host_stand_ins()
    arrays, api = {}, {}

    # -- tinycudann constructor calls of ngp_nerf.py, on the shim
    import tinycudann
    calls, shim_cls = [], tinycudann.NetworkWithInputEncoding

    class Recording(shim_cls):
        def __init__(self, *a, **k):
            kw = dict(zip(("n_input_dims", "n_output_dims", "encoding_config", "network_config"), a), **k)
            calls.append(kw)
            super().__init__(**kw)
    tinycudann.NetworkWithInputEncoding = Recording
    from modules.fields import ngp_nerf
    f = ngp_nerf.NGPNeRF(aabb=[-1.0, -1.0, -1.0, 1.0, 1.0, 1.0])
    api["tcnn_calls"] = {"NGPNeRF": calls[:]}
    api["nerf_state_dict"] = {k: {"shape": list(v.shape), "dtype": str(v.dtype)} for k, v in f.state_dict().items()}
    del calls[:]
    f.reset_geo()
    api["tcnn_calls"]["NGPNeRF.reset_geo"] = calls[:]
    del calls[:]
    try:
        ngp_nerf.NGPDensityField(aabb=[-1.0, -1.0, -1.0, 1.0, 1.0, 1.0])
    except RuntimeError:                                             # the shim refuses the proposal field's 10-wide input
        pass
    api["tcnn_calls"]["NGPDensityField"] = calls[:]
    tinycudann.NetworkWithInputEncoding = shim_cls
    api["shim_names"] = shim_names_used()
    from modules.scene import nerf_renderer
    from modules.scene import nerf as nerf_scene
    api["renderer_state_dict_keys"] = sorted(nerf_renderer.NeRFOCCRenderer(max_radius=2, bg_color="rand_noise").state_dict())

    # -- configs/nerf.yaml and the defaults it selects, parsed; the LR schedule of NeRFScene.update_lr on it
    root = yaml.safe_load(open(os.path.join(REF, "configs", "nerf.yaml")))
    api["configs"] = {"nerf.yaml": root}
    for item in root["defaults"]:
        for group, choice in (item.items() if isinstance(item, dict) else ()):
            api["configs"][f"{group}/{choice}.yaml"] = yaml.safe_load(open(os.path.join(REF, "configs", group, f"{choice}.yaml")))
    oc = SimpleNamespace(**{k: float(v) for k, v in root["scene"]["train_conf"]["geo_optimizer"].items()})
    opt = SimpleNamespace(param_groups=[{"lr": 0.0}])
    progress, lrs = [i / 3000 for i in range(0, 3000, 37)], []
    for p in progress:
        nerf_scene.NeRFScene.update_lr(None, opt, oc, p)
        lrs.append(opt.param_groups[0]["lr"])
    api["lr_schedule"] = {"progress": progress, "geo_optimizer_lr": lrs}

    # -- SupInfoPool.gen_occ_grid and to_bounded_rays (inputs of tests/test_shims_reference_import.py)
    from modules.dataset import sup_info as ref
    from utils.camera_utils import Rays as RefRays
    g = torch.Generator().manual_seed(0)
    n = 5000
    o = (torch.rand(n, 3, generator=g) - .5) * .2
    d = torch.nn.functional.normalize(torch.randn(n, 3, generator=g), dim=-1)
    dist = torch.rand(n, 1, generator=g) * .8 + .05
    grid, pts = ref.SupInfoPool.gen_occ_grid(SimpleNamespace(all_sup_rays=RefRays(o, d), all_sup_distances=dist), res=32)
    arrays["occ32_grid"], arrays["occ32_pts"] = grid.numpy(), pts.numpy()
    br = nerf_scene.NeRFScene.to_bounded_rays(None, RefRays(o, d))
    arrays["bounded_near"], arrays["bounded_far"] = br.near.numpy(), br.far.numpy()

    # -- pose samplers on the distance map of tests/test_runner_host.py (the reference hard-codes .cuda())
    saved_cuda = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self
    try:
        from modules.pose_sampler import circle_pose_sampler, dense_travel_pose_sampler
        circle = circle_pose_sampler.CirclePoseSampler(test_runner_host._distance_map(), traverse_ratios=[0.2, 0.4, 0.6],
                                                       n_anchors_per_ratio=[8, 8, 8])
        for name in ("plane_pts_raw", "plane_pts_filter", "plane_pts_smooth", "anchor_pts", "traverse_pts", "traverse_normals"):
            arrays[f"circle_{name}"] = getattr(circle, name).numpy()
        arrays["circle_n_anchors"] = np.array(circle.n_anchors)
        arrays["circle_sample_pose_5"] = circle.sample_pose(5).numpy()
        np.random.seed(0)
        arrays["dense_sample_poses"] = dense_travel_pose_sampler.DenseTravelPoseSampler(circle, n_dense_poses=12).sample_poses.numpy()
    finally:
        torch.Tensor.cuda = saved_cuda

    # -- SupInfoPool of tests/test_sup_info.py
    scene = T._scene()
    pool = T._pool(ref.SupInfoPool, *scene)
    for i, info in enumerate(pool.sup_infos):
        for name in T.POOL_INFO_FIELDS:
            arrays[f"pool{i}_{name}"] = getattr(info, name).numpy()
    arrays["pool_all_sup_colors"], arrays["pool_all_sup_dirs"] = pool.all_sup_colors.numpy(), pool.all_sup_rays.d.numpy()
    arrays["pool_all_sup_distances"], arrays["pool_all_sup_normals"] = pool.all_sup_distances.numpy(), pool.all_sup_normals.numpy()
    rays, distances = T._probe(pool, 40, 80, scene[4])
    arrays["pool_geo_check"] = pool.geo_check(ref.Rays(rays.o, rays.d), distances).numpy()
    grid, pts = pool.gen_occ_grid(32)
    arrays["pool_occ32_grid"], arrays["pool_occ32_pts"] = grid.numpy(), pts.numpy()
    torch.manual_seed(5)
    r, c, dd, nn = pool.rand_ray_color_data(64)
    arrays.update(pool_draw64_dirs=r.d.numpy(), pool_draw64_colors=c.numpy(), pool_draw64_distances=dd.numpy(), pool_draw64_normals=nn.numpy())
    for mode in ("only_first", "only_last"):
        torch.manual_seed(6)
        r, c, _, _ = pool.rand_ray_color_data(32, rand_mode=mode)
        arrays[f"pool_draw32_{mode}_dirs"], arrays[f"pool_draw32_{mode}_colors"] = r.d.numpy(), c.numpy()
    sd = pool.state_dict()
    api["sup_pool_state_dict_keys"] = {"pool": sorted(sd), "sup_info_0": sorted(sd["sup_info_0"])}
    np.savez_compressed(os.path.join(HERE, "sup_info.npz"), **T._golden_payload(T._pool(ref.SupInfoPool, *scene), scene))

    # the large float arrays of the pool are compared bit for bit: their digests keep the fixture small
    api["pool_sha256"] = {}
    for k in [k for k in arrays if k.startswith("pool") and arrays[k].dtype.kind == "f" and arrays[k].size >= 4096]:
        a = np.ascontiguousarray(arrays.pop(k))
        api["pool_sha256"][k] = {"shape": list(a.shape), "dtype": str(a.dtype), "sha256": hashlib.sha256(a.tobytes()).hexdigest()}
    np.savez_compressed(os.path.join(HERE, "reference_host.npz"), **arrays)
    with open(os.path.join(HERE, "reference_api.json"), "w") as fh:
        json.dump(api, fh, indent=1, sort_keys=True)
        fh.write("\n")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    REF = os.path.abspath(sys.argv[1])
    make_raygen()
    make_field_and_render()
    make_reference_host()
    for f in ("raygen.npz", "field.npz", "render.npz", "sup_info.npz", "reference_host.npz", "reference_api.json"):
        print(f, os.path.getsize(os.path.join(HERE, f)))
