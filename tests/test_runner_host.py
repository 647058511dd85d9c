"""CPU tests of the host-side callers of the path: pose samplers (against what the reference's own files
computed on the same distance map, tests/golden/reference_host.npz), dataset file formats, config -> runner
plumbing that does not need a GPU."""
import json
import os

import numpy as np
import pytest
import torch

from perf_b200 import pose_sampler as P
from perf_b200.synthetic import box_room_distance, smooth_rgb

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _distance_map(h=64, w=128):
    d = box_room_distance(h, w).reshape(h, w).clone()
    d[h // 2 - 3:h // 2 + 3, 10:14] = 0.0                       # a hole on the horizon: filled from its neighbours
    return d / (d.max() * 1.05)


def test_pose_samplers_match_reference_files():
    ref = np.load(os.path.join(GOLDEN, "reference_host.npz"))
    d = _distance_map()
    kw = dict(traverse_ratios=[0.2, 0.4, 0.6], n_anchors_per_ratio=[8, 8, 8])       # configs/nerf.yaml:16-18
    got = P.CirclePoseSampler(d.clone(), **kw)
    assert int(ref["circle_n_anchors"]) == got.n_anchors == 24 and got.n_poses == 24
    for name in ("plane_pts_raw", "plane_pts_filter", "plane_pts_smooth", "anchor_pts", "traverse_pts", "traverse_normals"):
        want = torch.from_numpy(ref[f"circle_{name}"])
        assert getattr(got, name).dtype == want.dtype and torch.equal(getattr(got, name), want), name
    assert torch.equal(torch.from_numpy(ref["circle_sample_pose_5"]), got.sample_pose(5))
    # anchors stay inside the room: closer to the origin than the wall in their direction
    assert got.anchor_pts.norm(dim=-1).max() < 0.7 * float(d.max())
    np.random.seed(0)
    dense_got = P.DenseTravelPoseSampler(got, n_dense_poses=12)
    dense_want = torch.from_numpy(ref["dense_sample_poses"])
    assert len(dense_want) == dense_got.n_poses and 10 <= dense_got.n_poses <= 14
    assert torch.equal(dense_want, dense_got.sample_poses)
    rot = dense_got.sample_poses[:, :3, :3]
    assert torch.allclose(rot @ rot.transpose(1, 2), torch.eye(3).expand_as(rot), atol=1e-5)


def test_wild_dataset_formats(tmp_path):
    import cv2
    from perf_b200.dataset import WildDataset, read_image
    h, w = 32, 64
    case = tmp_path / "room"
    case.mkdir()
    rgb = (smooth_rgb(h * 2, w * 2, seed=1) * 255).byte().numpy()
    cv2.imwrite(str(case / "image.png"), rgb[:, :, ::-1])
    dist = box_room_distance(h, w).reshape(h, w).numpy() * 3.0                  # metric scale: normalisation must remove it
    normal = np.zeros((h, w, 3), np.float32); normal[..., 2] = 1.0
    np.save(case / "image_ref_distance.npy", dist)
    np.save(case / "image_ref_normal.npy", normal)
    ds = WildDataset({"image_path": str(case / "image.png"), "image_resize": [w, h]}, device="cpu")
    assert ds.case_name == "room" and (ds.height, ds.width) == (h, w) and ds.image.shape == (h, w, 3)
    want_img = cv2.resize(read_image(str(case / "image.png")).numpy(), (w, h), cv2.INTER_AREA)
    assert np.array_equal(ds.image.numpy(), want_img)
    assert abs(float(ds.ref_distance.max()) - 1 / 1.05) < 1e-6                   # dataset.py:96-101
    # the normalised maps were written back and a point cloud exported (dataset.py:103-119)
    assert abs(float(np.load(case / "image_ref_distance.npy").max()) - 1 / 1.05) < 1e-6
    raw = (case / "image_ref_geometry.ply").read_bytes()
    head, _, body = raw.partition(b"end_header\n")
    assert b"element vertex %d" % (h * w) in head and b"property uchar alpha" in head and len(body) == h * w * 16
    pts = np.frombuffer(body, dtype=[("p", "<f4", 3), ("c", "u1", 4)])["p"]
    np.testing.assert_allclose(np.linalg.norm(pts, axis=-1).reshape(h, w), ds.ref_distance.numpy(), atol=1e-6)
    # missing reference geometry: the predictors are out of scope, say so
    os.remove(case / "image_ref_normal.npy")
    with pytest.raises(FileNotFoundError, match="predictors"):
        WildDataset({"image_path": str(case / "image.png")}, device="cpu")


def test_runner_config_plumbing_without_gpu(tmp_path):
    """The reference's YAML drives the runner unchanged; without a CUDA device constructing the scene fails loudly."""
    from perf_b200.config import load_config
    from test_shims_reference_import import write_reference_configs
    config_dir = write_reference_configs(tmp_path, json.load(open(os.path.join(GOLDEN, "reference_api.json"))))
    conf = load_config(config_dir, "nerf", ["exp_name=t", "scene.train_conf.raw_phase_iter_geo=10"])
    assert conf.scene.estimator_type == "occ" and conf.scene.train_conf.raw_phase_iter_geo == 10
    assert conf.pose_sampler.n_anchors_per_ratio == [8, 8, 8] and conf.device.base_exp_dir == "."
    assert conf.dataset.image_resize == [2048, 1024]


def test_inpainting_phase_loop_with_injected_priors(tmp_path, monkeypatch):
    """The orchestration of `core_exp_runner.py:126-177` (visibility -> inpaint -> geometric check -> mask arithmetic ->
    register -> re-fit -> checkpoint) with the scene and the 2-D priors replaced by CPU stand-ins."""
    from perf_b200 import runner as R
    from perf_b200.config import Conf
    from perf_b200.scene import Rays
    from perf_b200.sup_info import SupInfoPool, apply_rot, pano_dirs
    h, w = 32, 64
    dist0 = box_room_distance(h, w).reshape(h, w)
    dist0 = dist0 / (dist0.max() * 1.05)
    rgb0 = smooth_rgb(h, w, seed=3)

    def cpu_rays(pose, height, width, device="cpu"):
        pose = torch.as_tensor(pose, dtype=torch.float32)
        return Rays(pose[None, None, :3, 3].repeat(height, width, 1), apply_rot(pano_dirs(height, width, "cpu"), pose[:3, :3]))
    monkeypatch.setattr(R, "gen_pano_rays", cpu_rays)

    class FakeScene:
        fits = 0

        def get_pano_visibility_mask(self, pool, rays):
            m = torch.ones(h, w)
            m[8:20, 10:30] = 0.0                              # a region no registered panorama sees
            return m

        def render(self, rays, query_keys):
            return {"rgb": rgb0.clone(), "distance": dist0.clone()[..., None]}

        def fit(self, pool):
            FakeScene.fits += 1

        def set_train(self): pass
        def set_eval(self): pass
        def state_dict(self): return {"render": {}, "nerf": {}, "estimator": {}}

    class FakeInpainter:
        def inpaint(self, colors, mask):
            out = colors.clone()
            out[mask.squeeze() > 0.5] = torch.tensor([1.0, 0.0, 0.0])
            return out

    calls = []

    def fake_geo(img, distances, mask=None, reg_loss_weight=None, normal_loss_weight=None, normal_tv_loss_weight=None):
        calls.append((reg_loss_weight, normal_loss_weight, normal_tv_loss_weight))
        d = distances.clone()
        d[10:14, 12:20] = 0.05                                 # invented content too close to the camera: must be rejected
        return d, None

    class Anchors:
        n_anchors = 2

        def sample_pose(self, i):
            p = torch.eye(4)
            p[0, 3] = 0.05 * (i + 1)
            return p

    run = R.CoreRunner.__new__(R.CoreRunner)
    run.conf = Conf.wrap({"rgbd_inpaint": False})
    run.device, run.is_main, run.exp_dir, run.phase = torch.device("cpu"), True, str(tmp_path), 0
    run.dataset = type("D", (), {"height": h, "width": w})()
    run.scene, run.pose_sampler, run.inpainter, run.geo_predictor = FakeScene(), Anchors(), FakeInpainter(), fake_geo
    run.sup_pool = SupInfoPool(locality_sort=False)
    run.sup_pool.register_sup_info(pose=torch.eye(4), mask=torch.ones(h, w), rgb=rgb0, distance=dist0, normal=None)
    n0 = len(run.sup_pool.all_sup_colors)
    run.train()
    assert run.phase == 2 and FakeScene.fits == 2 and len(run.sup_pool.sup_infos) == 3
    assert calls == [(0., 5e-2, 5e-2)] * 2                       # the reference's keyword arguments (core_exp_runner.py:203-208)
    new = run.sup_pool.sup_infos[1]
    # only pixels that were invisible can become supervision, and the too-close invented block was rejected
    assert not new.mask_raw[:8].any() and not new.mask_raw[:, :10].any()
    assert not new.mask_raw[10:14, 12:20].any()
    assert len(run.sup_pool.all_sup_colors) > n0
    red = (new.sup_colors - torch.tensor([1.0, 0.0, 0.0])).abs().max()
    assert float(red) == 0.0                                      # the new supervision is exactly the inpainted content
    ck = torch.load(os.path.join(str(tmp_path), "checkpoints", "ckpt.pth"), weights_only=False)
    assert ck["phase"] == 2 and ck["sup_pool"]["n_sup_infos"] == 3
    for f in ("final_mask.jpg", "final_masked.jpg", "uninpainted_0.jpg", "mask_0.jpg", "inpainted_0.jpg", "aligned_disparity_0.jpg"):
        assert os.path.exists(os.path.join(str(tmp_path), "inpaint_vis", "0000", f)), f
    # resume: the pool saved at phase k comes back with its k+1 panoramas (ADVICE r1: it used to be dropped)
    FakeScene.load_state_dict = lambda self, sd: None
    n_all = len(run.sup_pool.all_sup_colors)
    run.sup_pool, run.phase = SupInfoPool(locality_sort=False), 0
    run.load_checkpoint("ckpt.pth")
    assert run.phase == 2 and len(run.sup_pool.sup_infos) == 3 and len(run.sup_pool.all_sup_colors) == n_all
    # without the priors the raw phase is all there is
    run.inpainter = None
    with pytest.raises(NotImplementedError, match="inpainter"):
        run.train()


def test_config_scalar_coercion_and_attribute_protocol(tmp_path):
    """ADVICE r1: only strings shaped like a float with an exponent (what PyYAML's YAML 1.1 misses: `1e-2`) become floats --
    `007`, names, dates stay strings -- and a missing key raises AttributeError (hasattr / deepcopy / pickle rely on it)."""
    import copy
    from perf_b200.config import Conf, load_config
    (tmp_path / "nerf.yaml").write_text("exp_name: '007'\nlr: 1e-2\nstep: 5e-4\nname: run_1e3x\nnested:\n  peak_lr: 1.5E-3\n  tag: '1_000'\n")
    conf = load_config(str(tmp_path), "nerf", ["nested.extra=3e-1"])
    assert conf.exp_name == "007" and conf.lr == 1e-2 and conf.step == 5e-4 and conf.name == "run_1e3x"
    assert conf.nested.peak_lr == 1.5e-3 and conf.nested.tag == "1_000" and conf.nested.extra == 0.3
    assert not hasattr(conf, "missing") and copy.deepcopy(conf).nested.peak_lr == 1.5e-3
    with pytest.raises(AttributeError):
        Conf.wrap({"a": 1}).b
