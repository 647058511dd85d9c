"""CPU tests of perf_b200/sup_info.py (SURVEY.md §8(f) row 3).

* the three kornia 0.7.0 functions restated there are pinned against OpenCV (an independent
  implementation of the same filters);
* ``PanoSupInfo`` / ``SupInfoPool`` are compared with what the reference's OWN `modules/dataset/sup_info.py`,
  imported unmodified with ``kornia`` bound to those restatements, computed on the same inputs: the
  fixtures ``tests/golden/reference_host.npz`` / ``reference_api.json`` and the summary
  ``tests/golden/sup_info.npz`` (all minted by tests/golden/make_golden.py).
"""
import hashlib
import json
import os

import cv2
import numpy as np
import pytest
import torch

from perf_b200 import sup_info as S
from perf_b200.synthetic import box_room_distance, smooth_rgb

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "sup_info.npz")
REFERENCE_HOST = os.path.join(os.path.dirname(__file__), "golden", "reference_host.npz")
REFERENCE_API = os.path.join(os.path.dirname(__file__), "golden", "reference_api.json")
POOL_INFO_FIELDS = ("mask_raw", "mask", "color_map", "distance_map", "normal_map", "sup_colors", "sup_distances",
                    "sup_normals", "sup_dirs", "sup_positions", "pose")


# ------------------------------------------------------------------ kornia restatements vs OpenCV
def test_laplacian_matches_opencv():
    g = torch.Generator().manual_seed(0)
    x = torch.rand(1, 1, 37, 53, generator=g)
    k = np.ones((3, 3), np.float32); k[1, 1] = -8.0; k /= 16.0
    want = cv2.filter2D(x[0, 0].numpy(), cv2.CV_32F, k, borderType=cv2.BORDER_REFLECT_101)
    np.testing.assert_allclose(S.laplacian3(x)[0, 0].numpy(), want, atol=1e-6)


@pytest.mark.parametrize("size", [3, 5, 9])
def test_morphology_and_ellipse_match_opencv(size):
    g = torch.Generator().manual_seed(size)
    x = (torch.rand(1, 1, 41, 67, generator=g) > 0.6).float()
    ell = cv2.getStructuringElement(cv2.MORPH_ELLIPSE, (size, size))
    assert np.array_equal(S.ellipse_kernel(size).numpy().astype(np.uint8), ell)
    for kern in (np.ones((size, size), np.uint8), ell):
        kt = torch.from_numpy(kern).float()
        # OpenCV's default border for erode / dilate is +inf / -inf: the border never wins (kornia 'geodesic')
        np.testing.assert_array_equal(S.erosion(x, kt)[0, 0].numpy(), cv2.erode(x[0, 0].numpy(), kern))
        np.testing.assert_array_equal(S.dilation(x, kt)[0, 0].numpy(), cv2.dilate(x[0, 0].numpy(), kern))
    # an asymmetric element: kornia's dilation reflects it (the set-theoretic definition), OpenCV's does not.
    # (The reference only passes symmetric elements: ones(3,3) and OpenCV ellipses.)
    asym = np.array([[1, 1, 0], [0, 1, 0], [0, 0, 0]], np.uint8)
    np.testing.assert_array_equal(S.dilation(x, torch.from_numpy(asym).float())[0, 0].numpy(),
                                  cv2.dilate(x[0, 0].numpy(), np.ascontiguousarray(asym[::-1, ::-1])))
    np.testing.assert_array_equal(S.erosion(x, torch.from_numpy(asym).float())[0, 0].numpy(), cv2.erode(x[0, 0].numpy(), asym))


# ------------------------------------------------------------------ scene shared by the comparisons
def _scene(h=48, w=96):
    rgb, dist = smooth_rgb(h, w, seed=2), box_room_distance(h, w)
    g = torch.Generator().manual_seed(4)
    dist = dist.reshape(h, w).clone()
    dist[10:20, 30:50] *= 0.6                                  # a depth edge the Laplacian mask must remove
    mask = torch.ones(h, w)
    mask[30:40, 5:25] = 0.0
    dirs = S.pano_dirs(h, w, "cpu")
    normal = -dirs + 0.3 * torch.randn(h, w, 3, generator=g)   # mostly facing the camera, some grazing
    normal = normal / normal.norm(dim=-1, keepdim=True)
    a = 0.4
    pose2 = torch.tensor([[np.cos(a), -np.sin(a), 0, 0.1], [np.sin(a), np.cos(a), 0, -0.05], [0, 0, 1, 0.02], [0, 0, 0, 1]], dtype=torch.float32)
    return rgb.reshape(h, w, 3), dist, mask, normal, pose2


def _pool(mod_pool_cls, rgb, dist, mask, normal, pose2):
    pool = mod_pool_cls()
    pool.register_sup_info(pose=torch.eye(4), mask=mask, rgb=rgb, distance=dist, normal=normal)
    pool.register_sup_info(pose=pose2, mask=mask.flip(1), rgb=rgb.flip(0), distance=dist * 0.9, normal=None)
    return pool


def _probe(pool, h, w, pose):
    """geo_check of a novel panorama's rays at a synthetic distance."""
    from perf_b200.scene import Rays
    dirs = S.apply_rot(S.pano_dirs(h, w, "cpu"), pose[:3, :3])
    rays = Rays(pose[None, None, :3, 3].repeat(h, w, 1), dirs)
    g = torch.Generator().manual_seed(9)
    distances = 0.2 + 0.5 * torch.rand(h, w, generator=g)
    return rays, distances


def test_pool_matches_reference_file():
    arrays, api = np.load(REFERENCE_HOST), json.load(open(REFERENCE_API))

    def _same(got: torch.Tensor, key: str, name: str):
        """Bit-identical to the reference's array (stored, or as shape, dtype and SHA-256 of its bytes)."""
        if key in arrays.files:
            want = torch.from_numpy(arrays[key])
            assert got.dtype == want.dtype and torch.equal(got, want), name
        else:
            a = np.ascontiguousarray(got.numpy())
            assert api["pool_sha256"][key] == {"shape": list(a.shape), "dtype": str(a.dtype),
                                               "sha256": hashlib.sha256(a.tobytes()).hexdigest()}, name
    scene = _scene()
    got = _pool(lambda: S.SupInfoPool(locality_sort=False), *scene)
    for i, b in enumerate(got.sup_infos):
        for name in POOL_INFO_FIELDS:
            _same(getattr(b, name), f"pool{i}_{name}", f"{name} of panorama {i}")
    assert 0.3 < got.sup_infos[0].mask.float().mean() < 0.95          # the masks do remove something
    _same(got.all_sup_colors, "pool_all_sup_colors", "all_sup_colors")
    _same(got.all_sup_rays.d, "pool_all_sup_dirs", "all_sup_rays.d")
    _same(got.all_sup_distances, "pool_all_sup_distances", "all_sup_distances")
    _same(got.all_sup_normals, "pool_all_sup_normals", "all_sup_normals")
    # geo_check on a novel view
    rays, distances = _probe(got, 40, 80, scene[4])
    m_got = got.geo_check(rays, distances)
    _same(m_got, "pool_geo_check", "geo_check")
    assert 0.02 < m_got.mean() < 0.98
    # occupancy pre-grid
    g_got, p_got = got.gen_occ_grid(32)
    _same(g_got, "pool_occ32_grid", "gen_occ_grid")
    _same(p_got, "pool_occ32_pts", "gen_occ_grid points")
    # batch sampler: the same draw from the same generator state
    got.use_default_generator = True
    torch.manual_seed(5)
    r_g, c_g, d_g, n_g = got.rand_ray_color_data(64)
    _same(r_g.d, "pool_draw64_dirs", "draw dirs")
    _same(c_g, "pool_draw64_colors", "draw colors")
    _same(d_g, "pool_draw64_distances", "draw distances")
    _same(n_g, "pool_draw64_normals", "draw normals")
    for mode in ("only_first", "only_last"):
        torch.manual_seed(6); b = got.rand_ray_color_data(32, rand_mode=mode)
        _same(b[1], f"pool_draw32_{mode}_colors", mode)
        _same(b[0].d, f"pool_draw32_{mode}_dirs", mode)
    # checkpoint keys (incl. the reference's unformatted height / width keys)
    keys = api["sup_pool_state_dict_keys"]
    assert sorted(got.state_dict()) == keys["pool"]
    assert sorted(got.state_dict()["sup_info_0"]) == keys["sup_info_0"]


def _golden_payload(pool, scene):
    rays, distances = _probe(pool, 40, 80, scene[4])
    occ, _ = pool.gen_occ_grid(32)
    return {"mask0": pool.sup_infos[0].mask.numpy(), "mask1": pool.sup_infos[1].mask.numpy(),
            "n_sup": np.array([len(i.sup_colors) for i in pool.sup_infos]),
            "color_sum": pool.all_sup_colors.double().sum(0).numpy(), "dir_sum": pool.all_sup_rays.d.double().sum(0).numpy(),
            "geo_check": pool.geo_check(rays, distances).numpy(), "occ_idx": torch.where(occ > 0)[0].numpy()}


def test_pool_matches_golden_fixture():
    """The fixture was written from the reference's own file (tests/golden/make_golden.py)."""
    scene = _scene()
    got = _golden_payload(_pool(lambda: S.SupInfoPool(locality_sort=False), *scene), scene)
    want = np.load(GOLDEN)
    for k in ("mask0", "mask1", "n_sup", "geo_check", "occ_idx"):
        np.testing.assert_array_equal(got[k], want[k], err_msg=k)
    for k in ("color_sum", "dir_sum"):
        np.testing.assert_allclose(got[k], want[k], rtol=1e-9, err_msg=k)


def test_locality_sort_keeps_the_multiset_and_checkpoint_roundtrip():
    scene = _scene()
    plain, sorted_ = _pool(lambda: S.SupInfoPool(locality_sort=False), *scene), _pool(lambda: S.SupInfoPool(locality_sort=True), *scene)
    plain.use_default_generator = sorted_.use_default_generator = True
    torch.manual_seed(11); a = plain.rand_ray_color_data(256)
    torch.manual_seed(11); b = sorted_.rand_ray_color_data(256)
    key = lambda t: t[torch.argsort(t[:, 0] * 7 + t[:, 1] * 3 + t[:, 2])]
    assert torch.equal(key(a[1]), key(b[1])) and not torch.equal(a[1], b[1])
    restored = S.SupInfoPool(locality_sort=True)
    restored.load_state_dict(sorted_.state_dict())
    assert torch.equal(restored.all_sup_colors, sorted_.all_sup_colors) and torch.equal(restored.locality_key, sorted_.locality_key)
    assert torch.equal(restored.all_sup_rays.d, sorted_.all_sup_rays.d)
    # visibility: a point on the registered surface is visible from its own panorama
    info = sorted_.sup_infos[0]
    from perf_b200.scene import Rays
    rays = Rays(torch.zeros(info.height, info.width, 3), S.pano_dirs(info.height, info.width, "cpu"))
    vis = sorted_.pano_visibility_mask(rays, info.distance_map)
    assert vis[info.mask[..., 0]].mean() > 0.9
    far_vis = sorted_.pano_visibility_mask(rays, info.distance_map * 1.5)          # behind the surface: hidden
    assert far_vis.mean() < 0.2


def test_factor_downsampling_is_opencv_inter_area():
    """`PanoSupInfo(factor=2)` (`sup_info.py:54-66`): the reference resizes with cv.INTER_AREA; for an integer factor
    that is the box average torch's 'area' mode computes."""
    rgb, dist, mask, normal, _ = _scene(32, 64)
    info = S.PanoSupInfo(torch.eye(4), mask, rgb, dist, normal, factor=2)
    assert (info.height, info.width) == (16, 32)
    want = cv2.resize(rgb.numpy(), (32, 16), interpolation=cv2.INTER_AREA)
    np.testing.assert_allclose(info.color_map.numpy(), want, atol=1e-6)
    want_d = cv2.resize(dist.numpy(), (32, 16), interpolation=cv2.INTER_AREA)
    np.testing.assert_allclose(info.distance_map[..., 0].numpy(), want_d, atol=1e-6)
    assert info.mask.shape == (16, 32, 1) and len(info.sup_colors) == int(info.mask.sum())
