"""The façade's generator-side helpers (MPIRenderer.get_xyz*, view_info_from_c2w_mat; gmpi/core/mpi_renderer.py:154-335)
against outputs of the unmodified reference (tests/golden/ffhq_xyz.npz, oracle/make_golden_xyz.py).  The plane table itself
is compared in test_host_geometry.py (<= 2e-6); here every array is rebuilt FROM that table with the reference's own fp32
operations, so the comparison is tight."""
import inspect
import json
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, load_golden
from ml_gmpi_b200 import geometry
from ml_gmpi_b200.renderer import MPIRenderer

KW = dict(plane_min_d=0.95, plane_max_d=1.12, plan_spatial_enlarge_factor=1.001, plane_distances_sample_method="inverse",
          cam_fov=12.6, sphere_center_z=1.0, sphere_r=1.0, horizontal_mean=0.0, horizontal_std=0.289, vertical_mean=0.0,
          vertical_std=0.127, cam_pose_n_truncated_stds=2, cam_sample_method="truncated_gaussian", use_confined_volume=True)
TOL = dict(rtol=3e-6, atol=3e-7)      # the table's 2e-6 + one rounding


@pytest.mark.parametrize("rng", ["-11", "01"])
def test_get_xyz_matches_reference(rng):
    ref = load_golden("ffhq_xyz")
    r = MPIRenderer(n_mpi_planes=8, use_normalized_xyz=True, normalized_xyz_range=rng, **KW)
    xyz, nxyz = r.get_xyz(16, 16)
    assert xyz.shape == (8, 16, 16, 3) and xyz.dtype == torch.float32
    np.testing.assert_allclose(xyz.numpy(), ref[f"xyz16_{rng}"], **TOL)
    np.testing.assert_allclose(nxyz.numpy(), ref[f"nxyz16_{rng}"], rtol=0, atol=3e-6)
    np.testing.assert_allclose(r.mpi_tex_pix_3d_coords.numpy(), ref[f"xyzd16_{rng}"], **TOL)
    assert r.mpi_tex_h == 16 and r.mpi_tex_w == 16
    z, nz = r.get_xyz(16, 16, only_z=True)
    np.testing.assert_allclose(z.numpy(), ref[f"z_{rng}"], **TOL)
    np.testing.assert_allclose(nz.numpy(), ref[f"nz_{rng}"], rtol=0, atol=3e-6)
    xd, nd = r.get_xyz(16, 16, ret_single_res=False)
    assert sorted(xd) == [4, 8, 16] == sorted(nd)
    for res in xd:
        np.testing.assert_allclose(xd[res].numpy(), ref[f"multi_xyz{res}_{rng}"], **TOL)
        np.testing.assert_allclose(nd[res].numpy(), ref[f"multi_nxyz{res}_{rng}"], rtol=0, atol=3e-6)
    # border texels sit ON the plane's edge (the align_corners=True convention of the sampler), normalised box is the last plane's
    dhw = r.static_mpi_plane_dhws
    assert torch.equal(xyz[:, 0, -1, 0], dhw[:, 2] / 2) and torch.equal(xyz[:, 0, 0, 1], -dhw[:, 1] / 2)
    lo = -1.0 if rng == "-11" else 0.0
    np.testing.assert_allclose(nxyz[-1, 0, 0].numpy(), [lo, lo, 1.0], atol=1e-6)


def test_get_xyz_from_the_reference_table_is_bit_identical():
    """Same fp32 operation sequence: fed the reference's own plane table, every output equals the reference's bit for bit."""
    ref, tab = load_golden("ffhq_xyz"), load_golden("ffhq_dhw")["n8"]
    r = MPIRenderer(n_mpi_planes=8, use_normalized_xyz=True, **KW)
    r.static_mpi_plane_dhws = r.dynamic_mpi_plane_dhws = torch.from_numpy(tab)
    xyz, nxyz = r.get_xyz(16, 16)
    assert np.array_equal(r.mpi_tex_pix_3d_coords.numpy(), ref["xyzd16_-11"])
    assert np.array_equal(nxyz.numpy(), ref["nxyz16_-11"])
    z, nz = r.get_xyz(16, 16, only_z=True)
    assert np.array_equal(z.numpy(), ref["z_-11"]) and np.array_equal(nz.numpy(), ref["nz_-11"])


def test_disparity_multi_res_and_cache():
    ref = load_golden("ffhq_xyz")
    r = MPIRenderer(n_mpi_planes=8, use_xyz_ztype="disparity", **KW)
    for _ in range(2):                                     # the cached tables are not inverted in place: a second call agrees
        xd, nd = r.get_xyz(8, 8, ret_single_res=False)
        assert nd[4] is None and nd[8] is None             # use_normalized_xyz=False
        np.testing.assert_allclose(xd[4].numpy(), ref["disp_xyz4"], **TOL)
        np.testing.assert_allclose(xd[8].numpy(), ref["disp_xyz8"], **TOL)
    a, _ = r.get_xyz(8, 8)
    b, _ = r.get_xyz(8, 8)
    assert a.data_ptr() == b.data_ptr()                    # built once (the reference rebuilds every resolution per iteration)
    assert float(a[0, 0, 0, 2]) == pytest.approx(0.95)     # single-res output stays metric depth
    r.dynamic_mpi_plane_dhws = r.static_mpi_plane_dhws * 2
    c, _ = r.get_xyz(8, 8)
    assert float(c[0, 0, 0, 2]) == pytest.approx(1.9)      # a new dynamic table invalidates the cache
    with pytest.raises(AssertionError, match="Only support square"):
        r.get_xyz(8, 16)
    with pytest.raises(AssertionError):
        r.get_xyz(12, 12)
    bad = MPIRenderer(n_mpi_planes=4, use_xyz_ztype="nope", **KW)
    with pytest.raises(ValueError):
        bad.get_xyz(8, 8, ret_single_res=False)


@pytest.mark.parametrize("s,t", [(8, 12), (32, 96), (8, 8), (96, 32)])
def test_interpolation_weights_match_reference(s, t):
    ref = load_golden("ffhq_xyz")[f"interp_{s}_{t}"]
    r = MPIRenderer(n_mpi_planes=4, **KW)
    ws = r.get_xyz_interpolate_ws(s, t)
    assert ws.shape == (t, s + 2) and ws.dtype == torch.float32
    assert np.array_equal(ws.numpy(), ref)
    assert int((ws != 0).sum(1).max()) <= 2
    np.testing.assert_allclose(ws.sum(1).numpy(), 1.0, atol=1e-5)
    # interpolating the source distances with the weights reproduces the target distances
    src = np.concatenate([[0], geometry.sample_distance(0.95, 1.12, s), [0]]).astype(np.float64)
    w = ws.numpy().astype(np.float64).copy()
    assert np.all(w[:, 0] == 0) and np.all(w[:-1, -1] == 0) and w[-1, -1] < 1e-6        # placeholder planes carry no weight
    np.testing.assert_allclose(w @ src, geometry.sample_distance(0.95, 1.12, t), rtol=2e-5)   # the 1e-8 in the denominator


def test_view_info_from_c2w_mat_matches_reference():
    ref = load_golden("ffhq_xyz")
    r = MPIRenderer(n_mpi_planes=4, **KW)
    r.set_cam(12.6, 12, 12)
    for c2w in (ref["vi_c2w"], torch.from_numpy(ref["vi_c2w"])):
        ray, eye, z, tf = r.view_info_from_c2w_mat(r.cam, c2w)
        assert ray.shape == (1, 3, 12, 12) and eye.shape == (1, 3) and z.shape == (1, 3) and tf.shape == (1, 4, 4)
        np.testing.assert_allclose(ray.numpy(), ref["vi_ray"], atol=2e-7)
        assert np.array_equal(eye.numpy(), ref["vi_eye"]) and np.array_equal(z.numpy(), ref["vi_z"])
        assert np.array_equal(tf.numpy(), ref["vi_tf"])


def test_facade_has_every_public_method_of_the_reference_with_its_signature():
    """tests/golden/reference_signatures.json: every function of the reference's MPIRenderer (oracle/make_golden_interface.py)."""
    with open(os.path.join(GOLDEN, "reference_signatures.json")) as f:
        ref = json.load(f)["MPIRenderer"]
    def params(fn):
        return [[n, p.kind.name, repr(p.default)] for n, p in inspect.signature(fn).parameters.items() if n != "self"]
    assert len(ref) > 1
    for name, rows in ref.items():
        if name == "__init__":
            continue
        assert hasattr(MPIRenderer, name), f"MPIRenderer.{name} missing"
        assert params(getattr(MPIRenderer, name)) == rows, name


@pytest.mark.parametrize("method", ["truncated_gaussian", "uniform", "normal"])
def test_seeded_random_poses_equal_the_reference(method):
    """Same torch seed -> the same cameras as the reference draws (RNG consumed in the same order and amounts:
    cam_utils.py:510-555, torch_utils.py:51-76), also on the second call from the same stream."""
    ref = load_golden("ffhq_xyz")
    r = MPIRenderer(n_mpi_planes=4, **dict(KW, cam_sample_method=method))
    r.set_cam(12.6, 8, 8)
    torch.manual_seed(3)
    y, p, c2w, rays, eyes, zs = r.sample_cam_poses(5, 0.0, 0.289, 0.0, 0.127, True)
    assert np.array_equal(y.numpy(), ref[f"rand_{method}_yaw"]) and np.array_equal(p.numpy(), ref[f"rand_{method}_pitch"])
    np.testing.assert_allclose(c2w.numpy(), ref[f"rand_{method}_c2w"], atol=2e-7)
    assert len(rays) == 5 and rays[0].shape == (1, 3, 8, 8) and eyes[0].shape == (1, 3) and zs[0].shape == (1, 3)
    y2, p2, *_ = r.sample_cam_poses(3, 0.1, 0.2, -0.05, 0.1, True)
    assert np.array_equal(y2.numpy(), ref[f"rand_{method}_yaw2"]) and np.array_equal(p2.numpy(), ref[f"rand_{method}_pitch2"])


def test_deterministic_sweep_equals_the_reference():
    ref = load_golden("ffhq_xyz")
    r = MPIRenderer(n_mpi_planes=4, **KW)
    r.set_cam(12.6, 8, 8)
    y, p, *_ = r.sample_cam_poses(5, 0.1, 0.289, 0.05, 0.127, False)
    assert np.array_equal(y.numpy(), ref["sweep_yaw"]) and np.array_equal(p.numpy(), ref["sweep_pitch"])


def test_light_renderer_draws_the_reference_light_from_the_same_seed():
    """LightRenderer.render blurs the depth (torchvision's GaussianBlur draws its sigma from torch's global generator: one
    uniform per call) and then samples the light with gen_sphere_path (light_renderer.py:112,136-149);
    tests/golden/light_2x6x32.npz recorded what the unmodified reference drew after torch.manual_seed(5).  The mirror must
    consume the generator identically, or every later draw of a seeded training run (lights, poses, latents) would differ."""
    from ml_gmpi_b200.light import LightRenderer, gaussian_blur
    ref = load_golden("light_2x6x32")
    lr = LightRenderer(sphere_center_z=1.0, sphere_r=1.0, ka_max=0.7, kd_max=0.6, n_grow_iters=10)
    img = torch.rand(2, 1, 32, 32, generator=torch.Generator().manual_seed(1))
    torch.manual_seed(5)
    blurred = lr._blur(img)                                   # what compute_pcl runs before the light is sampled
    assert torch.equal(blurred, gaussian_blur(img, lr.blur_ksize, lr.blur_sigma))
    d = lr.sample_light_directions(2, torch.device("cpu"))
    from ml_gmpi_b200.camera import sphere_poses
    c2w = sphere_poses(torch.from_numpy(ref["light_yaws"]).reshape(2, 1), torch.from_numpy(ref["light_pitches"]).reshape(2, 1),
                       (0, 0, 1.0), 1.0)
    want = torch.tensor([[0.0, 0.0, 1.0]]) - c2w[:, :3, 3]
    assert torch.equal(d, want / torch.norm(want, dim=-1, keepdim=True))
