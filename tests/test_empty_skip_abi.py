"""CPU checks of empty-space skipping's interface (no GPU needed): the new C entry points are declared, exported and bound,
the occupancy map's size formula, the argument checks that run before any CUDA call, the Python signatures and the `MPI`
attribute, and the pass-through of the render service."""
import ctypes
import inspect
import os
import re

import numpy as np
import pytest
import torch

import ml_gmpi_b200 as g
from ml_gmpi_b200 import _lib, service
from conftest import ROOT

NEW = ["gmpi_mpi_occupancy_plane_words", "gmpi_mpi_occupancy", "gmpi_mpi_render_fwd_skip_ex"]


@pytest.fixture(scope="module")
def lib():
    g.build_library()
    return _lib.load()


def test_new_entry_points_are_declared_exported_and_listed(lib):
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "gmpi_mpi_render.h")).read(), flags=re.S)
    assert re.search(r"size_t gmpi_mpi_occupancy_plane_words\(int Ht, int Wt\);", hdr)
    assert re.search(r"int gmpi_mpi_occupancy\(const float\* alpha, long long mpi_stride, long long plane_stride, int M, int N, int Ht, "
                     r"int Wt, float threshold,\s*uint64_t\* occupancy, void\* stream\);", hdr)
    assert re.search(r"int gmpi_mpi_render_fwd_skip_ex\(const gmpi_render_desc\* desc, const uint64_t\* occupancy, "
                     r"uint64_t\* empty_pixel_planes\);", hdr)
    for s in NEW:
        assert s in _lib.EXPORTS and hasattr(lib, s)
    assert lib.gmpi_mpi_occupancy_plane_words.restype is ctypes.c_size_t


@pytest.mark.parametrize("ht,wt", [(1, 1), (8, 512), (9, 513), (100, 36), (37, 101), (1023, 1025), (1024, 1024), (7, 2049)])
def test_plane_words_formula(lib, ht, wt):
    assert lib.gmpi_mpi_occupancy_plane_words(ht, wt) == -(-ht // 8) * -(-wt // 512)
    assert lib.gmpi_mpi_occupancy_plane_words(0, wt) == 0 and lib.gmpi_mpi_occupancy_plane_words(ht, -1) == 0


def _desc(**kw):
    buf = (ctypes.c_float * 64)()
    p = ctypes.addressof(buf)
    base = dict(M=1, V=1, N=1, Ht=4, Wt=4, H=4, W=4, rgba=p, view2mpi=p, dhw=p, ray_dir=p, eye=p, z_dir=p, color=p, depth=p, flags=p)
    base.update(kw)
    return _lib.make_desc(**base), buf


def test_skip_forward_rejects_a_null_map_and_the_training_forward(lib):
    d, buf = _desc()
    words = (ctypes.c_uint64 * 4)()
    assert lib.gmpi_mpi_render_fwd_skip_ex(ctypes.byref(d), None, None) == 1
    assert b"null occupancy" in lib.gmpi_last_error()
    d.transmittance = ctypes.addressof(buf)
    assert lib.gmpi_mpi_render_fwd_skip_ex(ctypes.byref(d), ctypes.addressof(words), None) == 1
    assert b"transmittance buffer" in lib.gmpi_last_error() and b"inference only" in lib.gmpi_last_error()
    assert lib.gmpi_mpi_render_fwd_skip_ex(None, ctypes.addressof(words), None) == 1 and b"null descriptor" in lib.gmpi_last_error()
    d, _ = _desc()
    d.V = 0                 # nothing to render: a valid call returns before any CUDA call
    assert lib.gmpi_mpi_render_fwd_skip_ex(ctypes.byref(d), ctypes.addressof(words), None) == 0


@pytest.mark.parametrize("threshold", [float("nan"), -0.1, 1.0, float("inf")])
def test_occupancy_rejects_a_threshold_outside_0_1(lib, threshold):
    buf = (ctypes.c_float * 64)()
    words = (ctypes.c_uint64 * 4)()
    rc = lib.gmpi_mpi_occupancy(ctypes.addressof(buf), 64, 16, 1, 4, 4, 4, threshold, ctypes.addressof(words), None)
    assert rc == 1 and b"threshold" in lib.gmpi_last_error() and b"[0, 1)" in lib.gmpi_last_error()


def test_occupancy_rejects_null_pointers_and_bad_sizes(lib):
    buf = (ctypes.c_float * 64)()
    words = (ctypes.c_uint64 * 4)()
    assert lib.gmpi_mpi_occupancy(None, 64, 16, 1, 4, 4, 4, 0.0, ctypes.addressof(words), None) == 1
    assert lib.gmpi_mpi_occupancy(ctypes.addressof(buf), 64, 16, 1, 4, 4, 4, 0.0, None, None) == 1
    assert lib.gmpi_mpi_occupancy(ctypes.addressof(buf), 64, 16, 1, 0, 4, 4, 0.0, ctypes.addressof(words), None) == 1
    assert b"bad sizes" in lib.gmpi_last_error()


def test_signatures_and_the_mpi_attribute():
    for fn in (g.render_views, g.render_views_factored, g.render_frames):
        assert inspect.signature(fn).parameters["skip_alpha"].default is None
    assert inspect.signature(g.render_frames).parameters["skipped_empty"].default is None
    assert "skip_alpha" not in inspect.signature(g.MPI.__init__).parameters      # stop_transmittance stays the last parameter
    mpi = g.MPI()
    assert mpi.skip_alpha is None
    for ok in (0.0, 2.0 ** -12, 0.5, None):
        mpi.skip_alpha = ok
        assert mpi.skip_alpha == ok
    mpi.skip_alpha = 0.25
    for bad in (-0.1, 1.0, float("nan"), float("inf")):
        with pytest.raises(ValueError, match="skip_alpha"):
            mpi.skip_alpha = bad
    assert mpi.skip_alpha == 0.25                 # a rejected value leaves the attribute as it was


def test_render_frames_validates_before_rendering():
    cpu = torch.zeros(1, 1, 4, 8, 8)
    with pytest.raises(RuntimeError, match="CUDA devices only"):
        g.render_frames(rgba=cpu, dhw=torch.zeros(1, 1, 3), view2mpi=torch.zeros(1, dtype=torch.int32), skip_alpha=0.0)


def test_video_service_passes_skip_alpha_only_when_set():
    seen = []

    def fake(rgba, dhw, c2w, img_size, fov, near, far, fast, factored, **kw):
        seen.append(kw)
        V = c2w.shape[0]
        img = torch.zeros((V, img_size, img_size, 3), dtype=torch.uint8)
        return img, img[..., :1].contiguous()

    def fake_old(rgba, dhw, c2w, img_size, fov, near, far, fast, factored):      # a render function from before the parameter
        return fake(rgba, dhw, c2w, img_size, fov, near, far, fast, factored)

    kw = dict(img_size=4, fov_deg=12.6, ray_start=0.95, ray_end=1.12, sphere_center=np.array([0, 0, 1.0]), sphere_r=1.0)
    angles = service.sweep_angles(3, True)
    service.render_video_frames(None, torch.zeros(1, 2, 3), angles, render_fn=fake, skip_alpha=0.0, **kw)
    assert seen[-1] == {"skip_alpha": 0.0}
    service.render_video_frames(None, torch.zeros(1, 2, 3), angles, render_fn=fake, skip_alpha=2.0 ** -12,
                                stop_transmittance=2.0 ** -24, **kw)
    assert seen[-1] == {"skip_alpha": 2.0 ** -12, "stop_transmittance": 2.0 ** -24}
    service.render_video_frames(None, torch.zeros(1, 2, 3), angles, render_fn=fake_old, **kw)
    assert seen[-1] == {}
    assert inspect.signature(service.render_video_frames).parameters["skip_alpha"].default is None
    assert inspect.signature(service._default_video_render).parameters["skip_alpha"].default is None
