"""CPU checks of early ray termination's interface (no GPU needed): the appended descriptor fields in the header and the
ctypes mirror, descriptors from before them still accepted, the argument checks that run before any CUDA call, the Python signatures, and the
pass-through of the render service."""
import ctypes
import inspect
import json
import os
import re

import numpy as np
import pytest
import torch

import ml_gmpi_b200 as g
from ml_gmpi_b200 import _lib, service
from conftest import GOLDEN, ROOT


@pytest.fixture(scope="module")
def lib():
    g.build_library()
    return _lib.load()


def test_header_and_ctypes_have_the_termination_fields():
    hdr = open(os.path.join(ROOT, "include", "gmpi_mpi_render.h")).read()
    assert re.search(r"#define GMPI_ABI_VERSION 2\b", hdr) and _lib.ABI_VERSION == 2      # appended, backward compatible
    body = re.search(r"typedef struct gmpi_render_desc \{(.*?)\} gmpi_render_desc;", hdr, re.S).group(1)
    assert re.search(r"void\* stream;\s*float stop_transmittance;\s*uint64_t\* skipped_pixel_planes;\s*$", body)
    f = dict(_lib.RenderDesc._fields_)
    assert f["stop_transmittance"] is ctypes.c_float and f["skipped_pixel_planes"] is ctypes.c_void_p
    assert _lib.DESC_BYTES_WITHOUT_STOP == _lib.RenderDesc.stream.offset + ctypes.sizeof(ctypes.c_void_p)
    assert ctypes.sizeof(_lib.RenderDesc) == _lib.DESC_BYTES_WITHOUT_STOP + 16
    d = _lib.make_desc(stop_transmittance=0.25, skipped_pixel_planes=1234)
    assert d.stop_transmittance == 0.25 and d.skipped_pixel_planes == 1234


def _desc(**kw):
    buf = (ctypes.c_float * 64)()
    p = ctypes.addressof(buf)
    base = dict(M=1, V=1, N=1, Ht=4, Wt=4, H=4, W=4, rgba=p, view2mpi=p, dhw=p, ray_dir=p, eye=p, z_dir=p, color=p, depth=p, flags=p)
    base.update(kw)
    return _lib.make_desc(**base), buf


def test_descriptor_without_the_fields_passes_the_size_check(lib):
    d = _lib.make_desc(M=1, V=1, N=1, Ht=4, Wt=4, H=4, W=4)
    d.struct_bytes = _lib.DESC_BYTES_WITHOUT_STOP
    assert lib.gmpi_mpi_render_fwd_ex(ctypes.byref(d)) == 1
    err = lib.gmpi_last_error()
    assert b"null input" in err and b"struct_bytes" not in err
    # the fields beyond a short descriptor are not read: a tau that would be rejected is ignored
    d, _ = _desc(stop_transmittance=float("nan"))
    d.struct_bytes = _lib.DESC_BYTES_WITHOUT_STOP
    d.V = 0                  # nothing to render: returns before any CUDA call
    assert lib.gmpi_mpi_render_fwd_ex(ctypes.byref(d)) == 0
    d.struct_bytes = _lib.DESC_BYTES_WITHOUT_STOP + 8
    assert lib.gmpi_mpi_render_fwd_ex(ctypes.byref(d)) == 1 and b"struct_bytes" in lib.gmpi_last_error()


@pytest.mark.parametrize("tau", [float("nan"), -0.25, 1.0, 3.0, float("inf")])
def test_out_of_range_tau_is_rejected(lib, tau):
    d, _ = _desc(stop_transmittance=tau)
    assert lib.gmpi_mpi_render_fwd_ex(ctypes.byref(d)) == 1
    assert b"stop_transmittance" in lib.gmpi_last_error() and b"[0, 1)" in lib.gmpi_last_error()
    assert lib.gmpi_mpi_render_host_ex(ctypes.byref(d), 0) == 1 and b"[0, 1)" in lib.gmpi_last_error()


def test_tau_with_the_training_transmittance_is_rejected(lib):
    d, buf = _desc(stop_transmittance=2.0 ** -24)
    d.transmittance = ctypes.addressof(buf)
    assert lib.gmpi_mpi_render_fwd_ex(ctypes.byref(d)) == 1
    assert b"transmittance buffer" in lib.gmpi_last_error() and b"inference only" in lib.gmpi_last_error()


def test_tau_in_the_backward_is_rejected(lib):
    d, buf = _desc(stop_transmittance=1.0 / 512)
    d.g_color = d.g_rgba = ctypes.addressof(buf)
    assert lib.gmpi_mpi_render_bwd_ex(ctypes.byref(d)) == 1
    assert b"in the backward" in lib.gmpi_last_error()
    d.stop_transmittance = 0.0          # (control: with tau = 0 the same descriptor gets past the argument checks)
    d.V = 0
    assert lib.gmpi_mpi_render_bwd_ex(ctypes.byref(d)) in (0, 2)


def test_mpi_signature_keeps_the_reference_prefix():
    with open(os.path.join(GOLDEN, "reference_signatures.json")) as f:
        ref = json.load(f)["MPI"]["__init__"]
    ours = [[n, p.kind.name, repr(p.default)] for n, p in inspect.signature(g.MPI.__init__).parameters.items() if n != "self"]
    assert ours[: len(ref)] == ref
    assert ours[-1] == ["stop_transmittance", "POSITIONAL_OR_KEYWORD", "0.0"]
    assert [n for n, _, _ in ours].index("stop_transmittance") > [n for n, _, _ in ours].index("validate")
    for fn in (g.render_views, g.render_views_factored):
        assert inspect.signature(fn).parameters["stop_transmittance"].default == 0.0
    p = inspect.signature(g.render_frames).parameters
    assert p["stop_transmittance"].default == 0.0 and p["skipped"].default is None
    assert g.MPI(stop_transmittance=2.0 ** -24).stop_transmittance == 2.0 ** -24
    for bad in (-0.1, 1.0, float("nan")):
        with pytest.raises(ValueError, match="stop_transmittance"):
            g.MPI(stop_transmittance=bad)


def test_video_service_passes_tau_through():
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
    service.render_video_frames(None, torch.zeros(1, 2, 3), angles, render_fn=fake, stop_transmittance=2.0 ** -24, **kw)
    assert seen[-1] == {"stop_transmittance": 2.0 ** -24}
    service.render_video_frames(None, torch.zeros(1, 2, 3), angles, render_fn=fake_old, **kw)
    assert seen[-1] == {}
    assert inspect.signature(service._default_video_render).parameters["stop_transmittance"].default == 0.0
