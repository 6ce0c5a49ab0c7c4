"""GPU tests of early ray termination (gmpi_render_desc.stop_transmittance, the inference forward), once per forward kernel
variant (direct gather, TMA-staged).  The contract of include/gmpi_mpi_render.h: tau = 0 changes nothing; at tau > 0 every
output lies in [full - tau * max(value), full], pixels whose T stays >= tau up to the last plane are bit-identical, the result
and the skip count are deterministic; renders with a gradient stay exact."""
import ctypes

import numpy as np
import pytest
import torch

import ml_gmpi_b200 as g
from ml_gmpi_b200 import _lib, synth
from ml_gmpi_b200.geometry import FFHQ
from conftest import MPI_CASES, load_golden, rel_err

pytestmark = pytest.mark.gpu
EXPECT = 2e-5
TAUS = [2.0 ** -24, 1.0 / 512]


def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


@pytest.fixture(params=["direct", "staged"])
def fwd_variant(request):
    lib = _lib.load()
    _lib.check(lib.gmpi_debug_set_fwd_variant({"direct": 1, "staged": 2}[request.param]))
    yield request.param
    _lib.check(lib.gmpi_debug_set_fwd_variant(0))


def render(case=None, *, tau=0.0, short=False, trans=None, video=None, factored=None, options=_lib.OPT_ALIGN_CORNERS):
    """One forward through gmpi_mpi_render_fwd_ex.  short: the descriptor as it was before stop_transmittance existed.
    Returns (colour or uint8 frames, depth, skip count)."""
    d = dev()
    lib = _lib.load()
    ref = factored[1] if factored is not None else case.rgba
    M, N = ref.shape[0], ref.shape[1]
    Ht, Wt = ref.shape[-2:]
    V, _, H, W = case.ray_dir.shape
    skipped = torch.zeros(1, dtype=torch.int64, device=d)
    flags = torch.zeros(1, dtype=torch.int32, device=d)
    color = depth = v_rgb = v_depth = None
    if video:
        v_rgb = torch.empty((V, H, W, 3), dtype=torch.uint8, device=d)
        v_depth = torch.empty((V, H, W, 1), dtype=torch.uint8, device=d)
        options |= _lib.OPT_COLOR_MINUS1_1
    else:
        color = torch.empty((V, 3, H, W), device=d)
        depth = torch.empty((V, 1, H, W), device=d)
    mpi = dict(rgb=factored[0], alpha=factored[1]) if factored is not None else dict(rgba=case.rgba)
    desc = _lib.make_desc(options=options, M=M, V=V, N=N, Ht=Ht, Wt=Wt, H=H, W=W, view_group=1, view2mpi=case.view2mpi, dhw=case.dhw,
                          ray_dir=case.ray_dir, eye=case.eye, z_dir=case.z_dir, color=color, depth=depth, transmittance=trans,
                          video_rgb=v_rgb, video_depth=v_depth, depth_near=FFHQ["plane_min_d"],
                          depth_range=FFHQ["plane_max_d"] - FFHQ["plane_min_d"], flags=flags, stop_transmittance=tau,
                          skipped_pixel_planes=None if short else skipped, **mpi)
    if short:
        desc.struct_bytes = _lib.DESC_BYTES_WITHOUT_STOP
    _lib.check(lib.gmpi_mpi_render_fwd_ex(ctypes.byref(desc)))
    torch.cuda.synchronize()
    if video:
        return v_rgb, v_depth, int(skipped.item())
    return color, depth, int(skipped.item())


def full_case(kind, seed=3):
    # 2 MPIs x 1 view, 96 planes, 1024^2: the headline plane count and resolution
    return synth.make_workload(kind, n_planes=96, tex=1024, img=1024, n_mpi=2, views_per_mpi=1, seed=seed, device=dev())


def test_tau_zero_is_bit_identical_to_a_descriptor_without_the_field(fwd_variant):
    case = synth.make_workload("noise", n_planes=32, tex=256, img=512, n_mpi=2, seed=5, device=dev())
    for kw in (dict(), dict(video=True)):
        a = render(case, short=True, **kw)
        b = render(case, tau=0.0, **kw)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and b[2] == 0
    gen = torch.Generator(device=dev()).manual_seed(2)
    rgb = torch.rand((2, 3, 256, 256), generator=gen, device=dev())
    alpha = torch.rand((2, 32, 1, 256, 256), generator=gen, device=dev())
    alpha[:, -1] = 1.0
    a = render(case, short=True, factored=(rgb, alpha))
    b = render(case, tau=0.0, factored=(rgb, alpha))
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and b[2] == 0


@pytest.mark.parametrize("kind", ["noise", "surface"])
def test_termination_bounds_identity_and_determinism(kind, fwd_variant):
    case = full_case(kind)
    V, _, H, W = case.ray_dir.shape
    N = case.rgba.shape[1]
    trans = torch.empty((V, N, H, W), device=dev())
    c0, d0, _ = render(case, trans=trans)                    # exact, with the saved T_i of every plane
    t_last = trans[:, -1:]                                   # T in front of the last plane
    del trans
    empty = synth.make_workload("empty", n_planes=96, tex=1024, img=1024, n_mpi=2, seed=3, device=dev())
    _, d_far, s_empty = render(empty, tau=TAUS[0])           # depth of the last plane: the largest per-plane depth of a pixel
    assert s_empty == 0
    for tau in TAUS:
        c, d, s = render(case, tau=tau)
        dc, dd = c0 - c, d0 - d
        assert float(dc.min()) >= 0.0 and float(dd.min()) >= 0.0, (float(dc.min()), float(dd.min()))
        assert float(dc.max()) <= tau * 1.0 + 1e-6
        assert float((dd - tau * d_far).max()) <= 1e-6
        keep = (t_last >= tau)              # the surface MPI: everything off the head; white noise: few pixels, or none at 2^-24
        assert bool(keep.any()) or kind == "noise"
        assert torch.equal(torch.where(keep, c, 0), torch.where(keep, c0, 0)) and torch.equal(torch.where(keep, d, 0), torch.where(keep, d0, 0))
        c2, d2, s2 = render(case, tau=tau)
        assert torch.equal(c, c2) and torch.equal(d, d2) and s == s2
        assert s > 0
        assert s <= V * H * W * N


def test_opaque_front_plane_ends_every_ray(fwd_variant):
    d = dev()
    N, S = 96, 1024
    case = synth.make_case(n_planes=N, tex=S, img=S, n_mpi=2, seed=9, device=d, yaws=np.zeros(2, np.float32),
                           pitches=np.zeros(2, np.float32))
    case.rgba[:, :, 3] = 1.0
    V, _, H, W = case.ray_dir.shape
    one = synth.Case(**{k: getattr(case, k) for k in case.__dataclass_fields__})     # plane 0 alone, as a one-plane MPI
    one.rgba = case.rgba[:, :1].contiguous()
    one.dhw = case.dhw[:, :1].contiguous()
    c1, d1, _ = render(one)
    for tau in TAUS:
        c, dp, s = render(case, tau=tau)
        # plane 0 up to the fp32 rounding of its bilinear weights: along the image border they sum to 1 - 2^-24, which leaves
        # T ~ 2^-24 behind plane 0 there (those rays stop one plane later)
        assert float((c - c1).abs().max()) <= 1e-6 and float((dp - d1).abs().max()) <= 1e-6
        assert s >= (N - 4) * H * W * V, (s, (N - 4) * H * W * V)


def test_video_frames_at_tau_equal_the_conversion_of_the_fp32_frames(fwd_variant):
    d = dev()
    case = synth.make_workload("surface", n_planes=96, tex=512, img=512, n_mpi=1, views_per_mpi=5, seed=12, device=d,
                               yaws=np.linspace(0.5, -0.5, 5).astype(np.float32), pitches=np.zeros(5, np.float32))
    near, far = FFHQ["plane_min_d"], FFHQ["plane_max_d"]
    tau = 1.0 / 512
    sk_f = torch.zeros(1, dtype=torch.int64, device=d)
    sk_v = torch.zeros(1, dtype=torch.int64, device=d)
    c, dp = g.render_frames(rgba=case.rgba, dhw=case.dhw, view2mpi=case.view2mpi, ray_dir=case.ray_dir, eye=case.eye, z_dir=case.z_dir,
                            stop_transmittance=tau, skipped=sk_f)
    u8, d8 = g.render_frames(rgba=case.rgba, dhw=case.dhw, view2mpi=case.view2mpi, ray_dir=case.ray_dir, eye=case.eye, z_dir=case.z_dir,
                             video={"near": near, "far": far}, stop_transmittance=tau, skipped=sk_v)
    img = ((c.permute(0, 2, 3, 1).cpu().numpy() + 1) / 2.0 * 255).astype(np.uint8)          # render_video.py:118-126
    dm = np.clip((dp.permute(0, 2, 3, 1).cpu().numpy() - near) / (far - near), 0, 1)
    assert np.array_equal(u8.cpu().numpy(), img) and np.array_equal(d8.cpu().numpy(), (dm * 255).astype(np.uint8))
    assert int(sk_f.item()) == int(sk_v.item()) > 0


def test_renders_with_a_gradient_stay_exact(fwd_variant):
    d = dev()
    case = synth.make_workload("noise", n_planes=32, tex=256, img=512, n_mpi=2, seed=6, device=d)
    rays, eyes, zs = [case.ray_dir[i:i + 1] for i in range(2)], [case.eye[i:i + 1] for i in range(2)], [case.z_dir[i:i + 1] for i in range(2)]
    gen = torch.Generator(device=d).manual_seed(1)
    gc = torch.randn((2, 3, 512, 512), generator=gen, device=d)
    out = []
    for tau in (0.0, 1.0 / 512):
        rgba = case.rgba.clone().requires_grad_(True)
        mpi = g.MPI(align_corners=True, validate="off", stop_transmittance=tau)
        c, dp = mpi(batch_rgba=rgba, batch_dhw=case.dhw, batch_ray_dir=rays, batch_eye_pos=eyes, batch_z_dir=zs, separate_background=None)
        ((c * gc).sum() + dp.sum()).backward()
        out.append((c.detach(), dp.detach(), rgba.grad))
    assert torch.equal(out[0][0], out[1][0]) and torch.equal(out[0][1], out[1][1])
    assert rel_err(out[1][2].cpu().numpy(), out[0][2].cpu().numpy()) <= 1e-6        # atomics: summation order only
    # the same MPI object without a gradient does terminate
    mpi = g.MPI(align_corners=True, validate="off", stop_transmittance=1.0 / 512)
    with torch.no_grad():
        c, _ = mpi(batch_rgba=case.rgba, batch_dhw=case.dhw, batch_ray_dir=rays, batch_eye_pos=eyes, batch_z_dir=zs, separate_background=None)
    assert not torch.equal(c, out[0][0]) and float((out[0][0] - c).min()) >= 0.0


@pytest.mark.parametrize("name", MPI_CASES)
def test_reference_goldens_at_tau_2_pow_minus_24(name, fwd_variant):
    gd = load_golden(name)
    d = dev()
    v2m = gd["view2mpi"]
    t = lambda a: torch.from_numpy(a).to(d)
    idx = [np.nonzero(v2m == m)[0] for m in range(gd["rgba"].shape[0])]
    mpi = g.MPI(align_corners=bool(gd["align_corners"]), validate="defer", stop_transmittance=2.0 ** -24)
    color, depth = mpi(batch_rgba=t(gd["rgba"]), batch_dhw=t(gd["dhw"]), batch_ray_dir=[t(gd["ray_dir"][i]) for i in idx],
                       batch_eye_pos=[t(gd["eye"][i]) for i in idx], batch_z_dir=[t(gd["z_dir"][i]) for i in idx],
                       separate_background=None)
    ec, ed = rel_err(color.cpu().numpy(), gd["color"]), rel_err(depth.cpu().numpy(), gd["depth"])
    assert ec <= EXPECT and ed <= EXPECT, (ec, ed)


def test_host_entry_point_honours_tau_and_returns_the_count():
    d = dev()
    case = synth.make_workload("noise", n_planes=32, tex=256, img=512, n_mpi=2, seed=7, device=d)
    tau = 1.0 / 512
    c_dev, d_dev, s_dev = render(case, tau=tau)
    h = case.to("cpu")
    V, _, H, W = h.ray_dir.shape
    color = torch.empty((V, 3, H, W))
    depth = torch.empty((V, 1, H, W))
    flags = ctypes.c_uint32(0)
    skipped = ctypes.c_uint64(5)
    desc = _lib.make_desc(options=_lib.OPT_ALIGN_CORNERS, M=2, V=V, N=32, Ht=256, Wt=256, H=H, W=W, rgba=h.rgba, view2mpi=h.view2mpi,
                          dhw=h.dhw, ray_dir=h.ray_dir, eye=h.eye, z_dir=h.z_dir, color=color, depth=depth,
                          flags=ctypes.addressof(flags), stop_transmittance=tau, skipped_pixel_planes=ctypes.addressof(skipped))
    _lib.check(_lib.load().gmpi_mpi_render_host_ex(ctypes.byref(desc), 0))
    assert skipped.value - 5 == s_dev > 0                   # accumulated into
    assert torch.equal(color, c_dev.cpu()) and torch.equal(depth, d_dev.cpu())
