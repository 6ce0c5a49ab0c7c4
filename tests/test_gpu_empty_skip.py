"""GPU tests of empty-space skipping (gmpi_mpi_occupancy + gmpi_mpi_render_fwd_skip_ex, the inference forward).  The contract
of include/gmpi_mpi_render.h: the occupancy map is one bit per 8x8 texels, set iff |alpha| > threshold or NaN; threshold 0
gives output bit-identical to gmpi_mpi_render_fwd_ex on the same descriptor (with early ray termination too, count included);
threshold eps moves every output by at most N * eps * max(value); the result and the count are deterministic; the direct
kernel ignores the map."""
import ctypes

import numpy as np
import pytest
import torch

import ml_gmpi_b200 as g
from ml_gmpi_b200 import _lib, synth
from ml_gmpi_b200.camera import cam_params, focal_from_fov
from ml_gmpi_b200.geometry import FFHQ
from conftest import MPI_CASES, load_golden, rel_err

pytestmark = pytest.mark.gpu
EXPECT = 2e-5
EPS = 2.0 ** -12
TAU = 2.0 ** -24


def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


@pytest.fixture
def staged():
    """Forces the TMA-staged kernel (small shapes would get the direct one), then restores auto."""
    lib = _lib.load()
    _lib.check(lib.gmpi_debug_set_fwd_variant(2))
    yield
    _lib.check(lib.gmpi_debug_set_fwd_variant(0))


@pytest.fixture(params=["direct", "staged"])
def fwd_variant(request):
    lib = _lib.load()
    _lib.check(lib.gmpi_debug_set_fwd_variant({"direct": 1, "staged": 2}[request.param]))
    yield request.param
    _lib.check(lib.gmpi_debug_set_fwd_variant(0))


def bits(t):
    return t.contiguous().view(torch.int32) if t.dtype == torch.float32 else t


def same(a, b):
    """Bit-identical (NaN in the same places with the same bits)."""
    return a.shape == b.shape and torch.equal(bits(a), bits(b))


def render(case, *, skip=None, tau=0.0, out="fp32", factored=None, cam=None, group=1):
    """One forward through the descriptor entry points: gmpi_mpi_render_fwd_ex, or with skip = threshold the occupancy map of
    the MPI and gmpi_mpi_render_fwd_skip_ex.  out: "fp32", "m11" (2c-1) or "video" (uint8).
    Returns (colour or uint8 frames, depth, termination count, empty count)."""
    d = dev()
    lib = _lib.load()
    rgba = None if factored is not None else case.rgba
    ref = factored[1] if factored is not None else rgba
    M, N = ref.shape[0], ref.shape[1]
    Ht, Wt = ref.shape[-2:]
    if cam is not None:
        V, H, W = cam.shape[0], case.ray_dir.shape[2], case.ray_dir.shape[3]
        rays = dict(cam=cam)
    else:
        V, _, H, W = case.ray_dir.shape
        rays = dict(ray_dir=case.ray_dir, eye=case.eye, z_dir=case.z_dir)
    counts = torch.zeros(2, dtype=torch.int64, device=d)
    flags = torch.zeros(1, dtype=torch.int32, device=d)
    color = depth = v_rgb = v_depth = None
    options = _lib.OPT_ALIGN_CORNERS
    if out == "video":
        v_rgb = torch.empty((V, H, W, 3), dtype=torch.uint8, device=d)
        v_depth = torch.empty((V, H, W, 1), dtype=torch.uint8, device=d)
        options |= _lib.OPT_COLOR_MINUS1_1
    else:
        color = torch.empty((V, 3, H, W), device=d)
        depth = torch.empty((V, 1, H, W), device=d)
        if out == "m11":
            options |= _lib.OPT_COLOR_MINUS1_1
    mpi = dict(rgb=factored[0], alpha=factored[1]) if factored is not None else dict(rgba=rgba)
    desc = _lib.make_desc(options=options, M=M, V=V, N=N, Ht=Ht, Wt=Wt, H=H, W=W, view_group=group, view2mpi=case.view2mpi, dhw=case.dhw,
                          color=color, depth=depth, video_rgb=v_rgb, video_depth=v_depth, depth_near=FFHQ["plane_min_d"],
                          depth_range=FFHQ["plane_max_d"] - FFHQ["plane_min_d"], flags=flags, stop_transmittance=tau,
                          skipped_pixel_planes=counts[0:1], **mpi, **rays)
    if skip is None:
        _lib.check(lib.gmpi_mpi_render_fwd_ex(ctypes.byref(desc)))
    else:
        occ = g.occupancy_map(skip, rgba=rgba, alpha=None if factored is None else factored[1])
        _lib.check(lib.gmpi_mpi_render_fwd_skip_ex(ctypes.byref(desc), occ.data_ptr(), counts[1:2].data_ptr()))
    torch.cuda.synchronize()
    c = counts.tolist()
    return (v_rgb, v_depth, c[0], c[1]) if out == "video" else (color, depth, c[0], c[1])


def headline(kind, seed=3, **kw):
    # 2 MPIs x 1 view, 96 planes, 1024^2: the headline plane count and resolution
    return synth.make_workload(kind, n_planes=96, tex=1024, img=1024, n_mpi=2, views_per_mpi=1, seed=seed, device=dev(), **kw)


def c4(kind):
    V = 120      # the video sweep: 120 views of ONE 96 x 512^2 MPI, view_group = 120
    return synth.make_workload(kind, n_planes=96, tex=512, img=512, n_mpi=1, views_per_mpi=V, seed=11, device=dev(),
                               yaws=np.linspace(0.5, -0.5, V).astype(np.float32), pitches=np.zeros(V, np.float32))


def factor(case):
    """The workload as a factored MPI: plane 0's colour shared by all planes, the workload's alpha per plane."""
    return case.rgba[:, 0, :3].contiguous(), case.rgba[:, :, 3:].contiguous()


# ------------------------------------------------------------------------------------------------------------------------------
# 1. the occupancy map
# ------------------------------------------------------------------------------------------------------------------------------
def occupancy_ref(alpha, threshold):
    """numpy reference: alpha [M,N,Ht,Wt] -> uint64 words [M,N,ceil(Ht/8),ceil(Wt/512)]."""
    M, N, Ht, Wt = alpha.shape
    wy, wx = -(-Ht // 8), -(-Wt // 512)
    occ = ~(np.abs(alpha) <= np.float32(threshold))                 # NaN: occupied
    pad = np.zeros((M, N, wy * 8, wx * 512), bool)
    pad[:, :, :Ht, :Wt] = occ
    blocks = pad.reshape(M, N, wy, 8, wx * 64, 8).any(axis=(3, 5)).reshape(M, N, wy, wx, 64)
    return (blocks.astype(np.uint64) << np.arange(64, dtype=np.uint64)).sum(axis=-1, dtype=np.uint64)


def sparse_alpha(M, N, Ht, Wt, seed):
    """Mostly 0 with scattered values around 2^-12 (below, exactly at, above), a NaN and -0.0 in otherwise empty blocks."""
    rng = np.random.default_rng(seed)
    a = np.zeros((M, N, Ht, Wt), np.float32)
    k = max(1, M * N * Ht * Wt // 300)
    idx = tuple(rng.integers(0, s, k) for s in a.shape)
    a[idx] = rng.choice(np.array([EPS, -EPS / 2, 2 * EPS, 0.5, 1.0, np.nextafter(np.float32(EPS), np.float32(1))], np.float32), k)
    a[0, 0, :8, :8] = 0.0
    a[0, 0, 3, 5] = np.nan
    a[-1, -1, -8:, -8:] = 0.0
    a[-1, -1, -1, -1] = -0.0
    return a


@pytest.mark.parametrize("ht,wt", [(100, 36), (37, 101), (1024, 1024)])
@pytest.mark.parametrize("layout", ["expanded", "factored"])
@pytest.mark.parametrize("threshold", [0.0, EPS])
def test_occupancy_equals_numpy_reference(ht, wt, layout, threshold):
    d = dev()
    M, N = 2, 3
    a = sparse_alpha(M, N, ht, wt, seed=ht + wt)
    if layout == "expanded":
        rgba = torch.rand((M, N, 4, ht, wt), device=d)
        rgba[:, :, 3] = torch.from_numpy(a).to(d)
        occ = g.occupancy_map(threshold, rgba=rgba)
    else:
        occ = g.occupancy_map(threshold, alpha=torch.from_numpy(a).to(d).unsqueeze(2).contiguous())
    torch.cuda.synchronize()
    want = occupancy_ref(a, threshold)
    got = occ.cpu().numpy().view(np.uint64)
    assert got.shape == want.shape and np.array_equal(got, want)
    assert got[0, 0, 0, 0] & 1                                        # the NaN's block
    assert not (got[-1, -1, -1, -1] >> np.uint64(((wt - 1) // 8) % 64)) & np.uint64(1)     # -0.0 alone leaves its block empty


# ------------------------------------------------------------------------------------------------------------------------------
# 2.-4. threshold 0 is the exact render, with and without early ray termination
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["noise", "surface", "empty"])
def test_threshold_zero_is_bit_identical_at_full_size(kind):
    case = headline(kind)
    for out in ("fp32", "m11", "video"):
        a = render(case, out=out)
        b = render(case, skip=0.0, out=out)
        assert same(a[0], b[0]) and same(a[1], b[1]), out
        if kind == "empty":
            assert b[3] > 0
        if kind == "noise":
            assert b[3] == 0                           # white noise: nothing is empty
    rgb, alpha = factor(case)
    a = render(case, factored=(rgb, alpha))
    b = render(case, skip=0.0, factored=(rgb, alpha))
    assert same(a[0], b[0]) and same(a[1], b[1]) and (b[3] > 0 or kind == "noise")
    cam = cam_params(case.c2w, focal_from_fov(FFHQ["fov_deg"], 1024), 1024, 1024)
    a = render(case, cam=cam)
    b = render(case, skip=0.0, cam=cam)
    assert same(a[0], b[0]) and same(a[1], b[1]) and (b[3] > 0 or kind == "noise")


@pytest.mark.parametrize("kind", ["surface", "empty"])
def test_threshold_zero_is_bit_identical_on_the_video_sweep(kind):
    case = c4(kind)
    for out in ("fp32", "video"):
        a = render(case, out=out, group=120)
        b = render(case, skip=0.0, out=out, group=120)
        assert same(a[0], b[0]) and same(a[1], b[1]) and b[3] > 0


def test_identity_pose_empty_mpi_skips_every_plane_but_the_last():
    z = np.zeros(2, np.float32)
    case = headline("empty", yaws=z, pitches=z)
    V, _, H, W = case.ray_dir.shape
    N = case.rgba.shape[1]
    a = render(case)
    b = render(case, skip=0.0)
    assert same(a[0], b[0]) and same(a[1], b[1])
    assert b[3] == (N - 1) * V * H * W


@pytest.mark.parametrize("kind", ["noise", "surface"])
def test_with_termination_output_and_count_equal_termination_alone(kind):
    case = headline(kind)
    a = render(case, tau=TAU)
    b = render(case, tau=TAU, skip=0.0)
    assert same(a[0], b[0]) and same(a[1], b[1]) and a[2] == b[2] > 0
    assert b[3] > 0 or kind == "noise"


# ------------------------------------------------------------------------------------------------------------------------------
# 5.-6. threshold eps: the bound, the count, determinism
# ------------------------------------------------------------------------------------------------------------------------------
def test_haze_threshold_eps_bound_and_determinism():
    case = headline("haze")
    N = case.rgba.shape[1]
    c0, d0, _, e0 = render(case, skip=0.0)
    assert e0 == 0                                     # haze everywhere: nothing is exactly empty
    _, d_far, _, _ = render(headline("empty"))         # depth of the last plane: the largest per-plane depth of a pixel
    c, dp, _, e = render(case, skip=EPS)
    assert e > 0
    assert float((c - c0).abs().max()) <= N * EPS * 1.0 + 1e-6
    assert float(((dp - d0).abs() - N * EPS * d_far).max()) <= 1e-6
    c2, dp2, _, e2 = render(case, skip=EPS)
    assert same(c, c2) and same(dp, dp2) and e == e2
    a = render(case, skip=EPS, tau=TAU)
    b = render(case, skip=EPS, tau=TAU)
    assert same(a[0], b[0]) and same(a[1], b[1]) and a[2] == b[2] and a[3] == b[3] > 0


# ------------------------------------------------------------------------------------------------------------------------------
# 7. safety: rays the footprint estimate does not describe, and the direct kernel
# ------------------------------------------------------------------------------------------------------------------------------
def hollow(case):
    """Alpha 0 on every other plane and in the left half of the rest (last plane 1): plenty of empty boxes."""
    case.rgba[:, 0::2, 3] = 0.0
    case.rgba[:, :, 3, :, : case.rgba.shape[-1] // 2] = 0.0
    case.rgba[:, -1, 3] = 1.0
    return case


def test_non_projective_rays_stay_bit_identical(staged):
    d = dev()
    case = hollow(synth.make_case(n_planes=12, tex=96, img=200, n_mpi=1, views_per_mpi=2, seed=3, device=d))
    gen = torch.Generator(device="cpu").manual_seed(0)
    perm = torch.randperm(200 * 200, generator=gen).to(d)
    case.ray_dir = case.ray_dir.reshape(2, 3, -1)[:, :, perm].reshape(2, 3, 200, 200).contiguous()     # shuffled rays
    a = render(case)
    b = render(case, skip=0.0)
    assert same(a[0], b[0]) and same(a[1], b[1])
    case = hollow(synth.make_case(n_planes=6, tex=64, img=128, n_mpi=1, views_per_mpi=2, seed=9, device=d))
    for ty in range(0, 128, 30):                       # tile corners far outside the planes, interiors unchanged
        for tx in range(0, 128, 64):
            for (cy, cx) in ((ty, tx), (ty, min(tx + 63, 127)), (min(ty + 29, 127), tx), (min(ty + 29, 127), min(tx + 63, 127))):
                case.ray_dir[:, 0, cy, cx] = 5.0
    a = render(case)
    b = render(case, skip=0.0)
    assert float(a[0].abs().max()) > 0.1 and same(a[0], b[0]) and same(a[1], b[1])


def test_degenerate_rays_keep_their_nan(staged):
    case = hollow(synth.make_case(n_planes=8, tex=64, img=64, n_mpi=1, seed=4, device=dev()))
    case.ray_dir[0, 2, 10, 10:14] = 0.0
    case.ray_dir[0, :, 20, 20] = float("nan")
    a = render(case)
    b = render(case, skip=0.0)
    assert same(a[0], b[0]) and same(a[1], b[1])      # (a NaN ray hits no texel: it renders 0 either way)
    assert b[3] > 0


def test_direct_kernel_ignores_the_map():
    lib = _lib.load()
    case = synth.make_workload("empty", n_planes=32, tex=256, img=512, n_mpi=2, seed=5, device=dev())
    _lib.check(lib.gmpi_debug_set_fwd_variant(1))
    try:
        a = render(case)
        b = render(case, skip=EPS)
    finally:
        _lib.check(lib.gmpi_debug_set_fwd_variant(0))
    assert same(a[0], b[0]) and same(a[1], b[1]) and b[3] == 0


# ------------------------------------------------------------------------------------------------------------------------------
# 8. the Python API and the MPI drop-in
# ------------------------------------------------------------------------------------------------------------------------------
def test_render_frames_and_render_views_factored_skip():
    d = dev()
    case = synth.make_workload("surface", n_planes=96, tex=512, img=512, n_mpi=1, views_per_mpi=5, seed=12, device=d,
                               yaws=np.linspace(0.5, -0.5, 5).astype(np.float32), pitches=np.zeros(5, np.float32))
    kw = dict(rgba=case.rgba, dhw=case.dhw, view2mpi=case.view2mpi, ray_dir=case.ray_dir, eye=case.eye, z_dir=case.z_dir)
    c0, d0 = g.render_frames(**kw)
    sk = torch.zeros(1, dtype=torch.int64, device=d)
    c1, d1 = g.render_frames(**kw, skip_alpha=0.0, skipped_empty=sk)
    assert same(c0, c1) and same(d0, d1) and int(sk.item()) > 0
    with pytest.raises(ValueError, match="skipped_empty"):
        g.render_frames(**kw, skip_alpha=0.0, skipped_empty=torch.zeros(1, dtype=torch.int32, device=d))
    with pytest.raises(ValueError, match="skip_alpha"):
        g.render_frames(**kw, skip_alpha=1.0)
    rgb, alpha = factor(case)
    a = g.render_views_factored(rgb, alpha, case.dhw, case.view2mpi, case.ray_dir, case.eye, case.z_dir)
    b = g.render_views_factored(rgb, alpha, case.dhw, case.view2mpi, case.ray_dir, case.eye, case.z_dir, skip_alpha=0.0)
    assert same(a[0], b[0]) and same(a[1], b[1])


def test_mpi_with_a_gradient_stays_exact_and_without_one_skips():
    d = dev()
    case = hollow(synth.make_workload("noise", n_planes=32, tex=256, img=512, n_mpi=2, seed=6, device=d))
    rays, eyes, zs = [case.ray_dir[i:i + 1] for i in range(2)], [case.eye[i:i + 1] for i in range(2)], [case.z_dir[i:i + 1] for i in range(2)]
    gen = torch.Generator(device=d).manual_seed(1)
    gc = torch.randn((2, 3, 512, 512), generator=gen, device=d)
    out = []
    for skip in (None, 0.0):
        rgba = case.rgba.clone().requires_grad_(True)
        mpi = g.MPI(align_corners=True, validate="off")
        mpi.skip_alpha = skip
        c, dp = mpi(batch_rgba=rgba, batch_dhw=case.dhw, batch_ray_dir=rays, batch_eye_pos=eyes, batch_z_dir=zs, separate_background=None)
        ((c * gc).sum() + dp.sum()).backward()
        out.append((c.detach(), dp.detach(), rgba.grad))
    assert same(out[0][0], out[1][0]) and same(out[0][1], out[1][1])
    assert rel_err(out[1][2].cpu().numpy(), out[0][2].cpu().numpy()) <= 1e-6        # atomics: summation order only
    # the same MPI object without a gradient skips (threshold 0: the output is still the exact one)
    mpi = g.MPI(align_corners=True, validate="off")
    res = []
    for skip in (None, 0.0):
        mpi.skip_alpha = skip
        with torch.no_grad():
            res.append(mpi(batch_rgba=case.rgba, batch_dhw=case.dhw, batch_ray_dir=rays, batch_eye_pos=eyes, batch_z_dir=zs,
                           separate_background=None))
    assert same(res[0][0], res[1][0]) and same(res[0][1], res[1][1])
    sk = torch.zeros(1, dtype=torch.int64, device=d)
    g.render_frames(rgba=case.rgba, dhw=case.dhw, view2mpi=case.view2mpi, ray_dir=case.ray_dir, eye=case.eye, z_dir=case.z_dir,
                    skip_alpha=0.0, skipped_empty=sk)
    assert int(sk.item()) > 0


def test_last_plane_flag_is_still_raised(staged):
    gd = load_golden("out_of_plane")
    d = dev()
    t = lambda a: torch.from_numpy(a).to(d)
    v2m = gd["view2mpi"]
    idx = [np.nonzero(v2m == m)[0] for m in range(gd["rgba"].shape[0])]
    rgba = t(gd["rgba"])
    rgba[:, : rgba.shape[1] // 2, 3] = 0.0              # empty front half
    mpi = g.MPI(align_corners=bool(gd["align_corners"]), validate="defer")
    mpi.skip_alpha = 0.0
    with torch.no_grad():
        mpi(batch_rgba=rgba, batch_dhw=t(gd["dhw"]), batch_ray_dir=[t(gd["ray_dir"][i]) for i in idx],
            batch_eye_pos=[t(gd["eye"][i]) for i in idx], batch_z_dir=[t(gd["z_dir"][i]) for i in idx], separate_background=None,
            assert_not_out_of_last_plane=True)
    assert mpi.last_flags() & _lib.FLAG_LAST_PLANE_OOB


@pytest.mark.parametrize("name", MPI_CASES)
def test_reference_goldens_with_skip_alpha_zero(name, fwd_variant):
    gd = load_golden(name)
    d = dev()
    v2m = gd["view2mpi"]
    t = lambda a: torch.from_numpy(a).to(d)
    idx = [np.nonzero(v2m == m)[0] for m in range(gd["rgba"].shape[0])]
    mpi = g.MPI(align_corners=bool(gd["align_corners"]), validate="defer")
    mpi.skip_alpha = 0.0
    with torch.no_grad():
        color, depth = mpi(batch_rgba=t(gd["rgba"]), batch_dhw=t(gd["dhw"]), batch_ray_dir=[t(gd["ray_dir"][i]) for i in idx],
                           batch_eye_pos=[t(gd["eye"][i]) for i in idx], batch_z_dir=[t(gd["z_dir"][i]) for i in idx],
                           separate_background=None)
    ec, ed = rel_err(color.cpu().numpy(), gd["color"]), rel_err(depth.cpu().numpy(), gd["depth"])
    assert ec <= EXPECT and ed <= EXPECT, (ec, ed)
