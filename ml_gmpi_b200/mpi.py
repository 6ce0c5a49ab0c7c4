"""Drop-in for `gmpi.core.mpi.MPI` (reference gmpi/core/mpi.py:156-436), backed by the sm_100a
kernels through the C ABI.  Same constructor, same keyword-only `forward`, same return values,
same assertion messages; differentiable w.r.t. `batch_rgba` (first order), which is all the
reference's callers need (the sampling grid and the depth are built under no_grad,
mpi.py:65,148).

No CPU path: tensors must live on a CUDA device, otherwise this raises.
"""
import ctypes
import warnings
from typing import List, Optional, Union

import numpy as np
import torch
from torch import nn

from . import _lib


class MPIOutOfPlaneError(AssertionError):
    """Rays leave the last plane (reference: prints the poses and sys.exit(1), mpi.py:103-128)."""


def _stream_ptr(device):
    return torch.cuda.current_stream(device).cuda_stream


def _as_f32c(t: torch.Tensor) -> torch.Tensor:
    if t.dtype != torch.float32:
        t = t.float()
    return t if t.is_contiguous() else t.contiguous()


class _RenderFn(torch.autograd.Function):
    """MPI.forward + its autograd through the C ABI's descriptor entry points (gmpi_mpi_render_fwd_ex / _bwd_ex).
    The MPI is either expanded (`rgba`) or factored (`rgb`, `alpha`, optional `bg_rgb`); the unused form is None."""

    @staticmethod
    def forward(ctx, rgba, rgb, alpha, bg_rgb, dhw, view2mpi, ray_dir, eye, z_dir, options, flags, view_group, stop_transmittance,
                skip_alpha):
        lib = _lib.load()
        factored = rgba is None
        ref = alpha if factored else rgba
        M, N = ref.shape[0], ref.shape[1]
        Ht, Wt = ref.shape[-2:]
        V, _, H, W = ray_dir.shape
        dev = ref.device
        color = torch.empty((V, 3, H, W), device=dev, dtype=torch.float32)
        depth = torch.empty((V, 1, H, W), device=dev, dtype=torch.float32)
        # training: the forward also saves the transmittance in front of every plane (4 B per pixel-plane) so that the
        # backward is ONE staged back-to-front sweep (torch autograd keeps ~30 such tensors alive for the reference)
        trans = None
        if any(ctx.needs_input_grad[:4]):
            trans = torch.empty((V, N, H, W), device=dev, dtype=torch.float32)
        # early ray termination only when no input needs a gradient: with one the render is exact (the backward needs every
        # plane's T), so one MPI object serves the no-grad D step and the G step alike
        tau = float(stop_transmittance) if trans is None else 0.0
        skip = skip_alpha if trans is None else None         # the same rule for empty-space skipping
        with torch.cuda.device(dev):
            d = _lib.make_desc(options=options, M=M, V=V, N=N, Ht=Ht, Wt=Wt, H=H, W=W, view_group=view_group, rgba=rgba, rgb=rgb,
                               alpha=alpha, bg_rgb=bg_rgb, view2mpi=view2mpi, dhw=dhw, ray_dir=ray_dir, eye=eye, z_dir=z_dir,
                               color=color, depth=depth, transmittance=trans, flags=flags, stream=_stream_ptr(dev),
                               stop_transmittance=tau)
            _render_fwd(lib, d, skip, rgba, alpha, V, H, W)
        ctx.save_for_backward(rgba, rgb, alpha, bg_rgb, dhw, view2mpi, ray_dir, eye, z_dir, trans)
        ctx.options, ctx.view_group = options, view_group
        ctx.set_materialize_grads(False)
        return color, depth

    @staticmethod
    @torch.autograd.function.once_differentiable     # raw kernels: a double backward (create_graph=True) must raise, not
    def backward(ctx, g_color, g_depth):             # silently treat the result as constant (the reference's R1 only differentiates D)
        rgba, rgb, alpha, bg_rgb, dhw, view2mpi, ray_dir, eye, z_dir, trans = ctx.saved_tensors
        none = (None,) * 14
        if not any(ctx.needs_input_grad[:4]):
            return none
        lib = _lib.load()
        factored = rgba is None
        ref = alpha if factored else rgba
        M, N = ref.shape[0], ref.shape[1]
        Ht, Wt = ref.shape[-2:]
        V, _, H, W = ray_dir.shape
        dev = ref.device
        if g_color is None:
            g_color = torch.zeros((V, 3, H, W), device=dev, dtype=torch.float32)
        g_color = _as_f32c(g_color)
        g_depth = _as_f32c(g_depth) if g_depth is not None else None
        # GMPI_ZERO_GRAD: the callee zeroes the buffers on the stream.  (Zeroing them on a side stream during the forward, as an
        # earlier version did, buys nothing: a memset cannot overlap the persistent kernels -- tools/zero_overlap_probe.py.)
        if factored:
            g_rgba = None
            g_rgb, g_alpha = torch.empty_like(rgb), torch.empty_like(alpha)
            g_bg = torch.empty_like(bg_rgb) if bg_rgb is not None else None
        else:
            g_rgb = g_alpha = g_bg = None
            g_rgba = torch.empty_like(rgba)
        with torch.cuda.device(dev):   # autograd worker threads do not inherit the device
            d = _lib.make_desc(options=ctx.options | _lib.OPT_ZERO_GRAD, M=M, V=V, N=N, Ht=Ht, Wt=Wt, H=H, W=W,
                               view_group=ctx.view_group, rgba=rgba, rgb=rgb, alpha=alpha, bg_rgb=bg_rgb, view2mpi=view2mpi, dhw=dhw,
                               ray_dir=ray_dir, eye=eye, z_dir=z_dir, transmittance=trans, g_color=g_color, g_depth=g_depth,
                               g_rgba=g_rgba, g_rgb=g_rgb, g_bg_rgb=g_bg, g_alpha=g_alpha, stream=_stream_ptr(dev))
            _lib.check(lib.gmpi_mpi_render_bwd_ex(ctypes.byref(d)))
        return (g_rgba, g_rgb, g_alpha, g_bg) + (None,) * 10


_warned_direct = set()


def _warn_if_direct(ref, V, H, W):
    """Surface the direct-kernel performance cliff (several times slower than the TMA-staged kernels) once per shape."""
    N, (Ht, Wt) = ref.shape[1], ref.shape[-2:]
    key = (V, N, Ht, Wt, H, W, ref.data_ptr() & 15)
    if key in _warned_direct:
        return
    _warned_direct.add(key)
    why = ctypes.c_uint32(0)
    if _lib.load().gmpi_mpi_render_fwd_plan(V, N, Ht, Wt, H, W, ref.data_ptr(), ctypes.byref(why)) == _lib.PLAN_DIRECT \
            and (why.value & ~2 or V * N * H * W >= 1 << 26):      # "few tiles" only matters when the problem is not tiny
        reasons = "; ".join(t for b, t in _lib.WHY.items() if why.value & b)
        warnings.warn(f"ml_gmpi_b200: rendering V={V} N={N} tex={Ht}x{Wt} img={H}x{W} with the direct (one thread per pixel) "
                      f"kernels, several times slower than the TMA-staged path: {reasons}", RuntimeWarning, stacklevel=3)


def _options(align_corners, check_last_plane, color_minus1_1, u8_round=False):
    return (_lib.OPT_ALIGN_CORNERS if align_corners else 0) | (_lib.OPT_CHECK_LAST_PLANE if check_last_plane else 0) \
        | (_lib.OPT_COLOR_MINUS1_1 if color_minus1_1 else 0) | (_lib.OPT_U8_ROUND_HALF_UP if u8_round else 0)


def _check_stop(stop_transmittance) -> float:
    tau = float(stop_transmittance)
    if not 0.0 <= tau < 1.0:
        raise ValueError(f"stop_transmittance must be in [0, 1), got {stop_transmittance}")
    return tau


def _check_skip(skip_alpha) -> Optional[float]:
    if skip_alpha is None:
        return None
    eps = float(skip_alpha)
    if not 0.0 <= eps < 1.0:
        raise ValueError(f"skip_alpha must be None or in [0, 1), got {skip_alpha}")
    return eps


def occupancy_map(threshold: float, *, rgba: Optional[torch.Tensor] = None, alpha: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Occupancy map of empty-space skipping (gmpi_mpi_occupancy), built on the current stream from the expanded stack rgba
    [M,N,4,Ht,Wt] (its channel 3, no copy) or the factored alpha [M,N,1,Ht,Wt] (contiguous fp32 CUDA tensors): one bit per 8x8-texel
    block of every plane, set iff some alpha of the block exceeds `threshold` in magnitude (or is NaN).  Returned as an int64 tensor
    [M, N, ceil(Ht/8), ceil(Wt/512)] holding the uint64 words of the C layout."""
    ref = alpha if rgba is None else rgba
    M, N = ref.shape[0], ref.shape[1]
    Ht, Wt = ref.shape[-2:]
    tex = Ht * Wt
    occ = torch.empty((M, N, (Ht + 7) // 8, (Wt + 511) // 512), dtype=torch.int64, device=ref.device)
    if rgba is not None:
        ptr, plane_stride = rgba.data_ptr() + 4 * 3 * tex, 4 * tex          # channel 3 of every plane
    else:
        ptr, plane_stride = alpha.data_ptr(), tex
    with torch.cuda.device(ref.device):
        _lib.check(_lib.load().gmpi_mpi_occupancy(ptr, N * plane_stride, plane_stride, M, N, Ht, Wt, float(threshold), occ.data_ptr(),
                                                  _stream_ptr(ref.device)))
    return occ


def _render_fwd(lib, d, skip_alpha, rgba, alpha, V, H, W, empty=None):
    """The forward of descriptor d: gmpi_mpi_render_fwd_ex, or -- skip_alpha set and the shapes take the staged kernel -- the
    skipping forward on an occupancy map built for this call (the direct kernel would ignore it: no map then).  `empty` (nullable
    int64 tensor of one element) receives the skipped pixel-planes.  Call on the render's device."""
    if skip_alpha is not None:
        ref = alpha if rgba is None else rgba
        N, (Ht, Wt) = ref.shape[1], ref.shape[-2:]
        if lib.gmpi_mpi_render_fwd_plan(V, N, Ht, Wt, H, W, ref.data_ptr(), None) == _lib.PLAN_STAGED:
            occ = occupancy_map(skip_alpha, rgba=rgba, alpha=alpha)
            _lib.check(lib.gmpi_mpi_render_fwd_skip_ex(ctypes.byref(d), occ.data_ptr(), None if empty is None else empty.data_ptr()))
            return
    _lib.check(lib.gmpi_mpi_render_fwd_ex(ctypes.byref(d)))


def render_views(rgba, dhw, view2mpi, ray_dir, eye, z_dir, *, align_corners=True, check_last_plane=False,
                 color_minus1_1=False, flags: Optional[torch.Tensor] = None, view_group: int = 1, stop_transmittance: float = 0.0,
                 skip_alpha: Optional[float] = None):
    """Functional form on packed tensors (no list handling, no host sync).
    rgba [M,N,4,Ht,Wt], dhw [M,N,3], view2mpi [V] int32, ray_dir [V,3,H,W], eye/z_dir [V,3].
    Returns (color [V,3,H,W], depth [V,1,H,W]); `flags` (uint32 tensor of 1, int32 storage) is OR-ed into.
    view_group > 1: every view_group consecutive views share one MPI (tile-order hint: L2 reuse, see the C header).
    stop_transmittance = tau in (0, 1): early ray termination when no input needs a gradient -- a pixel may drop the planes
    behind the point where its transmittance fell below tau, so every output is within tau * max(value) below the exact one
    (the contract in include/gmpi_mpi_render.h).  0 (default): exact.  Ignored (exact render) when rgba requires grad.
    skip_alpha = eps: empty-space skipping when no input needs a gradient -- the call builds an occupancy map of the MPI (one
    streaming read of alpha) and the kernel skips the (64x30 tile, plane) pairs whose alpha is within eps of 0 under the whole
    tile.  0.0 skips only exactly transparent space and is bit-identical to the exact render; eps in (0, 1) moves every output by
    at most N * eps * max(value) (colour and alpha in [0, 1]).  None (default): off.  Ignored (exact render) when rgba requires
    grad, like stop_transmittance."""
    if not rgba.is_cuda:
        raise RuntimeError("ml_gmpi_b200 renders on CUDA devices only (no CPU fallback); got a CPU tensor")
    if flags is None:
        flags = torch.zeros(1, dtype=torch.int32, device=rgba.device)
    _warn_if_direct(rgba, ray_dir.shape[0], ray_dir.shape[2], ray_dir.shape[3])
    return _RenderFn.apply(_as_f32c(rgba), None, None, None, _as_f32c(dhw), view2mpi, _as_f32c(ray_dir), _as_f32c(eye), _as_f32c(z_dir),
                           _options(align_corners, check_last_plane, color_minus1_1), flags, int(view_group),
                           _check_stop(stop_transmittance), _check_skip(skip_alpha))


def render_views_factored(rgb, alpha, dhw, view2mpi, ray_dir, eye, z_dir, *, bg_rgb=None, align_corners=True,
                          check_last_plane=False, color_minus1_1=False, flags: Optional[torch.Tensor] = None, view_group: int = 1,
                          stop_transmittance: float = 0.0, skip_alpha: Optional[float] = None):
    """The same render from the generator's FACTORED output (networks_cond_on_pos_enc.py:950-975,984): one colour image
    rgb [M,3,Ht,Wt] shared by all planes (bg_rgb [M,3,Ht,Wt]: the last plane's own colour under torgba_sep_background) and
    alpha [M,N,1,Ht,Wt] -- what the reference expands to [M,N,4,Ht,Wt] (and copies per view, train.py:553-558,733-738) before
    rendering.  Output identical to render_views on the expanded stack, 4x fewer HBM bytes; differentiable w.r.t. rgb, alpha
    and bg_rgb (d/d rgb is the sum over the planes that share it).  stop_transmittance, skip_alpha (the map is built from
    `alpha`): as in render_views."""
    if not alpha.is_cuda:
        raise RuntimeError("ml_gmpi_b200 renders on CUDA devices only (no CPU fallback); got a CPU tensor")
    assert rgb.ndim == 4 and rgb.shape[1] == 3 and alpha.ndim == 5 and alpha.shape[2] == 1 and rgb.shape[0] == alpha.shape[0] \
        and rgb.shape[-2:] == alpha.shape[-2:], f"expected rgb [M,3,Ht,Wt] and alpha [M,N,1,Ht,Wt], got {rgb.shape}, {alpha.shape}"
    assert bg_rgb is None or bg_rgb.shape == rgb.shape, f"bg_rgb must have rgb's shape, got {bg_rgb.shape}"
    if flags is None:
        flags = torch.zeros(1, dtype=torch.int32, device=alpha.device)
    _warn_if_direct(alpha, ray_dir.shape[0], ray_dir.shape[2], ray_dir.shape[3])
    return _RenderFn.apply(None, _as_f32c(rgb), _as_f32c(alpha), None if bg_rgb is None else _as_f32c(bg_rgb), _as_f32c(dhw), view2mpi,
                           _as_f32c(ray_dir), _as_f32c(eye), _as_f32c(z_dir), _options(align_corners, check_last_plane, color_minus1_1),
                           flags, int(view_group), _check_stop(stop_transmittance), _check_skip(skip_alpha))


def expand_factored(rgb, alpha, bg_rgb=None):
    """[M,3,Ht,Wt] + [M,N,1,Ht,Wt] -> [M,N,4,Ht,Wt], the generator's expand + cat (networks_cond_on_pos_enc.py:950-975):
    what the reference renders from; here only tests and callers that need the expanded stack use it."""
    N = alpha.shape[1]
    col = rgb.unsqueeze(1).expand(-1, N, -1, -1, -1)
    if bg_rgb is not None:
        col = torch.cat([col[:, : N - 1], bg_rgb.unsqueeze(1)], dim=1)
    return torch.cat([col, alpha], dim=2).contiguous()


def render_frames(*, dhw, view2mpi, rgba=None, rgb=None, alpha=None, bg_rgb=None, ray_dir=None, eye=None, z_dir=None, cam=None,
                  align_corners=True, check_last_plane=False, video: Optional[dict] = None, u8_round=False,
                  flags: Optional[torch.Tensor] = None, view_group: int = 1, H: Optional[int] = None, W: Optional[int] = None,
                  stop_transmittance: float = 0.0, skipped: Optional[torch.Tensor] = None, skip_alpha: Optional[float] = None,
                  skipped_empty: Optional[torch.Tensor] = None):
    """Inference-only render with the opt-in fast paths of the C ABI (no autograd):
      cam [V,16]     rays generated in the kernel from the pinhole camera (see camera.cam_params) instead of ray_dir/eye/z_dir;
      video={"near": ray_start, "far": ray_end, "depth": True}   uint8 HWC frames as render_video.py:118-126 builds them:
                     returns (rgb_u8 [V,H,W,3], depth_u8 [V,H,W,1] or None); otherwise (color in [-1,1], depth) fp32.
      stop_transmittance = tau in (0, 1)   early ray termination (see render_views; the [-1,1] colour moves by up to 2 tau);
      skipped        int64 CUDA tensor of one element: the number of pixel-planes not composited is added to it.
      skip_alpha = eps in [0, 1)   empty-space skipping (see render_views; one occupancy map per call, for all its views);
      skipped_empty  int64 CUDA tensor of one element: the number of pixel-planes skipped as empty is added to it.
    """
    ref = alpha if rgba is None else rgba
    if not ref.is_cuda:
        raise RuntimeError("ml_gmpi_b200 renders on CUDA devices only (no CPU fallback); got a CPU tensor")
    lib = _lib.load()
    dev = ref.device
    M, N = ref.shape[0], ref.shape[1]
    Ht, Wt = ref.shape[-2:]
    if cam is not None:
        V = cam.shape[0]
        assert H is not None and W is not None, "pass H and W with cam"
        cam = _as_f32c(cam)
    else:
        V, _, H, W = ray_dir.shape
        ray_dir, eye, z_dir = _as_f32c(ray_dir), _as_f32c(eye), _as_f32c(z_dir)
    if flags is None:
        flags = torch.zeros(1, dtype=torch.int32, device=dev)
    tau = _check_stop(stop_transmittance)
    eps = _check_skip(skip_alpha)
    for name, t in (("skipped", skipped), ("skipped_empty", skipped_empty)):
        if t is not None and not (t.is_cuda and t.dtype == torch.int64 and t.numel() == 1 and t.is_contiguous()):
            raise ValueError(f"{name} must be a contiguous int64 CUDA tensor of one element")
    color = depth = v_rgb = v_depth = None
    near = rng = 0.0
    if video is not None:
        v_rgb = torch.empty((V, H, W, 3), device=dev, dtype=torch.uint8)
        if video.get("depth", True):
            v_depth = torch.empty((V, H, W, 1), device=dev, dtype=torch.uint8)
        near = float(np.float32(video["near"]))
        rng = float(np.float32(video["far"] - video["near"]))            # the python-double difference, rounded once (numpy weak scalar)
    else:
        color = torch.empty((V, 3, H, W), device=dev, dtype=torch.float32)
        depth = torch.empty((V, 1, H, W), device=dev, dtype=torch.float32)
    keep = [_as_f32c(t) if t is not None else None for t in (rgba, rgb, alpha, bg_rgb, dhw)]
    with torch.cuda.device(dev):
        d = _lib.make_desc(options=_options(align_corners, check_last_plane, True, u8_round), M=M, V=V, N=N, Ht=Ht, Wt=Wt, H=H, W=W,
                           view_group=int(view_group), depth_near=near, depth_range=rng, rgba=keep[0], rgb=keep[1], alpha=keep[2],
                           bg_rgb=keep[3], view2mpi=view2mpi, dhw=keep[4], ray_dir=ray_dir, eye=eye, z_dir=z_dir, cam=cam, color=color,
                           depth=depth, video_rgb=v_rgb, video_depth=v_depth, flags=flags, stream=_stream_ptr(dev),
                           stop_transmittance=tau, skipped_pixel_planes=skipped)
        _render_fwd(lib, d, eps, keep[0], keep[2], V, H, W, skipped_empty)
    return (v_rgb, v_depth) if video is not None else (color, depth)


def check_range(rgba: torch.Tensor, flags: torch.Tensor) -> None:
    """One streaming pass: RGBA/alpha in [0,1] (mpi_renderer.py:447-449, mpi.py:185-187) -> flag bits."""
    lib = _lib.load()
    M, N, _, Ht, Wt = rgba.shape
    with torch.cuda.device(rgba.device):
        _lib.check(lib.gmpi_mpi_check_range(rgba.data_ptr(), M, N, Ht, Wt, flags.data_ptr(), _stream_ptr(rgba.device)))


class MPI(nn.Module):
    """`validate`:
         "full"  (default) every data-dependent assert of the reference is evaluated on the device
                 (alpha range scan, plane-behind-camera, rays leaving the last plane) and raised
                 after ONE host sync per call (the reference syncs six or more times);
         "defer" the geometric flags are still computed inside the render kernel (free) but nothing
                 is scanned or synced; read them later with `.raise_if_flagged()`;
         "off"   like "defer" without the last-plane check.
    `stop_transmittance` = tau in (0, 1): early ray termination of renders where no input needs a gradient (see render_views);
    renders with a gradient stay exact.  0 (default): exact.
    `skip_alpha` (attribute, not a constructor parameter): empty-space skipping threshold of the same renders (see render_views).
    None (default): off; 0.0: exactly transparent space only (bit-identical output).
    """

    def __init__(self, align_corners=True, validate: str = "full", stop_transmittance: float = 0.0):
        super().__init__()
        assert validate in ("full", "defer", "off"), validate
        self._align_corners = align_corners
        self.validate = validate
        self.stop_transmittance = _check_stop(stop_transmittance)
        self._skip_alpha = None
        self._flags = None
        self._flag_ctx = None

    @property
    def skip_alpha(self) -> Optional[float]:
        return self._skip_alpha

    @skip_alpha.setter
    def skip_alpha(self, value):
        self._skip_alpha = _check_skip(value)      # ValueError outside [0, 1)

    # -- reference: MPI.check_shapes, mpi.py:161-216 (shape part; the alpha range is checked on the device)
    def check_shapes(self, *, batch_rgba, batch_dhw, batch_ray_dir, batch_eye_pos, batch_z_dir, separate_background):
        assert (batch_rgba.ndim == 5) and (batch_rgba.shape[2] == 4), (
            f"Expected rgba to be of shape (#mpi, #planes, 4, texture_height, texture_width), "
            f"but instead got {batch_rgba.shape}")
        assert ((batch_dhw.ndim == 3) and (batch_dhw.shape[0] == batch_rgba.shape[0])
                and (batch_dhw.shape[1] == batch_rgba.shape[1]) and (batch_dhw.shape[2] == 3)), (
            f"Expected dhw to be of shape (#mpi, #planes, 3), but instead got {batch_dhw.shape} (rgba: {batch_rgba.shape})")
        assert len(batch_ray_dir) == batch_rgba.shape[0], f"{len(batch_ray_dir)}, {batch_rgba.shape[0]}"
        assert len(batch_eye_pos) == batch_rgba.shape[0], f"{len(batch_eye_pos)}, {batch_rgba.shape[0]}"
        assert len(batch_z_dir) == batch_rgba.shape[0], f"{len(batch_z_dir)}, {batch_rgba.shape[0]}"
        for i in range(len(batch_ray_dir)):
            assert (batch_ray_dir[i].ndim == 4) and (batch_ray_dir[i].shape[1] == 3), (
                f"Expected ray_dir to be of shape (minibatch, 3, image_height, image_width), "
                f"but instead got {batch_ray_dir[i].shape} for {i} th elem.")
            assert (batch_eye_pos[i].ndim == 2) and (batch_eye_pos[i].shape[1] == 3), (
                f"Expected eye_pos to be of shape (minibatch, 3), but instead got {batch_eye_pos[i].shape} for {i} th elem.")
            assert (batch_z_dir[i].ndim == 2) and (batch_z_dir[i].shape[1] == 3), (
                f"Expected z_dir to be of shape (minibatch, 3), but instead got {batch_z_dir[i].shape} for {i} th elem.")
        if separate_background is not None:
            assert separate_background.ndim == 4 and separate_background.shape[1] == 3, (
                f"Expect background to be of shape (#mpi, 3, h, w), but instead get {separate_background.shape}.")

    @staticmethod
    def pack_views(batch_ray_dir, batch_eye_pos, batch_z_dir, device):
        """mpi.py:334-354 without the copies of the MPI: views stay MPI-major and a [V] int32 index
        replaces expand+cat of rgba/dhw."""
        counts = [int(r.shape[0]) for r in batch_ray_dir]
        if all(c == 1 for c in counts):
            view2mpi = torch.arange(len(counts), dtype=torch.int32, device=device)
        else:
            view2mpi = torch.repeat_interleave(torch.arange(len(counts), dtype=torch.int32),
                                               torch.tensor(counts)).to(device=device, dtype=torch.int32)
        cat = (lambda xs: xs[0] if len(xs) == 1 else torch.cat(xs, dim=0))
        return view2mpi, cat(list(batch_ray_dir)), cat(list(batch_eye_pos)), cat(list(batch_z_dir))

    @staticmethod
    def view_group_of(batch_ray_dir) -> int:
        """k when every MPI is rendered from the same number k > 1 of views (the expand of train.py:733-738 /
        train_helpers.py:181-186, a video sweep of one MPI): the kernels then order tiles for L2 reuse.  Else 1."""
        counts = {int(r.shape[0]) for r in batch_ray_dir}
        k = counts.pop() if len(counts) == 1 else 1
        return k if k > 1 else 1

    def forward(self, *, batch_rgba: torch.Tensor, batch_dhw: torch.Tensor, batch_ray_dir: List[torch.Tensor],
                batch_eye_pos: List[torch.Tensor], batch_z_dir: List[torch.Tensor],
                separate_background: Union[None, torch.Tensor], assert_not_out_of_last_plane: bool = False,
                c2w_mat: torch.Tensor = None, sphere_c: np.ndarray = None):
        self.check_shapes(batch_rgba=batch_rgba, batch_dhw=batch_dhw, batch_ray_dir=batch_ray_dir,
                          batch_eye_pos=batch_eye_pos, batch_z_dir=batch_z_dir, separate_background=separate_background)
        if not batch_rgba.is_cuda:
            raise RuntimeError("ml_gmpi_b200.MPI renders on CUDA devices only (no CPU fallback); got a CPU tensor")
        dev = batch_rgba.device
        view2mpi, ray_dir, eye, z_dir = self.pack_views(batch_ray_dir, batch_eye_pos, batch_z_dir, dev)
        rgba = _as_f32c(batch_rgba)
        flags = torch.zeros(1, dtype=torch.int32, device=dev)
        if self.validate == "full":
            check_range(rgba.detach(), flags)
        color, depth = render_views(rgba, batch_dhw.to(dev), view2mpi, ray_dir.to(dev), eye.to(dev), z_dir.to(dev),
                                    align_corners=self._align_corners,
                                    check_last_plane=bool(assert_not_out_of_last_plane) and self.validate != "off",
                                    flags=flags, view_group=self.view_group_of(batch_ray_dir),
                                    stop_transmittance=self.stop_transmittance, skip_alpha=self.skip_alpha)
        self._flags = flags
        self._flag_ctx = (batch_dhw, eye, c2w_mat, sphere_c)
        if self.validate == "full":
            self.raise_if_flagged(ignore=_lib.FLAG_RGBA_RANGE)   # rgba range is MPIRenderer.render's assert
        return color, depth

    def last_flags(self) -> int:
        """Flag word of the most recent forward (one host sync)."""
        return 0 if self._flags is None else int(self._flags.item()) & 0xFFFFFFFF

    def raise_if_flagged(self, ignore: int = 0):
        f = self.last_flags() & ~ignore
        if f == 0:
            return
        dhw, eye, c2w, sphere_c = self._flag_ctx
        if f & _lib.FLAG_ALPHA_RANGE:
            raise AssertionError("Expected alpha to be within the the range [0, 1]")             # mpi.py:185-187
        if f & _lib.FLAG_RGBA_RANGE:
            raise AssertionError("MPI rgba outside [0, 1]")                                       # mpi_renderer.py:447-449
        if f & _lib.FLAG_PLANE_BEHIND_EYE:
            raise AssertionError(f"Camera must be placed closer to origin than MPI. {dhw[..., 0]}, {eye[0, ...]}")  # mpi.py:70-72
        if f & _lib.FLAG_LAST_PLANE_OOB:
            msg = f"Ray's U/V direction goes out of plane at {dhw[:, -1, 0]}"                    # mpi.py:106-109
            if c2w is not None and sphere_c is not None:
                msg += f"; c2w: {c2w.detach().cpu().numpy().tolist()}"
            raise MPIOutOfPlaneError(msg)
