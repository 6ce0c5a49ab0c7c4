"""Synthetic MPI workloads with the reference's FFHQ geometry (SURVEY.md section 8d): random RGBA
stacks, in-envelope poses, rays from the pinhole camera.  Used by bench.py, smoke() and the
full-size GPU tests; needs neither the reference nor the oracle."""
from dataclasses import dataclass

import numpy as np
import torch

from .camera import PinholeCamera, sphere_poses
from .geometry import FFHQ, plane_dhw_table

_DHW_CACHE = {}


def ffhq_dhw(n_planes: int) -> torch.Tensor:
    if n_planes not in _DHW_CACHE:
        _DHW_CACHE[n_planes] = torch.from_numpy(plane_dhw_table(n_planes=n_planes, **FFHQ))
    return _DHW_CACHE[n_planes]


@dataclass
class Case:
    rgba: torch.Tensor       # [M,N,4,T,T]
    dhw: torch.Tensor        # [M,N,3]
    view2mpi: torch.Tensor   # [V] int32
    ray_dir: torch.Tensor    # [V,3,H,W]
    eye: torch.Tensor        # [V,3]
    z_dir: torch.Tensor      # [V,3]
    c2w: torch.Tensor        # [V,4,4]
    yaws: torch.Tensor
    pitches: torch.Tensor

    def to(self, device, pin=False):
        f = (lambda t: t.pin_memory()) if pin else (lambda t: t.to(device))
        return Case(*[f(getattr(self, k)) for k in self.__dataclass_fields__])


def make_poses(n_views, img, seed=1234, yaws=None, pitches=None, device="cpu"):
    if yaws is None:   # U(-0.5,0.5) x U(-0.2,0.2): inside the 2-sigma envelope (BASELINE.md section 4)
        rng = np.random.default_rng(seed)
        yaws = rng.uniform(-0.5, 0.5, n_views).astype(np.float32)
        pitches = rng.uniform(-0.2, 0.2, n_views).astype(np.float32)
    yaws, pitches = torch.as_tensor(yaws, dtype=torch.float32), torch.as_tensor(pitches, dtype=torch.float32)
    c2w = sphere_poses(yaws, pitches, FFHQ["sphere_center"], FFHQ["sphere_r"]).to(device)
    cam = PinholeCamera.from_fov(FFHQ["fov_deg"], img, img)
    ray_dir, eye, z_dir = cam.generate_rays(c2w)
    return ray_dir, eye, z_dir, c2w, yaws, pitches


def make_case(*, n_planes, tex, img, n_mpi, views_per_mpi=1, seed=1234, device="cpu", last_alpha_one=False,
              yaws=None, pitches=None, rgba=True) -> Case:
    V = n_mpi * views_per_mpi
    ray_dir, eye, z_dir, c2w, yaws, pitches = make_poses(V, img, seed, yaws, pitches, device)
    gen = torch.Generator(device=device).manual_seed(seed)
    t = None
    if rgba:
        t = torch.rand((n_mpi, n_planes, 4, tex, tex), generator=gen, device=device, dtype=torch.float32)
        if last_alpha_one:
            t[:, -1, 3] = 1.0      # production MPIs: networks_cond_on_pos_enc.py:1307-1310
    dhw = ffhq_dhw(n_planes).to(device).unsqueeze(0).expand(n_mpi, -1, -1).contiguous()
    v2m = torch.arange(n_mpi, dtype=torch.int32, device=device).repeat_interleave(views_per_mpi)
    return Case(t, dhw, v2m, ray_dir, eye, z_dir, c2w, yaws, pitches)


def surface_alpha(n_mpi, n_planes, tex, *, device="cpu", front=0.2, back=0.75, band=6.0, peak=0.98, semi_axes=(0.55, 0.7)):
    """Alpha [M,N,1,T,T] of a "head": an ellipsoid heightfield over the texture centre, nearest (plane front*N) at the centre and
    reaching plane back*N at its rim; in front of the surface alpha = 0, then a soft band (alpha rising to `peak` over the first
    quarter of `band` planes, zero after it); outside the ellipse alpha = 0; the last plane alpha = 1 everywhere.  A stand-in for
    a trained generator's MPI: only rays through the head become opaque before the last plane."""
    u = torch.linspace(-1.0, 1.0, tex, device=device)
    r2 = (u.view(1, -1) / semi_axes[0]) ** 2 + (u.view(-1, 1) / semi_axes[1]) ** 2          # [T(y), T(x)]
    inside = r2 < 1.0
    s = (back - (back - front) * torch.sqrt(torch.clamp(1.0 - r2, min=0.0))) * (n_planes - 1)  # surface plane index
    i = torch.arange(n_planes, device=device, dtype=torch.float32).view(-1, 1, 1)
    d = i - s.unsqueeze(0)                                                                     # planes behind the surface
    a = torch.clamp((d + 1.0) / (0.25 * band), 0.0, 1.0) * peak * (d < band).float() * inside.unsqueeze(0).float()
    a[-1] = 1.0
    return a.unsqueeze(0).unsqueeze(2).expand(n_mpi, -1, -1, -1, -1).contiguous()


def make_workload(kind, *, n_planes, tex, img, n_mpi, views_per_mpi=1, seed=1234, device="cpu", yaws=None, pitches=None) -> Case:
    """Early-ray-termination and empty-space-skipping workloads, random colours and last plane alpha = 1 in all of them:
      "noise"   white-noise alpha (make_case(last_alpha_one=True)): T falls below 2^-24 after a few dozen planes everywhere;
      "surface" surface_alpha: only tiles inside the head can terminate;
      "empty"   alpha = 0 except the last plane: nothing can be skipped (the cost of the termination test alone);
      "haze"    "surface" with alpha uniform in [0, 2^-12) where it is 0 there: empty-space skipping at threshold 0 finds nothing
                to skip, at threshold 2^-12 everything in front of and around the head."""
    case = make_case(n_planes=n_planes, tex=tex, img=img, n_mpi=n_mpi, views_per_mpi=views_per_mpi, seed=seed, device=device,
                     last_alpha_one=True, yaws=yaws, pitches=pitches)
    if kind in ("surface", "haze"):
        case.rgba[:, :, 3:] = surface_alpha(n_mpi, n_planes, tex, device=device)
        if kind == "haze":
            gen = torch.Generator(device=device).manual_seed(seed + 1)
            a = case.rgba[:, :, 3]
            haze = torch.rand(a.shape, generator=gen, device=device, dtype=torch.float32) * 2.0 ** -12
            case.rgba[:, :, 3] = torch.where(a == 0, haze, a)
    elif kind == "empty":
        case.rgba[:, :, 3] = 0.0
        case.rgba[:, -1, 3] = 1.0
    elif kind != "noise":
        raise ValueError(f"unknown workload {kind!r}")
    return case
