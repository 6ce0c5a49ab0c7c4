"""Render service harness: the reference's two bulk-render drivers with their per-view Python loops, per-frame `.cpu()` syncs
and numpy conversions folded into batched launches -- SURVEY.md 8(f) row N4.

  render_video_frames   `generate_img`'s hot loop (gmpi/eval/vis/render_video.py:95-130): 100 renders of ONE MPI, one
                        `mpi_renderer.render` call, one `.cpu()` and one uint8 conversion per view.  Here: all views of a rank
                        in one launch (views grouped for L2 reuse of the shared MPI), uint8 HWC frames written by the kernel's
                        epilogue, one device->host copy; with world > 1 the views are sharded (dist.shard_range) and the uint8
                        frames all-gathered (NCCL; gloo in the CPU test).
  dump_fid_images       `fid_evaluation.output_images` (gmpi/fid_evaluation.py:60-135): image k is produced by rank k % world
                        (img_counter = rank; += world_size), rendered from a random pose, converted like torchvision's
                        save_image(normalize=True, range=(-1, 1)) and written as f"{k:0>5}.png".

  render_eval_views     `generate_img` of the evaluation-data dump (gmpi/eval/prepare_fake_data.py:17-95): every MPI of a batch from
                        n_imgs random poses -- the reference expands the batch to B*n_imgs copies of the MPI before rendering
                        (:59-64); here the views index their MPI (`view_group` = n_imgs orders the tiles for L2 reuse).  Returns
                        the reference's triple: uint8 images (truncating conversion, :72-74), fp32 metric depth maps, (pitch, yaw).

The MPI itself comes from the caller (`mpi_source`): the generator is outside the render path.  `render_fn` is injectable so
that the sharding / ordering logic is testable without a GPU (tests/test_service.py); the default is the CUDA renderer.
"""
import os
from typing import Callable, List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.distributed as dist

from .camera import PinholeCamera, cam_params, focal_from_fov, sample_yaw_pitch, sphere_poses
from .dist import shard_range


def sweep_angles(n_views: int = 100, horizontal: bool = True, mean: float = 0.0) -> List[float]:
    """render_video.py:235-240: linspace(0.5, -0.5, n) yaw sweep or linspace(0.3, -0.3, n) pitch sweep, around `mean`."""
    half = 0.5 if horizontal else 0.3
    return [float(a) + mean for a in np.linspace(half, -half, n_views).tolist()]


def _default_video_render(rgba, dhw, c2w, img_size, fov_deg, near, far, fast_rays, factored, stop_transmittance=0.0, skip_alpha=None):
    from .mpi import render_frames
    dev = dhw.device
    V = c2w.shape[0]
    v2m = torch.zeros(V, dtype=torch.int32, device=dev)
    kw = dict(rgb=factored[0], alpha=factored[1], bg_rgb=factored[2]) if factored is not None else dict(rgba=rgba)
    kw.update(stop_transmittance=stop_transmittance, skip_alpha=skip_alpha)     # one call: one occupancy map for the sweep
    if fast_rays:
        cam = cam_params(c2w.to(dev), focal_from_fov(fov_deg, img_size), img_size, img_size)
        return render_frames(dhw=dhw, view2mpi=v2m, cam=cam, H=img_size, W=img_size, video={"near": near, "far": far},
                             check_last_plane=True, view_group=V, **kw)
    ray_dir, eye, z_dir = PinholeCamera.from_fov(fov_deg, img_size, img_size).generate_rays(c2w.to(dev))
    return render_frames(dhw=dhw, view2mpi=v2m, ray_dir=ray_dir, eye=eye, z_dir=z_dir, video={"near": near, "far": far},
                         check_last_plane=True, view_group=V, **kw)


def render_video_frames(mpi_rgba: Optional[torch.Tensor], dhw: torch.Tensor, angles: Sequence[float], *, img_size: int, fov_deg: float,
                        ray_start: float, ray_end: float, sphere_center, sphere_r: float, horizontal: bool = True,
                        other_angle: float = 0.0, fast_rays: bool = False, factored: Optional[Tuple] = None,
                        rank: int = 0, world: int = 1, gather: bool = True, render_fn: Optional[Callable] = None,
                        stop_transmittance: float = 0.0, skip_alpha: Optional[float] = None):
    """All `angles` (yaw sweep if `horizontal`, else pitch sweep; the other angle fixed) of ONE MPI ([1,N,4,T,T], or
    factored=(rgb [1,3,T,T], alpha [1,N,1,T,T], bg_rgb or None)) as uint8 frames.
    Returns (img [V,H,W,3] uint8, depth [V,H,W,1] uint8) as CPU tensors: all V views when `gather` (every rank), else this rank's
    slice [lo, hi) of shard_range(V, rank, world).
    stop_transmittance: early ray termination of the render (see mpi.render_views); handed to `render_fn` as a keyword
    argument when it is not 0, so render functions without the parameter keep working for exact renders.  skip_alpha:
    empty-space skipping (see mpi.render_views), likewise handed on only when it is not None."""
    V = len(angles)
    lo, hi = shard_range(V, rank, world)
    a = torch.tensor(list(angles[lo:hi]), dtype=torch.float32).reshape(-1, 1)
    o = torch.full_like(a, float(other_angle))
    yaws, pitches = (a, o) if horizontal else (o, a)
    c2w = sphere_poses(yaws, pitches, sphere_center, sphere_r)
    fn = render_fn or _default_video_render
    if hi > lo:
        extra = {"stop_transmittance": float(stop_transmittance)} if stop_transmittance else {}
        if skip_alpha is not None:
            extra["skip_alpha"] = float(skip_alpha)
        img, depth = fn(mpi_rgba, dhw, c2w, img_size, fov_deg, ray_start, ray_end, fast_rays, factored, **extra)
    else:
        dev = dhw.device
        img = torch.empty((0, img_size, img_size, 3), dtype=torch.uint8, device=dev)
        depth = torch.empty((0, img_size, img_size, 1), dtype=torch.uint8, device=dev)
    if world == 1 or not gather:
        return img.cpu(), depth.cpu()
    # the one collective: all-gather of uint8 frames (4 bytes per pixel instead of 16), padded to the largest share
    per = -(-V // world)
    packed = torch.zeros((per, img_size, img_size, 4), dtype=torch.uint8, device=img.device)
    packed[: hi - lo, :, :, :3] = img
    packed[: hi - lo, :, :, 3:] = depth
    out = torch.empty((world * per, img_size, img_size, 4), dtype=torch.uint8, device=img.device)
    dist.all_gather_into_tensor(out, packed)
    keep = torch.cat([out[r * per: r * per + (shard_range(V, r, world)[1] - shard_range(V, r, world)[0])] for r in range(world)], 0)
    return keep[..., :3].contiguous().cpu(), keep[..., 3:].contiguous().cpu()


def fid_image_indices(num_imgs: int, rank: int, world: int) -> List[int]:
    """fid_evaluation.py:86,100,129-133: img_counter = rank; while img_counter < num_imgs: ...; img_counter += world_size."""
    return list(range(rank, num_imgs, world))


def _default_fid_render(renderer, batch_mpi, img_size, yaws, pitches):
    from .mpi import render_frames
    dev = batch_mpi.device
    B = batch_mpi.shape[0]
    c2w = sphere_poses(yaws, pitches, renderer.sphere_center, renderer.sphere_r).to(dev)
    cam = PinholeCamera.from_fov(renderer.cam_fov, img_size, img_size)
    ray_dir, eye, z_dir = cam.generate_rays(c2w)
    dhw = renderer.static_mpi_plane_dhws.to(dev).reshape(1, -1, 3).expand(B, -1, -1).contiguous()
    img, _ = render_frames(rgba=batch_mpi, dhw=dhw, view2mpi=torch.arange(B, dtype=torch.int32, device=dev), ray_dir=ray_dir, eye=eye,
                           z_dir=z_dir, video={"near": 0.0, "far": 1.0, "depth": False}, u8_round=True, check_last_plane=True)
    return img


def dump_fid_images(renderer, mpi_source: Callable[[int], torch.Tensor], num_imgs: int, rank: int, world: int, img_size: int,
                    output_dir: Optional[str] = None, writer: Optional[Callable[[int, np.ndarray], None]] = None,
                    h_mean: float = 0.0, h_std: float = 0.289, v_mean: float = 0.0, v_std: float = 0.127,
                    generator: Optional[torch.Generator] = None, render_fn: Optional[Callable] = None) -> List[int]:
    """Rank `rank`'s share of `num_imgs` images: for every call k, `mpi_source(k)` returns a batch [B,N,4,T,T] of MPIs; each is
    rendered from one random pose (truncated Gaussian, as MPIRenderer.render samples it) and converted to uint8 with
    save_image's rounding.  Images are numbered rank, rank + world, ... (the reference's strided file names) and handed to
    `writer(index, hwc_uint8)` or written to output_dir/{index:05d}.png.  Returns the indices written."""
    todo = fid_image_indices(num_imgs, rank, world)
    fn = render_fn or _default_fid_render
    done, k = [], 0
    while len(done) < len(todo):
        batch = mpi_source(k)
        k += 1
        B = batch.shape[0]
        yaws, pitches = sample_yaw_pitch(B, h_mean, h_std, v_mean, v_std, 2, "truncated_gaussian", True, generator=generator)
        imgs = fn(renderer, batch, img_size, yaws, pitches).cpu().numpy()
        for img in imgs:
            if len(done) == len(todo):
                break
            idx = todo[len(done)]
            if writer is not None:
                writer(idx, img)
            elif output_dir is not None:
                from PIL import Image
                os.makedirs(output_dir, exist_ok=True)
                Image.fromarray(img).save(os.path.join(output_dir, f"{idx:0>5}.png"))
            done.append(idx)
    return done


def to_uint8_truncating(img_m11: torch.Tensor) -> torch.Tensor:
    """[-1,1] fp32 -> uint8 as prepare_fake_data.py:72-74 / render_video.py:119-121 convert: clip((x + 1) / 2, 0, 1) * 255,
    truncated (numpy's astype(uint8)); the same fp32 operations, so the bytes are identical."""
    return (torch.clamp((img_m11 + 1) / 2.0, 0.0, 1.0) * 255).to(torch.uint8)


def _default_eval_render(renderer, batch_mpi, n_imgs, img_size, yaws, pitches):
    from .mpi import render_frames
    dev = batch_mpi.device
    B = batch_mpi.shape[0]
    c2w = sphere_poses(yaws, pitches, renderer.sphere_center, renderer.sphere_r).to(dev)
    ray_dir, eye, z_dir = PinholeCamera.from_fov(renderer.cam_fov, img_size, img_size).generate_rays(c2w)
    dhw = renderer.static_mpi_plane_dhws.to(dev).reshape(1, -1, 3).expand(B, -1, -1).contiguous()
    view2mpi = torch.arange(B, dtype=torch.int32, device=dev).repeat_interleave(n_imgs)
    return render_frames(rgba=batch_mpi, dhw=dhw, view2mpi=view2mpi, ray_dir=ray_dir, eye=eye, z_dir=z_dir, check_last_plane=True,
                         view_group=n_imgs)                              # (colour in [-1,1] [V,3,H,W], depth [V,1,H,W])


def render_eval_views(renderer, batch_mpi: torch.Tensor, n_imgs: int, img_size: int, *, generator: Optional[torch.Generator] = None,
                      render_fn: Optional[Callable] = None):
    """batch_mpi [B,N,4,T,T] -> (img uint8 [B*n_imgs,H,W,3], depth fp32 [B*n_imgs,H,W,1], angles fp32 [B*n_imgs,2] = (pitch,
    yaw)) as numpy arrays, views MPI-major (the n_imgs views of MPI 0 first) like the reference's expand.  Poses are drawn
    as MPIRenderer.render draws them for a batch of B*n_imgs (same generator consumption: mpi_renderer.py:418-434)."""
    B = batch_mpi.shape[0]
    V = B * int(n_imgs)
    yaws, pitches = sample_yaw_pitch(V, renderer.horizontal_mean, renderer.horizontal_std, renderer.vertical_mean, renderer.vertical_std,
                                     renderer.cam_pose_n_truncated_stds, renderer.cam_sample_method, True, generator=generator)
    fn = render_fn or _default_eval_render
    img, depth = fn(renderer, batch_mpi, int(n_imgs), img_size, yaws, pitches)
    assert img.shape[0] == V and depth.shape[0] == V, f"{img.shape}, {depth.shape}, {V}"
    img_u8 = to_uint8_truncating(img.permute(0, 2, 3, 1)).cpu().numpy()
    angles = torch.cat([pitches, yaws], dim=-1).numpy()                 # mpi_renderer.py:464
    return img_u8, depth.permute(0, 2, 3, 1).float().cpu().numpy(), angles
