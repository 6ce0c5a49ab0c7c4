#!/usr/bin/env python
"""Empty-space skipping (skip_alpha: gmpi_mpi_occupancy + gmpi_mpi_render_fwd_skip_ex) measured on synthetic workloads:
    python tools/empty_skip_bench.py [--rounds R] [--iters K] [--out FILE]
Shapes: the headline forward (4 MPIs x 1 view, 96 planes, 1024^2), expanded and factored, and the C4 sweep (120 views of ONE
96-plane 512^2 MPI, view_group = 120).  Inputs (synth.make_workload): white-noise alpha (nothing is empty), the "surface" head
MPI, alpha = 0 except the last plane, and "haze" (the head with alpha uniform in [0, 2^-12) where it was 0: threshold 0 skips
nothing, 2^-12 skips the haze).  Arms: exact; skip eps = 0; skip eps = 2^-12; tau = 2^-24 (early ray termination alone); skip
eps = 0 with tau = 2^-24.  The occupancy builds (eps = 0 and 2^-12) are timed as arms of their own.  Every round times each arm
with CUDA events over K launches after warm-ups, the order rotating between rounds (the boxes throttle under sustained load);
medians over rounds.  Prints ONE JSON line: kernel time and frames/s per arm, the build time, the per-call sum (build + kernel:
the Python API builds the map on every call), the fractions of pixel-planes skipped as empty and by termination, the largest
deviation from the exact render (colour, depth), and the device name, power limit and SM clocks read in the same run.  The MPIs are
synthetic: what trained-generator MPIs would gain is not measured here."""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

from ml_gmpi_b200 import _lib, synth

EPS = 2.0 ** -12
TAU = 2.0 ** -24
ARMS = [("exact", None, 0.0), ("skip0", 0.0, 0.0), ("skip2^-12", EPS, 0.0), ("tau2^-24", None, TAU), ("skip0+tau2^-24", 0.0, TAU)]
BUILDS = [("build0", 0.0), ("build2^-12", EPS)]
KINDS = ["noise", "surface", "empty", "haze"]


def device_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["sm_max_mhz"], info["sm_mhz_at_start"] = float(out[0]), float(out[1]), float(out[2])
    except Exception as e:      # the numbers are then reported without it, and say so
        info["power_limit_w"] = f"unavailable: {e}"
    return info


class Workload:
    def __init__(self, shape, kind, dev):
        if shape == "c4_video_512":
            V = 120
            case = synth.make_workload(kind, n_planes=96, tex=512, img=512, n_mpi=1, views_per_mpi=V, seed=1234, device=dev,
                                       yaws=np.linspace(0.5, -0.5, V).astype(np.float32), pitches=np.zeros(V, np.float32))
            group = V
        else:
            case = synth.make_workload(kind, n_planes=96, tex=1024, img=1024, n_mpi=4, seed=1234, device=dev)
            group = 1
        M, N, _, Ht, Wt = case.rgba.shape
        V, _, H, W = case.ray_dir.shape
        tex = Ht * Wt
        mpi = dict(rgba=case.rgba)
        # the alpha planes as gmpi_mpi_occupancy reads them: channel 3 of the expanded stack, or the factored alpha
        self.alpha_view = (case.rgba.data_ptr() + 4 * 3 * tex, N * 4 * tex, 4 * tex)
        if shape == "headline_factored":      # one colour image per MPI (plane 0's), the workload's alpha per plane
            self.rgb = case.rgba[:, 0, :3].contiguous()
            self.alpha = case.rgba[:, :, 3:].contiguous()
            mpi = dict(rgb=self.rgb, alpha=self.alpha)
            self.alpha_view = (self.alpha.data_ptr(), N * tex, tex)
            case.rgba = None
        self.case, self.dims = case, (M, N, Ht, Wt)
        self.alpha_bytes = M * N * tex * 4
        self.color = torch.empty((V, 3, H, W), device=dev)
        self.depth = torch.empty((V, 1, H, W), device=dev)
        self.flags = torch.zeros(1, dtype=torch.int32, device=dev)
        self.counts = torch.zeros(2, dtype=torch.int64, device=dev)      # termination, empty
        self.pixel_planes = V * H * W * N
        self.occ = {eps: torch.empty((M, N, (Ht + 7) // 8, (Wt + 511) // 512), dtype=torch.int64, device=dev) for _, eps in BUILDS}
        self.stream = torch.cuda.current_stream().cuda_stream
        self.descs = {}
        for name, _, tau in ARMS:
            self.descs[name] = _lib.make_desc(options=_lib.OPT_ALIGN_CORNERS | _lib.OPT_COLOR_MINUS1_1, M=M, V=V, N=N, Ht=Ht, Wt=Wt,
                                              H=H, W=W, view_group=group, view2mpi=case.view2mpi, dhw=case.dhw, ray_dir=case.ray_dir,
                                              eye=case.eye, z_dir=case.z_dir, color=self.color, depth=self.depth, flags=self.flags,
                                              stream=self.stream, stop_transmittance=tau, skipped_pixel_planes=self.counts[0:1], **mpi)
        self.skip = {name: eps for name, eps, _ in ARMS}
        self.V = V

    def build(self, lib, eps):
        M, N, Ht, Wt = self.dims
        ptr, mpi_stride, plane_stride = self.alpha_view
        _lib.check(lib.gmpi_mpi_occupancy(ptr, mpi_stride, plane_stride, M, N, Ht, Wt, eps, self.occ[eps].data_ptr(), self.stream))

    def run(self, lib, name):
        if name.startswith("build"):
            return self.build(lib, dict(BUILDS)[name])
        eps = self.skip[name]
        if eps is None:
            _lib.check(lib.gmpi_mpi_render_fwd_ex(ctypes.byref(self.descs[name])))
        else:
            _lib.check(lib.gmpi_mpi_render_fwd_skip_ex(ctypes.byref(self.descs[name]), self.occ[eps].data_ptr(), self.counts[1:2].data_ptr()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--shapes", default="headline_expanded,headline_factored,c4_video_512")
    ap.add_argument("--kinds", default=",".join(KINDS))
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "empty_skip_bench measures on a CUDA device"
    dev = torch.device("cuda:0")
    lib = _lib.load()
    res = {"what": "empty-space skipping (skip_alpha), synthetic MPIs; kernel time from CUDA events; frames/s = views rendered per "
                   "second of kernel time; per_call_ms = occupancy build + kernel (what one Python call costs); colour in [-1,1] "
                   "(deviation bound 2 N eps), depth metric; *_fraction = pixel-planes skipped / all pixel-planes",
           **device_info(), "rounds": a.rounds, "iters_per_round": a.iters, "results": {}}
    for shape in a.shapes.split(","):
        for kind in a.kinds.split(","):
            w = Workload(shape, kind, dev)
            for _, eps in BUILDS:
                w.build(lib, eps)
            out, frac = {}, {}
            for name, _, _ in ARMS:          # outputs + counts (one launch each) before timing
                w.counts.zero_()
                w.run(lib, name)
                torch.cuda.synchronize()
                out[name] = (w.color.clone(), w.depth.clone())
                c = w.counts.tolist()
                frac[name] = (c[1] / w.pixel_planes, c[0] / w.pixel_planes)
            names = [n for n, _, _ in ARMS] + [n for n, _ in BUILDS]
            times = {n: [] for n in names}
            for r in range(a.rounds):
                order = names[r % len(names):] + names[: r % len(names)]
                for n in order:
                    for _ in range(a.warmup):
                        w.run(lib, n)
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for _ in range(a.iters):
                        w.run(lib, n)
                    e1.record()
                    torch.cuda.synchronize()
                    times[n].append(e0.elapsed_time(e1) / a.iters)
                time.sleep(0.2)
            med = {n: statistics.median(times[n]) for n in names}
            row = {"builds": {n: {"ms": round(med[n], 4), "ms_min_max": [round(min(times[n]), 4), round(max(times[n]), 4)],
                                  "alpha_gb_per_s": round(w.alpha_bytes / med[n] / 1e6, 1)} for n, _ in BUILDS}}
            for name, eps, tau in ARMS:
                ms = med[name]
                build = med["build0" if eps == 0.0 else "build2^-12"] if eps is not None else 0.0
                row[name] = {"ms": round(ms, 4), "frames_per_s": round(w.V / ms * 1e3, 1),
                             "ms_min_max": [round(min(times[name]), 4), round(max(times[name]), 4)],
                             "per_call_ms": round(ms + build, 4),
                             "speedup_kernel": round(med["exact"] / ms, 3), "speedup_per_call": round(med["exact"] / (ms + build), 3),
                             "empty_fraction": round(frac[name][0], 4), "terminated_fraction": round(frac[name][1], 4),
                             "max_dev_color": float((out["exact"][0] - out[name][0]).abs().max()),
                             "max_dev_depth": float((out["exact"][1] - out[name][1]).abs().max())}
            res["results"][f"{shape}/{kind}"] = row
            print(f"# {shape}/{kind}: build {row['builds']['build0']['ms']} ms; " +
                  ", ".join(f"{n} {row[n]['ms']} ms (x{row[n]['speedup_kernel']}) empty {row[n]['empty_fraction']}" for n, _, _ in ARMS),
                  file=sys.stderr, flush=True)
            del w, out
            torch.cuda.empty_cache()
    res["sm_mhz_at_end"] = device_info().get("sm_mhz_at_start")
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
