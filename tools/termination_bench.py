#!/usr/bin/env python
"""Early ray termination (stop_transmittance) measured on synthetic workloads:
    python tools/termination_bench.py [--rounds R] [--iters K] [--out FILE]
Shapes: the headline forward (4 MPIs x 1 view, 96 planes, 1024^2), expanded and factored, and the C4 sweep (120 views of ONE
96-plane 512^2 MPI, view_group = 120).  Inputs (synth.make_workload): white-noise alpha, the "surface" head MPI, and alpha = 0
except the last plane (nothing to skip: the cost of the vote alone).  tau in {0, 2^-24, 1/512}.  Every round times each tau
with CUDA events over K launches after warm-ups, the order rotating between rounds so that tau = 0 and tau > 0 alternate (the
boxes throttle under sustained load); medians over rounds.  Prints ONE JSON line: frames/s, the fraction of pixel-planes
skipped, the largest deviation from the tau = 0 render (colour, depth), and the device name and power limit read in the same
run.  No HBM-roofline share: with work skipped the algorithmic byte count no longer applies.  The MPIs are synthetic: what
trained-generator MPIs would gain is not measured here."""
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

TAUS = [("0", 0.0), ("2^-24", 2.0 ** -24), ("1/512", 1.0 / 512)]
KINDS = ["noise", "surface", "empty"]


def device_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["sm_max_mhz"] = float(out[0]), float(out[1])
    except Exception as e:      # the numbers are then reported without it, and say so
        info["power_limit_w"] = f"unavailable: {e}"
    return info


class Workload:
    def __init__(self, shape, kind, dev):
        self.shape = shape
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
        mpi = dict(rgba=case.rgba)
        if shape == "headline_factored":      # one colour image per MPI (plane 0's), the workload's alpha per plane
            self.rgb = case.rgba[:, 0, :3].contiguous()
            self.alpha = case.rgba[:, :, 3:].contiguous()
            mpi = dict(rgb=self.rgb, alpha=self.alpha)
            case.rgba = None
        self.case = case
        self.color = torch.empty((V, 3, H, W), device=dev)
        self.depth = torch.empty((V, 1, H, W), device=dev)
        self.flags = torch.zeros(1, dtype=torch.int32, device=dev)
        self.skipped = torch.zeros(1, dtype=torch.int64, device=dev)
        self.pixel_planes = V * H * W * N
        self.descs = {}
        for name, tau in TAUS:
            self.descs[name] = _lib.make_desc(options=_lib.OPT_ALIGN_CORNERS | _lib.OPT_COLOR_MINUS1_1, M=M, V=V, N=N, Ht=Ht, Wt=Wt,
                                              H=H, W=W, view_group=group, view2mpi=case.view2mpi, dhw=case.dhw, ray_dir=case.ray_dir,
                                              eye=case.eye, z_dir=case.z_dir, color=self.color, depth=self.depth, flags=self.flags,
                                              stream=torch.cuda.current_stream().cuda_stream, stop_transmittance=tau,
                                              skipped_pixel_planes=self.skipped, **mpi)
        self.V = V

    def run(self, lib, name):
        _lib.check(lib.gmpi_mpi_render_fwd_ex(ctypes.byref(self.descs[name])))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--shapes", default="headline_expanded,headline_factored,c4_video_512")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "termination_bench measures on a CUDA device"
    dev = torch.device("cuda:0")
    lib = _lib.load()
    res = {"what": "early ray termination (stop_transmittance), synthetic MPIs; frames/s = views rendered per second "
                   "(kernel time, CUDA events); colour in [-1,1] (deviation bound 2 tau), depth metric",
           **device_info(), "rounds": a.rounds, "iters_per_round": a.iters, "results": {}}
    for shape in a.shapes.split(","):
        for kind in KINDS:
            w = Workload(shape, kind, dev)
            ref = {}
            skip_frac = {}
            for name, _ in TAUS:          # outputs + skip counts (one launch each) before timing
                w.skipped.zero_()
                w.run(lib, name)
                torch.cuda.synchronize()
                ref[name] = (w.color.clone(), w.depth.clone())
                skip_frac[name] = int(w.skipped.item()) / w.pixel_planes
            times = {n: [] for n, _ in TAUS}
            names = [n for n, _ in TAUS]
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
            row = {}
            for n, _ in TAUS:
                ms = statistics.median(times[n])
                row[n] = {"ms": round(ms, 4), "frames_per_s": round(w.V / ms * 1e3, 1),
                          "ms_min_max": [round(min(times[n]), 4), round(max(times[n]), 4)],
                          "skipped_fraction": round(skip_frac[n], 4),
                          "max_dev_color": float((ref["0"][0] - ref[n][0]).abs().max()),
                          "max_dev_depth": float((ref["0"][1] - ref[n][1]).abs().max())}
                row[n]["speedup_vs_tau0"] = round(statistics.median(times["0"]) / ms, 3)
            res["results"][f"{shape}/{kind}"] = row
            print(f"# {shape}/{kind}: " + ", ".join(f"tau={n} {row[n]['frames_per_s']} f/s skip {row[n]['skipped_fraction']}"
                                                     for n, _ in TAUS), file=sys.stderr, flush=True)
            del w
            torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
