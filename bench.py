#!/usr/bin/env python
"""bench.py -- MPI frames/s (96 planes, 1024^2) on N B200s, with roofline, end-to-end, CPU-baseline and config legs.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Headline workload (BASELINE.json configs[2], "FFHQ1024"): per GPU a batch of 4 MPIs, 96 planes, 1024^2 textures, one
1024^2 view per MPI, random RGBA in [0,1), FFHQ geometry, in-envelope poses (SURVEY.md section 8d).  One "step" renders
the batch (4 frames: RGB + depth).  Views are sharded across ranks (weak scaling: 4 frames per GPU) and the step ends
with the ONE collective of the path, the all-gather of frames, fused into the render kernel's epilogue (peer stores into
symmetric memory) or, where symmetric memory is unavailable, an ncclAllGather.  `value` = frames/s, whole job, inputs
resident in HBM.

Keys beyond the base contract:
  roofline      dominant kernel vs the measured HBM copy peak (MEASURED_PEAKS.json), algorithmic bytes of SURVEY.md 8(d)
  e2e           host buffers -> C-ABI host entry point -> host frames, copies inside the timed region
  train_step    forward+backward through the autograd Function (BASELINE configs[2] is fwd+bwd)
  configs       the other BASELINE configs, briefly: C2 (32 planes, 256^2, batch 8), C4 (video: 120 views of ONE 96x512^2 MPI
                sharded over the ranks, strong scaling), C5 (train step at 96x512^2, batch 4 per GPU)
  cpu_baseline  the reference's PyTorch op sequence (oracle/torch_port.py) on this box's host cores (N=1 only)
  reference_on_gpu  the same op sequence on one B200 (torch kernels): the honest competitor (N=1 only)

The GPU-specific calls live behind a small backend object so that tests/test_bench_flow.py can drive this file's whole
control flow for world_size 2 on CPU (gloo) with a fake backend: the N>1 path must never again ship untested.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_PLANES, RES, BATCH = 96, 1024, 4
WORKLOAD = "FFHQ1024: 96 planes, 1024^2 textures and views, 4 MPIs x 1 view per GPU, forward render"
METRIC = "MPI frames/s (96 planes, 1024^2)"
VIDEO_VIEWS = 120
DUMP_MAX_BYTES = 64 * 10**6       # --dump-outputs: the headline's 4 x 1024^2 frames (67 MB) are sampled to fit


def algorithmic_bytes_fwd(n, ht, wt, h, w):
    return 16 * n * ht * wt + 16 * h * w            # SURVEY.md 8(d): read every texel once, write RGB+depth


def algorithmic_bytes_bwd(n, ht, wt, h, w):
    return 2 * 16 * n * ht * wt + 16 * h * w        # re-read the MPI, write d rgba once, read upstream grads


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy kernel)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def usable_cores():
    """Host threads this process may really use: CPU affinity, capped by the cgroup CPU quota (a container with 128
    visible CPUs and a 32-CPU quota runs 128 torch threads 4x oversubscribed: the 10x box-to-box spread of round 1)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period))))
    except Exception:
        pass
    return n


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0=None, t1=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        inside = [r for (ts, r) in self.rows if t0 is not None and t0 <= ts <= t1 + 0.03]
        window = "timed region"
        if not inside:      # timed region shorter than the sampling period: use everything since warm-up started
            inside, window = [r for (_, r) in self.rows], "warm-up + timed region"
        for r in inside:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": window}


# ----------------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's torch op sequence on the host cores
# ----------------------------------------------------------------------------------------------------------------
def cpu_reference_frames_per_s(steps, warmup, budget_s, planes=N_PLANES, res=RES):
    """Times oracle/torch_port (== MPIRenderer.render's arithmetic) for ONE frame of the headline workload on the host.

    A frame = the per-call range scan of the MPI (mpi_renderer.py:447-449, timed on its own, once per frame) + the render
    of all `res` image rows.  If a full frame fits the budget it is timed whole; otherwise the render is timed on row
    blocks SPREAD over the frame (8-row blocks at evenly spaced offsets, so oblique border rows are represented) and
    scaled by res/rows -- the scan is not scaled.  Threads = the cores this process can actually use.
    Returns dict(value frames/s, sample, cores, ms_per_step, spread)."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import torch_port
    from ml_gmpi_b200 import synth
    cores = usable_cores()
    torch.set_num_threads(cores)
    case = synth.make_case(n_planes=planes, tex=res, img=res, n_mpi=1, seed=1234, device="cpu")
    dhw = case.dhw[:1]

    def scan():
        t0 = time.perf_counter()
        ok = bool(torch.min(case.rgba) >= 0.0) and bool(torch.max(case.rgba) <= 1.0)          # mpi_renderer.py:447-449
        assert ok
        return time.perf_counter() - t0

    def rows_index(rows):
        nblk = max(1, rows // 8)
        starts = [int(round(k * (res - 8) / max(nblk - 1, 1))) for k in range(nblk)] if nblk > 1 else [(res - 8) // 2]
        return torch.tensor([s + j for s in starts for j in range(8)], dtype=torch.long)

    def render_rows(idx):
        ray = case.ray_dir if idx is None else case.ray_dir[:, :, idx, :].contiguous()
        t0 = time.perf_counter()
        with torch.no_grad():
            color, depth = torch_port.render_views(case.rgba, dhw, [ray], [case.eye], [case.z_dir], True)
            img = 2 * color - 1                                                               # mpi_renderer.py:467
        del img, depth
        return time.perf_counter() - t0

    scan()
    render_rows(rows_index(8))                                                                 # page in
    t_scan = min(scan() for _ in range(2))
    per_row = render_rows(rows_index(32)) / 32.0
    n_runs = max(steps + warmup, 1)
    est_full = t_scan + per_row * res
    if est_full * n_runs <= budget_s:
        idx, rows = None, res
    else:
        rows = int(max(8, min(res, (budget_s / n_runs - t_scan) / per_row)))
        rows -= rows % 8
        rows = max(rows, 8)
        idx = rows_index(rows) if rows < res else None
        rows = res if idx is None else rows
    for _ in range(warmup):
        render_rows(idx)
    ts = [render_rows(idx) for _ in range(max(steps, 1))]
    frame_ts = [t_scan + t * (res / rows) for t in ts]
    t = statistics.median(frame_ts)
    spread = (max(frame_ts) - min(frame_ts)) / t if len(frame_ts) > 1 else 0.0
    what = "whole frame" if rows == res else f"{rows} of {res} rows in 8-row blocks spread over the frame, scaled by {res}/{rows}"
    sample = (f"1 frame (1 MPI, {planes} planes, {res}^2 texture and view), forward, no_grad: range scan {t_scan * 1e3:.0f} ms (once per "
              f"frame, not scaled) + render of {what}; torch {torch.__version__} CPU ops on {cores} threads; {len(ts)} timed runs, "
              f"median {t:.2f} s per frame, run-to-run spread {100 * spread:.0f} %")
    return {"value": 1.0 / t, "sample": sample, "cores": cores, "ms_per_step": t * 1e3, "spread": spread}


def headline_config(NP, R, B, world):
    """`config` of the JSON line: the workload only, so that both arms (`--impl reference` included) print the same object."""
    default = (NP, R, B) == (N_PLANES, RES, BATCH)
    return {"workload": WORKLOAD if default else f"{NP} planes, {R}^2, {B} MPIs x 1 view per GPU, forward render",
            "planes": NP, "tex": R, "img": R, "mpis_per_gpu": B, "views_per_gpu": B,
            "parallelism": f"views sharded x{world}: every GPU renders its own {B} MPIs x 1 view; one all-gather of frames per step when x > 1",
            "l2": f"inputs {B * NP * 4 * R * R * 4 / 1e9:.2f} GB per GPU >> 126 MB L2 (no flush needed)"}


def run_reference_arm(args, out):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference_frames_per_s(args.steps, args.warmup, budget_s=args.ref_budget_s)
    fps = r["value"]
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": headline_config(N_PLANES, RES, BATCH, args.gpus), "device": "host CPU",
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": r["cores"], "kind": "port", "sample": r["sample"],
                         "spread": r["spread"], "stable": r["spread"] < 0.2},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    out.emit(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------------
# backends: everything that touches a GPU (or pretends to, for the CPU control-flow test)
# ----------------------------------------------------------------------------------------------------------------
class CudaBackend:
    """The real thing: cuda:LOCAL_RANK, NCCL, the C-ABI library.  No CPU fallback."""
    name = "cuda"

    def __init__(self, local):
        import torch
        import ml_gmpi_b200 as g
        from ml_gmpi_b200 import _lib, synth, dist as gdist, host_api
        assert torch.cuda.is_available(), "bench.py (impl ours) needs a CUDA device; there is no CPU fallback"
        self.torch, self.g, self._lib, self.synth, self.gdist, self.host_api = torch, g, _lib, synth, gdist, host_api
        torch.cuda.set_device(local)
        self.local = local
        self.device = torch.device("cuda", local)
        self.lib = _lib.load()
        self.stream = torch.cuda.current_stream(self.device)
        self.dist_backend = "nccl"

    def init_dist(self):
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=self.device)

    def sizes(self, planes, res, batch):
        return planes, res, batch

    def make_case(self, **kw):
        return self.synth.make_case(device=self.device, **kw)

    def empty(self, shape):
        return self.torch.empty(shape, device=self.device, dtype=self.torch.float32)

    def event(self):
        return self.torch.cuda.Event(enable_timing=True)

    def record(self, ev):
        ev.record(self.stream)

    def elapsed_ms(self, a, b):
        return a.elapsed_time(b)

    def synchronize(self):
        self.torch.cuda.synchronize(self.device)

    def opts(self, check_last=True, minus1_1=True):
        L = self._lib
        return L.OPT_ALIGN_CORNERS | (L.OPT_CHECK_LAST_PLANE if check_last else 0) | (L.OPT_COLOR_MINUS1_1 if minus1_1 else 0)

    def render(self, case, color, depth, flags, view_group=1, factored=None):
        """One forward launch through the descriptor entry point.  factored = (rgb, alpha): the generator's factored MPI."""
        import ctypes
        V, _, H, W = case.ray_dir.shape
        ref = factored[1] if factored is not None else case.rgba
        M, N = ref.shape[0], ref.shape[1]
        Ht, Wt = ref.shape[-2:]
        d = self._lib.make_desc(options=self.opts(), M=M, V=V, N=N, Ht=Ht, Wt=Wt, H=H, W=W, view_group=view_group,
                                rgba=None if factored is not None else case.rgba, rgb=factored[0] if factored is not None else None,
                                alpha=factored[1] if factored is not None else None, view2mpi=case.view2mpi, dhw=case.dhw,
                                ray_dir=case.ray_dir, eye=case.eye, z_dir=case.z_dir, color=color, depth=depth, flags=flags,
                                stream=self.stream.cuda_stream)
        self._lib.check(self.lib.gmpi_mpi_render_fwd_ex(ctypes.byref(d)))

    def make_factored(self, n_mpi, n_planes, tex, seed):
        t = self.torch
        gen = t.Generator(device=self.device).manual_seed(seed)
        rgb = t.rand((n_mpi, 3, tex, tex), generator=gen, device=self.device)
        alpha = t.rand((n_mpi, n_planes, 1, tex, tex), generator=gen, device=self.device)
        return rgb, alpha

    def render_host_video(self, h, n_views, res, near, far):
        """Host buffers (factored MPI + cam [V,16]) -> uint8 video frames in host memory, one C-ABI call."""
        import ctypes
        import numpy as np
        flags = np.zeros(1, np.uint32)
        N = h["alpha"].shape[1]
        T = h["alpha"].shape[-1]
        d = self._lib.make_desc(options=self.opts(), M=1, V=n_views, N=N, Ht=T, Wt=T, H=res, W=res, view_group=n_views,
                                depth_near=float(np.float32(near)), depth_range=float(np.float32(far - near)), rgb=h["rgb"],
                                alpha=h["alpha"], view2mpi=h["view2mpi"], dhw=h["dhw"], cam=h["cam"], video_rgb=h["out_rgb"],
                                video_depth=h["out_depth"], flags=flags.ctypes.data)
        self._lib.check(self.lib.gmpi_mpi_render_host_ex(ctypes.byref(d), self.local))
        return int(flags[0])

    def render_host_factored(self, h, case_shapes):
        import ctypes
        import numpy as np
        flags = np.zeros(1, np.uint32)
        M, N, T, V, R = case_shapes
        d = self._lib.make_desc(options=self.opts(), M=M, V=V, N=N, Ht=T, Wt=T, H=R, W=R, rgb=h["rgb"], alpha=h["alpha"],
                                view2mpi=h["view2mpi"], dhw=h["dhw"], ray_dir=h["ray_dir"], eye=h["eye"], z_dir=h["z_dir"],
                                color=h["color"], depth=h["depth"], flags=flags.ctypes.data)
        self._lib.check(self.lib.gmpi_mpi_render_host_ex(ctypes.byref(d), self.local))
        return int(flags[0])

    def pin(self, t):
        return t.detach().cpu().pin_memory()

    def make_gather(self, frames_per_rank, H, W):
        return self.gdist.FrameGather(frames_per_rank, H, W, self.device)

    def gather_render(self, gather, case, flags):
        gather.render(case.rgba, case.dhw, case.view2mpi, case.ray_dir, case.eye, case.z_dir, flags, check_last_plane=True,
                      color_minus1_1=True)

    def render_views(self, rgba, case):
        return self.g.render_views(rgba, case.dhw, case.view2mpi, case.ray_dir, case.eye, case.z_dir, color_minus1_1=True)

    def host_case(self, case):
        t = self.torch
        h_rgba = t.empty(case.rgba.shape, dtype=t.float32).pin_memory()
        h_rgba.copy_(case.rgba)
        hc = {k: getattr(case, k).cpu().pin_memory() for k in ("dhw", "view2mpi", "ray_dir", "eye", "z_dir")}
        hc["rgba"] = h_rgba
        V, _, H, W = case.ray_dir.shape
        hc["color"] = t.empty((V, 3, H, W), dtype=t.float32).pin_memory()
        hc["depth"] = t.empty((V, 1, H, W), dtype=t.float32).pin_memory()
        return hc

    def render_host(self, hc):
        return self.host_api.render_host(hc["rgba"], hc["dhw"], hc["view2mpi"], hc["ray_dir"], hc["eye"], hc["z_dir"],
                                         check_last_plane=True, color_minus1_1=True, device=self.local, out_color=hc["color"],
                                         out_depth=hc["depth"])

    def release_host(self):
        self.lib.gmpi_mpi_release_host_cache()
        self.torch.cuda.empty_cache()

    def fwd_variant(self, N, Ht, Wt, H, W):
        return self.lib.gmpi_mpi_render_fwd_variant(N, Ht, Wt, H, W).decode()

    def reference_on_gpu(self, planes, res):
        """oracle/torch_port (the reference's op sequence) on this GPU, one view: the library-kernel competitor."""
        t = self.torch
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import torch_port
        case = self.make_case(n_planes=planes, tex=res, img=res, n_mpi=1, seed=1234)

        def run():
            with t.no_grad():
                assert bool(t.min(case.rgba) >= 0.0) and bool(t.max(case.rgba) <= 1.0)       # mpi_renderer.py:447-449 (2 syncs)
                c, d = torch_port.render_views(case.rgba, case.dhw[:1], [case.ray_dir], [case.eye], [case.z_dir], True)
                return 2 * c - 1, d
        run(); run()
        self.synchronize()
        e0, e1 = self.event(), self.event()
        n = 3
        self.record(e0)
        for _ in range(n):
            run()
        self.record(e1)
        self.synchronize()
        ms = self.elapsed_ms(e0, e1) / n
        peak_gb = t.cuda.max_memory_allocated(self.device) / 1e9
        del case
        t.cuda.empty_cache()
        return {"value": 1e3 / ms, "unit": "frames/s", "ms_per_frame": ms, "kind": "port on cuda (torch ATen kernels: grid_sampler_2d, "
                "cumprod, elementwise)", "sample": f"1 view, {planes} planes, {res}^2, forward, no_grad, incl. the range scan; {n} timed runs",
                "peak_mem_gb": peak_gb}


class FakeBackend:
    """CPU stand-in used ONLY by tests/test_bench_flow.py (--fake): gloo, tiny sizes, deterministic fills instead of
    renders.  It exercises this file's control flow (legs, gather modes, checks, JSON), not the renderer."""
    name = "fake"

    def __init__(self, local):
        import torch
        from ml_gmpi_b200 import synth, dist as gdist
        self.torch, self.synth, self.gdist = torch, synth, gdist
        self.local = local
        self.device = torch.device("cpu")
        self.dist_backend = "gloo"
        self.rank = int(os.environ.get("RANK", "0"))
        print("[fake backend] a library banner on stdout, as NCCL prints one")     # must not reach the real stdout

    def init_dist(self):
        import torch.distributed as dist
        dist.init_process_group("gloo")

    def sizes(self, planes, res, batch):
        return 2, 16, 2

    def make_case(self, **kw):
        return self.synth.make_case(device="cpu", **kw)

    def empty(self, shape):
        return self.torch.empty(shape, dtype=self.torch.float32)

    def event(self):
        return [0.0]

    def record(self, ev):
        ev[0] = time.perf_counter()

    def elapsed_ms(self, a, b):
        return max((b[0] - a[0]) * 1e3, 1e-6)

    def synchronize(self):
        pass

    def _fill(self, case):
        V, _, H, W = case.ray_dir.shape
        base = case.ray_dir[:, :1].abs() + float(case.rgba.flatten()[0])
        return base.expand(V, 3, H, W).contiguous(), base.clone()

    def render(self, case, color, depth, flags, view_group=1, factored=None):
        c, d = self._fill(case) if factored is None else self._fill_from(case, factored[1])
        color.copy_(c); depth.copy_(d)

    def _fill_from(self, case, ref):
        V, _, H, W = case.ray_dir.shape
        base = case.ray_dir[:, :1].abs() + float(ref.flatten()[0])
        return base.expand(V, 3, H, W).contiguous(), base.clone()

    def make_factored(self, n_mpi, n_planes, tex, seed):
        gen = self.torch.Generator().manual_seed(seed)
        return self.torch.rand((n_mpi, 3, tex, tex), generator=gen), self.torch.rand((n_mpi, n_planes, 1, tex, tex), generator=gen)

    def render_host_video(self, h, n_views, res, near, far):
        h["out_rgb"].fill_(7); h["out_depth"].fill_(9)
        return 0

    def render_host_factored(self, h, case_shapes):
        c, d = self._fill_from(h["_case"], h["alpha"])
        h["color"].copy_(c); h["depth"].copy_(d)
        return 0

    def pin(self, t):
        return t.detach().clone()

    def make_gather(self, frames_per_rank, H, W):
        if os.environ.get("GMPI_FAKE_NO_SYMM"):
            raise RuntimeError("symmetric memory unavailable (fake)")
        return _FakeGather(self, frames_per_rank, H, W)

    def gather_render(self, gather, case, flags):
        c, d = self._fill(case)
        gather.local = self.torch.cat([c, d], 1)

    def render_views(self, rgba, case):
        c, d = self._fill(case)
        s = rgba.mean()
        return c * s, d * s

    def host_case(self, case):
        hc = {k: getattr(case, k) for k in ("rgba", "dhw", "view2mpi", "ray_dir", "eye", "z_dir")}
        V, _, H, W = case.ray_dir.shape
        hc["color"], hc["depth"], hc["_case"] = self.empty((V, 3, H, W)), self.empty((V, 1, H, W)), case
        return hc

    def render_host(self, hc):
        self.render(hc["_case"], hc["color"], hc["depth"], None)
        return hc["color"], hc["depth"], 0

    def release_host(self):
        pass

    def fwd_variant(self, *a):
        return "fake"

    def reference_on_gpu(self, planes, res):
        return None


class _FakeGather:
    def __init__(self, be, frames_per_rank, H, W):
        import torch.distributed as dist
        self.be, self.dist = be, dist
        self.world, self.rank = dist.get_world_size(), dist.get_rank()
        self.frames_per_rank = frames_per_rank
        self.frames = be.empty((self.world * frames_per_rank, 4, H, W))
        self.local = None

    def finish(self):
        t = self.be.torch
        pad = t.zeros((self.frames_per_rank,) + tuple(self.frames.shape[1:]))
        pad[: self.local.shape[0]] = self.local
        self.dist.all_gather_into_tensor(self.frames, pad)


# ----------------------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------------------
class Job:
    """One bench process: rank bookkeeping + barrier/reduction helpers shared by all legs."""

    def __init__(self, be, world, rank):
        self.be, self.world, self.rank = be, world, rank

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        self.be.synchronize()

    def max_over_ranks(self, values):
        t = self.be.torch.tensor(list(values), dtype=self.be.torch.float64, device=self.be.device)
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t]

    def timed(self, fn, steps, warmup=2):
        """ms per call of fn(), CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks."""
        for _ in range(warmup):
            fn()
        self.barrier()
        e0, e1 = self.be.event(), self.be.event()
        self.be.record(e0)
        for _ in range(steps):
            fn()
        self.be.record(e1)
        self.barrier()
        return self.max_over_ranks([self.be.elapsed_ms(e0, e1) / steps])[0]


def make_gather_or_fallback(job, frames_per_rank, H, W):
    """(gather, mode text).  gather is None when symmetric memory is unavailable: render, then ncclAllGather."""
    be = job.be
    if job.world == 1:
        return None, "none"
    try:    # all-gather fused into the render epilogue: peer stores into symmetric memory over NVLink
        gather = be.make_gather(frames_per_rank, H, W)
        how = ("one float4 store per quad to the NVLS multicast address, the switch replicates" if getattr(gather, "multicast", False)
               else "float4 peer stores into every rank's symmetric-memory buffer")
        return gather, f"fused: render epilogue, {how} (NVLink), double-buffered, 1 device barrier per step"
    except Exception as ex:
        if job.rank == 0:
            print(f"[bench] symmetric memory unavailable ({type(ex).__name__}: {ex}); using ncclAllGather", file=sys.stderr)
        return None, "render, then one ncclAllGather of [V,4,H,W] frames"


def leg_headline(job, args, NP, R, B):
    """The metric: forward render of B MPIs x 1 view per GPU (+ the fused all-gather at N>1).  Returns the result dict and
    the state later legs reuse (case, device-resident result of the last step)."""
    import torch.distributed as dist
    be, world, rank = job.be, job.world, job.rank
    torch = be.torch
    case = be.make_case(n_planes=NP, tex=R, img=R, n_mpi=B, seed=1234 + rank)
    flags = torch.zeros(1, dtype=torch.int32, device=be.device)
    color, depth = be.empty((B, 3, R, R)), be.empty((B, 1, R, R))
    gather, gather_mode = make_gather_or_fallback(job, B, R, R)
    frames_all = frames_local = None
    if world > 1 and gather is None:
        frames_all, frames_local = be.empty((world * B, 4, R, R)), be.empty((B, 4, R, R))
    launches = [0]

    def step(kev=None):
        if gather is not None:   # the one collective of the path, fused into the kernel
            be.gather_render(gather, case, flags)
            launches[0] += 1
            if kev is not None:
                be.record(kev)
            gather.finish()
        else:
            be.render(case, color, depth, flags)
            launches[0] += 1
            if kev is not None:
                be.record(kev)
            if world > 1:
                frames_local[:, :3].copy_(color); frames_local[:, 3:].copy_(depth)
                dist.all_gather_into_tensor(frames_all, frames_local)

    sampler = ClockSampler(be.local)
    if rank == 0 and be.name == "cuda":
        sampler.start()
    # W warm-up steps, then K timed ones: a BURST measurement, like the copy peak it is compared with (MEASURED_PEAKS.json: best of
    # 10).  These boxes shed ~5 % of kernel speed within a few hundred ms of sustained load (tools/fwd_ab.py shows it for any
    # build), so no extra spin-up here: it would only move the timed region into the throttled regime.
    for _ in range(args.warmup):
        step()
    job.barrier()
    assert int(flags.item()) == 0, f"render flagged {int(flags.item())} on the synthetic workload"

    # --- timed region: whole step (render [+ all-gather]), CUDA events, max over ranks ---
    ev0, ev1 = be.event(), be.event()
    kev = [(be.event(), be.event()) for _ in range(args.steps)]
    job.barrier()
    launches[0] = 0
    t_wall0 = time.time()
    be.record(ev0)
    for i in range(args.steps):
        be.record(kev[i][0])
        step(kev[i][1])
    be.record(ev1)
    job.barrier()
    t_wall1 = time.time()
    clocks = sampler.stop(t_wall0, t_wall1) if (rank == 0 and be.name == "cuda") else None
    total_ms = be.elapsed_ms(ev0, ev1)
    kernel_ms = sum(be.elapsed_ms(a, b) for a, b in kev) / args.steps
    total_ms, kernel_ms = job.max_over_ranks([total_ms, kernel_ms])
    ms_per_step = total_ms / args.steps
    # device-resident result of the last step, for the e2e cross-check; `frames` = every rank's frames after the all-gather
    if gather is not None:
        mine = gather.frames[rank * B:(rank + 1) * B]
        res_color, res_depth = mine[:, :3], mine[:, 3:]
        frames = gather.frames
    else:
        res_color, res_depth = color, depth
        frames = frames_all
    peak, peak_src = measured_peak()
    alg = algorithmic_bytes_fwd(NP, R, R, R, R) * B
    achieved = alg / (kernel_ms * 1e-3) / 1e9
    traffic, traffic_src = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f)
        traffic = tj.get("fwd_dram_bytes_per_launch")
        traffic_src = "static: " + tj.get("source", "ncu --set full capture committed under profiles/ (not measured in this run)")
    except Exception:
        pass
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_source": traffic_src, "kernel": be.fwd_variant(NP, R, R, R, R), "kernel_ms": kernel_ms,
                "algorithmic_bytes_per_launch": alg, "peak_source": peak_src}
    out = {"frames_per_s": world * B / (ms_per_step * 1e-3), "ms_per_step": ms_per_step, "clocks": clocks, "launches": launches[0],
           "roofline": roofline, "gather_mode": gather_mode}
    return out, {"case": case, "color": res_color, "depth": res_depth, "gather": gather, "frames": frames}


def dump_outputs(dirname, color, depth, max_bytes=DUMP_MAX_BYTES):
    """Writes a headline step's frames as float32 .npy files, so that two builds run with the same arguments (hence the same
    seeded inputs) can be compared output for output.  Pixels p = (view * H + y) * W + x of color [V,3,H,W] and depth
    [V,1,H,W] go to color.npy [P,3], depth.npy [P] and pixel_index.npy [P] (p as float64).  When all pixels would exceed
    max_bytes, P is a fixed sample (seed 0, sorted) of as many pixels as fit.  Returns {name: shape}."""
    import numpy as np
    import torch
    V, _, H, W = color.shape
    n_pix = V * H * W
    per_pixel = 3 * 4 + 4 + 8
    budget = max_bytes - 3 * 1024                  # room for the three .npy headers
    if n_pix * per_pixel <= budget:
        idx = np.arange(n_pix)
    else:
        idx = np.sort(np.random.default_rng(0).choice(n_pix, budget // per_pixel, replace=False))
    sel = torch.from_numpy(idx).to(color.device)
    out = {"color": color.permute(0, 2, 3, 1).reshape(n_pix, 3).index_select(0, sel),
           "depth": depth.reshape(n_pix).index_select(0, sel)}
    out = {k: v.float().cpu().numpy() for k, v in out.items()}
    out["pixel_index"] = idx.astype(np.float64)
    os.makedirs(dirname, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(dirname, k + ".npy"), v)
    return {k: list(v.shape) for k, v in out.items()}


def leg_train(job, case, steps, NP, R, B):
    """forward+backward (BASELINE configs[2] and [4] are fwd+bwd): autograd Function, grad w.r.t. rgba."""
    be = job.be
    torch = be.torch
    peak, _ = measured_peak()
    rg = case.rgba.requires_grad_(True)
    gcol = torch.randn((B, 3, R, R), device=be.device)

    def fb():
        rg.grad = None
        c, _ = be.render_views(rg, case)
        (c * gcol).sum().backward()
    ms = job.timed(fb, steps, warmup=2)
    assert rg.grad is not None and bool(torch.isfinite(rg.grad.flatten()[:1024]).all())
    algfb = (algorithmic_bytes_fwd(NP, R, R, R, R) + algorithmic_bytes_bwd(NP, R, R, R, R)) * B
    case.rgba.requires_grad_(False)
    rg.grad = None
    return {"value": job.world * B / (ms * 1e-3), "unit": "frames/s (forward+backward, d/d rgba)", "ms_per_step": ms,
            "steps": steps, "roofline_frac": algfb / (ms * 1e-3) / 1e9 / peak,
            "note": "includes the torch (c*g).sum() loss kernels; the gradient buffer is zeroed inside the step"}


def leg_e2e(job, state, steps, B):
    """pinned HOST buffers -> C-ABI host entry point -> pinned host frames; compared with the device-resident result."""
    be = job.be
    torch = be.torch
    hc = be.host_case(state["case"])
    be.render_host(hc)
    job.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        _, _, fl = be.render_host(hc)
    job.barrier()
    dt = job.max_over_ranks([(time.perf_counter() - t0) / steps])[0]
    assert fl == 0
    same = torch.equal(hc["color"].to(be.device), state["color"]) and torch.equal(hc["depth"].to(be.device), state["depth"])
    assert same, "e2e result differs from the device-resident run"
    h2d = sum(int(hc[k].numel()) * hc[k].element_size() for k in ("rgba", "dhw", "view2mpi", "ray_dir", "eye", "z_dir"))
    d2h = (hc["color"].numel() + hc["depth"].numel()) * 4 + 4
    # the same step from the generator's FACTORED output (shared colour + per-plane alpha): 4x fewer bytes over PCIe
    case = state["case"]
    M, N = case.rgba.shape[0], case.rgba.shape[1]
    T, R = case.rgba.shape[-1], case.ray_dir.shape[-1]
    rgb, alpha = be.make_factored(M, N, T, 4242 + job.rank)
    hf = {"rgb": be.pin(rgb), "alpha": be.pin(alpha), "color": hc["color"], "depth": hc["depth"], "_case": case}
    for k in ("dhw", "view2mpi", "ray_dir", "eye", "z_dir"):
        hf[k] = hc[k]
    shapes = (M, N, T, B, R)
    be.render_host_factored(hf, shapes)
    fcol, fdep = be.empty((B, 3, R, R)), be.empty((B, 1, R, R))
    fflags = torch.zeros(1, dtype=torch.int32, device=be.device)
    be.render(case, fcol, fdep, fflags, factored=(rgb, alpha))
    be.synchronize()
    same_f = torch.equal(hf["color"].to(be.device), fcol) and torch.equal(hf["depth"].to(be.device), fdep)
    assert same_f, "factored e2e result differs from the device-resident factored run"
    job.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        flf = be.render_host_factored(hf, shapes)
    job.barrier()
    dtf = job.max_over_ranks([(time.perf_counter() - t0) / steps])[0]
    assert flf == 0
    h2df = sum(int(hf[k].numel()) * hf[k].element_size() for k in ("rgb", "alpha", "dhw", "view2mpi", "ray_dir", "eye", "z_dir"))
    factored = {"value": job.world * B / dtf, "unit": "frames/s", "h2d_bytes_per_step": h2df, "d2h_bytes_per_step": d2h,
                "ms_per_step": dtf * 1e3, "h2d_gbs": h2df / dtf / 1e9, "matches_device_resident_run": True,
                "form": "rgb [M,3,T,T] + alpha [M,N,1,T,T] (networks_cond_on_pos_enc.py:950-975) -> gmpi_mpi_render_host_ex"}
    del hc, hf, rgb, alpha, fcol, fdep
    be.release_host()
    return {"factored_input": factored, "value": job.world * B / dt, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": steps,
            "ms_per_step": dt * 1e3, "api": "ml_gmpi_b200.host_api.render_host -> gmpi_mpi_render_fwd_host (C ABI)",
            "h2d_gbs": h2d / dt / 1e9, "matches_device_resident_run": True}


def leg_configs(job, args):
    """The other BASELINE.json configs, a few steps each (the headline keeps the step budget)."""
    import torch.distributed as dist
    be, world, rank = job.be, job.world, job.rank
    torch = be.torch
    peak, _ = measured_peak()
    out = {}
    steps = max(3, min(args.steps, 10))

    # C2: FFHQ256, 32 planes, 256^2, batch 8, forward only
    NP, R, B = be.sizes(32, 256, 8)
    case = be.make_case(n_planes=NP, tex=R, img=R, n_mpi=B, seed=1234 + rank)
    flags = torch.zeros(1, dtype=torch.int32, device=be.device)
    color, depth = be.empty((B, 3, R, R)), be.empty((B, 1, R, R))
    ms = job.timed(lambda: be.render(case, color, depth, flags), steps * 5, warmup=3)
    alg = algorithmic_bytes_fwd(NP, R, R, R, R) * B
    out["C2_ffhq256_fwd"] = {"workload": f"{NP} planes, {R}^2, batch {B} per GPU, forward", "frames_per_s": world * B / (ms * 1e-3),
                             "ms_per_step": ms, "roofline_frac": alg / (ms * 1e-3) / 1e9 / peak,
                             "note": "34.6 MB per frame: the whole batch sits in L2, launch/tail bound", "kernel": be.fwd_variant(NP, R, R, R, R)}
    assert int(flags.item()) == 0
    del case, color, depth

    # N1: the headline shape rendered from the generator's FACTORED output (shared colour + per-plane alpha): same frames, a
    # quarter of the HBM bytes (the colour image lives in L2) -- the kernel is bound by its shared-memory tap path, so frames/s
    # barely moves while the DRAM traffic drops (ncu: profiles/README.md)
    NP, R, B = be.sizes(args.planes, args.res, args.batch)
    case = be.make_case(n_planes=NP, tex=R, img=R, n_mpi=B, seed=1234 + rank, rgba=False)
    rgb, alpha = be.make_factored(B, NP, R, 99 + rank)
    color, depth = be.empty((B, 3, R, R)), be.empty((B, 1, R, R))
    ms = job.timed(lambda: be.render(case, color, depth, flags, factored=(rgb, alpha)), steps, warmup=3)
    alg_f = (4 * NP * R * R + 12 * R * R + 16 * R * R) * B
    out["N1_factored_fwd"] = {"workload": f"{NP} planes, {R}^2, batch {B} per GPU, forward from rgb [B,3,T,T] + alpha [B,N,1,T,T]",
                              "frames_per_s": world * B / (ms * 1e-3), "ms_per_step": ms, "algorithmic_bytes_per_step": alg_f,
                              "roofline_frac_of_factored_bytes": alg_f / (ms * 1e-3) / 1e9 / peak,
                              "bytes_vs_expanded": alg_f / (algorithmic_bytes_fwd(NP, R, R, R, R) * B)}
    assert int(flags.item()) == 0
    if be.name == "cuda":       # the factored TRAIN step: gradients per factor (g_rgb [B,3,T,T] summed over planes, g_alpha [B,N,1,T,T])
        torch = be.torch
        rgb_g, alpha_g = rgb.requires_grad_(True), alpha.requires_grad_(True)
        gcol = torch.randn((B, 3, R, R), device=be.device)

        def fb_factored():
            rgb_g.grad = alpha_g.grad = None
            c, _ = be.g.render_views_factored(rgb_g, alpha_g, case.dhw, case.view2mpi, case.ray_dir, case.eye, case.z_dir,
                                              color_minus1_1=True)
            (c * gcol).sum().backward()
        ms_t = job.timed(fb_factored, max(3, steps // 4), warmup=2)
        assert alpha_g.grad is not None and bool(torch.isfinite(alpha_g.grad.flatten()[:1024]).all())
        out["N1_factored_train"] = {"workload": f"{NP} planes, {R}^2, batch {B} per GPU, forward + backward from / to the factors",
                                    "value": world * B / (ms_t * 1e-3), "unit": "frames/s (forward+backward)", "ms_per_step": ms_t}
        rgb_g.requires_grad_(False); alpha_g.requires_grad_(False)
        rgb_g.grad = alpha_g.grad = None
        del gcol
    # N3: LightRenderer.compute_depth on the same alpha stack (light_renderer.py:82-100): one streaming pass, 4 B per texel-plane
    if be.name == "cuda":
        from ml_gmpi_b200.light import alpha_depth
        pd = case.dhw[0, :, 0].contiguous()
        ms_d = job.timed(lambda: alpha_depth(alpha, pd), steps, warmup=3)
        bytes_d = (4 * NP * R * R + 4 * R * R) * B
        out["N3_light_compute_depth"] = {"workload": f"alpha [{B},{NP},1,{R},{R}] -> depth [{B},1,{R},{R}]", "ms_per_step": ms_d,
                                         "gbs": bytes_d / (ms_d * 1e-3) / 1e9, "roofline_frac": bytes_d / (ms_d * 1e-3) / 1e9 / peak}
    del case, rgb, alpha, color, depth

    # C4: video render: ONE 96-plane 512^2 MPI (replicated: every rank regenerates it from the same seed), 120 novel views
    # yaw = linspace(0.5, -0.5, 120) sharded over the ranks, frames all-gathered: strong scaling
    NP, R, _ = be.sizes(96, 512, 1)
    import numpy as np
    from ml_gmpi_b200.dist import shard_range
    lo, hi = shard_range(VIDEO_VIEWS, rank, world)
    yaws = np.linspace(0.5, -0.5, VIDEO_VIEWS).astype(np.float32)
    case = be.make_case(n_planes=NP, tex=R, img=R, n_mpi=1, views_per_mpi=hi - lo, seed=1234, yaws=yaws[lo:hi],
                        pitches=np.zeros(hi - lo, np.float32))
    per_rank = -(-VIDEO_VIEWS // world)
    gather, mode = make_gather_or_fallback(job, per_rank, R, R)
    color, depth = be.empty((hi - lo, 3, R, R)), be.empty((hi - lo, 1, R, R))
    frames_all = frames_local = None
    if world > 1 and gather is None:
        frames_all, frames_local = be.empty((world * per_rank, 4, R, R)), torch.zeros((per_rank, 4, R, R), device=be.device)

    def video():
        if gather is not None:
            be.gather_render(gather, case, flags)
            gather.finish()
        else:
            be.render(case, color, depth, flags, view_group=hi - lo)     # all views share the MPI: tiles ordered for L2 reuse
            if world > 1:
                frames_local[: hi - lo, :3].copy_(color); frames_local[: hi - lo, 3:].copy_(depth)
                dist.all_gather_into_tensor(frames_all, frames_local)
    ms = job.timed(video, steps, warmup=2)
    alg = algorithmic_bytes_fwd(NP, R, R, R, R) * VIDEO_VIEWS
    out["C4_video_512"] = {"workload": f"{NP} planes, {R}^2, {VIDEO_VIEWS} views of one MPI over {world} GPU(s), forward + all-gather of frames",
                           "frames_per_s": VIDEO_VIEWS / (ms * 1e-3), "ms_per_step": ms, "scaling": "strong", "gather": mode,
                           "roofline_frac_per_view_bytes": alg / (ms * 1e-3) / 1e9 / (peak * world),
                           "note": "per-view algorithmic bytes; views share one MPI, so DRAM traffic can be below them (L2 reuse)"}
    assert int(flags.item()) == 0
    # the same sweep end to end as the service renders it: factored MPI and cameras from HOST memory, rays generated in the
    # kernel, uint8 frames back in host memory (render_video.py:95-126 incl. its .cpu() and uint8 conversion), this rank's share
    if not args.no_e2e:
        from ml_gmpi_b200.camera import cam_params, focal_from_fov
        from ml_gmpi_b200.geometry import FFHQ
        rgb, alpha = be.make_factored(1, NP, R, 77)
        cam = cam_params(case.c2w, focal_from_fov(FFHQ["fov_deg"], R), R, R)
        nv = hi - lo
        h = {"rgb": be.pin(rgb), "alpha": be.pin(alpha), "dhw": be.pin(case.dhw), "view2mpi": be.pin(case.view2mpi), "cam": be.pin(cam),
             "out_rgb": be.pin(torch.empty((nv, R, R, 3), dtype=torch.uint8)), "out_depth": be.pin(torch.empty((nv, R, R, 1), dtype=torch.uint8))}
        be.render_host_video(h, nv, R, FFHQ["plane_min_d"], FFHQ["plane_max_d"])
        job.barrier()
        t0 = time.perf_counter()
        n_rep = 3
        for _ in range(n_rep):
            fl = be.render_host_video(h, nv, R, FFHQ["plane_min_d"], FFHQ["plane_max_d"])
        job.barrier()
        dt = job.max_over_ranks([(time.perf_counter() - t0) / n_rep])[0]
        assert fl == 0
        h2d = sum(int(h[k].numel()) * h[k].element_size() for k in ("rgb", "alpha", "dhw", "view2mpi", "cam"))
        out["C4_video_512"]["e2e"] = {"frames_per_s": VIDEO_VIEWS / dt, "ms_per_sweep": dt * 1e3, "h2d_bytes_per_rank": h2d,
                                      "d2h_bytes_per_rank": nv * R * R * 4, "form": "factored MPI (rgb + alpha) + cam [V,16] in, uint8 HWC "
                                      "frames + depth out (gmpi_mpi_render_host_ex); the replicated MPI is uploaded by every rank"}
        del h, rgb, alpha
        be.release_host()
    del case, color, depth, gather, frames_all, frames_local

    # C5: train step at 512^2: per GPU 4 MPIs x 1 view, 96 planes, forward+backward
    if not args.no_train_step:
        NP, R, B = be.sizes(96, 512, 4)
        case = be.make_case(n_planes=NP, tex=R, img=R, n_mpi=B, seed=4321 + rank, last_alpha_one=True)
        t = leg_train(job, case, steps, NP, R, B)
        t["workload"] = f"{NP} planes, {R}^2, batch {B} per GPU, forward+backward (global batch {B * world})"
        out["C5_train_512"] = t
        del case
    if be.name == "cuda":
        torch.cuda.empty_cache()
    return out


class OneLineStdout:
    """The contract is ONE JSON line on stdout.  Libraries print there too (NCCL writes its version banner to stdout at the first
    communicator): during the run file descriptor 1 points at stderr, and the line goes to the real stdout at the end."""

    def __init__(self):
        sys.stdout.flush()
        self.real = os.dup(1)
        os.dup2(2, 1)

    def emit(self, text):
        sys.stdout.flush()
        os.write(self.real, (text + "\n").encode())

    def close(self):
        sys.stdout.flush()
        os.dup2(self.real, 1)
        os.close(self.real)


def main(argv=None):
    out = OneLineStdout()
    try:
        return _main(argv, out)
    finally:
        out.close()


def _main(argv, out):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--ref-budget-s", type=float, default=150.0, help="wall-clock budget of the --impl reference run")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-train-step", action="store_true")
    ap.add_argument("--no-configs", action="store_true")
    ap.add_argument("--no-reference-on-gpu", action="store_true")
    ap.add_argument("--planes", type=int, default=N_PLANES)
    ap.add_argument("--res", type=int, default=RES)
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the frames of the last one (colour and depth "
                    "of every view, float32 .npy; a fixed sample of pixels beyond 64 MB) to DIR")
    ap.add_argument("--fake", action="store_true", help=argparse.SUPPRESS)     # tests/test_bench_flow.py only
    args = ap.parse_args(argv)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.impl == "reference":
        return run_reference_arm(args, out)
    args.warmup = max(args.warmup, 3)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    be = (FakeBackend if args.fake else CudaBackend)(local)
    if world > 1:
        be.init_dist()
    job = Job(be, world, rank)
    NP, R, B = be.sizes(args.planes, args.res, args.batch)

    head, state = leg_headline(job, args, NP, R, B)
    if args.dump_outputs and rank == 0:
        frames = state["frames"]
        color, depth = (state["color"], state["depth"]) if frames is None else (frames[:, :3], frames[:, 3:])
        written = dump_outputs(args.dump_outputs, color, depth)
        print(f"[bench] wrote {written} to {args.dump_outputs}", file=sys.stderr)
    train = None
    if not args.no_train_step:
        train = leg_train(job, state["case"], max(3, min(args.steps, 5)), NP, R, B)
        if be.name == "cuda":
            be.torch.cuda.empty_cache()
    e2e = None
    if not args.no_e2e:
        e2e = leg_e2e(job, state, max(2, min(args.steps, 4)), B)
    state = None
    if be.name == "cuda":
        be.torch.cuda.empty_cache()
    configs = None if args.no_configs else leg_configs(job, args)
    ref_gpu = None
    if rank == 0 and world == 1 and not args.no_reference_on_gpu:
        try:
            ref_gpu = be.reference_on_gpu(NP, R)
        except Exception as ex:     # e.g. out of memory on a smaller part: report, never fail the bench for a comparison column
            ref_gpu = {"unavailable": f"{type(ex).__name__}: {ex}"[:200]}
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and not args.fake:
        r = cpu_reference_frames_per_s(steps=3, warmup=1, budget_s=25.0, planes=NP, res=R)
        cpu = {"value": r["value"], "unit": "frames/s", "cores": r["cores"], "kind": "port", "sample": r["sample"],
               "spread": r["spread"], "stable": r["spread"] < 0.2}

    if rank == 0:
        line = {
            "metric": METRIC, "value": head["frames_per_s"], "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": headline_config(NP, R, B, world), "collective": f"all-gather of frames: {head['gather_mode']}",
            "validate": "geometric flags fused in-kernel; range scan off in the timed region",
            "clocks": head["clocks"], "e2e": e2e, "gpu_launches": head["launches"], "roofline": head["roofline"], "cpu_baseline": cpu,
            "train_step": train, "configs": configs, "reference_on_gpu": ref_gpu,
        }
        out.emit(json.dumps(line))
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
