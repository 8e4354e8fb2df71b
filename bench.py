#!/usr/bin/env python
"""bench.py — rasterizer fwd+bwd Mpix/s @1080p (1M Gaussians) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One "step" = one forward + one backward of the splat rasterizer over the
BASELINE.json configs[1] workload on synthetic data: the JAX_004-shaped scene of
sfgs.synthetic.city_scene (1M Gaussians, SH degree 3) seen by frame 0 of the
reference's JAX_004 camera path at 1920x1080, with fixed N(0,1) pixel cotangents.

Printed (rank 0, ONE JSON line):
  value    fwd+bwd Mpix/s through the C ABI (ctypes, same call the diff_gauss._C
           stand-in makes) with every input resident in HBM; per-step CUDA events
           on the launching stream, L2 flushed between steps, max over ranks.
  e2e      the same metric through the public autograd API (diff_gauss.GaussianRasterizer
           -> loss -> backward); per step the camera matrices and the target image are
           copied host->device from pinned memory and the loss is read back.
  roofline the dominant kernel: algorithmic bytes per launch (SURVEY.md §8d / DESIGN.md)
           / its mean launch duration measured live with CUDA events around the launch.
  cpu_baseline  the CPU oracle (oracle/sfgs_oracle.c, a port: the reference has no CPU
           path) timed on this box's host cores on a bounded sample.
`--dump-outputs DIR` writes what the last timed step of `value` returned to its caller as DIR/<name>.npy (see
dump_outputs); the inputs are seeded, so two builds given the same arguments can be compared output for output.
`--impl reference` times the UNMODIFIED reference through its own stock code path: its pybind module `diff_gauss._C`
(RAST/ext.cpp, rasterize_points.cu, cuda_rasterizer/*.cu) for `value` and its own autograd wrapper
`diff_gauss.GaussianRasterizer` for `e2e`, installed into oracle/_ref by oracle/build_ref_torch.py; if that install is
absent it falls back to the reference core behind the ctypes shim (oracle/_ref/libref_rasterizer.so), and to the CPU
oracle port if nothing was built.  `reference_kind` in the line says which.

Extra records in the same line (single-GPU run only; they never change `value`).  extra_frames, ssim and tilerows
time K steps like the headline; knn (5 calls), train_loop (300 iterations) and next_ops (3-20 calls per op) keep
their own fixed counts:
  extra_frames  the SURVEY 8d whole-scene orbit camera, the BASELINE configs[3] 5M-Gaussian scene and its dense variant:
                Mpix/s, V, R and (this library) per-stage times, device-resident leg;
  ssim          fused-ssim forward(train)+backward at 1x3x1080x1920 with the 72N / 84N-byte roofline of SURVEY 8d, this
                library next to the reference's compiled kernel (when oracle/_ref has it);
  train_loop    a bounded sample (300 iterations) of the BASELINE configs[2] Stage-1 loop, it/s, either arm with its own packages;
  next_ops      (this library) the fused appearance path and compute_3D_filter next to their torch formulations;
  roofline.traffic  dram__bytes_read + dram__bytes_write of the dominant kernel measured in THIS run by an `ncu`
                subprocess (falls back to profiles/traffic.json and says so in `traffic_source`).
Multi-GPU: the headline is the "views" mode — ranks render different cameras of the replicated scene (weak scaling, no
data-path collective).  In the same invocation every rank then also runs the tile-row sharded mode (ONE frame split by
balanced bands of tile rows, image all-gather and [P,16] reduce-scatter fused into the kernels over NVLink peer memory,
sfgs/multigpu.py) on the 1M scene and on BASELINE configs[3] (5M Gaussians); those strong-scaling records are attached
as `tilerows`.  `--shard tilerows` prints only that mode.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "skyfall-gs_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)
sys.dont_write_bytecode = True     # the benchmark leaves the source tree as it found it (it may be read-only)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from sfgs import synthetic as S  # noqa: E402

W_IMG, H_IMG = 1920, 1080
P_GAUSS = 1_000_000
SH_DEGREE = 3
METRIC = "rasterizer fwd+bwd Mpix/s @1080p (1M Gaussians)"


# ----------------------------------------------------------------------------- helpers
def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock and throttle reasons for the timed loop.

    The clock is measured IN-STREAM, in the un-timed gap between two steps while the previous step's backward
    is still in flight: a one-thread kernel (sfgs_sm_clock_probe) counts SM cycles against %globaltimer for
    ~20 us.  NVML is only touched before the warm-up (max clock) and once right after the last timed step
    (throttle reasons): polling NVML or nvidia-smi from the host DURING the loop was measured to inflate the
    median step from 1.8 ms to 3.8-4.7 ms with 30-70 ms outliers on these boxes."""

    def __init__(self, index: int, dev):
        self.index, self.dev = index, dev
        self.buf = torch.zeros(64, dtype=torch.float32, device=dev)
        self.n = 0

    def sample(self):
        from sfgs import native
        if self.n < 64:
            native.lib().sfgs_sm_clock_probe(self.buf.data_ptr() + 4 * self.n, torch.cuda.current_stream(self.dev).cuda_stream)
            self.n += 1

    def stop(self):
        reasons, src, max_mhz = [], "in-stream cycle counter between steps of the timed loop", None
        try:   # NVML is initialised only now; the GPU is still executing the last step's backward
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.index]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else self.index
            h = nv.nvmlDeviceGetHandleByIndex(phys)
            names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                     "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                     "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                     "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            reasons = sorted(k for k, bit in names.items() if r & bit)
            max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            nvml_now = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
            src += "; throttle reasons, max clock and one NVML clock sample read right after the last timed step"
            nv.nvmlShutdown()
        except Exception:  # noqa: BLE001
            reasons, nvml_now = ["nvml unavailable"], None
        torch.cuda.synchronize(self.dev)
        vals = self.buf[: self.n].cpu().numpy() if self.n else np.zeros(0)
        sm = float(np.median(vals)) if len(vals) else nvml_now
        return {"sm_mhz": sm, "sm_max_mhz": max_mhz, "reasons": reasons, "samples": int(len(vals)) if len(vals) else 1,
                "source": src if len(vals) else "one NVML read right after the last timed step"}


def camera_for_rank(rank: int, world: int) -> S.Camera:
    """Rank 0 sees the JAX_004 frame-0 camera; other ranks the same orbit rotated about the scene's z axis."""
    if rank == 0:
        return S.jax004_camera(W_IMG, H_IMG)
    ang = 2.0 * math.pi * rank / max(world, 1)
    rot = np.array([[math.cos(ang), -math.sin(ang), 0, 0], [math.sin(ang), math.cos(ang), 0, 0], [0, 0, 1, 0], [0, 0, 0, 1.0]])
    return S.camera_from_c2w_opengl(rot @ S.JAX004_FRAME0_C2W, S.JAX004_FOV_DEG, W_IMG, H_IMG)


def algorithmic_bytes(P, V, R, N, M, tiles):
    """SURVEY.md §8d compulsory traffic, split by stage (each input read once, each output written once)."""
    return {
        "preprocess": 20 * P + (111 + 12 * M) * V,
        "tile_scan": 8 * tiles + 8 * P,
        "emit_keys": 20 * V + 12 * R,
        "tile_sort": 32 * R,
        "render_fwd": 56 * R + 36 * N + 8 * tiles,
        "render_bwd": 56 * R + 40 * N + 120 * V,
        "gauss_bwd": (124 + 12 * M) * P + (291 + 24 * M) * V,
    }


class L2Flusher:
    def __init__(self, dev):
        self.buf = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)   # > 126 MB L2

    def __call__(self):
        self.buf.add_(1)


# ----------------------------------------------------------------------------- device-resident leg ("value")
def make_inputs(scene, cam, dev):
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    d = dict(means3D=t(scene.means3D), scales=t(scene.scales), rotations=t(scene.rotations),
             opacities=t(scene.opacities), shs=t(scene.shs), viewmatrix=t(cam.viewmatrix),
             projmatrix=t(cam.projmatrix), campos=t(cam.campos), bg=torch.zeros(3, device=dev))
    d["cot"] = [t(c) for c in S.cotangents(cam.width, cam.height, seed=1)]
    d["empty"] = torch.empty(0, device=dev)
    d["cpu_empty"] = torch.Tensor([])
    return d


def step_ours(d, cam):
    from sfgs import rasterizer as R
    e = d["empty"]
    f = R.rasterize_gaussians(d["bg"], d["means3D"], e, d["opacities"], d["scales"], d["rotations"], 1.0, e, e, e, 0,
                              d["viewmatrix"], d["projmatrix"], cam.tanfovx, cam.tanfovy, 0.1, cam.height, cam.width,
                              d["shs"], SH_DEGREE, d["campos"], False, False)
    c = d["cot"]
    g = R.rasterize_gaussians_backward(d["bg"], d["means3D"], f[5], e, d["scales"], d["rotations"], e, 1.0, e, e,
                                       d["viewmatrix"], d["projmatrix"], cam.tanfovx, cam.tanfovy, 0.1, c[0], c[1],
                                       c[2], c[3], e, d["shs"], SH_DEGREE, d["campos"], f[7], f[0], f[8], f[9], f[4],
                                       False)
    return f, g


def step_ref(d, cam):
    from oracle import ref_cuda
    e = d["empty"]
    f = ref_cuda.forward(d["bg"], d["means3D"], e, d["opacities"], d["scales"], d["rotations"], 1.0, e, e, e,
                         d["viewmatrix"], d["projmatrix"], cam.tanfovx, cam.tanfovy, 0.1, cam.height, cam.width,
                         d["shs"], SH_DEGREE, d["campos"])
    c = d["cot"]
    g = ref_cuda.backward(d["bg"], d["means3D"], f["radii"], e, d["scales"], d["rotations"], e, 1.0, e, e,
                          d["viewmatrix"], d["projmatrix"], cam.tanfovx, cam.tanfovy, 0.1, c[0], c[1], c[2], c[3], e,
                          d["shs"], SH_DEGREE, d["campos"], f["geom"], f["num_rendered"], f["binning"], f["img"],
                          f["alpha"])
    return f, g


_REF_PKGS = None


def ref_packages():
    """(ref_diff_gauss, ref_fused_ssim): the reference's own packages as installed by oracle/build_ref_torch.py."""
    global _REF_PKGS
    if _REF_PKGS is None:
        from oracle import build_ref_torch
        _REF_PKGS = build_ref_torch.import_reference_packages()
    return _REF_PKGS


def reference_kind():
    from oracle import build_ref_torch, ref_cuda
    if build_ref_torch.built():
        return "stock"
    return "shim" if ref_cuda.available() else "cpu"


def step_ref_stock(d, cam):
    """The reference's own pybind entry points, called the way its diff_gauss/__init__.py calls them (positional
    orders of RAST/rasterize_points.h:17-73; `None` arguments arrive as empty CPU tensors there)."""
    C_ = ref_packages()[0]._C
    e = d["cpu_empty"]
    f = C_.rasterize_gaussians(d["bg"], d["means3D"], e, d["opacities"], d["scales"], d["rotations"], 1.0, e, e, e, 0,
                               d["viewmatrix"], d["projmatrix"], cam.tanfovx, cam.tanfovy, 0.1, cam.height, cam.width,
                               d["shs"], SH_DEGREE, d["campos"], False, False)
    num_rendered, color, depth, norm, alpha, radii, extra, geom, binning, img = f
    c = d["cot"]
    g = C_.rasterize_gaussians_backward(d["bg"], d["means3D"], radii, e, d["scales"], d["rotations"], e, 1.0, e, e,
                                        d["viewmatrix"], d["projmatrix"], cam.tanfovx, cam.tanfovy, 0.1, c[0], c[1], c[2],
                                        c[3], e, d["shs"], SH_DEGREE, d["campos"], geom, num_rendered, binning, img, alpha,
                                        False)
    return (num_rendered, color, depth, norm, alpha, radii), g


def settle(step_fn, flush, dev, min_seconds=0.5, max_seconds=3.0):
    """UNTIMED extra warm-up after the W requested steps.  A freshly set-up loop (or one resumed after the GPU sat idle
    while the host prepared the next scene) runs its first 0.1-0.3 s in a slow mode on these boxes — steps of 5-8 ms,
    sometimes bursts of 20-40 ms, then 1.08 ms flat for good (gpurun_out/v1_bench.err, v3_bench.err) — which five
    warm-up steps do not outlast.  So steps are run four at a time for at least `min_seconds` of wall clock and until a
    group is within 5 % of the fastest group seen (at most `max_seconds`).  Nothing here is reported."""
    best, n, t0 = None, 0, time.perf_counter()
    while True:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(4):
            flush()
            step_fn()
        b.record()
        torch.cuda.synchronize(dev)
        t = a.elapsed_time(b)
        n += 4
        el = time.perf_counter() - t0
        if el >= max_seconds or (el >= min_seconds and best is not None and t <= 1.05 * best):
            break
        best = t if best is None else min(best, t)
    return n


def timed_steps(step_fn, steps, warmup, flush, dev, between=None):
    for _ in range(warmup):
        step_fn()
    torch.cuda.synchronize(dev)
    settle(step_fn, flush, dev)
    evs = []
    for i in range(steps):
        if between is not None and i % 4 == 2:
            between()          # un-timed gap: the previous step's backward is still executing
        flush()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        step_fn()
        b.record()
        evs.append((a, b))
    torch.cuda.synchronize(dev)
    ms = [a.elapsed_time(b) for a, b in evs]   # ms per step
    if os.environ.get("SFGS_BENCH_VERBOSE"):
        srt = sorted(ms)
        print(f"[bench] steps={steps} min={srt[0]:.3f} med={srt[len(srt) // 2]:.3f} max={srt[-1]:.3f} ms; "
              + " ".join(f"{m:.2f}" for m in ms), file=sys.stderr)
    return ms


def measure(step_fn, steps, warmup, flush, dev, between=None, max_attempts=8):
    """Time exactly `steps` steps; a pass disturbed from outside is rejected and re-measured.

    Every step launches ~10 kernels from Python and the forward waits once for the instance count, so a host
    core that is descheduled for a few ms leaves the GPU idle inside the timed step; the boxes are shared
    (load average 40-60 on 128 cores observed) and single steps of 5-250 ms appear at random in either leg.
    A pass counts as clean when its MEAN step is within 5 % of its fastest step (one large spike is enough to
    fail it); the reported pass is the first clean one, or the pass with the smallest total if none of
    `max_attempts` is.  Every attempt is listed in the JSON line.  Each pass starts with W untimed warm-up steps and the
    untimed `settle` loop above."""
    attempts = []
    for k in range(max_attempts):
        ms = timed_steps(step_fn, steps, warmup if k == 0 else 3, flush, dev, between)
        attempts.append(ms)
        if sum(ms) / len(ms) <= 1.05 * min(ms):
            break
    best = min(attempts, key=sum)
    if sum(attempts[-1]) / len(attempts[-1]) <= 1.05 * min(attempts[-1]):
        best = attempts[-1]
    info = {"attempts": len(attempts), "ms_per_step_of_each_attempt": [round(sum(a) / len(a), 4) for a in attempts],
            "reported_min_ms": round(min(best), 4), "reported_median_ms": round(sorted(best)[len(best) // 2], 4)}
    return best, info


# ----------------------------------------------------------------------------- public-API leg ("e2e")
class E2E:
    """render -> L1-style loss -> backward through a `diff_gauss` package (this library's drop-in, or the reference's
    own package), with per-step H2D of camera + target image and a D2H read of the loss."""

    def __init__(self, scene, cam, dev, pkg):
        self.GRS, self.GR = pkg.GaussianRasterizationSettings, pkg.GaussianRasterizer
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
        self.dev, self.cam = dev, cam
        self.params = [t(scene.means3D).requires_grad_(True), t(scene.opacities).requires_grad_(True),
                       t(scene.shs).requires_grad_(True), t(scene.scales).requires_grad_(True),
                       t(scene.rotations).requires_grad_(True)]
        self.means2D = torch.zeros((scene.P, 3), device=dev, requires_grad=True)
        rng = np.random.default_rng(5)
        self.h_cam = torch.from_numpy(np.concatenate([cam.viewmatrix.ravel(), cam.projmatrix.ravel(), cam.campos])).pin_memory()
        # the target image travels as 8-bit RGB, the way image datasets are stored, and is converted on the device
        self.h_gt = torch.from_numpy(rng.integers(0, 256, size=(3, cam.height, cam.width), dtype=np.uint8)).pin_memory()
        self.h_loss = torch.zeros(1).pin_memory()
        self.bg = torch.zeros(3, device=dev)
        self.sub = torch.zeros(1, device=dev)
        self.h2d_bytes = self.h_cam.numel() * 4 + self.h_gt.numel()
        self.d2h_bytes = 4
        self.copy_stream = torch.cuda.Stream(dev)

    def step(self):
        cam = self.cam
        cur = torch.cuda.current_stream(self.dev)
        dcam = self.h_cam.to(self.dev, non_blocking=True)
        # the target image is only needed by the loss: copy it on a side stream while the forward runs
        self.copy_stream.wait_stream(cur)
        with torch.cuda.stream(self.copy_stream):
            gt = self.h_gt.to(self.dev, non_blocking=True)
        rs = self.GRS(cam.height, cam.width, cam.tanfovx, cam.tanfovy, 0.1, self.sub, self.bg, 1.0,
                      dcam[0:16].view(4, 4), dcam[16:32].view(4, 4), SH_DEGREE, dcam[32:35], False, False)
        means3D, opac, shs, scales, rots = self.params
        color, depth, norm, alpha, radii, _ = self.GR(rs)(means3D, self.means2D, opac, shs=shs, scales=scales,
                                                          rotations=rots)
        cur.wait_stream(self.copy_stream)
        gt.record_stream(cur)
        gt = torch.mul(gt, 1.0 / 255.0)          # uint8 -> float32 in [0,1], one kernel
        loss = torch.nn.functional.l1_loss(color, gt) + 0.01 * depth.mean() + 0.01 * (1 - alpha).mean() + 0.01 * norm.mean()
        for p in self.params:
            p.grad = None
        self.means2D.grad = None
        loss.backward()
        self.h_loss.copy_(loss.detach().reshape(1), non_blocking=True)


class E2ERefShim:
    """Fallback when the reference's own torch extension was not installed: the reference CUDA core behind the ctypes
    shim (no autograd wrapper: gradients of the same loss are formed by hand and fed to its backward)."""

    def __init__(self, scene, cam, dev):
        self.d = make_inputs(scene, cam, dev)
        self.dev, self.cam = dev, cam
        rng = np.random.default_rng(5)
        self.h_cam = torch.from_numpy(np.concatenate([cam.viewmatrix.ravel(), cam.projmatrix.ravel(), cam.campos])).pin_memory()
        self.h_gt = torch.from_numpy(rng.integers(0, 256, size=(3, cam.height, cam.width), dtype=np.uint8)).pin_memory()
        self.h_loss = torch.zeros(1).pin_memory()
        self.copy_stream = torch.cuda.Stream(dev)

    def step(self):
        from oracle import ref_cuda
        d, cam, e = self.d, self.cam, self.d["empty"]
        cur = torch.cuda.current_stream(self.dev)
        dcam = self.h_cam.to(self.dev, non_blocking=True)
        self.copy_stream.wait_stream(cur)
        with torch.cuda.stream(self.copy_stream):
            gt = self.h_gt.to(self.dev, non_blocking=True)
        view, proj, campos = dcam[0:16].view(4, 4), dcam[16:32].view(4, 4), dcam[32:35]
        f = ref_cuda.forward(d["bg"], d["means3D"], e, d["opacities"], d["scales"], d["rotations"], 1.0, e, e, e, view,
                             proj, cam.tanfovx, cam.tanfovy, 0.1, cam.height, cam.width, d["shs"], SH_DEGREE, campos)
        cur.wait_stream(self.copy_stream)
        gt.record_stream(cur)
        gt = torch.mul(gt, 1.0 / 255.0)
        n = float(cam.height * cam.width)
        norm_raw = f["norm"].detach().requires_grad_(True)
        norm = torch.nn.functional.normalize(norm_raw, p=2, dim=0)
        loss = torch.nn.functional.l1_loss(f["color"], gt) + 0.01 * f["depth"].mean() + 0.01 * (1 - f["alpha"]).mean() + 0.01 * norm.mean()
        (g_norm,) = torch.autograd.grad(0.01 * norm.mean(), norm_raw)
        g_color = torch.sign(f["color"] - gt) / (3 * n)
        g_depth = torch.full_like(f["depth"], 0.01 / n)
        g_alpha = torch.full_like(f["alpha"], -0.01 / n)
        ref_cuda.backward(d["bg"], d["means3D"], f["radii"], e, d["scales"], d["rotations"], e, 1.0, e, e, view, proj,
                          cam.tanfovx, cam.tanfovy, 0.1, g_color, g_depth, g_norm, g_alpha, e, d["shs"], SH_DEGREE,
                          campos, f["geom"], f["num_rendered"], f["binning"], f["img"], f["alpha"])
        self.h_loss.copy_(loss.detach().reshape(1), non_blocking=True)


# ----------------------------------------------------------------------------- CPU baseline
def cpu_baseline(scene, cam, max_seconds=25.0):
    """CPU oracle (port of the reference algorithm; the reference itself has no CPU path) on this box's cores."""
    from oracle import cpu_oracle as O
    cot = S.cotangents(cam.width, cam.height, seed=1)
    bg = np.zeros(3, np.float32)
    times = []
    t_start = time.perf_counter()
    while True:
        t0 = time.perf_counter()
        f = O.forward(scene.means3D, scene.scales, scene.rotations, scene.opacities, scene.shs, scene.sh_degree,
                      cam.viewmatrix, cam.projmatrix, cam.campos, cam.width, cam.height, cam.tanfovx, cam.tanfovy, bg)
        O.backward(f, *cot)
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_start > max_seconds * 0.6 or len(times) >= 4:
            break
    best = min(times)
    return {"value": cam.width * cam.height / best / 1e6, "unit": "Mpix/s", "cores": O.num_threads(), "kind": "port",
            "sample": f"{len(times)} full fwd+bwd step(s) of the same workload (P={scene.P}, {cam.width}x{cam.height}), "
                      f"best of {len(times)}, OpenMP over {O.num_threads()} threads"}


# ----------------------------------------------------------------------------- extra records (N = 1 only)
EXTRA_FRAMES = {
    # name: (P, extent, camera)   — the same (scene, camera) pairs tests/test_gpu_parity.py diffs against the reference
    "configs1_1M_orbit": (1_000_000, 256.0, "orbit"),      # SURVEY 8d: whole scene in view, fov 60, radius 300, elevation 85
    "configs3_5M_jax004": (5_000_000, 256.0 * 5 ** 0.5, "jax"),   # BASELINE configs[3]: same generator, extent x sqrt(5)
    "dense_5M_jax004": (5_000_000, 256.0, "jax"),          # 5x the density in the same extent: long tile lists
}


def frame_record(name, impl_kind, dev, steps):
    """Device-resident fwd+bwd of one extra frame: Mpix/s (median step), V, R and, for this library, stage times."""
    from sfgs import native
    P, extent, camname = EXTRA_FRAMES[name]
    scene = S.city_scene(P, seed=0, sh_degree=SH_DEGREE, extent=extent)
    cam = S.jax004_camera(W_IMG, H_IMG) if camname == "jax" else S.orbit_camera(width=W_IMG, height=H_IMG)
    d = make_inputs(scene, cam, dev)
    flush = L2Flusher(dev)
    step = {"ours": lambda: step_ours(d, cam), "stock": lambda: step_ref_stock(d, cam), "shim": lambda: step_ref(d, cam)}[impl_kind]
    ms, timing = measure(step, steps, 5, flush, dev, max_attempts=6)      # same disturbance rule as the headline
    med = float(np.median(ms))
    f, _ = step()
    torch.cuda.synchronize(dev)
    if impl_kind == "shim":
        R, radii = int(f["num_rendered"]), f["radii"]
    else:
        R, radii = int(f[0]), f[5]
    rec = {"name": name, "P": P, "extent": round(extent, 2), "camera": camname, "value": round(cam.width * cam.height / med / 1e3, 2),
           "unit": "Mpix/s", "ms_per_step": round(med, 4), "ms_min": round(min(ms), 4), "ms_all": [round(m, 3) for m in ms], "timing": timing, "steps": steps,
           "V": int((radii > 0).sum().item()), "R": R}
    if impl_kind == "ours":
        per_stage = {}
        for _ in range(5):
            flush()
            native.profile_enable(True)
            step()
            torch.cuda.synchronize(dev)
            for k, v in native.profile_read().items():
                per_stage.setdefault(k, []).append(v[0] / v[1] if v[1] else 0.0)
        native.profile_enable(False)
        rec["stages_ms"] = {k: round(float(np.median(v)), 4) for k, v in per_stage.items()}
    del d, scene
    torch.cuda.empty_cache()
    return rec


def knn_record(impl_kind, dev):
    """distCUDA2 over the 1M scene's positions (scene initialisation, scene/gaussian_model.py:25): this library's grid
    search vs the reference's Morton-order kernel (KNN/simple_knn.cu:186-222, compiled from its own sources)."""
    pts = torch.from_numpy(S.city_scene(P_GAUSS, seed=0).means3D).to(dev)
    if impl_kind == "ours":
        from simple_knn._C import distCUDA2 as fn
    else:
        from oracle import ref_cuda
        if not ref_cuda.available():
            return None
        fn = ref_cuda.knn
    for _ in range(2):
        out = fn(pts)
    torch.cuda.synchronize(dev)
    ts = []
    for _ in range(5):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); out = fn(pts); b.record()
        torch.cuda.synchronize(dev)
        ts.append(a.elapsed_time(b))
    return {"P": P_GAUSS, "ms": round(float(np.median(ts)), 3), "mean_dist2": float(out.mean()),
            "timing": "CUDA events around the call (the reference's includes its own cudaMalloc/cudaMemcpy), median of 5"}


def ssim_record(impl_kind, dev, steps=20):
    """fused-ssim forward(train) and backward at the training shape [1,3,1080,1920]; bytes per SURVEY 8d:
    forward reads 2 and writes 4 planes (72*N bytes at 3 channels), backward reads 6 and writes 1 (84*N)."""
    if impl_kind == "ours":
        import fused_ssim as fs
    elif impl_kind == "stock":
        fs = ref_packages()[1]
    else:
        return None
    H, W, C = H_IMG, W_IMG, 3
    g = torch.Generator(device="cpu").manual_seed(2)
    a = torch.rand((1, C, H, W), generator=g).to(dev)
    b = (a + 0.1 * torch.randn((1, C, H, W), generator=g).to(dev)).clamp(0, 1)
    dL = torch.full((1, C, H, W), 1.0 / (C * H * W), device=dev)
    flush = L2Flusher(dev)
    C1, C2 = 0.01 ** 2, 0.03 ** 2
    t_f, t_b = [], []
    for i in range(steps + 3):
        flush()
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record()
        m, d1, d2, d3 = fs.fusedssim(C1, C2, a, b, True)
        e1.record()
        gimg = fs.fusedssim_backward(C1, C2, a, b, dL, d1, d2, d3)
        e2.record()
        torch.cuda.synchronize(dev)
        if i >= 3:
            t_f.append(e0.elapsed_time(e1)); t_b.append(e1.elapsed_time(e2))
    N = H * W
    peak, _ = peaks()
    mf, mb = float(np.median(t_f)), float(np.median(t_b))
    return {"shape": [1, C, H, W], "fwd_ms": round(mf, 4), "bwd_ms": round(mb, 4),
            "fwd_algorithmic_bytes": 24 * C * N, "bwd_algorithmic_bytes": 28 * C * N,
            "fwd_GBps": round(24 * C * N / mf / 1e6, 1), "bwd_GBps": round(28 * C * N / mb / 1e6, 1),
            "fwd_frac_of_hbm_peak": round(24 * C * N / mf / 1e6 / peak, 4), "bwd_frac_of_hbm_peak": round(28 * C * N / mb / 1e6 / peak, 4),
            "timing": "CUDA events around each call (includes the output allocations of the op), L2 flushed, median",
            "mean_ssim": round(float(m.mean().item()), 6), "grad_abs_max": float(gimg.abs().max().item())}


def train_loop_record(kind, dev, iters=300):
    """BASELINE configs[2] shape — the per-iteration work of train.py Stage 1 (train.py:195-260) around the rasterizer:
    activations -> render one of 8 orbit views at 1920x1080 -> 0.8 L1 + 0.2 (1 - SSIM) -> backward -> Adam on
    (xyz, scaling, rotation, opacity, SH) — as a bounded sample of `iters` iterations of the 7000 (synthetic scene and
    targets; no JAX_068 data here).  ours: the drop-in packages + fused activations; reference: ITS OWN diff_gauss and
    fused_ssim packages (oracle/_ref) + the torch activations of scene/gaussian_model.py:207-249."""
    if kind == "ours":
        import diff_gauss as dg
        import fused_ssim as fs
        from sfgs.activations import fused_activations
    elif kind == "stock":
        dg, fs = ref_packages()
        fused_activations = None
    else:
        return None
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    scene = S.city_scene(P_GAUSS, seed=0, sh_degree=SH_DEGREE)
    cams = [S.orbit_camera(azimuth_deg=45.0 * k) for k in range(8)]
    P = scene.P
    bg = torch.zeros(3, device=dev)
    sub = torch.zeros(1, device=dev)
    cam_t = [(c, t(c.viewmatrix), t(c.projmatrix), t(c.campos)) for c in cams]
    m2d = torch.zeros((P, 3), device=dev, requires_grad=True)
    base = [t(scene.means3D), t(scene.opacities), t(scene.shs), t(scene.scales), t(scene.rotations)]
    targets = []
    with torch.no_grad():
        for c, view, proj, campos in cam_t:
            rs = dg.GaussianRasterizationSettings(c.height, c.width, c.tanfovx, c.tanfovy, 0.1, sub, bg, 1.0, view, proj,
                                                  SH_DEGREE, campos, False, False)
            targets.append(dg.GaussianRasterizer(rs)(base[0], m2d.detach(), base[1], shs=base[2], scales=base[3],
                                                     rotations=base[4])[0].clone())
    rng = np.random.default_rng(1)
    xyz = t((scene.means3D + rng.normal(0, 0.05, scene.means3D.shape)).astype(np.float32)).requires_grad_(True)
    scaling = torch.log(t(scene.scales)).requires_grad_(True)
    rotation = t(scene.rotations).clone().requires_grad_(True)
    opacity = torch.logit(t(scene.opacities).clamp(1e-4, 1 - 1e-4)).reshape(P, 1).clone().requires_grad_(True)
    shs = (t(scene.shs) * 0.9).requires_grad_(True)
    filter_3D = torch.full((P, 1), 0.05, dtype=torch.float64, device=dev)
    opt = torch.optim.Adam([{"params": [xyz], "lr": 1.6e-4}, {"params": [scaling], "lr": 5e-3},
                            {"params": [rotation], "lr": 1e-3}, {"params": [opacity], "lr": 5e-2},
                            {"params": [shs], "lr": 2.5e-3}], eps=1e-15)

    def step(i):
        cam, view, proj, campos = cam_t[i % len(cam_t)]
        if fused_activations is not None:
            op, sc, rot = fused_activations(opacity, scaling, rotation, filter_3D)
        else:
            sq = torch.square(torch.exp(scaling))                    # scene/gaussian_model.py:207-249
            a2 = sq + torch.square(filter_3D)
            sc = torch.sqrt(a2).float()
            op = (torch.sigmoid(opacity) * torch.sqrt(sq.prod(dim=1) / a2.prod(dim=1))[..., None]).float()
            rot = torch.nn.functional.normalize(rotation)
        rs = dg.GaussianRasterizationSettings(cam.height, cam.width, cam.tanfovx, cam.tanfovy, 0.1, sub, bg, 1.0, view, proj,
                                              SH_DEGREE, campos, False, False)
        color = dg.GaussianRasterizer(rs)(xyz, m2d, op, shs=shs, scales=sc, rotations=rot)[0]
        gt = targets[i % len(targets)]
        loss = 0.8 * torch.nn.functional.l1_loss(color, gt) + 0.2 * (1.0 - fs.fused_ssim(color[None], gt[None]))
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        return loss

    for i in range(10):
        step(i)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    first = last = None
    for i in range(iters):
        loss = step(i)
        if i == 0:
            first = loss.detach()
        last = loss.detach()
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1)
    return {"workload": f"BASELINE configs[2] shape: {iters} of the 7000 Stage-1 iterations (activations, render 1 of 8 orbit "
                        "views 1920x1080, 0.8 L1 + 0.2 (1-SSIM), backward, Adam), 1M Gaussians, SH 3, synthetic targets",
            "iterations": iters, "it_per_s": round(iters / (ms / 1e3), 1), "ms_per_it": round(ms / iters, 3),
            "loss_first": round(float(first), 5), "loss_last": round(float(last), 5)}


def next_ops_record(dev):
    """SURVEY 8f rows built this round, each next to the torch formulation it replaces (this library only)."""
    from sfgs import appearance as AP
    from sfgs import filter3d as F3
    import types
    out = {}
    P = P_GAUSS
    g = torch.Generator(device="cpu").manual_seed(3)
    feats = (torch.randn(P, 16, 3, generator=g) * 0.3).to(dev); feats[:, 0] += 0.6
    gemb = torch.sin(torch.randn(P, 24, generator=g) * 3).to(dev)
    aemb = (torch.randn(32, generator=g) * 0.5).to(dev)
    xyz = (torch.randn(P, 3, generator=g) * 80).to(dev)
    campos = torch.tensor([10.0, -300.0, 120.0], device=dev)
    lin = [torch.nn.Linear(59, 128), torch.nn.Linear(128, 128), torch.nn.Linear(128, 6)]
    W = [x.to(dev) for l in lin for x in (l.weight.detach(), l.bias.detach())]

    def timeit(fn, n=10):
        for _ in range(3):
            fn()
        torch.cuda.synchronize(dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        torch.cuda.synchronize(dev)
        return a.elapsed_time(b) / n
    with torch.no_grad():
        t_fused = timeit(lambda: AP.fused_appearance_colors(feats, gemb, aemb, tuple(W), xyz, campos, 3))
        t_torch = timeit(lambda: AP.reference_colors(feats, gemb, aemb, *W, xyz, campos, 3))
        err = float((AP.fused_appearance_colors(feats, gemb, aemb, tuple(W), xyz, campos, 3)
                     - AP.reference_colors(feats, gemb, aemb, *W, xyz, campos, 3)).abs().max())
    peak, _ = peaks()
    out["appearance_forward"] = {"P": P, "fused_ms": round(t_fused, 4), "torch_eager_ms": round(t_torch, 4),
                                 "speedup": round(t_torch / t_fused, 1), "max_abs_diff_vs_torch_f32": err,
                                 "algorithmic_bytes": 324 * P, "GBps": round(324 * P / t_fused / 1e6, 1),
                                 "frac_of_hbm_peak": round(324 * P / t_fused / 1e6 / peak, 4),
                                 "tensor_core_flops": 3 * 2 * P * (32 * 128 + 128 * 128 + 128 * 16),
                                 "note": "tcgen05 kernel (split-bf16 operands, fp32 accumulate in TMEM) vs the reference's statements in torch"}
    # compute_3D_filter: 64 cameras
    rng = np.random.default_rng(2)
    cams = []
    for c in range(64):
        cam = S.orbit_camera(azimuth_deg=float(rng.uniform(0, 360)), elevation_deg=float(rng.uniform(40, 88)), radius=float(rng.uniform(200, 400)))
        w2c = cam.viewmatrix.T.astype(np.float64)
        cams.append(types.SimpleNamespace(R=w2c[:3, :3].T.copy(), T=w2c[:3, 3].copy(), focal_x=cam.width / (2 * cam.tanfovx),
                                          focal_y=cam.height / (2 * cam.tanfovy), cx=0.0, cy=0.0, image_width=cam.width, image_height=cam.height))
    xyz_city = torch.from_numpy(S.city_scene(P, seed=0).means3D).to(dev)

    def torch_filter():      # the reference's statements (scene/gaussian_model.py:254-308) on the GPU in torch
        x = xyz_city.double()
        dist = torch.ones(P, device=dev, dtype=torch.float64) * 1e8
        valid_pts = torch.zeros(P, device=dev, dtype=torch.bool)
        fl = 0.0
        for cam in cams:
            R = torch.tensor(cam.R, device=dev, dtype=torch.float64); T = torch.tensor(cam.T, device=dev, dtype=torch.float64)
            xc = x @ R + T[None, :]
            vd = xc[:, 2] > 0.2
            z = torch.clamp(xc[:, 2], min=0.001)
            px = xc[:, 0] / z * cam.focal_x + cam.image_width / 2; py = xc[:, 1] / z * cam.focal_y + cam.image_height / 2
            ins = (px >= -0.15 * cam.image_width) & (px <= cam.image_width * 1.15) & (py >= -0.15 * cam.image_height) & (py <= 1.15 * cam.image_height)
            v = vd & ins
            dist[v] = torch.min(dist[v], z[v]); valid_pts |= v
            fl = max(fl, cam.focal_x)
        dist[~valid_pts] = dist[valid_pts].max()
        return (dist / fl * (0.2 ** 0.5))[..., None]
    t_f = timeit(lambda: F3.compute_3D_filter(xyz_city, cams), n=5)
    t_t = timeit(torch_filter, n=2)
    d = float((F3.compute_3D_filter(xyz_city, cams) - torch_filter()).abs().max())
    out["compute_3D_filter"] = {"P": P, "cameras": len(cams), "fused_ms": round(t_f, 4), "torch_eager_ms": round(t_t, 3),
                                "speedup": round(t_t / t_f, 1), "max_abs_diff": d}
    out.update(density_control_record(dev, timeit))
    return out


def density_control_record(dev, timeit):
    """Per-iteration densification statistics and densify_and_prune (train.py:311-322, scene/gaussian_model.py:564-749):
    this library's kernels next to the reference's torch statements on the same tensors."""
    from sfgs import densify as D
    P = P_GAUSS
    g = torch.Generator(device=dev).manual_seed(9)
    r = lambda *s: torch.randn(*s, generator=g, device=dev)   # noqa: E731
    par = {"xyz": r(P, 3) * 50, "f_dc": r(P, 1, 3), "f_rest": r(P, 15, 3) * 0.1, "opacity": r(P, 1) * 3,
           "scaling": torch.log(torch.exp(r(P, 3) * 1.2) * 0.5), "rotation": r(P, 4)}
    m = {k: r(*v.shape) * 1e-3 for k, v in par.items()}
    v = {k: (r(*t.shape) * 1e-3) ** 2 for k, t in par.items()}
    denom = torch.randint(0, 4, (P, 1), generator=g, device=dev).float()
    accum = torch.rand((P, 1), generator=g, device=dev) * 3e-4 * denom
    accum_abs = torch.rand((P, 1), generator=g, device=dev) * 6e-4 * denom
    radii = torch.randint(-2, 30, (P,), generator=g, device=dev, dtype=torch.int32).clamp_min(0)
    grad4 = r(P, 4) * 2e-4
    stats = [torch.zeros(P, device=dev)] + [torch.zeros((P, 1), device=dev) for _ in range(4)]

    def torch_stats():            # train.py:314 + gaussian_model.py:744-749
        mr, a, aa, am, dn = stats
        vis = radii > 0
        mr[vis] = torch.max(mr[vis], radii[vis])
        a[vis] += torch.norm(grad4[vis, :2], dim=-1, keepdim=True)
        aa[vis] += torch.norm(grad4[vis, 2:], dim=-1, keepdim=True)
        am[vis] = torch.max(am[vis], torch.norm(grad4[vis, 2:], dim=-1, keepdim=True))
        dn[vis] += 1
    t_stats = timeit(lambda: D.densification_stats(grad4, radii, *stats), n=20)
    t_stats_torch = timeit(torch_stats, n=10)
    extent, max_grad, pd = 120.0, 0.0002, 0.01
    kw = dict(max_grad=max_grad, min_opacity=0.005, extent=extent, max_screen_size=20, percent_dense=pd)
    Q = D.gradient_thresholds(accum, accum_abs, denom, max_grad)
    _, _, _, t0 = D.densify_tensors(par, m, v, accum, accum_abs, denom, abs_threshold=Q, **kw)
    noise = torch.randn((2 * t0["S"], 3), generator=g, device=dev)

    def torch_densify():          # gaussian_model.py:653-735 with the optimizer surgery of :564-651, on the same tensors
        st = {k: [par[k], m[k], v[k]] for k in par}

        def append(new):
            for k in st:
                st[k] = [torch.cat((st[k][0], new[k])), torch.cat((st[k][1], torch.zeros_like(new[k]))),
                         torch.cat((st[k][2], torch.zeros_like(new[k])))]

        def prune(mask):
            keep = ~mask
            for k in st:
                st[k] = [t[keep] for t in st[k]]
        grads = accum / denom; grads[grads.isnan()] = 0.0
        gabs = accum_abs / denom; gabs[gabs.isnan()] = 0.0
        if not torch.isinf(gabs).any() and not torch.isnan(gabs).any():
            q = torch.quantile(gabs.reshape(-1), 1 - (torch.norm(grads, dim=-1) >= max_grad).float().mean())
        sel = (torch.norm(grads, dim=-1) >= max_grad) | (torch.norm(gabs, dim=-1) >= q)
        sel = sel & (torch.exp(st["scaling"][0]).max(dim=1).values <= pd * extent)
        append({k: st[k][0][sel] for k in st})
        n = st["xyz"][0].shape[0]
        pg = torch.zeros(n, device=dev); pg[:P] = grads.squeeze()
        pa = torch.zeros(n, device=dev); pa[:P] = gabs.squeeze()
        sel = ((pg >= max_grad) | (pa >= q)) & (torch.exp(st["scaling"][0]).max(dim=1).values > pd * extent)
        stds = torch.exp(st["scaling"][0])[sel].repeat(2, 1)
        samples = noise * stds
        q4 = st["rotation"][0][sel]
        q4 = q4 / q4.norm(dim=1, keepdim=True)
        w, x, y, z = q4.unbind(1)
        R = torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y), 2 * (x * y + w * z), 1 - 2 * (x * x + z * z),
                         2 * (y * z - w * x), 2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)], dim=1).reshape(-1, 3, 3).repeat(2, 1, 1)
        new = {k: st[k][0][sel].repeat(2, *([1] * (st[k][0].dim() - 1))) for k in st}
        new["xyz"] = torch.bmm(R, samples.unsqueeze(-1)).squeeze(-1) + st["xyz"][0][sel].repeat(2, 1)
        new["scaling"] = torch.log(stds / 1.6)
        ns = int(sel.sum())
        append(new)
        prune(torch.cat((sel, torch.zeros(2 * ns, device=dev, dtype=torch.bool))))
        pm = (torch.sigmoid(st["opacity"][0]) < 0.005).squeeze(-1) | (torch.exp(st["scaling"][0]).max(dim=1).values > 0.1 * extent)
        prune(pm)
        return st["xyz"][0].shape[0]
    t_dens = timeit(lambda: D.densify_tensors(par, m, v, accum, accum_abs, denom, noise=noise, **kw), n=5)
    t_dens_torch = timeit(torch_densify, n=3)
    _, _, _, t = D.densify_tensors(par, m, v, accum, accum_abs, denom, noise=noise, **kw)
    return {"densification_stats": {"P": P, "fused_ms": round(t_stats, 4), "torch_eager_ms": round(t_stats_torch, 3),
                                    "speedup": round(t_stats_torch / t_stats, 1), "algorithmic_bytes": 52 * P,
                                    "GBps": round(52 * P / t_stats / 1e6, 1), "note": "runs every training iteration below densify_until_iter"},
            "densify_and_prune": {"P": P, "new_P": t["new_P"], "cloned": t["C"], "split": t["S"], "fused_ms": round(t_dens, 3),
                                  "torch_eager_ms": round(t_dens_torch, 2), "speedup": round(t_dens_torch / t_dens, 1),
                                  "same_point_count_as_torch": bool(torch_densify() == t["new_P"]),
                                  "note": "both include the quantile (torch.quantile) and one host synchronisation; Adam moments moved with the rows"}}


def live_traffic(kernel_regex, timeout_s=240):
    """dram__bytes_read + dram__bytes_write (and issue-slot utilisation) of ONE launch of the dominant kernel, captured in
    this run by an ncu subprocess over tests/gpu_profile_case.py (same scene, camera and cotangents as the timed loop).
    Returns None when ncu is unavailable."""
    import csv
    import shutil
    import tempfile
    ncu = shutil.which("ncu") or "/usr/local/cuda/bin/ncu"
    if not os.path.exists(ncu):
        return None
    with tempfile.TemporaryDirectory() as td:
        log = os.path.join(td, "t.csv")
        cmd = [ncu, "--metrics", "dram__bytes_read.sum,dram__bytes_write.sum,sm__issue_active.avg.pct_of_peak_sustained_elapsed,"
               "smsp__inst_executed.sum,gpu__time_duration.sum", "--clock-control", "none", "-k", f"regex:{kernel_regex}",
               "-s", "1", "-c", "1", "--csv", "--log-file", log, sys.executable, os.path.join(ROOT, "tests", "gpu_profile_case.py"),
               "--iters", "2"]
        try:
            subprocess.run(cmd, capture_output=True, text=True, timeout=timeout_s, check=True)
            vals = {}
            with open(log) as fh:
                rows = [r for r in csv.reader(l for l in fh if not l.startswith("=="))]
            h0 = next(i for i, r in enumerate(rows) if "Metric Name" in r and "Metric Value" in r)
            hdr = rows[h0]
            for r in rows[h0 + 1:]:
                row = dict(zip(hdr, r))
                v = float(row["Metric Value"].replace(",", ""))
                unit = row.get("Metric Unit", "")
                scale = {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(unit, 1)
                vals[row["Metric Name"]] = v * scale
            return {"traffic": int(vals["dram__bytes_read.sum"] + vals["dram__bytes_write.sum"]),
                    "issue_active_pct": round(vals["sm__issue_active.avg.pct_of_peak_sustained_elapsed"], 1),
                    "warp_instructions": int(vals["smsp__inst_executed.sum"])}
        except Exception as exc:  # noqa: BLE001
            print(f"[bench] live ncu capture failed: {type(exc).__name__}: {str(exc)[:200]}", file=sys.stderr)
            return None


# ----------------------------------------------------------------------------- --dump-outputs
DUMP_MAX_ELEMENTS = 1 << 20        # per array: 14 float32 arrays of <= 4 MB and radii as float64 (8 MB), ~60 MB in all
FWD_NAMES = ("num_rendered", "color", "depth", "norm", "alpha", "radii")
BWD_NAMES = ("grad_means2D", "grad_colors", "grad_opacity", "grad_means3D", "grad_cov3D", "grad_norm3D", "grad_sh",
             "grad_scales", "grad_rotations")
SHIM_BWD_KEYS = ("means2D", "colors", "opacity", "means3D", "cov3D", "norm3D", "sh", "scales", "rot")


def dump_outputs(out, kind, path):
    """The arrays one fwd+bwd step hands its caller: num_rendered, the four images and radii of the forward, and the
    nine gradient tensors of the backward (the forward's opaque scratch buffers are left out).  Floating arrays are
    written as float32, integer ones as float64.  An array of more than DUMP_MAX_ELEMENTS elements is written as a
    sample: the elements at DUMP_MAX_ELEMENTS flat indices drawn without replacement by numpy's default_rng(0), in
    increasing order — the same indices for every run of the same shape."""
    f, g = out
    if kind == "shim":
        fwd = [f[k] for k in FWD_NAMES]
        bwd = [g[k] for k in SHIM_BWD_KEYS]
    else:
        fwd, bwd = list(f[:6]), list(g[:9])
    os.makedirs(path, exist_ok=True)
    for name, t in zip(FWD_NAMES + BWD_NAMES, fwd + bwd):
        t = torch.as_tensor(t).detach().reshape(-1)
        if t.numel() > DUMP_MAX_ELEMENTS:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), DUMP_MAX_ELEMENTS, replace=False))
            t = t[torch.from_numpy(idx).to(t.device)]
        a = t.cpu().numpy()
        a = a.astype(np.float32) if a.dtype.kind == "f" else a.astype(np.float64)
        np.save(os.path.join(path, name + ".npy"), a)


# ----------------------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--shard", default="views", choices=["views", "tilerows"])
    ap.add_argument("--P", type=int, default=P_GAUSS)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-clocks", action="store_true", help="do not sample SM clocks during the timed region")
    ap.add_argument("--no-extras", action="store_true", help="skip the extra frames / ssim / ncu / tile-row records")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    steps, warmup = max(1, args.steps), max(3, args.warmup)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    dev = torch.device(f"cuda:{local_rank}")
    torch.cuda.set_device(dev)

    kind = "ours" if args.impl == "ours" else reference_kind()
    if kind == "cpu":
        return reference_cpu_arm(args, rank, world, steps, warmup)

    if args.shard == "tilerows" and world > 1 and args.impl == "ours":
        from sfgs import multigpu
        return multigpu.bench_tilerows(args, rank, world, dev, steps, warmup, METRIC)

    scene = S.city_scene(args.P, seed=0, sh_degree=SH_DEGREE)
    cam = camera_for_rank(rank, world)
    N = cam.width * cam.height
    d = make_inputs(scene, cam, dev)
    flush = L2Flusher(dev)

    from sfgs import native
    if kind == "ours":
        native.lib()
        step = lambda: step_ours(d, cam)  # noqa: E731
    elif kind == "stock":
        step = lambda: step_ref_stock(d, cam)  # noqa: E731
    else:
        step = lambda: step_ref(d, cam)   # noqa: E731
    last = {}
    if args.dump_outputs:
        timed_step = step

        def step():
            last["out"] = timed_step()
            return last["out"]

    # ---- value: device-resident inputs, per-step events, max over ranks
    sampler = ClockSampler(local_rank, dev)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    ms, value_info = measure(step, steps, warmup, flush, dev,
                             between=sampler.sample if (args.impl == "ours" and not args.no_clocks) else None)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(last.pop("out"), kind, args.dump_outputs)
    total_ms = torch.tensor([sum(ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.barrier()
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms.item())
    value = world * steps * N / (total_ms / 1e3) / 1e6

    # ---- e2e: public API with host<->device copies inside the timed region
    if kind == "ours":
        import diff_gauss as pkg
        e2e_obj = E2E(scene, cam, dev, pkg)
    elif kind == "stock":
        e2e_obj = E2E(scene, cam, dev, ref_packages()[0])
    else:
        e2e_obj = E2ERefShim(scene, cam, dev)
    e2e_ms, e2e_info = measure(e2e_obj.step, steps, warmup, flush, dev)
    e2e_total = torch.tensor([sum(e2e_ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_total, op=dist.ReduceOp.MAX)
    e2e_value = world * steps * N / (float(e2e_total.item()) / 1e3) / 1e6
    del e2e_obj

    # ---- tile-row sharded mode, same invocation (every rank takes part; strong scaling; SURVEY 8e / BASELINE configs[3])
    tilerows = None
    if kind == "ours" and not args.no_extras:        # at N = 1 the same loop runs unsharded: the strong-scaling baseline
        from sfgs import multigpu
        del d
        torch.cuda.empty_cache()
        tilerows = []
        for label, P_t, extent in (("1M", P_GAUSS, 256.0), ("configs3_5M", 5_000_000, 256.0 * 5 ** 0.5)):
            try:
                tsamp = ClockSampler(local_rank, dev)
                rec = multigpu.run_tilerows(P_t, extent, rank, world, dev, steps, warmup)
                tsamp.sample()
                rec["clocks"] = tsamp.stop()
                rec["label"] = label
                tilerows.append(rec)
            except Exception as exc:  # noqa: BLE001
                tilerows.append({"label": label, "error": f"{type(exc).__name__}: {exc}"[:300]})
        d = make_inputs(scene, cam, dev)

    # ---- IDU render set sharded by view (SURVEY 8f rank 4 / BASELINE configs[4], rasterizer side): every rank takes part
    renderset = None
    if kind == "ours" and not args.no_extras:
        try:
            from sfgs import renderset as RS
            renderset = RS.run_renderset(P_GAUSS, rank, world, dev)
        except Exception as exc:  # noqa: BLE001
            renderset = {"error": f"{type(exc).__name__}: {exc}"[:300]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    out = {"metric": METRIC, "value": round(value, 2), "unit": "Mpix/s", "n_gpus": world, "steps": steps,
           "warmup": warmup, "ms_per_step": round(total_ms / steps, 4), "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": "BASELINE configs[1]: JAX_004-shaped synthetic scene, 1M Gaussians, SH degree 3, "
                                  "1920x1080, JAX_004 frame-0 camera, fwd+bwd, fixed N(0,1) cotangents",
                      "P": scene.P, "width": cam.width, "height": cam.height, "sh_degree": SH_DEGREE,
                      "parallelism": f"views x{world} (one camera per GPU, scene replicated, no collective)",
                      "l2": "flushed between steps (256 MB write)", "timing": "per-step CUDA events, max over ranks"},
           "e2e": {"value": round(e2e_value, 2), "unit": "Mpix/s", "h2d_bytes_per_step": (16 + 16 + 3) * 4 + 3 * N,
                   "d2h_bytes_per_step": 4},
           "clocks": clocks}
    out["timing"] = {"value": value_info, "e2e": e2e_info,
                     "rule": "W warm-up steps, then untimed steps in groups of 4 for >= 0.5 s and until a group is within 5 % of the fastest group (<= 3 s), then exactly K timed steps; a pass whose mean step exceeds 1.05x its fastest step is re-measured (<= 8 passes)"}
    out["e2e"]["api"] = {"ours": "diff_gauss.GaussianRasterizer + autograd (this library's drop-in package)",
                         "stock": "the reference's own diff_gauss.GaussianRasterizer + autograd over its own pybind module",
                         "shim": "reference CudaRasterizer::Rasterizer forward/backward behind the ctypes shim"}[kind]
    if tilerows is not None:
        out["tilerows"] = tilerows
    if renderset is not None:
        out["renderset"] = renderset
    if kind == "ours":
        l0 = native.lib().sfgs_launch_count()
        f, _ = step()
        torch.cuda.synchronize(dev)
        # kernels of this library launched inside the reported timed pass (steps x launches of one step)
        out["gpu_launches"] = int(native.lib().sfgs_launch_count() - l0) * steps
        R, V = int(f[0]), int((f[5] > 0).sum().item())
        M = (SH_DEGREE + 1) ** 2
        tiles = ((cam.width + 15) // 16) * ((cam.height + 15) // 16)
        # per-stage CUDA-event times, one read per step; the MEDIAN over the steps is reported (the boxes are
        # shared: a mean is ruined by one step that was disturbed)
        per_stage = {}
        for _ in range(steps):
            flush()
            native.profile_enable(True)
            step()
            torch.cuda.synchronize(dev)
            for k, v in native.profile_read().items():
                per_stage.setdefault(k, []).append(v[0] / v[1] if v[1] else 0.0)
        native.profile_enable(False)
        alg = algorithmic_bytes(scene.P, V, R, N, M, tiles)
        stage_ms = {k: float(np.median(v)) for k, v in per_stage.items()}
        dom = max((k for k in stage_ms if k in alg), key=lambda k: stage_ms[k])
        peak, peak_src = peaks()
        ach = alg[dom] / (stage_ms[dom] / 1e3) / 1e9
        b_total = sum(alg.values())
        t_kernels = sum(stage_ms.values())
        out["roofline"] = {"bound": "hbm", "kernel": dom, "achieved": round(ach, 1), "peak": peak, "unit": "GB/s",
                           "frac": round(ach / peak, 4), "traffic": None, "peak_source": peak_src,
                           "algorithmic_bytes": int(alg[dom]), "kernel_ms": round(stage_ms[dom], 4),
                           "share_of_step": round(stage_ms[dom] / t_kernels, 3)}
        out["roofline_pipeline"] = {"algorithmic_bytes": int(b_total), "kernels_ms": round(t_kernels, 4),
                                    "achieved": round(b_total / (t_kernels / 1e3) / 1e9, 1), "unit": "GB/s",
                                    "frac": round(b_total / (t_kernels / 1e3) / 1e9 / peak, 4)}
        out["stages_ms"] = {k: round(v, 4) for k, v in stage_ms.items()}
        out["counts"] = {"P": scene.P, "V": V, "R": R, "N": N}
    else:
        out["impl"] = "reference"
        out["reference_kind"] = {"stock": "unmodified reference through its own pybind module and autograd wrapper (oracle/_ref, "
                                          "installed by oracle/build_ref_torch.py), same GPU, same inputs",
                                 "shim": "unmodified reference CUDA core behind a ctypes shim (oracle/_ref/libref_rasterizer.so)"}[kind]
        out["e2e"]["note"] = "same host<->device copies and the same loss code as the product arm"

    # ---- extra records: other frames, fused-ssim, live DRAM traffic (single-GPU run only)
    if world == 1 and not args.no_extras:
        del d
        torch.cuda.empty_cache()
        frames = []
        for name in EXTRA_FRAMES:
            try:
                frames.append(frame_record(name, kind, dev, steps))
            except Exception as exc:  # noqa: BLE001
                frames.append({"name": name, "error": f"{type(exc).__name__}: {exc}"[:300]})
        out["extra_frames"] = frames
        try:
            out["ssim"] = ssim_record(kind, dev, steps)
        except Exception as exc:  # noqa: BLE001
            out["ssim"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        try:
            out["knn"] = knn_record(kind, dev)
        except Exception as exc:  # noqa: BLE001
            out["knn"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        try:
            out["train_loop"] = train_loop_record(kind, dev)
        except Exception as exc:  # noqa: BLE001
            out["train_loop"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        if kind == "ours":
            try:
                out["next_ops"] = next_ops_record(dev)
            except Exception as exc:  # noqa: BLE001
                out["next_ops"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        if kind == "ours":
            torch.cuda.synchronize(dev)
            lt = live_traffic({"render_bwd": "render_bwd", "render_fwd": "render_fwd"}.get(dom, dom))
            if lt is not None:
                out["roofline"].update(traffic=lt["traffic"], traffic_source="ncu subprocess in this run (one launch, "
                                       "dram__bytes_read.sum + dram__bytes_write.sum)")
                out["roofline"]["limiter"] = (f"instruction issue: {lt['issue_active_pct']}% of issue slots active, "
                                              f"{lt['warp_instructions']} warp instructions (same ncu capture)")
            else:
                tpath = os.path.join(ROOT, "profiles", "traffic.json")
                if os.path.exists(tpath):
                    with open(tpath) as fh:
                        tj = json.load(fh)
                    out["roofline"].update(traffic=tj.get("kernels", {}).get(dom),
                                           traffic_source="profiles/traffic.json (committed ncu capture; live capture unavailable)")
    if not args.no_cpu_baseline and world == 1:   # the CPU port is timed on rank 0 of the single-GPU run only
        out["cpu_baseline"] = cpu_baseline(scene, cam)
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def reference_cpu_arm(args, rank, world, steps, warmup):
    """Fallback reference arm when oracle/_ref is absent: the CPU oracle port on the host cores (rank 0 only)."""
    if rank != 0:
        return
    scene = S.city_scene(args.P, seed=0, sh_degree=SH_DEGREE)
    cam = S.jax004_camera(W_IMG, H_IMG)
    cb = cpu_baseline(scene, cam, max_seconds=60.0)
    out = {"metric": METRIC, "value": round(cb["value"], 4), "unit": "Mpix/s", "n_gpus": world, "steps": steps,
           "warmup": warmup, "ms_per_step": round(cam.width * cam.height / cb["value"] / 1e3, 2),
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "impl": "reference", "config": {"workload": "BASELINE configs[1] (same as the product arm)"},
           "cpu_baseline": cb,
           "e2e": {"value": round(cb["value"], 4), "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
