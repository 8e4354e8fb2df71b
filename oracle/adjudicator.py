"""float64 adjudicator of the gradient parity tests — ctypes face of oracle/adjudicator_f64.cu.

TEST INFRASTRUCTURE.  Only tests/ import this module.  See the header of adjudicator_f64.cu for what it computes
(the reference's backward algorithm, RAST/cuda_rasterizer/backward.cu, evaluated in double precision with the
float32 control flow) and why it runs on the GPU (its alpha-threshold decisions must use the same `expf` as the
reference CUDA build and the product).

`backward_f64(internals, ...)` takes the float32 forward intermediates in the reference's vocabulary — the dict
`oracle.ref_cuda.internals()` returns for the reference CUDA build, or `tests/helpers.our_internals()` for the
product (bit-identical on every indexing quantity) — and returns the ten gradient tensors of the reference's
backward as float64, keyed like `oracle.ref_cuda.backward()`.

`error_report(ours, ref, f64)` is the comparison the tests assert on: error of each implementation against the
float64 values, per tensor, as max / 99.9th percentile / rms.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "adjudicator_f64.cu")
OUT_DIR = os.path.join(HERE, "_build")
LIB = os.path.join(OUT_DIR, "libadjudicator_f64.so")
_lib = None


def build(force: bool = False) -> str:
    os.makedirs(OUT_DIR, exist_ok=True)
    if force or not os.path.exists(LIB) or os.path.getmtime(LIB) < os.path.getmtime(SRC):
        # no fast-math, default FMA contraction: the flags the reference rasterizer is built with (oracle/build_ref.py)
        cmd = [os.environ.get("NVCC", "nvcc"), "-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a",
               "-Xcompiler", "-fPIC", "-shared", SRC, "-o", LIB]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("adjudicator build failed:\n" + r.stderr)
    return LIB


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB):
            build()
        L = C.CDLL(LIB)
        L.adj_backward_f64.restype = C.c_int
        _lib = L
    return _lib


def _p(t):
    return None if (t is None or t.numel() == 0) else C.c_void_p(t.data_ptr())


def backward_f64(I, means3D, radii, shs, scales, rotations, scale_modifier, viewmatrix, projmatrix, campos, tan_fovx,
                 tan_fovy, kernel_size, sh_degree, bg, out_alpha, cot, colors_precomp=None):
    """I: forward intermediates (means2D [P,2], conic_opacity [P,4], rgb [P,3], depths [P], norm3D [P,3], cov3D [P,6],
    clamped [P,3] uint8, n_contrib [H*W], ranges [tiles,2], point_list [R]); cot: (dL_color [3,H,W], dL_depth [1,H,W],
    dL_norm [3,H,W] w.r.t. the UN-normalised normal map, dL_alpha [1,H,W])."""
    L = lib()
    dev = means3D.device
    P = int(means3D.shape[0])
    H, W = int(cot[0].shape[1]), int(cot[0].shape[2])
    use_sh = colors_precomp is None
    M = int(shs.shape[1]) if use_sh else 0
    f32 = lambda t: t.contiguous().float()  # noqa: E731
    colors = f32(I["rgb"]) if use_sh else f32(colors_precomp)
    clamped = I["clamped"]
    if clamped.ndim == 1:      # this library packs the three flags into bits 0..2
        clamped = torch.stack([(clamped >> k) & 1 for k in range(3)], 1)
    clamped = clamped.to(torch.uint8).contiguous()
    z = lambda *s: torch.zeros(s, dtype=torch.float64, device=dev)  # noqa: E731
    g = dict(means2D=z(P, 3), conic=z(P, 4), opacity=z(P), colors=z(P, 3), depths=z(P), norm3D=z(P, 3),
             means3D=z(P, 3), cov3D=z(P, 6), sh=z(P, M, 3), scales=z(P, 3), rot=z(P, 4))
    keep = [f32(I["means2D"]), f32(I["conic_opacity"]), colors, f32(I["depths"]), f32(I["norm3D"]), f32(I["cov3D"]),
            I["ranges"].contiguous().to(torch.int32), I["point_list"].contiguous().to(torch.int32),
            I["n_contrib"].contiguous().to(torch.int32), f32(out_alpha), [f32(c) for c in cot], f32(bg),
            f32(means3D), radii.contiguous().to(torch.int32), f32(shs) if use_sh else None, f32(scales),
            f32(rotations), f32(viewmatrix), f32(projmatrix), f32(campos)]
    (m2d, con, col, dep, nrm, cov, ranges, plist, ncon, alpha, c4, bgf, m3d, rad, shf, sc, rot, vm, pm, cam) = keep
    torch.cuda.synchronize(dev)
    with torch.cuda.device(dev):
        rc = L.adj_backward_f64(
            C.c_int(P), C.c_int(int(sh_degree)), C.c_int(M), C.c_int(W), C.c_int(H), _p(ranges), _p(plist), _p(bgf),
            _p(m2d), _p(con), _p(col), _p(dep), _p(nrm), _p(alpha), _p(ncon), _p(c4[0]), _p(c4[1]), _p(c4[2]),
            _p(c4[3]), _p(m3d), _p(rad), _p(shf), _p(clamped), _p(sc), _p(rot), C.c_float(float(scale_modifier)),
            _p(cov), _p(vm), _p(pm), C.c_float(float(tan_fovx)), C.c_float(float(tan_fovy)),
            C.c_float(float(kernel_size)), _p(cam), _p(g["means2D"]), _p(g["conic"]), _p(g["opacity"]),
            _p(g["colors"]), _p(g["depths"]), _p(g["norm3D"]), _p(g["means3D"]), _p(g["cov3D"]), _p(g["sh"]),
            _p(g["scales"]), _p(g["rot"]), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
    if rc != 0:
        raise RuntimeError(f"adjudicator: CUDA error {rc}")
    g["opacity"] = g["opacity"].view(P, 1)
    return g


GRAD_KEYS = ("means2D", "colors", "opacity", "means3D", "cov3D", "norm3D", "sh", "scales", "rot")


def error_report(ours, ref, f64, keys=GRAD_KEYS, ref_stats=None):
    """Per tensor: the error of `ours` and of `ref` against the float64 adjudicator, as max / 99.9th percentile /
    mean / rms of the absolute error.  `ref` may be a list of runs of the reference CUDA build (its float atomics make
    it non-deterministic): every statistic is then the largest over the runs.  `ours` may be a list of runs too (its
    vector reductions are unordered as well): mean / p99.9 / rms are then the LARGEST over the runs, and the worst
    element — an extreme-value statistic whose single draws scatter by a factor of five between runs of either
    implementation — the MEDIAN over the runs (every run's value is kept in `ours_max_runs`).
    `ref_stats` ({tensor: statistics}, from `reference_stats` of an earlier run) stands in for `ref` where given."""
    refs = [] if ref is None else (list(ref) if isinstance(ref, (list, tuple)) else [ref])
    ours_runs = list(ours) if isinstance(ours, (list, tuple)) else [ours]

    def stats(e):
        # "p999": the 99.9th percentile, or, for tensors with fewer than 100 000 elements, the quantile that leaves 100
        # elements above it — a percentile defined by a dozen elements is as noisy as the maximum
        qq = 1.0 - max(1e-3, 100.0 / max(e.numel(), 101))
        if e.numel() > 4_000_000:      # torch.quantile is limited to 16M elements: subsample for the percentile only
            idx = torch.randint(0, e.numel(), (4_000_000,), device=e.device, generator=None)
            q = float(torch.quantile(e[idx], qq))
        else:
            q = float(torch.quantile(e, qq)) if e.numel() > 1 else float(e.max())
        return dict(max=float(e.max()), p999=q, mean=float(e.mean()), rms=float((e * e).mean().sqrt()))

    rep = {}
    for k in keys:
        t = f64[k].double().flatten()
        if t.numel() == 0:
            continue
        runs = [stats((o[k].double().flatten() - t).abs()) for o in ours_runs]
        so = {m: max(r_[m] for r_ in runs) for m in runs[0]}
        so["max"] = sorted(r_["max"] for r_ in runs)[len(runs) // 2]
        sr = None
        for r in refs:
            s1 = stats((r[k].double().flatten() - t).abs())
            sr = s1 if sr is None else {m: max(sr[m], s1[m]) for m in s1}
        if ref_stats is not None:
            sr = ref_stats[k]
        rep[k] = dict(ours=so, ref=sr, scale=float(t.abs().max()), n=int(t.numel()), ref_runs=len(refs),
                      ours_runs=len(runs), ours_max_runs=[r_["max"] for r_ in runs])
    return rep


def reference_stats(ref, f64, keys=GRAD_KEYS):
    """{tensor: error statistics of the reference runs `ref` against `f64`} — the `ref` half of error_report."""
    rep = error_report(ref, ref, f64, keys)
    return {k: r["ref"] for k, r in rep.items()}


def format_report(rep) -> str:
    lines = ["tensor        max|f64|   ours: max / p99.9 / mean / rms                 reference: max / p99.9 / mean / rms"]
    for k, r in rep.items():
        o, f = r["ours"], r["ref"]
        lines.append(f"{k:10s} {r['scale']:11.4e}   {o['max']:9.2e} {o['p999']:9.2e} {o['mean']:9.2e} {o['rms']:9.2e}      "
                     + (f"{f['max']:9.2e} {f['p999']:9.2e} {f['mean']:9.2e} {f['rms']:9.2e}" if f else "-"))
    return "\n".join(lines)
