"""Shared helpers for the parity tests (test infrastructure)."""
from __future__ import annotations

import numpy as np
import torch

from sfgs import synthetic as S


def to_torch(scene: S.Scene, cam: S.Camera, device):
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(device)  # noqa: E731
    return dict(means3D=t(scene.means3D), scales=t(scene.scales), rotations=t(scene.rotations),
                opacities=t(scene.opacities), shs=t(scene.shs), viewmatrix=t(cam.viewmatrix),
                projmatrix=t(cam.projmatrix), campos=t(cam.campos))


def run_ours_forward(d, cam, sh_degree, bg, kernel_size=0.1, scale_modifier=1.0, colors=None, debug=False):
    from sfgs import rasterizer as R
    e = torch.empty(0, device=d["means3D"].device)
    sh = e if colors is not None else d["shs"]
    col = colors if colors is not None else e
    out = R.rasterize_gaussians(bg, d["means3D"], col, d["opacities"], d["scales"], d["rotations"], scale_modifier,
                                e, e, e, 0, d["viewmatrix"], d["projmatrix"], cam.tanfovx, cam.tanfovy, kernel_size,
                                cam.height, cam.width, sh, sh_degree, d["campos"], False, debug)
    keys = ("num_rendered", "color", "depth", "norm", "alpha", "radii", "extra", "geom", "binning", "img")
    return dict(zip(keys, out))


def run_ours_backward(d, cam, sh_degree, bg, fwd, cot, kernel_size=0.1, scale_modifier=1.0, colors=None, debug=False,
                      **kw):
    from sfgs import rasterizer as R
    e = torch.empty(0, device=d["means3D"].device)
    sh = e if colors is not None else d["shs"]
    col = colors if colors is not None else e
    out = R.rasterize_gaussians_backward(bg, d["means3D"], fwd["radii"], col, d["scales"], d["rotations"], e,
                                         scale_modifier, e, e, d["viewmatrix"], d["projmatrix"], cam.tanfovx,
                                         cam.tanfovy, kernel_size, cot[0], cot[1], cot[2], cot[3], e, sh, sh_degree,
                                         d["campos"], fwd["geom"], fwd["num_rendered"], fwd["binning"], fwd["img"],
                                         fwd["alpha"], debug, **kw)
    if kw.get("phase") == 1:
        return out                      # the [P,16] blend-adjoint sums
    keys = ("means2D", "colors", "opacity", "means3D", "cov3D", "norm3D", "sh", "scales", "rot", "extra")
    return dict(zip(keys, out))


def run_ref_forward(d, cam, sh_degree, bg, kernel_size=0.1, scale_modifier=1.0, colors=None):
    from oracle import ref_cuda
    e = torch.empty(0, device=d["means3D"].device)
    sh = e if colors is not None else d["shs"]
    col = colors if colors is not None else e
    return ref_cuda.forward(bg, d["means3D"], col, d["opacities"], d["scales"], d["rotations"], scale_modifier, e, e,
                            e, d["viewmatrix"], d["projmatrix"], cam.tanfovx, cam.tanfovy, kernel_size, cam.height,
                            cam.width, sh, sh_degree, d["campos"])


def run_ref_backward(d, cam, sh_degree, bg, fwd, cot, kernel_size=0.1, scale_modifier=1.0, colors=None):
    from oracle import ref_cuda
    e = torch.empty(0, device=d["means3D"].device)
    sh = e if colors is not None else d["shs"]
    col = colors if colors is not None else e
    return ref_cuda.backward(bg, d["means3D"], fwd["radii"], col, d["scales"], d["rotations"], e, scale_modifier, e,
                             e, d["viewmatrix"], d["projmatrix"], cam.tanfovx, cam.tanfovy, kernel_size, cot[0],
                             cot[1], cot[2], cot[3], e, sh, sh_degree, d["campos"], fwd["geom"],
                             fwd["num_rendered"], fwd["binning"], fwd["img"], fwd["alpha"])


def our_internals(fwd, P, H, W):
    """Unpack this library's scratch buffers into the reference's vocabulary."""
    import ctypes as C
    from sfgs import native as N
    L = N.lib()
    dev = fwd["geom"].device
    gv, iv, bv = N.GeomView(), N.ImageView(), N.BinningView()
    N.check(L.sfgs_geom_layout(fwd["geom"].data_ptr(), P, C.byref(gv)), "geom_layout")
    N.check(L.sfgs_image_layout(fwd["img"].data_ptr(), W, H, C.byref(iv)), "image_layout")
    # the binning layout depends on the capacity THIS forward used; it is recorded in the image header (words 2,3)
    hdr = fwd["img"][:32].view(torch.int32).cpu().numpy().astype(np.uint32)
    assert fwd["img"].data_ptr() % 256 == 0
    cap = int(hdr[2]) | (int(hdr[3]) << 32)
    N.check(L.sfgs_binning_layout(fwd["binning"].data_ptr(), cap, C.byref(bv)), "binning_layout")
    tiles = ((W + 15) // 16) * ((H + 15) // 16)
    R = fwd["num_rendered"]

    def view(ptr, base_t, shape, dtype):
        off = ptr - base_t.data_ptr()
        n = int(np.prod(shape)) * torch.empty(0, dtype=dtype).element_size()
        return base_t[off:off + n].view(dtype).view(*shape).clone()

    rec = view(gv.rec, fwd["geom"], (P, 16), torch.float32)
    out = dict(rec=rec, means2D=rec[:, 0:2], conic_opacity=torch.cat([rec[:, 2:5], rec[:, 5:6]], 1),
               depths=rec[:, 6], rgb=rec[:, 8:11], norm3D=rec[:, 11:14],
               cov3D=view(gv.cov3D, fwd["geom"], (P, 6), torch.float32),
               clamped=view(gv.clamped, fwd["geom"], (P,), torch.uint8),
               tiles_touched=view(gv.tiles_touched, fwd["geom"], (P,), torch.int32),
               n_contrib=view(iv.n_contrib, fwd["img"], (H * W,), torch.int32),
               ranges=view(iv.ranges, fwd["img"], (tiles, 2), torch.int32),
               keys=view(bv.keys, fwd["binning"], (R,), torch.int64),
               point_list=view(bv.point_list, fwd["binning"], (R,), torch.int32))
    return out


def ref_style_keys(ranges, keys_depth_id):
    """Rebuild the reference's (tile << 32 | depth_bits) keys from our per-tile (depth_bits << 32 | id) keys."""
    R = keys_depth_id.shape[0]
    counts = (ranges[:, 1] - ranges[:, 0]).long()
    tile_of = torch.repeat_interleave(torch.arange(ranges.shape[0], device=ranges.device), counts)
    assert tile_of.shape[0] == R
    depth_bits = (keys_depth_id >> 32) & 0xFFFFFFFF
    return (tile_of << 32) | depth_bits


# ----------------------------------------------------------------------------- float64-adjudicated gradient parity
# Our error against the float64 values may be at most this multiple of the reference CUDA build's own error against
# them, per gradient tensor.  The bulk statistics (mean, 99.9th percentile) are held to tight factors; the worst
# single element is an extreme-value statistic of a heavy-tailed error distribution (the ill-conditioned covariance /
# rotation chain) and is compared with the worst element of the reference over several of its (non-deterministic)
# runs, with a wider factor.  Nothing is exempt: the maximum is over every element.
ADJ_FACTORS = {"mean": 1.5, "p999": 2.0, "max": 4.0}
ADJ_FLOOR = 1e-5      # north_star: 1e-5 abs on gradient tensors


def adjudicate_gradients(d, cam, sh_degree, bg, I, out_alpha, radii, cot, ours, ref, tag, kernel_size=0.1,
                         scale_modifier=1.0, colors=None, factors=None, floor=ADJ_FLOOR, ref_stats=None):
    """The gradient gate of the parity tests.

    The reference's backward is itself an approximation (float atomics in a run-dependent order, transmittance
    recovered by repeated float division), so `|ours - ref|` cannot say whose error a deviation is.  The float64
    adjudicator (oracle/adjudicator_f64.cu: the reference's algorithm in double with the float32 control flow)
    can: for every gradient tensor the error of this library against the float64 values must not exceed
    ADJ_FACTORS x the reference CUDA build's own error against them (+ the 1e-5 absolute floor of the north star)
    in the mean, at the 99.9th percentile and in the worst element.  No element is exempt.

    I: forward intermediates in the reference's vocabulary (oracle.ref_cuda.internals or helpers.our_internals).
    ref: one run of the reference's gradients, or a list of runs (every statistic: the largest over the runs); or None
    with `ref_stats`, the reference's statistics as stored by tests/golden/make_parity_golden.py.
    ours: one run of this library's gradients, or a list of runs (mean / p99.9: the largest over the runs; the worst
    element: the median over the runs — see oracle.adjudicator.error_report).
    Returns the report (also appended to gpurun_out/adjudication.jsonl when that directory exists)."""
    import json
    import os
    from oracle import adjudicator as A
    factors = factors or ADJ_FACTORS
    f64 = A.backward_f64(I, d["means3D"], radii, d["shs"], d["scales"], d["rotations"], scale_modifier,
                         d["viewmatrix"], d["projmatrix"], d["campos"], cam.tanfovx, cam.tanfovy, kernel_size,
                         sh_degree, bg, out_alpha, cot, colors_precomp=colors)
    keys = [k for k in A.GRAD_KEYS if not (colors is not None and k == "sh")]
    rep = A.error_report(ours, ref, f64, keys, ref_stats=ref_stats)
    print(f"\n[adjudication] {tag}\n" + A.format_report(rep))
    out_dir = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
    if os.path.isdir(out_dir):
        with open(os.path.join(out_dir, "adjudication.jsonl"), "a") as fh:
            fh.write(json.dumps({"case": tag, "report": rep}) + "\n")
    failures = []
    for k, r in rep.items():
        for stat, factor in factors.items():
            lim = factor * r["ref"][stat] + floor
            if not r["ours"][stat] <= lim:
                failures.append(f"{k}.{stat}: ours {r['ours'][stat]:.3e} > {factor} x ref {r['ref'][stat]:.3e} + {floor}")
    assert not failures, f"{tag}: " + "; ".join(failures)
    return rep
