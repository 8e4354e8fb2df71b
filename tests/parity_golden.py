"""Stored results of the unmodified reference CUDA rasterizer for the parity tests (tests/golden/parity_*.npz).

The reference build cannot be assumed on the machine that runs the tests, so what each parity test compared against
is recorded once by tests/golden/make_parity_golden.py and compared here:
  * quantities the tests require bit for bit (radii, indexing arrays, depth bits, ...) as SHA-256 digests of their
    bytes — equal digests mean equal arrays;
  * the four images as a fixed, seeded sample of SAMPLE_PIXELS pixels (every pixel of smaller frames), compared with
    the tests' absolute tolerance;
  * gradients as the reference build's own error statistics against the float64 adjudicator (the largest over three
    of its runs): the tests compute this library's error against the same float64 evaluation and compare the two.
"""
from __future__ import annotations

import hashlib
import os

import numpy as np
import torch

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SAMPLE_PIXELS = 4096
IMAGES = ("color", "depth", "norm", "alpha")
STATS = ("max", "p999", "mean", "rms")


def digest(t) -> str:
    """SHA-256 of the shape and raw bytes; integers are widened to int64 and booleans to uint8 first."""
    a = t.detach().contiguous().cpu().numpy() if isinstance(t, torch.Tensor) else np.ascontiguousarray(t)
    if a.dtype == np.bool_:
        a = a.astype(np.uint8)
    elif np.issubdtype(a.dtype, np.integer):
        a = a.astype(np.int64)
    h = hashlib.sha256(repr(a.shape).encode())
    h.update(a.tobytes())
    return h.hexdigest()


def pixel_sample(H: int, W: int) -> np.ndarray:
    n = H * W
    if n <= SAMPLE_PIXELS:
        return np.arange(n)
    return np.sort(np.random.default_rng(H * 100_003 + W).choice(n, SAMPLE_PIXELS, replace=False))


def record(fwd, I, P, H, W):
    """Everything the parity tests compare, from a forward pass (`fwd`: num_rendered, radii and the four images) and
    its intermediates in the reference's vocabulary (`I`: keys as tile << 32 | depth bits, clamped as [P,3] flags)."""
    vis = fwd["radii"] > 0
    rec = {"num_rendered": np.int64(int(fwd["num_rendered"])), "radii": digest(fwd["radii"])}
    for k in ("tiles_touched", "ranges", "point_list", "keys", "n_contrib"):
        rec[k] = digest(I[k])
    for k in ("depths", "means2D", "cov3D", "conic_opacity", "rgb", "norm3D"):
        rec[k] = digest(I[k][vis])
    rec["clamped"] = digest(I["clamped"].bool()[vis])
    rec["depth_image"], rec["alpha_image"] = digest(fwd["depth"]), digest(fwd["alpha"])
    ranges = I["ranges"]
    rec["longest"] = np.int64(int((ranges[:, 1] - ranges[:, 0]).max()) if ranges.numel() else 0)
    idx = torch.from_numpy(pixel_sample(H, W)).to(fwd["color"].device)
    for k in IMAGES:
        img = fwd[k]
        rec["px_" + k] = img.reshape(img.shape[0], -1)[:, idx].cpu().numpy()
    return rec


def ours_vocabulary(oi):
    """helpers.our_internals() with keys and clamp flags in the reference's form."""
    import helpers as Hh
    out = dict(oi)
    out["keys"] = Hh.ref_style_keys(oi["ranges"], oi["keys"])
    out["clamped"] = torch.stack([(oi["clamped"] >> k) & 1 for k in range(3)], 1).bool()
    return out


def timed(fn, dev, min_warmup_s=0.5, passes=7):
    """Time of one call in ms: the median over `passes` passes of the mean of 10 calls, after untimed calls for at
    least `min_warmup_s` of wall clock (a freshly started process runs its first few hundred milliseconds of GPU work
    noticeably slower).  The median keeps one pass disturbed by other work on a shared machine from setting it."""
    import time
    t0, n = time.perf_counter(), 0
    while n < 3 or time.perf_counter() - t0 < min_warmup_s:
        fn()
        torch.cuda.synchronize(dev)
        n += 1
    ms = []
    for _ in range(passes):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(10):
            fn()
        b.record()
        torch.cuda.synchronize(dev)
        ms.append(a.elapsed_time(b) / 10)
    return float(np.median(ms))


def save(directory, stem, cases):
    """cases: {case id: {field: value}} -> <stem>.npz (or <stem>-N.npz, see golden_io) with keys '<case id>/<field>'."""
    import golden_io
    flat = {}
    for cid, fields in cases.items():
        for f, v in fields.items():
            flat[f"{cid}/{f}"] = np.asarray(v)
    return golden_io.save(stem, flat, directory)


_CACHE = {}


def load(stem: str, cid: str) -> dict:
    """The stored fields of case `cid` in tests/golden/<stem>.npz (or <stem>-N.npz)."""
    import golden_io
    if stem not in _CACHE:
        _CACHE[stem] = golden_io.load(stem, GOLD)
    z = _CACHE[stem]
    pre = cid + "/"
    got = {k[len(pre):]: v for k, v in z.items() if k.startswith(pre)}
    assert got, f"no stored reference results for {cid} in {stem}"
    return got


def check(rec, gold, fields, img_atol=None, exact_images=()):
    """Assert `rec` (this library) equals the stored reference results on `fields`, and the sampled images within
    `img_atol` (None: no image comparison); `exact_images` are compared bit for bit over the whole image."""
    for f in fields:
        want = gold[f]
        got = rec[f]
        if want.dtype.kind in "US":
            assert got == str(want), f"{f} differs from the reference"
        else:
            assert int(got) == int(want), (f, int(got), int(want))
    for k in exact_images:
        assert rec[k + "_image"] == str(gold[k + "_image"]), f"{k} image differs from the reference"
    if img_atol is not None:
        for k in IMAGES:
            err = float(np.abs(rec["px_" + k] - gold["px_" + k]).max())
            assert err <= img_atol, (k, err)


def ref_stats(gold) -> dict:
    """The reference's error statistics against the float64 adjudicator, as oracle.adjudicator.error_report wants."""
    out = {}
    for f, v in gold.items():
        if f.startswith("refstat_"):
            out[f[len("refstat_"):]] = {s: float(x) for s, x in zip(STATS, v)}
    return out


def stats_fields(stats: dict) -> dict:
    return {"refstat_" + k: np.array([s[m] for m in STATS], np.float64) for k, s in stats.items()}
