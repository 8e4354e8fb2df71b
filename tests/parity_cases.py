"""Seeded scenes of the parity tests against the reference CUDA rasterizer, shared by tests/test_gpu_parity.py and
tests/golden/make_parity_golden.py (which records the reference's results on them)."""
import numpy as np

from sfgs import synthetic as S

SORT_SIZES = [1, 2, 31, 33, 127, 128, 129, 255, 256, 257, 511, 512, 513, 1023, 1024, 1025, 4095, 4096, 4097]
BENCHED = ["configs1_1M_jax004", "configs1_1M_orbit", "configs3_5M_jax004", "dense_5M_jax004"]
NEEDLE_KERNELS = (0.1, 0.0005)       # the second filter size leaves the conic nearly singular
FAMILIES = {
    "indexing": ["blob", "city", "precomp", "modifier"],
    "backward": ["blob", "city"],
    "random": [str(s) for s in range(10)],
    "long": ["long"],
    "sort": [str(n) for n in SORT_SIZES],
    "benched": BENCHED,
    "needles": [str(k) for k in NEEDLE_KERNELS],
}


class Case:
    def __init__(self, scene, cam, bg=(0.1, 0.2, 0.3), colors=None, cot_seed=None, kernel_size=0.1,
                 scale_modifier=1.0, sh_degree=None):
        self.scene, self.cam, self.bg, self.colors, self.cot_seed = scene, cam, bg, colors, cot_seed
        self.kw = dict(kernel_size=kernel_size, scale_modifier=scale_modifier,
                       sh_degree=scene.sh_degree if sh_degree is None else sh_degree)


def benched_config(name):
    """(scene, camera) of every frame bench.py reports a number on (BASELINE.json configs[1] and configs[3], plus the
    SURVEY 8d whole-scene orbit stress frame and the dense 5M variant the round-1 numbers were quoted on)."""
    if name == "configs1_1M_jax004":       # bench.py's headline frame, exactly
        return S.city_scene(1_000_000, seed=0), S.jax004_camera(1920, 1080)
    if name == "configs1_1M_orbit":        # SURVEY 8d second camera: fov 60, radius 300, elevation 85
        return S.city_scene(1_000_000, seed=0), S.orbit_camera(width=1920, height=1080)
    if name == "configs3_5M_jax004":       # SURVEY 8d config 4: same generator, extent x sqrt(5)
        return S.city_scene(5_000_000, seed=0, extent=256.0 * 5 ** 0.5), S.jax004_camera(1920, 1080)
    if name == "dense_5M_jax004":          # 5x the density of configs[1] in the same extent (long tile lists)
        return S.city_scene(5_000_000, seed=0), S.jax004_camera(1920, 1080)
    raise KeyError(name)


def build(family: str, cid: str) -> Case:
    if family == "indexing":
        if cid == "blob":
            return Case(S.blob_scene(6000, seed=21), S.simple_camera(333, 217))
        if cid == "city":
            return Case(S.city_scene(200_000, seed=2), S.jax004_camera(1920, 1080))
        if cid == "precomp":
            scene = S.blob_scene(3000, seed=22, sh_degree=0)
            colors = np.random.default_rng(0).uniform(0, 1, (scene.P, 3)).astype(np.float32)
            return Case(scene, S.simple_camera(256, 256), colors=colors)
        if cid == "modifier":
            return Case(S.blob_scene(3000, seed=23), S.simple_camera(200, 120), kernel_size=0.3, scale_modifier=1.7,
                        sh_degree=2)
    if family == "backward":
        if cid == "blob":
            return Case(S.blob_scene(6000, seed=31), S.simple_camera(320, 200), cot_seed=4)
        if cid == "city":
            return Case(S.city_scene(300_000, seed=3), S.jax004_camera(1920, 1080), cot_seed=4)
    if family == "random":
        # image sizes off the tile grid, every SH degree, scale modifiers, filter sizes, backgrounds, cluster tightness
        seed = int(cid)
        rng = np.random.default_rng(1000 + seed)
        P = int(rng.integers(1, 5000))
        W, H = int(rng.integers(17, 400)), int(rng.integers(17, 300))
        deg = int(rng.integers(0, 4))
        scene = S.blob_scene(P, seed=200 + seed, sh_degree=3, spread=float(rng.uniform(0.2, 3.0)),
                             scale=float(rng.uniform(0.01, 0.4)))
        cam = S.simple_camera(W, H, fov_deg=float(rng.uniform(30, 90)), distance=float(rng.uniform(3.0, 10.0)))
        ks, sm = float(rng.choice([0.05, 0.1, 0.3])), float(rng.uniform(0.5, 2.0))
        bg = tuple(float(x) for x in rng.uniform(0, 1, 3))
        return Case(scene, cam, bg=bg, cot_seed=seed, kernel_size=ks, scale_modifier=sm, sh_degree=deg)
    if family == "long":
        # > 1024 and > 4096 instances in one tile: the heavy sort window and the global radix fallback
        return Case(S.blob_scene(9000, seed=77, spread=0.25, scale=0.05), S.simple_camera(64, 64, distance=10.0),
                    bg=(0, 0, 0))
    if family == "sort":
        # ONE tile whose list has exactly n instances; a third of the Gaussians duplicate others (depth ties)
        n = int(cid)
        scene = S.blob_scene(n, seed=1000 + n, spread=0.05, scale=0.08)
        dup = np.arange(n) % 3 == 2
        scene.means3D[dup] = scene.means3D[np.maximum(np.flatnonzero(dup) - 1, 0)]      # exact copies: depth ties
        return Case(scene, S.simple_camera(16, 16, distance=6.0), bg=(0, 0, 0))
    if family == "benched":
        scene, cam = benched_config(cid)
        return Case(scene, cam, bg=(0.0, 0.0, 0.0), cot_seed=1)                        # bench.py's cotangents
    if family == "needles":
        rng = np.random.default_rng(7)
        scene = S.blob_scene(4000, seed=91, spread=2.0, scale=0.02)
        scene.scales[:, 0] = np.exp(rng.uniform(np.log(0.5), np.log(8.0), scene.P)).astype(np.float32)    # long axis
        scene.scales[:, 1] = np.exp(rng.uniform(np.log(0.002), np.log(0.02), scene.P)).astype(np.float32)  # needle
        scene.scales[:, 2] = scene.scales[:, 1]
        scene.opacities[:] = rng.uniform(0.004, 1.0, (scene.P, 1)).astype(np.float32)   # includes values near 1/255
        scene.opacities[::97] = np.float32(1.0) / np.float32(255.0)                      # exactly the threshold
        return Case(scene, S.simple_camera(640, 400, fov_deg=50.0, distance=9.0), bg=(0.2, 0.1, 0.0), cot_seed=12,
                    kernel_size=float(cid))
    raise KeyError((family, cid))
