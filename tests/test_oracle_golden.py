"""Pin the CPU oracle (oracle/sfgs_oracle.c) against the UNMODIFIED reference CUDA rasterizer.

tests/golden/ref_*.npz were produced on a B200 by the reference's own code (oracle/_ref, built from
/root/reference by oracle/build_ref.py) with tests/golden/make_golden.py.  No GPU is needed here."""
import os

import numpy as np
import pytest

import golden_io
from golden_cases import CASES, build_case
from oracle import cpu_oracle as O

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


@pytest.mark.parametrize("name", CASES)
def test_oracle_matches_reference_cuda(name):
    if not golden_io.exists(f"ref_{name}"):
        pytest.skip("fixture not generated")
    g = golden_io.load(f"ref_{name}")
    scene, cam, bg, kw = build_case(name)
    f = O.forward(scene.means3D, scene.scales, scene.rotations, scene.opacities, scene.shs, kw["sh_degree"],
                  cam.viewmatrix, cam.projmatrix, cam.campos, cam.width, cam.height, cam.tanfovx, cam.tanfovy, bg,
                  kernel_size=kw["kernel_size"], scale_modifier=kw["scale_modifier"], colors_precomp=kw.get("colors"))
    # ---- integer / index work: bit-exact
    assert f["num_rendered"] == int(g["num_rendered"])
    assert np.array_equal(f["radii"], g["radii"])
    assert np.array_equal(f["tiles_touched"], g["int_tiles_touched"].astype(np.uint32))
    assert np.array_equal(f["point_offsets"], g["int_point_offsets"].astype(np.uint32))
    assert np.array_equal(f["point_list"], g["int_point_list"].astype(np.uint32))
    assert np.array_equal(f["keys"], g["int_keys"].astype(np.uint64))
    assert np.array_equal(f["ranges"], g["int_ranges"].astype(np.uint32))
    vis = g["radii"] > 0
    # ---- the floats that decide the indexing: bit-exact as well (the oracle spells out the GPU's FMA split)
    for k in ("depths", "means2D", "cov3D", "conic_opacity"):
        assert np.array_equal(bits(f[k][vis]), bits(g["int_" + k][vis])), k
    if not kw.get("colors_precomp"):
        assert np.abs(f["rgb"][vis] - g["int_rgb"][vis]).max() < 1e-6
        assert np.array_equal(f["clamped"][vis].astype(bool), g["int_clamped"][vis].astype(bool))
    assert np.abs(f["norm3D"][vis] - g["int_norm3D"][vis]).max() < 1e-6
    # ---- blended images: glibc expf vs CUDA expf differ by <= 2 ulp; a borderline alpha/T test may flip a pixel
    for k in ("color", "depth", "norm", "alpha"):
        d = np.abs(f[k] - g[k])
        scale = max(1.0, float(np.abs(g[k]).max()))       # depth is un-normalised (hundreds of scene units)
        assert np.quantile(d, 0.999) <= 1e-5 * scale and d.max() <= 5e-3 * scale, (k, d.max())
    assert (f["n_contrib"] != g["int_n_contrib"].astype(np.uint32)).mean() < 1e-3
    # ---- gradients: within the reference's own atomic-order noise
    gb = O.backward(f, *kw["cot"])
    for k in ("means2D", "colors", "opacity", "means3D", "cov3D", "norm3D", "sh", "scales", "rot"):
        a, b = gb[k].astype(np.float64).ravel(), g["grad_" + k].astype(np.float64).ravel()
        if b.size == 0:
            continue
        tol = 1e-5 + 2e-4 * np.abs(b) + 4.0 * float(g["gradspread_" + k]) + 5e-6 * np.abs(b).max()
        bad = np.abs(a - b) > tol
        assert bad.mean() < 2e-3, (k, int(bad.sum()), float(np.abs(a - b).max()))
