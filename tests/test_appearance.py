"""SURVEY.md 8f rank 2 — the appearance path (EmbeddingModel MLP + tone map + eval_sh -> colors_precomp).

Golden vectors: tests/golden/appearance_ref-*.npz, produced by the reference's OWN EmbeddingModel and eval_sh
(tests/golden/make_appearance_golden.py, float32 and float64).
  * CPU: the torch formulation in sfgs/appearance.py (used for the backward pass) equals the reference modules' output;
  * GPU: the tcgen05 kernel equals it within the stated bf16 tolerance, for every SH degree, ragged P, and the
    gradients of the autograd wrapper are those of the torch formulation.
"""
import os

import numpy as np
import pytest
import torch

import golden_io


COLOR_ATOL = 1e-4      # split-bf16 (hi + lo) tensor-core operands, fp32 accumulation: ~2^-16 relative per product


def _load(dev, dtype=torch.float32):
    g = golden_io.load("appearance_ref")
    t = {k: torch.from_numpy(g[k]).to(dev) for k in ("features", "gemb", "aemb", "xyz", "campos", "W1", "b1", "W2", "b2", "W3", "b3")}
    return g, {k: v.to(dtype) for k, v in t.items()}


def test_torch_formulation_matches_the_reference_modules():
    from sfgs.appearance import reference_colors
    g, t = _load("cpu", torch.float64)
    for deg in (0, 1, 2, 3):
        got = reference_colors(t["features"], t["gemb"], t["aemb"], t["W1"], t["b1"], t["W2"], t["b2"], t["W3"], t["b3"],
                               t["xyz"], t["campos"], deg)
        assert np.abs(got.numpy() - g[f"colors_deg{deg}_f64"]).max() < 1e-12, deg
    g, t = _load("cpu", torch.float32)
    got = reference_colors(*(t[k] for k in ("features", "gemb", "aemb", "W1", "b1", "W2", "b2", "W3", "b3", "xyz", "campos")), 3)
    assert np.abs(got.numpy() - g["colors_deg3_f32"]).max() < 2e-6


@pytest.mark.gpu
@pytest.mark.parametrize("deg", [0, 1, 2, 3])
def test_fused_appearance_kernel_matches_the_reference_modules(cuda_device, deg):
    from sfgs.appearance import fused_appearance_colors
    g, t = _load(cuda_device)
    mlp = (t["W1"], t["b1"], t["W2"], t["b2"], t["W3"], t["b3"])
    got = fused_appearance_colors(t["features"], t["gemb"], t["aemb"], mlp, t["xyz"], t["campos"], deg)
    err = np.abs(got.cpu().numpy().astype(np.float64) - g[f"colors_deg{deg}_f64"])
    assert got.shape == (t["features"].shape[0], 3)
    assert err.max() <= COLOR_ATOL, (deg, float(err.max()))
    assert err.mean() <= 1e-5, float(err.mean())
    # zeros where the reference clamps (clamp_min(. + 0.5, 0)) except within the tolerance of the threshold
    ref = g[f"colors_deg{deg}_f64"]
    assert np.all(got.cpu().numpy()[ref == 0.0] <= COLOR_ATOL)


@pytest.mark.gpu
def test_fused_appearance_ragged_sizes_and_gradients(cuda_device):
    from sfgs.appearance import fused_appearance_colors, reference_colors
    g, t = _load(cuda_device)
    keys = ("features", "gemb", "aemb", "W1", "b1", "W2", "b2", "W3", "b3", "xyz", "campos")
    for P in (1, 127, 128, 129, 1000, 2999):
        sub = {k: (v[:P].contiguous() if k in ("features", "gemb", "xyz") else v) for k, v in t.items()}
        got = fused_appearance_colors(sub["features"], sub["gemb"], sub["aemb"], tuple(sub[k] for k in keys[3:9]), sub["xyz"],
                                      sub["campos"], 3)
        want = reference_colors(*(sub[k] for k in keys), 3)
        assert float((got - want).abs().max()) <= COLOR_ATOL, P
    # gradients: the autograd wrapper differentiates the torch formulation
    leaves = {k: t[k].clone().requires_grad_(True) for k in keys if k != "campos"}
    out = fused_appearance_colors(leaves["features"], leaves["gemb"], leaves["aemb"], tuple(leaves[k] for k in keys[3:9]),
                                  leaves["xyz"], t["campos"], 3)
    w = torch.randn_like(out)
    (out * w).sum().backward()
    ref_leaves = {k: t[k].clone().requires_grad_(True) for k in keys if k != "campos"}
    (reference_colors(*(ref_leaves[k] for k in keys[:10]), t["campos"], 3) * w).sum().backward()
    for k in leaves:
        assert torch.allclose(leaves[k].grad, ref_leaves[k].grad, rtol=1e-5, atol=1e-7), k
