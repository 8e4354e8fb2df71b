"""SURVEY.md §8 row a1 / §8b: the reference's OWN caller runs unmodified on the drop-in packages.

`gaussian_renderer.render()` (gaussian_renderer/__init__.py:19-164) and `scene.gaussian_model.GaussianModel`
(scene/gaussian_model.py) are imported from the reference source tree ($SFGS_REFERENCE, by default REF_DEFAULT below)
as they are — nothing is copied or edited — with
`skyfall-gs_b200/` on sys.path so that `from diff_gauss import ...` (gaussian_renderer/__init__.py:14) and
`from simple_knn._C import distCUDA2` (scene/gaussian_model.py:25) resolve to this repository's packages.

There is no GPU in this container, so the native layer below the pybind boundary (`diff_gauss._C`, i.e.
sfgs.rasterizer over libsfgs.so) is replaced by a RECORDING FAKE that
  * checks every positional argument of `rasterize_gaussians` / `rasterize_gaussians_backward` for position, python
    type, dtype and shape against the reference's binding (RAST/rasterize_points.h:17-73, .cu:35-243), and
  * returns correctly shaped tensors (10-tuple forward, 10-tuple backward),
and the reference's hard-coded `device="cuda"` / `.to("cuda")` are redirected to the CPU by a TorchFunctionMode.
Everything above that boundary is the real code: the reference's render(), its GaussianModel properties (3D-filter
opacity / scale, rotation normalise, appearance MLP), this repository's `diff_gauss` autograd wrapper, and the
reference's `add_densification_stats`, which consumes `viewspace_points.grad` (scene/gaussian_model.py:744-749).

The test fails if any name, argument order, default, dtype or return arity drifts from what
gaussian_renderer/__init__.py:132-140 and the reference's diff_gauss/__init__.py expect.  (Where that tree is absent
the two tests that need it skip; there the same call sequence runs on the real kernels as a restatement:
tests/test_gpu_parity.py::test_training_loop_with_all_three_ops.)
"""
import os
import sys
import types

import pytest
import torch

REF_DEFAULT = "/root/reference"      # where the build environment keeps the reference checkout; override with SFGS_REFERENCE
REF = os.environ.get("SFGS_REFERENCE", REF_DEFAULT)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "skyfall-gs_b200")

needs_reference = pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "gaussian_renderer")),
                                     reason="needs the reference source tree (set SFGS_REFERENCE)")


class _CudaToCpu(torch.overrides.TorchFunctionMode):
    """Redirect explicit CUDA placements of the reference code to the CPU (no GPU in this container)."""

    @staticmethod
    def _fix(v):
        if isinstance(v, str) and v.startswith("cuda"):
            return "cpu"
        if isinstance(v, torch.device) and v.type == "cuda":
            return torch.device("cpu")
        return v

    def __torch_function__(self, func, types_, args=(), kwargs=None):
        kwargs = dict(kwargs or {})
        if "device" in kwargs:
            kwargs["device"] = self._fix(kwargs["device"])
        if func in (torch.Tensor.cuda,):
            return args[0]
        if func is torch.Tensor.to:
            args = tuple(self._fix(a) for a in args)
        return func(*args, **kwargs)


def _stub(name):
    m = types.ModuleType(name)

    class _Any:
        def __getattr__(self, k):
            return _Any()

        def __call__(self, *a, **k):
            return _Any()
    m.__getattr__ = lambda k: _Any()
    m.__path__ = []
    return m


@pytest.fixture()
def reference_stack(monkeypatch):
    """Import the reference's caller against the drop-in packages; yields (render, GaussianModel, records)."""
    for p in (REF, PKG):
        monkeypatch.syspath_prepend(p)
    for name in ("plyfile", "OpenEXR"):          # I/O dependencies of modules the hot path never calls
        if name not in sys.modules:
            monkeypatch.setitem(sys.modules, name, _stub(name))
    for name in [k for k in sys.modules if k.split(".")[0] in ("gaussian_renderer", "scene", "utils", "arguments")]:
        monkeypatch.delitem(sys.modules, name)
    import diff_gauss
    from diff_gauss import _C
    import gaussian_renderer
    from scene.gaussian_model import GaussianModel
    assert os.path.realpath(gaussian_renderer.__file__).startswith(os.path.realpath(REF))
    assert os.path.realpath(diff_gauss.__file__).startswith(os.path.realpath(PKG))
    assert gaussian_renderer.GaussianRasterizer is diff_gauss.GaussianRasterizer

    rec = {"fwd": [], "bwd": []}
    f32 = torch.float32

    def is_f32(t, shape=None):
        assert isinstance(t, torch.Tensor) and t.dtype == f32, (type(t), getattr(t, "dtype", None))
        if shape is not None:
            assert tuple(t.shape) == tuple(shape), (tuple(t.shape), shape)

    def empty(t):
        assert isinstance(t, torch.Tensor) and t.numel() == 0

    def fake_forward(*a, fuse_normalize=False):
        # RasterizeGaussiansCUDA, RAST/rasterize_points.h:17-41: 23 positional arguments in this order
        assert len(a) == 23, len(a)
        (bg, means3D, colors, opacity, scales, rotations, scale_modifier, cov3D_precomp, norm3D_precomp, extra_attrs,
         attr_degree, viewmatrix, projmatrix, tan_fovx, tan_fovy, kernel_size, image_height, image_width, sh, degree,
         campos, prefiltered, debug) = a
        P = means3D.shape[0]
        is_f32(bg, (3,)); is_f32(means3D, (P, 3)); is_f32(opacity, (P, 1)); is_f32(scales, (P, 3)); is_f32(rotations, (P, 4))
        assert isinstance(scale_modifier, float) and isinstance(attr_degree, int) and attr_degree == 0
        empty(cov3D_precomp); empty(norm3D_precomp); empty(extra_attrs)
        is_f32(viewmatrix, (4, 4)); is_f32(projmatrix, (4, 4)); is_f32(campos, (3,))
        for v in (tan_fovx, tan_fovy, kernel_size):
            assert isinstance(v, float)
        assert isinstance(image_height, int) and isinstance(image_width, int) and isinstance(degree, int)
        assert prefiltered is False and debug is False
        if sh.numel():
            is_f32(sh); assert sh.ndim == 3 and sh.shape[0] == P and sh.shape[2] == 3; empty(colors)
        else:
            is_f32(colors, (P, 3))
        H, W = image_height, image_width
        rec["fwd"].append(dict(P=P, H=H, W=W, M=int(sh.shape[1]) if sh.numel() else 0, degree=degree,
                               kernel_size=kernel_size, scale_modifier=scale_modifier, fused=fuse_normalize,
                               opacity_max=float(opacity.max())))
        g = torch.Generator().manual_seed(0)
        img = lambda c: torch.rand((c, H, W), generator=g)  # noqa: E731
        radii = torch.randint(0, 5, (P,), generator=g, dtype=torch.int32)
        byte = lambda n: torch.zeros(n, dtype=torch.uint8)  # noqa: E731
        out = (int((radii > 0).sum()) * 3, img(3), img(1), img(3), img(1), radii, torch.empty(0), byte(64), byte(64), byte(64))
        return out + (img(3),) if fuse_normalize else out

    def fake_backward(*a, norm_raw=None):
        # RasterizeGaussiansBackwardCUDA, RAST/rasterize_points.h:43-73: 29 positional arguments in this order
        assert len(a) == 29, len(a)
        (bg, means3D, radii, colors, scales, rotations, extra_attrs, scale_modifier, cov3D_precomp, norm3D_precomp,
         viewmatrix, projmatrix, tan_fovx, tan_fovy, kernel_size, dL_color, dL_depth, dL_norm, dL_alpha, dL_extra, sh,
         degree, campos, geom, R, binning, img, out_alpha, debug) = a
        P = means3D.shape[0]
        f = rec["fwd"][-1]
        H, W = f["H"], f["W"]
        is_f32(bg, (3,)); is_f32(means3D, (P, 3)); is_f32(scales, (P, 3)); is_f32(rotations, (P, 4))
        assert radii.dtype == torch.int32 and tuple(radii.shape) == (P,)
        is_f32(dL_color, (3, H, W)); is_f32(dL_depth, (1, H, W)); is_f32(dL_norm, (3, H, W)); is_f32(dL_alpha, (1, H, W))
        is_f32(out_alpha, (1, H, W))
        assert isinstance(R, int) and isinstance(degree, int) and debug is False
        for b in (geom, binning, img):
            assert b.dtype == torch.uint8
        M = f["M"]
        rec["bwd"].append(dict(P=P, R=R, norm_raw=norm_raw is not None))
        g = torch.Generator().manual_seed(1)
        r = lambda *s: torch.rand(s, generator=g) - 0.5  # noqa: E731
        # (dL_dmeans2D, dL_dcolors, dL_dopacity, dL_dmeans3D, dL_dcov3D, dL_dnorm3D, dL_dsh, dL_dscales, dL_drotations,
        #  dL_dextra_attrs), RAST/rasterize_points.cu:242
        return (r(P, 3), r(P, 3), r(P, 1), r(P, 3), r(P, 6), r(P, 3), r(P, M, 3), r(P, 3), r(P, 4), torch.empty(0))

    monkeypatch.setattr(_C, "rasterize_gaussians", fake_forward)
    monkeypatch.setattr(_C, "rasterize_gaussians_fused", lambda *a: fake_forward(*a, fuse_normalize=True))
    monkeypatch.setattr(_C, "rasterize_gaussians_backward", fake_backward)
    monkeypatch.setattr(_C, "rasterize_gaussians_backward_fused", fake_backward)
    with _CudaToCpu():
        yield gaussian_renderer.render, GaussianModel, rec


def _fill(pc, P, appearance):
    """Populate a reference GaussianModel the way create_from_pcd / training_setup leave it (scene/gaussian_model.py:
    310-420), without the point-cloud and optimizer plumbing."""
    g = torch.Generator().manual_seed(5)
    M = (pc.max_sh_degree + 1) ** 2
    leaf = lambda *s: torch.nn.Parameter(torch.randn(*s, generator=g) * 0.3)  # noqa: E731
    pc._xyz, pc._scaling, pc._rotation, pc._opacity = leaf(P, 3), leaf(P, 3), leaf(P, 4), leaf(P, 1)
    pc._features_dc, pc._features_rest = leaf(P, 1, 3), leaf(P, M - 1, 3)
    pc.filter_3D = torch.rand((P, 1), generator=g, dtype=torch.float64) * 0.05      # float64, like compute_3D_filter
    pc.active_sh_degree = pc.max_sh_degree
    pc.xyz_gradient_accum = torch.zeros((P, 1))
    pc.xyz_gradient_accum_abs = torch.zeros((P, 1))
    pc.xyz_gradient_accum_abs_max = torch.zeros((P, 1))
    pc.denom = torch.zeros((P, 1))
    if appearance:
        pc._embeddings = leaf(P, 6 * pc.appearance_n_fourier_freqs)
        pc.appearance_embeddings = leaf(4, pc.appearance_embedding_dim)


def _camera(W=80, H=48):
    from sfgs import synthetic as S
    c = S.simple_camera(W, H)
    import math
    return types.SimpleNamespace(FoVx=2 * math.atan(c.tanfovx), FoVy=2 * math.atan(c.tanfovy), image_height=H,
                                 image_width=W, world_view_transform=torch.from_numpy(c.viewmatrix),
                                 full_proj_transform=torch.from_numpy(c.projmatrix),
                                 camera_center=torch.from_numpy(c.campos), uid=1)


@needs_reference
@pytest.mark.parametrize("appearance", [False, True])
def test_reference_render_and_model_run_unmodified_on_the_dropin(reference_stack, appearance):
    render, GaussianModel, rec = reference_stack
    P = 300
    pc = GaussianModel(3, appearance, 4, 32)
    _fill(pc, P, appearance)
    cam = _camera()
    pipe = types.SimpleNamespace(debug=False, compute_cov3D_python=False, convert_SHs_python=False)
    bg = torch.tensor([0.0, 0.0, 0.0])
    out = render(cam, pc, pipe, bg, kernel_size=0.1)
    # the dict the training loop reads (train.py:195-210)
    assert set(out) == {"render", "render_depth", "render_norm", "render_alpha", "viewspace_points", "visibility_filter",
                        "radii", "extra"}
    assert out["render"].shape == (3, 48, 80) and out["render_depth"].shape == (1, 48, 80)
    assert out["render_norm"].shape == (3, 48, 80) and out["render_alpha"].shape == (1, 48, 80)
    assert out["radii"].dtype == torch.int32 and out["visibility_filter"].dtype == torch.bool
    f = rec["fwd"][-1]
    assert (f["P"], f["H"], f["W"], f["degree"], f["kernel_size"], f["scale_modifier"]) == (P, 48, 80, 3, 0.1, 1.0)
    assert f["M"] == (0 if appearance else 16)          # appearance path feeds colors_precomp, plain path the SHs
    assert 0.0 < f["opacity_max"] <= 1.0                 # the 3D-filtered, activated opacity arrived as float32 [P,1]

    loss = out["render"].mean() + out["render_depth"].mean() + out["render_alpha"].mean() + out["render_norm"].mean()
    loss.backward()
    assert len(rec["bwd"]) == 1 and rec["bwd"][0]["P"] == P
    # gradients reached the reference's raw parameters through its own activation code
    for name in ("_xyz", "_scaling", "_rotation", "_opacity", "_features_dc"):
        g = getattr(pc, name).grad
        assert g is not None and g.shape == getattr(pc, name).shape and bool(torch.isfinite(g).all()), name
    if appearance:
        assert pc._embeddings.grad is not None and pc.appearance_embeddings.grad is not None
        assert all(p.grad is not None for p in pc.appearance_mlp.parameters())
    else:
        assert pc._features_rest.grad is not None
    # viewspace_points.grad is [P,3] = (d/dx * W/2, d/dy * H/2, sum |.|) and is consumed by the densification statistics
    vsp = out["viewspace_points"]
    assert vsp.grad is not None and tuple(vsp.grad.shape) == (P, 3)
    pc.add_densification_stats(vsp, out["visibility_filter"])
    vis = out["visibility_filter"]
    assert bool((pc.denom[vis] == 1).all()) and bool((pc.denom[~vis] == 0).all())
    assert torch.allclose(pc.xyz_gradient_accum[vis], vsp.grad[vis, :2].norm(dim=-1, keepdim=True))
    assert torch.allclose(pc.xyz_gradient_accum_abs[vis], vsp.grad[vis, 2:].norm(dim=-1, keepdim=True))


@needs_reference
def test_reference_callers_of_the_sibling_ops_resolve_to_the_dropins(reference_stack):
    """train.py:42 `from fused_ssim import fused_ssim` and scene/gaussian_model.py:25 `from simple_knn._C import distCUDA2`."""
    import fused_ssim
    import simple_knn._C as knn_c
    import inspect
    assert os.path.realpath(fused_ssim.__file__).startswith(os.path.realpath(PKG))
    assert os.path.realpath(knn_c.__file__).startswith(os.path.realpath(PKG))
    sig = inspect.signature(fused_ssim.fused_ssim)
    assert list(sig.parameters)[:2] == ["img1", "img2"] and sig.parameters["padding"].default == "same"
    assert sig.parameters["train"].default is True
    assert callable(knn_c.distCUDA2)
    import scene.gaussian_model as gm
    assert gm.distCUDA2 is knn_c.distCUDA2


def test_integration_stub_compiles_against_the_header():
    """The reference-side C++ binding shown in INTEGRATION.md section 2 is real code: extract it and compile it
    (syntax + types only) against include/sfgs.h."""
    import re
    import subprocess
    import tempfile
    text = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    blocks = re.findall(r"```cpp\n(.*?)```", text, flags=re.S)
    assert blocks, "INTEGRATION.md has no ```cpp block"
    from torch.utils import cpp_extension
    inc = [os.path.join(ROOT, "include"), "/usr/local/cuda/include"] + cpp_extension.include_paths()
    import sysconfig
    inc.append(sysconfig.get_paths()["include"])
    with tempfile.TemporaryDirectory() as td:
        src = os.path.join(td, "stub.cpp")
        with open(src, "w") as fh:
            fh.write("#define TORCH_EXTENSION_NAME _C\n" + "\n".join(blocks))
        cmd = ["g++", "-std=c++17", "-fsyntax-only", "-w"] + [x for i in inc for x in ("-I", i)] + [src]
        r = subprocess.run(cmd, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-4000:]
