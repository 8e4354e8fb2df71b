"""GPU tests of the two sibling ops: fused SSIM and simple-knn's distCUDA2."""
import os

import numpy as np
import pytest
import torch

import parity_golden as PG

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def torch_ssim_map(a, b):
    """conv2d SSIM, the construction the reference's own test compares against (SSIM/tests/test.py:47-76)."""
    import torch.nn.functional as F
    from oracle.ssim_oracle import GAUSS
    g = torch.tensor(GAUSS, dtype=a.dtype, device=a.device)
    C = a.shape[1]
    w = (g[:, None] * g[None, :])[None, None].expand(C, 1, 11, 11).contiguous()
    mu1, mu2 = F.conv2d(a, w, padding=5, groups=C), F.conv2d(b, w, padding=5, groups=C)
    s1 = F.conv2d(a * a, w, padding=5, groups=C) - mu1 * mu1
    s2 = F.conv2d(b * b, w, padding=5, groups=C) - mu2 * mu2
    s12 = F.conv2d(a * b, w, padding=5, groups=C) - mu1 * mu2
    return ((2 * mu1 * mu2 + 1e-4) * (2 * s12 + 9e-4)) / ((mu1 * mu1 + mu2 * mu2 + 1e-4) * (s1 + s2 + 9e-4))


def test_fused_ssim_matches_golden_and_torch(cuda_device):
    from fused_ssim import fused_ssim
    dev = cuda_device
    g = np.load(os.path.join(GOLD, "ssim_ref.npz"))
    a = torch.from_numpy(g["img1"]).to(dev).requires_grad_(True)
    b = torch.from_numpy(g["img2"]).to(dev)
    v = fused_ssim(a, b)
    v.backward()
    assert abs(v.item() - float(g["mean"])) < 2e-6
    assert np.abs(a.grad.cpu().numpy() - g["grad"]).max() < 1e-7 + 1e-3 * np.abs(g["grad"]).max()
    # the reference's own test shapes (B,CH,H,W = 5,5,1080,1920 there; smaller here) and its isclose criterion
    torch.manual_seed(0)
    x = torch.rand(2, 3, 270, 333, device=dev, requires_grad=True)
    y = torch.rand(2, 3, 270, 333, device=dev)
    got = fused_ssim(x, y)
    want = torch_ssim_map(x.double(), y.double()).mean()
    assert torch.isclose(got.double(), want, rtol=1e-5, atol=1e-6)
    got.backward()
    gx = x.grad.clone()
    xd = x.detach().double().requires_grad_(True)
    torch_ssim_map(xd, y.double()).mean().backward()
    assert (gx.double() - xd.grad).abs().max().item() < 1e-9 + 1e-3 * xd.grad.abs().max().item()
    # "valid" padding crops 5 px and inference mode skips the derivative maps
    vv = fused_ssim(x.detach(), y, padding="valid", train=False)
    want_v = torch_ssim_map(x.detach().double(), y.double())[:, :, 5:-5, 5:-5].mean()
    assert torch.isclose(vv.double(), want_v, rtol=1e-5, atol=1e-6)


def knn_clouds():
    rng = np.random.default_rng(3)
    return {
        "uniform": rng.uniform(-5, 5, size=(20000, 3)),
        "clustered": np.concatenate([rng.normal(0, 0.05, (5000, 3)), rng.normal(3, 1.0, (5000, 3)), [[40.0, -30.0, 9.0]]]),
        "flat": np.concatenate([rng.uniform(-2, 2, (8000, 2)), np.zeros((8000, 1))], 1),
        "dupes": np.repeat(rng.uniform(0, 1, (300, 3)), 4, axis=0),
        "tiny": rng.uniform(0, 1, (5, 3)),
    }


def knn_cloud():
    """The cloud the reference's distCUDA2 was recorded on (tests/golden/siblings_ref.npz, at KNN_SAMPLE)."""
    return knn_clouds()["uniform"].astype(np.float32)


KNN_SAMPLE = np.sort(np.random.default_rng(5).choice(20000, 1024, replace=False))


def test_dist_cuda2_matches_bruteforce_and_reference(cuda_device):
    from oracle import knn_oracle
    from simple_knn._C import distCUDA2
    dev = cuda_device
    for name, pts in knn_clouds().items():
        pts = pts.astype(np.float32)
        got = distCUDA2(torch.from_numpy(pts).to(dev)).cpu().numpy()
        want = knn_oracle.dist2_knn3(pts)
        assert np.allclose(got, want, rtol=2e-6, atol=1e-12), name
    # the reference's distCUDA2 on the uniform cloud: same 3-NN set; the squared distance may contract differently (1 ulp)
    got = distCUDA2(torch.from_numpy(knn_cloud()).to(dev)).cpu().numpy()[KNN_SAMPLE]
    want = PG.load("siblings_ref", "knn")["value"]
    assert np.allclose(got, want, rtol=1e-6, atol=0)


def test_expf_replica_is_bit_exact(cuda_device):
    """The blend kernels evaluate expf through a hand-scheduled replica of the compiler's routine (constants pinned in
    registers, csrc/sfgs_common.cuh).  The alpha thresholds that decide n_contrib sit on its result, so it must equal
    expf() bit for bit: a dense sweep of the range the kernels use, every exponent/sign pattern, and special values."""
    from sfgs import native as N
    dev = cuda_device
    g = torch.Generator(device="cpu").manual_seed(3)
    parts = [torch.linspace(-110.0, 0.0, 8_000_001, dtype=torch.float64).float(),          # the kernels' range
             -torch.rand(4_000_000, generator=g).mul(20.0),                                 # where alpha is decided
             -torch.exp(torch.rand(2_000_000, generator=g) * 60.0 - 50.0),                  # log-uniform magnitudes
             torch.randint(-2 ** 31, 2 ** 31 - 1, (4_000_000,), generator=g, dtype=torch.int64).to(torch.int32).view(torch.float32),
             torch.tensor([0.0, -0.0, 1.0, -1.0, 88.7, 88.8, -87.3, -87.4, -103.9, -104.1, float("inf"), float("-inf"),
                           1e-45, -1e-45, 1.1754944e-38, -1.1754944e-38, 3.0e38, -3.0e38])]
    x = torch.cat(parts).to(dev)
    yr, ye = torch.empty_like(x), torch.empty_like(x)
    N.check(N.lib().sfgs_selftest_expf(x.numel(), x.data_ptr(), yr.data_ptr(), ye.data_ptr(),
                                       torch.cuda.current_stream(dev).cuda_stream), "selftest_expf")
    torch.cuda.synchronize(dev)
    ok = (yr.view(torch.int32) == ye.view(torch.int32)) | (torch.isnan(yr) & torch.isnan(ye))
    # the kernels only ever use the value for arguments <= 0 (a positive `power` is rejected before/independently)
    neg = x <= 0
    bad = (~ok) & neg
    assert int(bad.sum()) == 0, f"{int(bad.sum())} mismatches for x <= 0, e.g. x = {x[bad][:5].tolist()}"
    assert float(ok.float().mean()) > 0.999, "replica should agree with expf on (almost) every bit pattern"


SSIM_SHAPES = [(5, 5, 1080, 1920), (1, 3, 1080, 1920), (2, 3, 270, 333), (1, 1, 17, 19), (1, 2, 64, 4), (1, 3, 33, 130)]
SSIM_C1, SSIM_C2 = 0.01 ** 2, 0.03 ** 2
SSIM_SAMPLE = 1024


def ssim_inputs(shape, dev):
    g = torch.Generator(device="cpu").manual_seed(sum(shape))
    a = torch.rand(shape, generator=g).to(dev)
    b = (a + 0.2 * torch.randn(shape, generator=g).to(dev)).clamp(0, 1) if shape[2] > 20 else torch.rand(shape, generator=g).to(dev)
    dL = torch.randn(shape, generator=g).to(dev)
    # derivative maps fed to the backward kernel on its own: seeded, of the magnitude the forward produces (up to ~1/C2)
    maps = [(torch.randn(shape, generator=g) * s).to(dev) for s in (30.0, 300.0, 300.0)]
    n = int(np.prod(shape))
    idx = np.arange(n) if n <= SSIM_SAMPLE else np.sort(np.random.default_rng(n).choice(n, SSIM_SAMPLE, replace=False))
    return a, b, dL, maps, torch.from_numpy(idx).to(dev)


def ssim_record(fs, shape, dev):
    """What the fused-ssim test compares, computed with the package `fs` (the reference's, when the golden file is
    written; this library's in the test): the forward maps and the backward (on fixed maps) at a seeded sample of
    elements with each tensor's largest magnitude, the end-to-end value and gradient, and the 'valid' value."""
    a, b, dL, maps, idx = ssim_inputs(shape, dev)
    C1, C2 = SSIM_C1, SSIM_C2
    rec = {}
    for name, t in zip(("ssim_map", "dm_dmu1", "dm_dsigma1_sq", "dm_dsigma12"), fs.fusedssim(C1, C2, a, b, True)):
        rec[name], rec[name + "_absmax"] = t.flatten()[idx].cpu().numpy(), np.float64(t.abs().max())
    g = fs.fusedssim_backward(C1, C2, a, b, dL, *maps)
    rec["backward"], rec["backward_absmax"] = g.flatten()[idx].cpu().numpy(), np.float64(g.abs().max())
    x = a.clone().requires_grad_(True)
    v = fs.fused_ssim(x, b)
    v.backward()
    rec["value"] = np.float64(v.item())
    rec["grad"], rec["grad_absmax"] = x.grad.flatten()[idx].cpu().numpy(), np.float64(x.grad.abs().max())
    if a.numel() <= 20_000_000:
        # whose error a deviation is, is decided by a float64 torch evaluation
        xd = a.double().requires_grad_(True)
        vd = torch_ssim_map(xd, b.double()).mean()
        vd.backward()
        rec["value_err_f64"] = np.float64(abs(v.item() - vd.item()))
        rec["grad_err_f64"] = np.float64((x.grad.double() - xd.grad).abs().max())
        rec["grad_f64_absmax"] = np.float64(xd.grad.abs().max())
    if shape[2] > 10 and shape[3] > 10:
        rec["valid_value"] = np.float64(fs.fused_ssim(a, b, padding="valid", train=False).item())
    return rec


@pytest.mark.parametrize("shape", SSIM_SHAPES)
def test_fused_ssim_against_the_reference_cuda_kernel(cuda_device, shape):
    """The reference's own compiled fused-ssim (SSIM/ssim.cu, built with its setup.py's flags; its results stored in
    tests/golden/siblings_ref.npz) as the oracle, first on its own test workload (SSIM/tests/test.py:81-83: B=5, CH=5,
    1080x1920), then on the training shape and on sizes that are off the tile grid, odd, narrower than a tile or not
    16-byte rows (the non-TMA load path).  The reference kernel is compiled with --use_fast_math (approximate
    divisions): the map agrees within 1e-5 (the image tolerance of the north star), and for the end-to-end value and
    gradient a float64 torch evaluation decides whose error a deviation is (ours <= 2x the reference kernel's)."""
    import fused_ssim
    ref = PG.load("siblings_ref", "ssim_" + "x".join(map(str, shape)))
    ours = ssim_record(fused_ssim, shape, cuda_device)
    # the value map is O(1); the derivative maps reach ~1/C2 and dm_dmu1 is a difference of terms far larger than the
    # result (the reference sums four of them with approximate divisions), so they are compared relative to the
    # largest magnitude in the tensor
    for name, rel in (("ssim_map", 1e-5), ("dm_dmu1", 2e-5), ("dm_dsigma1_sq", 2e-5), ("dm_dsigma12", 2e-5)):
        tol = rel * max(1.0, float(ref[name + "_absmax"]))
        err = float(np.abs(ours[name] - ref[name]).max())
        assert err <= tol, (name, err, tol)
        assert abs(float(ours[name + "_absmax"]) - float(ref[name + "_absmax"])) <= tol, name
    # same derivative maps in: isolates the backward kernel
    tol = 2e-6 * max(1.0, float(ref["backward_absmax"]))
    assert float(np.abs(ours["backward"] - ref["backward"]).max()) <= tol
    # the public entry point end to end
    assert abs(float(ours["value"]) - float(ref["value"])) < 2e-6
    if "grad_err_f64" in ref:
        assert float(ours["value_err_f64"]) <= 2 * float(ref["value_err_f64"]) + 1e-6
        e_ours, e_ref = float(ours["grad_err_f64"]), float(ref["grad_err_f64"])
        assert e_ours <= 2 * e_ref + 1e-9 * float(ref["grad_f64_absmax"]) + 1e-12, (e_ours, e_ref)
    else:
        assert float(np.abs(ours["grad"] - ref["grad"]).max()) <= 2e-5 * float(ref["grad_absmax"]) + 1e-12
    if "valid_value" in ref:
        assert abs(float(ours["valid_value"]) - float(ref["valid_value"])) < 2e-6
