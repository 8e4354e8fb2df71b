"""Record the UNMODIFIED reference CUDA rasterizer (oracle/_ref) on the parity tests' scenes -> tests/golden/parity_*.npz,
plus the reference's simple-knn and fused-ssim kernels -> tests/golden/siblings_ref.npz.

Needs a B200 and oracle/_ref (built by __graft_entry__.build() where the reference sources exist):
    python tests/golden/make_parity_golden.py OUT_DIR
then copy OUT_DIR/*.npz into tests/golden/ in place of the parity_* and siblings_ref* files there.  What is stored is described in tests/parity_golden.py; inputs are not
stored, they are regenerated from the seeds in tests/parity_cases.py.
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, "skyfall-gs_b200"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import helpers as Hh  # noqa: E402
import parity_cases as PC  # noqa: E402
import parity_golden as PG  # noqa: E402
from oracle import adjudicator as A  # noqa: E402
from oracle import ref_cuda  # noqa: E402
from sfgs import synthetic as S  # noqa: E402

GRADIENT_FAMILIES = ("backward", "random", "benched", "needles")


def reference_case(family, cid, dev):
    c = PC.build(family, cid)
    scene, cam, kw = c.scene, c.cam, c.kw
    d = Hh.to_torch(scene, cam, dev)
    bg = torch.tensor(c.bg, device=dev, dtype=torch.float32)
    col = None if c.colors is None else torch.from_numpy(c.colors).to(dev)
    f = Hh.run_ref_forward(d, cam, kw["sh_degree"], bg, kernel_size=kw["kernel_size"],
                           scale_modifier=kw["scale_modifier"], colors=col)
    ri = ref_cuda.internals(f, scene.P, cam.height, cam.width)
    rec = PG.record(f, ri, scene.P, cam.height, cam.width)
    if family in GRADIENT_FAMILIES:
        cot = [torch.from_numpy(x).to(dev) for x in S.cotangents(cam.width, cam.height, seed=c.cot_seed)]
        runs = [Hh.run_ref_backward(d, cam, kw["sh_degree"], bg, f, cot, kernel_size=kw["kernel_size"],
                                    scale_modifier=kw["scale_modifier"], colors=col) for _ in range(3)]
        f64 = A.backward_f64(ri, d["means3D"], f["radii"], d["shs"], d["scales"], d["rotations"], kw["scale_modifier"],
                             d["viewmatrix"], d["projmatrix"], d["campos"], cam.tanfovx, cam.tanfovy, kw["kernel_size"],
                             kw["sh_degree"], bg, f["alpha"], cot, colors_precomp=col)
        keys = [k for k in A.GRAD_KEYS if not (col is not None and k == "sh")]
        rec.update(PG.stats_fields(A.reference_stats(runs, f64, keys)))
    if family == "long":
        # median of several timed passes after a time-based warm-up (parity_golden.timed), like the test's own timing
        rec["forward_ms"] = np.float64(PG.timed(lambda: Hh.run_ref_forward(d, cam, 3, bg), dev))
    return rec


def siblings(dev):
    """distCUDA2 on the knn test's uniform cloud, and fused-ssim on the shapes of the ssim test."""
    import test_gpu_siblings as TS
    from oracle import build_ref_torch
    out = {}
    pts = TS.knn_cloud()
    out["knn"] = {"value": ref_cuda.knn(torch.from_numpy(pts).to(dev)).cpu().numpy()[TS.KNN_SAMPLE]}
    ref = build_ref_torch.import_reference_packages()[1]
    for shape in TS.SSIM_SHAPES:
        out["ssim_" + "x".join(map(str, shape))] = TS.ssim_record(ref, shape, dev)
    return out


def main(out_dir):
    os.makedirs(out_dir, exist_ok=True)
    dev = torch.device("cuda:0")
    for family, cids in PC.FAMILIES.items():
        cases = {}
        for cid in cids:
            cases[cid] = reference_case(family, cid, dev)
            torch.cuda.empty_cache()
            print(family, cid, "R =", int(cases[cid]["num_rendered"]), flush=True)
        for path in PG.save(out_dir, f"parity_{family}", cases):
            print("wrote", path, os.path.getsize(path), "bytes", flush=True)
    for path in PG.save(out_dir, "siblings_ref", siblings(dev)):
        print("wrote", path, os.path.getsize(path), "bytes", flush=True)


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
