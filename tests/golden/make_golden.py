"""Generate tests/golden/*.npz from the UNMODIFIED reference CUDA rasterizer (oracle/_ref) on a B200.

Run on the GPU box (the reference cannot execute in the CPU-only container):
    python tests/golden/make_golden.py OUT_DIR
then copy OUT_DIR/*.npz into tests/golden/.  The fixtures pin the CPU oracle
(tests/test_oracle_golden.py, no GPU needed) and are checked again against the product on the GPU.
Inputs are not stored: they are regenerated from the seeds with sfgs.synthetic (numpy PCG64).
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, "skyfall-gs_b200"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import numpy as np
import torch

import golden_io
import helpers as Hh
from golden_cases import CASES, build_case
from oracle import ref_cuda


def main(out_dir):
    os.makedirs(out_dir, exist_ok=True)
    dev = torch.device("cuda:0")
    for name in CASES:
        scene, cam, bg, kw = build_case(name)
        d = Hh.to_torch(scene, cam, dev)
        bg_t = torch.from_numpy(bg).to(dev)
        colors = None
        if kw.get("colors_precomp"):
            colors = torch.from_numpy(kw["colors"]).to(dev)
        f = Hh.run_ref_forward(d, cam, kw["sh_degree"], bg_t, kernel_size=kw["kernel_size"],
                               scale_modifier=kw["scale_modifier"], colors=colors)
        it = ref_cuda.internals(f, scene.P, cam.height, cam.width)
        cot = [torch.from_numpy(c).to(dev) for c in kw["cot"]]
        g = Hh.run_ref_backward(d, cam, kw["sh_degree"], bg_t, f, cot, kernel_size=kw["kernel_size"],
                                scale_modifier=kw["scale_modifier"], colors=colors)
        g2 = Hh.run_ref_backward(d, cam, kw["sh_degree"], bg_t, f, cot, kernel_size=kw["kernel_size"],
                                 scale_modifier=kw["scale_modifier"], colors=colors)
        out = dict(num_rendered=np.int64(f["num_rendered"]), radii=f["radii"].cpu().numpy())
        for k in ("color", "depth", "norm", "alpha"):
            out[k] = f[k].cpu().numpy()
        for k in ("depths", "means2D", "cov3D", "conic_opacity", "rgb", "norm3D", "clamped", "tiles_touched",
                  "point_offsets", "n_contrib", "ranges", "keys", "point_list"):
            out["int_" + k] = it[k].cpu().numpy()
        for k in ("means2D", "colors", "opacity", "means3D", "cov3D", "norm3D", "sh", "scales", "rot", "conic", "depths"):
            out["grad_" + k] = g[k].cpu().numpy()
            out["gradspread_" + k] = np.float32((g[k] - g2[k]).abs().max().item() if g[k].numel() else 0.0)
        paths = golden_io.save(f"ref_{name}", out, out_dir)
        print(name, "R=", f["num_rendered"], "visible=", int((f["radii"] > 0).sum()), [os.path.getsize(p) for p in paths], "bytes")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
