"""Golden vectors for adaptive density control, produced by the reference's OWN GaussianModel (scene/gaussian_model.py)
running unmodified on CPU (run where /root/reference exists):

  * add_densification_stats (:744-749) + the max_radii2D statement of train.py:314,
  * densify_and_prune (:694-735) including the optimizer surgery (:564-651),

for two models: plain (with the screen-size rule) and appearance-enabled (extra per-Gaussian `embeddings` group, no
screen-size rule).  The only intervention: torch.normal is wrapped so that the standard-normal draw behind
torch.normal(mean=0, std=stds) (:668) is recorded next to the result (eps * std + mean, which is what torch computes).
"""
import os
import sys
import types
from argparse import Namespace

import numpy as np
import torch

REF = os.environ.get("SFGS_REFERENCE", "/root/reference")
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REF)
sys.path.insert(0, os.path.join(HERE, "..", "..", "skyfall-gs_b200"))


def _stub(name):
    m = types.ModuleType(name)
    m.__file__ = name + ".py"

    def _getattr(k):
        if k.startswith("__"):
            raise AttributeError(k)
        return lambda *a, **k2: None
    m.__getattr__ = _getattr
    return m


for name in ("plyfile", "OpenEXR"):          # I/O dependencies of modules this script never calls
    sys.modules.setdefault(name, _stub(name))


class _CudaToCpu(torch.overrides.TorchFunctionMode):
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
        if func is torch.Tensor.to:
            args = tuple(self._fix(a) for a in args)
        return func(*args, **kwargs)


NAMES = ("xyz", "f_dc", "f_rest", "opacity", "scaling", "rotation")
ATTR = {"xyz": "_xyz", "f_dc": "_features_dc", "f_rest": "_features_rest", "opacity": "_opacity", "scaling": "_scaling",
        "rotation": "_rotation", "embeddings": "_embeddings"}
OPT = Namespace(percent_dense=0.01, position_lr_init=1.6e-4, position_lr_final=1.6e-6, position_lr_delay_mult=0.01,
                position_lr_max_steps=30000, idu_position_lr_max_steps=30000, feature_lr=2.5e-3, opacity_lr=0.05, scaling_lr=5e-3,
                rotation_lr=1e-3, appearance_embedding_lr=1e-3, appearance_embedding_regularization=0.0, embedding_lr=5e-3,
                appearance_mlp_lr=1e-3)
EXTENT = 10.0
MAX_GRAD = 0.0002


def build(GaussianModel, P, appearance, seed):
    g = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=g)    # noqa: E731
    pc = GaussianModel(3, appearance, 4, 32)
    pc.spatial_lr_scale = 1.0
    pc._xyz = torch.nn.Parameter(r(P, 3) * 5)
    pc._features_dc = torch.nn.Parameter(r(P, 1, 3))
    pc._features_rest = torch.nn.Parameter(r(P, 15, 3) * 0.1)
    pc._opacity = torch.nn.Parameter(r(P, 1) * 4)
    pc._scaling = torch.nn.Parameter(torch.log(torch.exp(r(P, 3) * 1.3) * 0.04))       # straddles 0.1 and 1.0
    pc._rotation = torch.nn.Parameter(r(P, 4))
    if appearance:
        pc._embeddings = torch.nn.Parameter(r(P, 24))
    pc.max_radii2D = torch.rand(P, generator=g) * 40
    pc.training_setup(OPT, num_train_cameras=3)
    names = NAMES + (("embeddings",) if appearance else ())
    for _ in range(2):                                     # two Adam steps so that both moments are populated
        for n in names:
            p = getattr(pc, ATTR[n])
            p.grad = r(*p.shape) * 1e-3
        pc.optimizer.step()
    pc.optimizer.zero_grad(set_to_none=True)
    return pc, names, g


def snapshot(pc, names, tag, out):
    groups = {gr["name"]: gr for gr in pc.optimizer.param_groups}
    for n in names:
        p = groups[n]["params"][0]
        assert p is getattr(pc, ATTR[n])
        st = pc.optimizer.state[p]
        out[f"{tag}_{n}"] = p.detach().numpy().copy()
        out[f"{tag}_{n}_m"] = st["exp_avg"].numpy().copy()
        out[f"{tag}_{n}_v"] = st["exp_avg_sq"].numpy().copy()


def main():
    out = {}
    with _CudaToCpu():
        from scene.gaussian_model import GaussianModel
        for case, (P, appearance, screen) in {"plain": (640, False, 20), "appearance": (400, True, None)}.items():
            pc, names, g = build(GaussianModel, P, appearance, seed=11 if appearance else 5)
            # ---- statistics: three iterations of train.py:314-315
            for it in range(3):
                radii = torch.randint(-1, 30, (P,), generator=g, dtype=torch.int32).clamp_min(0)
                vsp = torch.zeros(P, 4, requires_grad=True)
                vsp.grad = torch.randn(P, 4, generator=g) * 1.3e-4
                out[f"{case}_stats_in{it}_radii"] = radii.numpy().copy()
                out[f"{case}_stats_in{it}_grad"] = vsp.grad.numpy().copy()
                if it == 0:
                    out[f"{case}_stats_start_max_radii2D"] = pc.max_radii2D.numpy().copy()
                vis = radii > 0
                pc.max_radii2D[vis] = torch.max(pc.max_radii2D[vis], radii[vis])          # train.py:314
                pc.add_densification_stats(vsp, vis)                                      # train.py:315
            for k in ("max_radii2D", "xyz_gradient_accum", "xyz_gradient_accum_abs", "xyz_gradient_accum_abs_max", "denom"):
                out[f"{case}_stats_{k}"] = getattr(pc, k).numpy().copy()
            # ---- densify_and_prune
            snapshot(pc, names, f"{case}_before", out)
            rec = []
            real_normal = torch.normal

            def normal(mean, std):
                eps = torch.randn(std.shape, generator=g)
                rec.append(eps)
                return eps * std + mean
            torch.normal = normal
            try:
                counts = pc.densify_and_prune(MAX_GRAD, 0.005, EXTENT, screen)
            finally:
                torch.normal = real_normal
            snapshot(pc, names, f"{case}_after", out)
            out[f"{case}_noise"] = rec[0].numpy().copy()
            out[f"{case}_counts"] = np.array(counts, dtype=np.int64)
            out[f"{case}_after_max_radii2D"] = pc.max_radii2D.numpy().copy()
            print(case, "P", P, "->", pc.get_xyz.shape[0], "counts (cloned, split, pruned)", counts, "noise", tuple(rec[0].shape))
    out["meta"] = np.array([EXTENT, MAX_GRAD, 0.005, OPT.percent_dense])
    sys.path.insert(0, os.path.join(HERE, ".."))
    import golden_io
    golden_io.save("densify_ref", out, HERE)
    print("wrote densify_ref")


if __name__ == "__main__":
    main()
