"""Adaptive density control (SURVEY.md 8f rank 3): per-iteration statistics + densify_and_prune.

CPU (`-m "not gpu"`): the torch restatement oracle/densify_oracle.py is pinned against tests/golden/densify_ref-*.npz, which
the reference's own GaussianModel produced (tests/golden/make_densify_golden.py) — bit-exact, both cases.
GPU: the kernels (through the C ABI) against the restatement running on the same GPU (= what the reference's torch ops
compute there) and against the fixture.  Bar: masks, row order, every copied value and both Adam moments bit-exact;
a split child's position (the reference's cuBLAS bmm) within 1e-6 relative; a child's scale bit-exact against the GPU
restatement and within 1 ulp of the CPU-generated fixture (torch divides by a scalar differently on the two devices).
"""
import os
import sys
import types

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "skyfall-gs_b200"))
sys.path.insert(0, ROOT)
import golden_io  # noqa: E402
from oracle import densify_oracle as O  # noqa: E402

GOLD = golden_io.load("densify_ref")
EXTENT, MAX_GRAD, MIN_OPACITY, PERCENT_DENSE = (float(v) for v in GOLD["meta"])
CASES = {"plain": dict(extra=(), screen=20), "appearance": dict(extra=("embeddings",), screen=None)}
STAT_KEYS = ("max_radii2D", "xyz_gradient_accum", "xyz_gradient_accum_abs", "xyz_gradient_accum_abs_max", "denom")


def names_of(case):
    return list(O.FIELDS) + list(CASES[case]["extra"])


def load(case, tag, dev):
    p, m, v = {}, {}, {}
    for n in names_of(case):
        p[n] = torch.from_numpy(GOLD[f"{case}_{tag}_{n}"]).to(dev)
        m[n] = torch.from_numpy(GOLD[f"{case}_{tag}_{n}_m"]).to(dev)
        v[n] = torch.from_numpy(GOLD[f"{case}_{tag}_{n}_v"]).to(dev)
    return p, m, v


def stats_inputs(case, dev):
    P = GOLD[f"{case}_stats_in0_radii"].shape[0]
    st = [torch.from_numpy(GOLD[f"{case}_stats_start_max_radii2D"]).to(dev)] + [torch.zeros((P, 1), device=dev) for _ in range(4)]
    its = [(torch.from_numpy(GOLD[f"{case}_stats_in{i}_grad"]).to(dev), torch.from_numpy(GOLD[f"{case}_stats_in{i}_radii"]).to(dev))
           for i in range(3)]
    return st, its


def stats_final(case, dev):
    return [torch.from_numpy(GOLD[f"{case}_stats_{k}"]).to(dev) for k in STAT_KEYS]


# ----------------------------------------------------------------------------------------------------------------------
# CPU: the oracle is the reference
@pytest.mark.parametrize("case", list(CASES))
def test_oracle_statistics_match_the_reference_model(case):
    st, its = stats_inputs(case, "cpu")
    for grad, radii in its:
        st = list(O.stats_update(grad, radii, *st))
    for got, want, k in zip(st, stats_final(case, "cpu"), STAT_KEYS):
        assert torch.equal(got, want), k


@pytest.mark.parametrize("case", list(CASES))
def test_oracle_densify_matches_the_reference_model(case):
    p, m, v = load(case, "before", "cpu")
    _, accum, accum_abs, _, denom = stats_final(case, "cpu")
    noise = torch.from_numpy(GOLD[f"{case}_noise"])
    np_, nm, nv, counts = O.densify_and_prune(p, m, v, accum, accum_abs, denom, max_grad=MAX_GRAD, min_opacity=MIN_OPACITY,
                                              extent=EXTENT, max_screen_size=CASES[case]["screen"], percent_dense=PERCENT_DENSE,
                                              noise=noise, extra=CASES[case]["extra"])
    assert (counts["cloned"], counts["split"], counts["pruned"]) == tuple(int(c) for c in GOLD[f"{case}_counts"])
    wp, wm, wv = load(case, "after", "cpu")
    for n in names_of(case):
        assert torch.equal(np_[n], wp[n]), n
        assert torch.equal(nm[n], wm[n]), n + " exp_avg"
        assert torch.equal(nv[n], wv[n]), n + " exp_avg_sq"


# ----------------------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu


def close_rel(a, b, rel):
    scale = float(b.abs().max()) + 1e-30
    return float((a - b).abs().max()) <= rel * scale


@gpu
@pytest.mark.parametrize("case", list(CASES))
def test_statistics_kernel_is_bit_exact(case):
    from sfgs import densify as D
    dev = torch.device("cuda:0")
    st, its = stats_inputs(case, dev)
    ora = [t.clone() for t in st]
    for grad, radii in its:
        D.densification_stats(grad.contiguous(), radii.contiguous(), *st)
        ora = list(O.stats_update(grad, radii, *ora))
    torch.cuda.synchronize()
    for got, o, want, k in zip(st, ora, stats_final(case, dev), STAT_KEYS):
        assert torch.equal(got, o), k + " vs the restatement on this GPU"
        # the fixture was produced on the CPU, whose two-element torch.norm rounds differently from the GPU's
        if k in ("max_radii2D", "denom"):
            assert torch.equal(got, want), k + " vs the reference fixture"
        else:
            assert close_rel(got, want, 3e-7), k + " vs the reference fixture"


def run_ours(case, dev, noise):
    from sfgs import densify as D
    p, m, v = load(case, "before", dev)
    _, accum, accum_abs, _, denom = stats_final(case, dev)
    return D.densify_tensors(p, m, v, accum, accum_abs, denom, max_grad=MAX_GRAD, min_opacity=MIN_OPACITY, extent=EXTENT,
                             max_screen_size=CASES[case]["screen"], percent_dense=PERCENT_DENSE, noise=noise,
                             extra=CASES[case]["extra"])


@gpu
@pytest.mark.parametrize("case", list(CASES))
def test_densify_kernels_match_restatement_and_fixture(case):
    dev = torch.device("cuda:0")
    noise = torch.from_numpy(GOLD[f"{case}_noise"]).to(dev)
    gp, gm, gv, t = run_ours(case, dev, noise)
    p, m, v = load(case, "before", dev)
    _, accum, accum_abs, _, denom = stats_final(case, dev)
    op, om, ov, counts = O.densify_and_prune(p, m, v, accum, accum_abs, denom, max_grad=MAX_GRAD, min_opacity=MIN_OPACITY,
                                             extent=EXTENT, max_screen_size=CASES[case]["screen"], percent_dense=PERCENT_DENSE,
                                             noise=noise, extra=CASES[case]["extra"])
    wp, wm, wv = load(case, "after", dev)
    assert (t["C"], t["S"]) == (counts["cloned"], counts["split"]) == tuple(int(c) for c in GOLD[f"{case}_counts"][:2])
    assert t["P"] + t["C"] + t["S"] - t["new_P"] == counts["pruned"] == int(GOLD[f"{case}_counts"][2])
    for n in names_of(case):
        assert gp[n].shape == op[n].shape == wp[n].shape, n
        if n == "xyz":
            assert close_rel(gp[n], op[n], 1e-6) and close_rel(gp[n], wp[n], 1e-6)
            kept = t["K"] + t["KC"]
            assert torch.equal(gp[n][:kept], wp[n][:kept])          # everything but the children is a copy
        elif n == "scaling":
            assert torch.equal(gp[n], op[n])
            assert close_rel(gp[n], wp[n], 2e-7)
        else:
            assert torch.equal(gp[n], op[n]), n
            assert torch.equal(gp[n], wp[n]), n
        assert torch.equal(gm[n], om[n]) and torch.equal(gm[n], wm[n]), n + " exp_avg"
        assert torch.equal(gv[n], ov[n]) and torch.equal(gv[n], wv[n]), n + " exp_avg_sq"


class _Model:
    """The attributes of the reference's GaussianModel that densify_and_prune touches (scene/gaussian_model.py)."""
    appearance_enabled = False
    percent_dense = PERCENT_DENSE


@gpu
def test_model_level_call_rebuilds_the_optimizer_like_the_reference():
    """densify.densify_and_prune(pc, ...) on an object shaped like the reference's GaussianModel with a real torch Adam:
    parameters, per-parameter Adam state, statistics and return value as gaussian_model.py:564-651, 694-735 leave them;
    the noise comes from the generator exactly as torch.normal(mean=0, std=stds) would draw it."""
    from sfgs import densify as D
    dev = torch.device("cuda:0")
    case = "plain"
    p, m, v = load(case, "before", dev)
    pc = _Model()
    groups = []
    for n in O.FIELDS:
        par = torch.nn.Parameter(p[n].clone())
        setattr(pc, D.ATTRS[n], par)
        groups.append({"params": [par], "lr": 1e-3, "name": n})
    pc.optimizer = torch.optim.Adam(groups, lr=0.0, eps=1e-15)
    for g in pc.optimizer.param_groups:
        par = g["params"][0]
        pc.optimizer.state[par] = {"step": torch.tensor(2.0), "exp_avg": m[g["name"]].clone(), "exp_avg_sq": v[g["name"]].clone()}
    pc.max_radii2D, pc.xyz_gradient_accum, pc.xyz_gradient_accum_abs, pc.xyz_gradient_accum_abs_max, pc.denom = stats_final(case, dev)
    accum, accum_abs, denom = pc.xyz_gradient_accum.clone(), pc.xyz_gradient_accum_abs.clone(), pc.denom.clone()

    torch.manual_seed(123)
    ret = D.densify_and_prune(pc, MAX_GRAD, MIN_OPACITY, EXTENT, 20)
    S = int(GOLD[f"{case}_counts"][1])
    torch.manual_seed(123)
    stds = torch.ones((2 * S, 3), device=dev)
    noise = torch.normal(mean=torch.zeros((2 * S, 3), device=dev), std=stds)      # the reference's draw (:666-668) for unit stds
    op, om, ov, counts = O.densify_and_prune(p, m, v, accum, accum_abs, denom, max_grad=MAX_GRAD, min_opacity=MIN_OPACITY,
                                             extent=EXTENT, max_screen_size=20, percent_dense=PERCENT_DENSE, noise=noise)
    assert ret == (counts["cloned"], counts["split"], counts["pruned"])
    newP = op["xyz"].shape[0]
    by_name = {g["name"]: g for g in pc.optimizer.param_groups}
    for n in O.FIELDS:
        par = by_name[n]["params"][0]
        assert par is getattr(pc, D.ATTRS[n]) and isinstance(par, torch.nn.Parameter) and par.requires_grad
        st = pc.optimizer.state[par]
        assert len(pc.optimizer.state) == len(O.FIELDS) and float(st["step"]) == 2.0
        if n == "xyz":
            assert close_rel(par.data, op[n], 1e-6)
        else:
            assert torch.equal(par.data, op[n]), n
        assert torch.equal(st["exp_avg"], om[n]) and torch.equal(st["exp_avg_sq"], ov[n]), n
    for k in STAT_KEYS:
        t = getattr(pc, k)
        assert t.shape[0] == newP and float(t.abs().max()) == 0.0
    # the rebuilt optimizer steps
    for g in pc.optimizer.param_groups:
        g["params"][0].grad = torch.ones_like(g["params"][0])
    pc.optimizer.step()


@gpu
def test_densify_edge_cases():
    from sfgs import densify as D
    dev = torch.device("cuda:0")
    g = torch.Generator(device="cpu").manual_seed(3)

    def scene(P):
        r = lambda *s: torch.randn(*s, generator=g).to(dev)   # noqa: E731
        return {"xyz": r(P, 3), "f_dc": r(P, 1, 3), "f_rest": r(P, 15, 3), "opacity": r(P, 1) * 4,
                "scaling": torch.log(torch.exp(r(P, 3)) * 0.04), "rotation": r(P, 4)}
    kw = dict(max_grad=MAX_GRAD, min_opacity=MIN_OPACITY, extent=EXTENT, percent_dense=PERCENT_DENSE)
    # empty model
    p = scene(0)
    z = torch.zeros((0, 1), device=dev)
    np_, nm, nv, t = D.densify_tensors(p, None, None, z, z, z, max_screen_size=None, **kw)
    assert t["new_P"] == 0 and nm is None and np_["f_rest"].shape == (0, 15, 3)
    # nothing visible yet: denom = 0 -> NaN gradients -> 0; the quantile falls on 0, so every Gaussian is selected (as in the reference)
    for P in (1, 1023, 1024, 1025, 5000):
        p = scene(P)
        z = torch.zeros((P, 1), device=dev)
        noise_free = dict(max_screen_size=None, **kw)
        np_, nm, nv, t = D.densify_tensors(p, None, None, z, z.clone(), z.clone(), **noise_free)
        op, _, _, counts = O.densify_and_prune({k: v.clone() for k, v in p.items()}, None, None, z.clone(), z.clone(), z.clone(),
                                               max_grad=MAX_GRAD, min_opacity=MIN_OPACITY, extent=EXTENT, max_screen_size=None,
                                               percent_dense=PERCENT_DENSE, noise=torch.zeros((2 * t["S"], 3), device=dev))
        assert t["new_P"] == op["xyz"].shape[0], P
        assert (t["C"], t["S"]) == (counts["cloned"], counts["split"])
        for n in ("f_dc", "f_rest", "opacity", "rotation", "scaling"):
            assert torch.equal(np_[n], op[n]), (P, n)
    # wrong noise shape is refused
    p = scene(2000)
    a = torch.rand((2000, 1), device=dev) * 1e-3
    d = torch.ones((2000, 1), device=dev)
    with pytest.raises(ValueError):
        D.densify_tensors(p, None, None, a, a.clone(), d, max_screen_size=20, noise=torch.zeros((1, 3), device=dev), **kw)
    with pytest.raises(ValueError):
        D.densify_tensors(p, {k: v.clone() for k, v in p.items()}, None, a, a.clone(), d, max_screen_size=20, **kw)


@gpu
def test_densify_at_training_size_against_the_restatement():
    """1M Gaussians: same counts, same copied rows as the torch restatement (= the reference's op sequence) on this GPU,
    and the time of both (reported by bench.py as `next_ops`; here only a sanity bound)."""
    from sfgs import densify as D
    dev = torch.device("cuda:0")
    P = 1_000_000
    g = torch.Generator(device=dev).manual_seed(9)
    r = lambda *s: torch.randn(*s, generator=g, device=dev)   # noqa: E731
    p = {"xyz": r(P, 3) * 50, "f_dc": r(P, 1, 3), "f_rest": r(P, 15, 3) * 0.1, "opacity": r(P, 1) * 3,
         "scaling": torch.log(torch.exp(r(P, 3) * 1.2) * 0.5), "rotation": r(P, 4)}
    m = {k: r(*v.shape) * 1e-3 for k, v in p.items()}
    v = {k: (r(*t.shape) * 1e-3) ** 2 for k, t in p.items()}
    denom = torch.randint(0, 4, (P, 1), generator=g, device=dev).float()
    accum = torch.rand((P, 1), generator=g, device=dev) * 3e-4 * denom
    accum_abs = torch.rand((P, 1), generator=g, device=dev) * 6e-4 * denom
    extent = 120.0
    kw = dict(max_grad=MAX_GRAD, min_opacity=MIN_OPACITY, extent=extent, max_screen_size=20, percent_dense=PERCENT_DENSE)
    Q = D.gradient_thresholds(accum, accum_abs, denom, MAX_GRAD)
    _, _, _, t0 = D.densify_tensors(p, m, v, accum, accum_abs, denom, abs_threshold=Q, noise=None, **kw)
    noise = torch.randn((2 * t0["S"], 3), generator=g, device=dev)
    # one untimed call of each first: whichever runs first otherwise pays the allocator's growth to the output sizes
    D.densify_tensors(p, m, v, accum, accum_abs, denom, noise=noise, **kw)
    O.densify_and_prune(dict(p), dict(m), dict(v), accum, accum_abs, denom, noise=noise, **kw)
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    ev[0].record()
    gp, gm, gv, t = D.densify_tensors(p, m, v, accum, accum_abs, denom, noise=noise, **kw)
    ev[1].record()
    op, om, ov, counts = O.densify_and_prune(dict(p), dict(m), dict(v), accum, accum_abs, denom, noise=noise, **kw)
    ev[2].record()
    torch.cuda.synchronize()
    assert t["S"] > 1000 and t["C"] > 1000 and t["new_P"] != P
    assert (t["C"], t["S"], t["P"] + t["C"] + t["S"] - t["new_P"]) == (counts["cloned"], counts["split"], counts["pruned"])
    for n in O.FIELDS:
        if n == "xyz":
            assert close_rel(gp[n], op[n], 1e-6)
        else:
            assert torch.equal(gp[n], op[n]), n
        assert torch.equal(gm[n], om[n]) and torch.equal(gv[n], ov[n]), n
    ours_ms, ref_ms = ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2])
    print(f"densify_and_prune 1M: ours {ours_ms:.2f} ms, torch op sequence {ref_ms:.2f} ms")
    assert ours_ms < ref_ms
