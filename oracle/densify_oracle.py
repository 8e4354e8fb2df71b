"""TEST INFRASTRUCTURE — torch restatement of the reference's adaptive density control, on plain tensors.

Not imported by the product (skyfall-gs_b200/); only tests/ use it.  Each function restates, statement by statement and
with the same torch calls (so that it computes what the reference computes on whichever device it runs on), the
reference code it cites.  Pinned against the reference's own GaussianModel by tests/golden/make_densify_golden.py
(fixture tests/golden/densify_ref-*.npz, checked in tests/test_densify.py).
"""
import torch

FIELDS = ("xyz", "f_dc", "f_rest", "opacity", "scaling", "rotation")


def stats_update(grad4, radii, max_radii2D, accum, accum_abs, accum_abs_max, denom):
    """train.py:314-315 and GaussianModel.add_densification_stats (scene/gaussian_model.py:744-749); returns new tensors."""
    vis = radii > 0
    max_radii2D, accum, accum_abs, accum_abs_max, denom = (t.clone() for t in (max_radii2D, accum, accum_abs, accum_abs_max, denom))
    max_radii2D[vis] = torch.max(max_radii2D[vis], radii[vis])
    accum[vis] += torch.norm(grad4[vis, :2], dim=-1, keepdim=True)
    accum_abs[vis] += torch.norm(grad4[vis, 2:], dim=-1, keepdim=True)
    accum_abs_max[vis] = torch.max(accum_abs_max[vis], torch.norm(grad4[vis, 2:], dim=-1, keepdim=True))
    denom[vis] += 1
    return max_radii2D, accum, accum_abs, accum_abs_max, denom


def build_rotation(r):
    """utils/general_utils.py:78-99."""
    norm = torch.sqrt(r[:, 0] * r[:, 0] + r[:, 1] * r[:, 1] + r[:, 2] * r[:, 2] + r[:, 3] * r[:, 3])
    q = r / norm[:, None]
    R = torch.zeros((q.size(0), 3, 3), device=r.device, dtype=r.dtype)
    w, x, y, z = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
    R[:, 0, 0] = 1 - 2 * (y * y + z * z)
    R[:, 0, 1] = 2 * (x * y - w * z)
    R[:, 0, 2] = 2 * (x * z + w * y)
    R[:, 1, 0] = 2 * (x * y + w * z)
    R[:, 1, 1] = 1 - 2 * (x * x + z * z)
    R[:, 1, 2] = 2 * (y * z - w * x)
    R[:, 2, 0] = 2 * (x * z - w * y)
    R[:, 2, 1] = 2 * (y * z + w * x)
    R[:, 2, 2] = 1 - 2 * (x * x + y * y)
    return R


class _State:
    """The tensors densify_and_prune rewrites: parameters, both Adam moments (or None), max_radii2D."""

    def __init__(self, params, m, v, names):
        self.names = names
        self.p = {n: params[n] for n in names}
        self.m = {n: m[n] for n in names} if m is not None else None
        self.v = {n: v[n] for n in names} if v is not None else None
        self.max_radii2D = None

    def n(self):
        return self.p["xyz"].shape[0]

    def append(self, new):
        """densification_postfix + cat_tensors_to_optimizer (gaussian_model.py:603-651)."""
        for k in self.names:
            ext = new[k]
            if self.m is not None:
                self.m[k] = torch.cat((self.m[k], torch.zeros_like(ext)), dim=0)
                self.v[k] = torch.cat((self.v[k], torch.zeros_like(ext)), dim=0)
            self.p[k] = torch.cat((self.p[k], ext), dim=0)
        self.max_radii2D = torch.zeros((self.n(),), device=self.p["xyz"].device)

    def prune(self, mask):
        """prune_points + _prune_optimizer (gaussian_model.py:564-601)."""
        valid = ~mask
        for k in self.names:
            if self.m is not None:
                self.m[k] = self.m[k][valid]
                self.v[k] = self.v[k][valid]
            self.p[k] = self.p[k][valid]
        self.max_radii2D = self.max_radii2D[valid]


def densify_and_prune(params, exp_avg, exp_avg_sq, accum, accum_abs, denom, *, max_grad, min_opacity, extent, max_screen_size,
                      percent_dense, noise, extra=()):
    """scene/gaussian_model.py:694-735 (with :653-692 split, :694 clone).  `noise` [2S,3] stands for the standard-normal draw
    inside torch.normal(mean=0, std=stds) (:668).  Returns (params, exp_avg, exp_avg_sq, counts)."""
    names = list(FIELDS) + list(extra)
    st = _State(params, exp_avg, exp_avg_sq, names)
    grads = accum / denom
    grads[grads.isnan()] = 0.0
    grads_abs = accum_abs / denom
    grads_abs[grads_abs.isnan()] = 0.0
    if grads_abs.numel() > 0 and not torch.isinf(grads_abs).any() and not torch.isnan(grads_abs).any():
        ratio = (torch.norm(grads, dim=-1) >= max_grad).float().mean()
        try:
            Q = torch.quantile(grads_abs.reshape(-1), 1 - ratio)
        except Exception:
            Q = 0.99
    else:
        Q = 0.99
    before = st.n()
    # ---- densify_and_clone
    sel = torch.where(torch.norm(grads, dim=-1) >= max_grad, True, False)
    sel_abs = torch.where(torch.norm(grads_abs, dim=-1) >= Q, True, False)
    sel = torch.logical_or(sel, sel_abs)
    sel = torch.logical_and(sel, torch.max(torch.exp(st.p["scaling"]), dim=1).values <= percent_dense * extent)
    st.append({k: st.p[k][sel] for k in names})
    clone = st.n()
    # ---- densify_and_split
    N = 2
    n_init = st.n()
    padded = torch.zeros((n_init,), device=grads.device)
    padded[:grads.shape[0]] = grads.squeeze()
    sel = torch.where(padded >= max_grad, True, False)
    padded_abs = torch.zeros((n_init,), device=grads.device)
    padded_abs[:grads_abs.shape[0]] = grads_abs.squeeze()
    sel = torch.logical_or(sel, torch.where(padded_abs >= Q, True, False))
    sel = torch.logical_and(sel, torch.max(torch.exp(st.p["scaling"]), dim=1).values > percent_dense * extent)
    stds = torch.exp(st.p["scaling"])[sel].repeat(N, 1)
    samples = noise * stds + torch.zeros((stds.size(0), 3), device=stds.device)          # torch.normal(mean=means, std=stds)
    rots = build_rotation(st.p["rotation"][sel]).repeat(N, 1, 1)
    new = {k: st.p[k][sel].repeat(N, *([1] * (st.p[k].dim() - 1))) for k in names}
    new["xyz"] = torch.bmm(rots, samples.unsqueeze(-1)).squeeze(-1) + st.p["xyz"][sel].repeat(N, 1)
    new["scaling"] = torch.log(torch.exp(st.p["scaling"])[sel].repeat(N, 1) / (0.8 * N))
    n_split = int(sel.sum())
    st.append(new)
    st.prune(torch.cat((sel, torch.zeros(N * n_split, device=sel.device, dtype=torch.bool))))
    split = st.n()
    # ---- prune
    prune_mask = (torch.sigmoid(st.p["opacity"]) < min_opacity).squeeze(-1)
    if max_screen_size:
        big_vs = st.max_radii2D > max_screen_size
        big_ws = torch.exp(st.p["scaling"]).max(dim=1).values > 0.1 * extent
        prune_mask = torch.logical_or(torch.logical_or(prune_mask, big_vs), big_ws)
    st.prune(prune_mask)
    return st.p, st.m, st.v, dict(cloned=clone - before, split=split - clone, pruned=split - st.n(), n_split_sources=n_split,
                                  Q=float(Q))
