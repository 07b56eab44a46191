"""CPU oracle of eims_attribute_peaks  --  TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Integrated gradients of each graph's top predicted peak with respect to its atom features, by torch autograd through
`gcn_oracle.forward` (eval mode), with the definition of include/eims_b200.h:
  - baseline: all-zero atom features on the same graph;
  - the peak bin m_r of graph r: the (r mod k)-th largest bin of its own spectrum at alpha = 1, value descending, exact
    ties to the higher bin (eims_topk_peaks);
  - midpoint rule, alpha_s = (s + 1/2) / S, weight 1/S:  ig = x * (1/S) sum_s  d prob_{m_r} / d x  at alpha_s X.
"""
from __future__ import annotations

from collections import OrderedDict

import numpy as np
import torch

from . import gcn_oracle as O


def path_alphas(steps: int):
    """The S midpoint-rule points, as float32 values (what the device computes: (s + 0.5f) / S)."""
    return [float(np.float32(np.float32(s + 0.5) / np.float32(steps))) for s in range(steps)]


def topk_bins(prob: np.ndarray, k: int) -> np.ndarray:
    """[B, k] bins of the k largest values per row, value descending, exact ties to the higher bin."""
    B, M = prob.shape
    order = np.lexsort((-np.broadcast_to(np.arange(M), (B, M)), -prob), axis=1)
    return order[:, :k]


def _decisions_of(aux, sd, d: O.Dims):
    """The discrete choices a forward took (the keys `gcn_oracle.forward` accepts as `decisions`)."""
    sp = "spectrum_predictor"
    dec = {("relu", l): (aux[f"r{l}"] > 0) for l in range(d.num_gcn_layers)}
    for i, (u, j) in enumerate([("u1", 1), ("u2", 5)]):
        x = aux[u]
        ln = torch.nn.functional.layer_norm(x, (x.shape[1],), sd[f"{sp}.{j}.weight"].to(x.dtype),
                                            sd[f"{sp}.{j}.bias"].to(x.dtype), 1e-5)
        dec[("head_relu", i)] = ln > 0
    if "argmax" in aux:
        dec["argmax"] = aux["argmax"]
    return dec


def _forward(sd, g, x, d, dtype, dec, keep=False):
    work = OrderedDict((n, t.clone() if O.is_buffer(n) else t.detach().to(dtype)) for n, t in sd.items())
    return O.forward(work, g, x, d, False, update_running=False, dtype=dtype, keep=keep, decisions=dec)


def integrated_gradients(sd, g: O.Graph, feat, d: O.Dims, k: int, steps: int, *, decisions=None, dtype=torch.float64,
                         alphas=None):
    """Returns dict(bins [B], peak_prob [B], base_prob [B], ig [N, F], decisions {alpha: the forward's own choices}).

    `decisions`: optional {alpha: decisions dict of `gcn_oracle.forward`} - the choices to take at that path point
    (alpha 1.0 for the peak bins, 0.0 for the baseline, the path points otherwise); points without an entry run free.
    `alphas`: the path points (default `path_alphas(steps)`)."""
    dec = decisions or {}
    feat = torch.as_tensor(feat)
    x = feat.to(dtype)
    own = {}
    with torch.no_grad():
        p1, aux = _forward(sd, g, x, d, dtype, dec.get(1.0), keep=True)
        own[1.0] = _decisions_of(aux, sd, d)
        tab = topk_bins(p1.numpy(), k)
        B = g.batch_size
        bins = torch.as_tensor(tab[np.arange(B), np.arange(B) % k])
        rows = torch.arange(B)
        peak = p1[rows, bins]
        p0, aux = _forward(sd, g, torch.zeros_like(x), d, dtype, dec.get(0.0), keep=True)
        own[0.0] = _decisions_of(aux, sd, d)
        base = p0[rows, bins]
    alphas = path_alphas(steps) if alphas is None else alphas
    acc = torch.zeros_like(x)
    for a in alphas:
        xa = (a * x).detach().requires_grad_(True)
        p, aux = _forward(sd, g, xa, d, dtype, dec.get(a), keep=True)
        own[a] = _decisions_of({kk: (v.detach() if torch.is_tensor(v) else v) for kk, v in aux.items()}, sd, d)
        gx, = torch.autograd.grad(p[rows, bins].sum(), xa)
        acc += gx
    ig = x * acc / len(alphas)
    return dict(bins=bins.numpy().astype(np.int32), peak_prob=peak.numpy(), base_prob=base.numpy(), ig=ig.detach().numpy(),
                decisions=own)


def decisions_change(decs) -> dict:
    """For a list of decision dicts of one batch (e.g. along a path): per key, the number of entries that are not the
    same in all of them."""
    out = {}
    for key in decs[0]:
        first = decs[0][key]
        changed = torch.zeros_like(first, dtype=torch.bool)
        for dd in decs[1:]:
            changed |= dd[key] != first
        out[key] = int(changed.sum())
    return out
