"""The integrated-gradients oracle (oracle/ig_oracle.py) on the CPU: the midpoint rule, and completeness on a model and
molecules whose integrand is smooth along the whole path."""
from collections import OrderedDict

import numpy as np
import torch

from eims_b200.synth import synth_molecules
from oracle import gcn_oracle as O
from oracle import ig_oracle as IG


def _model(seed, pooling="sum", H=32, M=40):
    d = O.Dims(hidden_dim=H, max_mz=M, pooling=pooling, num_gcn_layers=2)
    sd = O.init_params(d, seed)
    g = torch.Generator().manual_seed(seed)
    for l in range(d.num_gcn_layers):
        sd[f"batch_norms.{l}.running_mean"] = torch.randn(H, generator=g) * 0.3
        sd[f"batch_norms.{l}.running_var"] = torch.rand(H, generator=g) + 0.5
    return d, sd


def _batch(n, seed):
    t = synth_molecules(n, max_atoms=10, seed=seed)
    return O.Graph.from_mols([t.mol(i) for i in range(n)])


def test_one_point_is_x_times_the_gradient_at_half():
    d, sd = _model(3, "combined")
    g, feat = _batch(6, 4)
    k = 3
    res = IG.integrated_gradients(sd, g, feat, d, k, 1)
    x = feat.double()
    xa = (0.5 * x).requires_grad_(True)
    work = OrderedDict((n, t.clone() if O.is_buffer(n) else t.double()) for n, t in sd.items())
    p, _ = O.forward(work, g, xa, d, False, update_running=False, dtype=torch.float64)
    rows = torch.arange(g.batch_size)
    gx, = torch.autograd.grad(p[rows, torch.as_tensor(res["bins"]).long()].sum(), xa)
    assert np.allclose(res["ig"], (x * gx).numpy(), rtol=1e-12, atol=1e-15)
    # the bins are each graph's (r mod k)-th largest, ties to the higher bin
    with torch.no_grad():
        p1, _ = O.forward(OrderedDict((n, t.clone()) for n, t in work.items()), g, x, d, False, update_running=False,
                          dtype=torch.float64)
    for r in range(g.batch_size):
        row = p1[r].numpy()
        order = sorted(range(d.max_mz), key=lambda m: (-row[m], -m))
        assert res["bins"][r] == order[r % k]
        assert res["peak_prob"][r] == row[res["bins"][r]]


def test_topk_ties_go_to_the_higher_bin():
    prob = np.array([[0.5, 0.9, 0.5, 0.9, 0.1]])
    assert IG.topk_bins(prob, 4).tolist() == [[3, 1, 2, 0]]


def test_completeness_on_a_smooth_path():
    """Sum pooling, one GraphConv layer whose bias keeps every ReLU open along the path (BatchNorm centred on the
    baseline's activation), and LayerNorm affines that keep the head's ReLUs open.  The oracle must report that no
    decision changes at any path point; the integrand is then smooth, so the completeness residual of the midpoint rule
    shrinks as S grows, at its second-order rate."""
    d = O.Dims(hidden_dim=32, max_mz=40, pooling="sum", num_gcn_layers=1)
    sd = O.init_params(d, 5)
    sd["gcn_layers.0.weight"] = sd["gcn_layers.0.weight"] * 0.3
    sd["gcn_layers.0.bias"] = torch.full((d.hidden_dim,), 4.0)
    sd["batch_norms.0.running_mean"] = torch.full((d.hidden_dim,), 4.0)
    sp = "spectrum_predictor"
    for j in (1, 5):
        sd[f"{sp}.{j}.weight"] = sd[f"{sp}.{j}.weight"] * 0.05
        sd[f"{sp}.{j}.bias"] = torch.ones_like(sd[f"{sp}.{j}.bias"])
    g, feat = _batch(5, 6)
    k = 2
    resid = []
    for S in (4, 32, 256):
        res = IG.integrated_gradients(sd, g, feat, d, k, S)
        changes = IG.decisions_change(list(res["decisions"].values()))
        assert all(v == 0 for v in changes.values()), changes
        total = np.zeros(g.batch_size)
        np.add.at(total, g.gid.numpy(), res["ig"].sum(1))
        delta = res["peak_prob"] - res["base_prob"]
        assert np.abs(delta).min() > 1e-4
        resid.append(float(np.abs(total - delta).max() / np.abs(delta).max()))
    assert resid[0] > resid[1] > resid[2], resid
    assert resid[1] / resid[2] > 30 and resid[2] < 1e-3, resid
