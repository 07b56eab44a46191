"""Gradients w.r.t. the atom features, and the backward of eval-mode forwards (eims_backward_feat, GCNSpectrum with
node_features), against the fp64 oracle on poisoned plans.

What these gradients are for: per-atom attribution of predicted peaks, `prob[:, m].sum().backward()` on features that
require grad, then `(x.grad * x).sum(1)`.  In eval mode BatchNorm is the affine map of the running statistics and
nothing couples molecules, so one backward over a batch gives every molecule's attribution.

The rows reuse the shapes of test_gpu_dispatch (one layer, odd and wide feature widths, hidden 1024, the planes path of
batch-4096 plans) plus the batch-512 / hidden-256 / 1000-bin shape in eval mode.  Each row runs, on a NaN-poisoned plan
each time, a training forward with a random dprob, a training forward with the MSE loss (dprob NULL) and an eval
forward with a random dprob.  The GPU's ReLU, head-ReLU and arg-max decisions are checked to be near-ties of the
free-running fp64 oracle and then injected into it (the flip-aware protocol of test_gpu_dispatch); every parameter
gradient and the feature gradient are then held to 1e-4 of the oracle, two-dimensional ones also column by column."""
import ctypes as C
import json
from collections import OrderedDict

import numpy as np
import pytest
import torch

from eims_b200 import _lib
from eims_b200 import script as S
from eims_b200.engine import DeviceDataset, FlatParams, Plan, make_step
from eims_b200.synth import dense_spectra, synth_molecules, synth_peaks
from oracle import gcn_oracle as O
from test_gpu_dispatch import (BACKENDS, COL_REL, ORDER_REL, REL, ROWS, _dims, col_err, dropout_masks, kernel_names,
                               make_plan, make_table, odims, poison, random_running_stats, rel_err)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
NEW_KERNELS = ["bn_bwd_apply_q0_kernel", "layer0_dgrad_kernel", "feat_grad_kernel", "bn_eval_zstat_kernel"]

# the dispatch rows this feature runs on, and batch 512 / hidden 256 / 1000 bins in eval mode
FROWS = {n: dict(ROWS[n], modes=("train", "mse", "eval"))
         for n in ("one_layer", "odd_width", "wide_odd", "dropin_defaults", "wide", "big_batch")}
FROWS["eval_512"] = dict(d=_dims(256, 3, 6, 1000, "combined", 0.2), B=512, atoms=40, paths=["tcgen05", "simt"], modes=("eval",))
FSEEDS = {name: 700 + 11 * k for k, name in enumerate(FROWS)}


def fcases():
    return [pytest.param(n, p, id=f"{n}-{p}") for n, r in FROWS.items() for p in r["paths"] if p.split("+")[0] in BACKENDS]


def setup(name):
    r = FROWS[name]
    d, B, seed = r["d"], r["B"], FSEEDS[name]
    table = make_table(B, r["atoms"], seed, d.node_feat_dim)
    targets = dense_spectra(*synth_peaks(B, d.max_mz, seed=seed + 2), d.max_mz)
    N, E = int(table.node_ptr[-1]), int(2 * table.bond_ptr[-1])
    Bc, Nc = r.get("cap") or (B, N)
    Ec = E if "cap" not in r else 2 * (Nc + 3 * Bc)
    sd = random_running_stats(O.init_params(odims(d), seed + 3), d, seed + 4)
    return d, table, targets, (Bc, Nc, Ec), sd


def gpu_decisions(plan, d, B, N):
    H, L = d.hidden_dim, d.num_gcn_layers
    dec = {("relu", l): (plan.buffer(f"z{l}", torch.float32, (N, H)) > 0).cpu() for l in range(L)}
    dec[("head_relu", 0)] = (plan.buffer("y1", torch.float32, (B, 2 * H)) > 0).cpu()
    dec[("head_relu", 1)] = (plan.buffer("y2", torch.float32, (B, H)) > 0).cpu()
    if d.pooling in ("max", "combined"):
        dec["argmax"] = plan.buffer("argmax", torch.int32, (B, H)).cpu().to(torch.int64)
    return dec


def gpu_backward(plan, ds, fp, mode, step, dprob, canary_rows=0):
    """Batch build, forward of `mode` ("train": dprob given, "mse": the loss kernel's gradient, "eval": dprob given,
    BatchNorm from the running statistics) and eims_backward_feat with dfeat.  dfeat has `canary_rows` rows past N
    filled with 7."""
    B, d = ds.num_mols, plan.d
    plan.batch_build(ds, None, B)
    N, _ = plan.check()
    plan.forward(fp, mode != "eval", step)
    if mode == "train":
        plan.sigmoid()
    elif mode == "mse":
        plan.loss(ds.targets, None, "mse", True)
    # eval: no eims_sigmoid - the backward must compute prob itself
    dfeat = torch.full((N + canary_rows, d.node_feat_dim), 7.0, device=DEV)
    fp.grads.zero_()
    plan.backward_feat(fp, None if mode == "mse" else dprob, dfeat)
    torch.cuda.synchronize()
    return dict(prob=plan.buffer("prob", torch.float32, (B, d.max_mz)).cpu().numpy().copy(),
                grads={k: v.cpu().numpy().copy() for k, v in fp.named_grads().items()},
                dfeat=dfeat[:N].cpu().numpy().copy(), canary=dfeat[N:].cpu(), dec=gpu_decisions(plan, d, B, N), N=N)


def flip_report(sd, graph, feat, d, training, masks, dec):
    """The GPU's decisions that differ from the free-running fp64 oracle's must be near-ties (test_gpu_dispatch)."""
    L, sp = d.num_gcn_layers, "spectrum_predictor"
    work = OrderedDict((n, t.clone()) for n, t in sd.items())
    with torch.no_grad():
        _, aux = O.forward(work, graph, feat, odims(d), training, dropout_masks=masks, update_running=False,
                           dtype=torch.float64, keep=True)
    rep, bad = {}, []
    for l in range(L):
        r = aux[f"r{l}"]
        diff = dec[("relu", l)] != (r > 0)
        worst = float((r.abs() / r.abs().amax(dim=0, keepdim=True).clamp_min(1e-30))[diff].max()) if diff.any() else 0.0
        rep[f"relu{l}"] = (int(diff.sum()), worst)
        if int(diff.sum()) > 4096 or worst >= 1e-4:
            bad.append(f"relu{l} flips")
    for i, (u, k) in enumerate([("u1", 1), ("u2", 5)]):
        x = aux[u]
        ln = torch.nn.functional.layer_norm(x, (x.shape[1],), sd[f"{sp}.{k}.weight"].double(), sd[f"{sp}.{k}.bias"].double(), 1e-5)
        live = masks[("head", i)].bool() if masks is not None else torch.ones_like(ln, dtype=torch.bool)
        diff = (dec[("head_relu", i)] != (ln > 0)) & live
        worst = float((ln.abs() / ln.abs().amax(dim=0, keepdim=True).clamp_min(1e-30))[diff].max()) if diff.any() else 0.0
        rep[f"head_relu{i}"] = (int(diff.sum()), worst)
        if worst >= 1e-4:
            bad.append(f"head_relu{i} flips")
    if "argmax" in dec:
        hbn = aux[f"bn{L - 1}"]
        gap = (hbn.gather(0, aux["argmax"]) - hbn.gather(0, dec["argmax"])).abs() / hbn.abs().amax(dim=0, keepdim=True).clamp_min(1e-30)
        rep["argmax"] = float(gap.max())
        if float(gap.max()) >= 1e-4:
            bad.append("argmax flips")
    return rep, bad


def oracle_grads(sd, graph, feat, d, training, masks, dec, dprob, targets, dtype):
    """(spectra, {parameter name: gradient}, feature gradient) of the oracle on the GPU's branch."""
    work = OrderedDict((n, t.clone() if O.is_buffer(n) else t.detach().to(dtype).clone().requires_grad_(True))
                       for n, t in sd.items())
    x = feat.detach().to(dtype).clone().requires_grad_(True)
    pred, _ = O.forward(work, graph, x, odims(d), training, dropout_masks=masks, update_running=False, dtype=dtype,
                        decisions=dec)
    loss = O.mse_loss(pred, targets.to(dtype)) if dprob is None else (pred * dprob.to(dtype)).sum()
    names = O.trainable(work)
    gs = torch.autograd.grad(loss, [work[n] for n in names] + [x])
    return pred.detach(), OrderedDict((n, g.numpy()) for n, g in zip(names, gs[:-1])), gs[-1].numpy()


def compare(res, g64, x64, g32, x32, L):
    """oracle_check's gradient rules, with the feature gradient as one more tensor."""
    rep, bad = {}, []
    got = dict(res["grads"], dfeat=res["dfeat"])
    ref, own = dict(g64, dfeat=x64), dict(g32, dfeat=x32)
    gmax = max(float(np.abs(g).max()) for g in g64.values())
    for n, g in got.items():
        r, o = ref[n], own[n]
        if n != "dfeat" and np.abs(r).max() < 1e-6 * gmax:   # zero in exact arithmetic: rounding noise on both sides
            rep[n] = ("abs", float(np.abs(g - r).max() / gmax))
            if rep[n][1] >= REL:
                bad.append(f"grad {n} (abs)")
            continue
        e = rel_err(g, r)
        rep[n] = ("rel", e)
        if not e < REL:
            bad.append(f"grad {n}")
        if g.ndim == 2:
            ce = max(col_err(g, r, 0), col_err(g, r, 1))
            floor = max(col_err(o, r, 0), col_err(o, r, 1))
            rep[n] = ("rel", e, ce, floor)
            if not ce < max(COL_REL, 16 * floor):
                bad.append(f"grad {n} (column-scaled)")
    if len(res["grads"]) != 4 * L + 10:
        bad.append("gradient count")
    if not all(np.isfinite(g).all() for g in got.values()) or not np.isfinite(res["prob"]).all():
        bad.append("NaN / Inf in an output")
    return rep, bad


# ------------------------------------------------------------------------------------------------ oracle parity
@pytest.mark.parametrize("name,path", fcases())
def test_feature_and_parameter_gradients_match_the_oracle(name, path, tmp_path):
    d, table, targets, caps, sd = setup(name)
    B, L = table.num_mols, d.num_gcn_layers
    graph, feat = O.Graph.from_mols([table.mol(i) for i in range(B)])
    dprob = torch.from_numpy(np.random.default_rng(FSEEDS[name] + 5).standard_normal((B, d.max_mz)).astype(np.float32))
    step = make_step(step=3, seed=11)
    ds = DeviceDataset(table, targets, DEV)
    tt = torch.from_numpy(targets)
    report, failures = {}, {}
    for mode in FROWS[name]["modes"]:
        plan = make_plan(d, *caps, path)
        fp = FlatParams(d, DEV)
        fp.load_state_dict(sd)
        res = gpu_backward(plan, ds, fp, mode, step, dprob.to(DEV), canary_rows=3)
        training = mode != "eval"
        masks = dropout_masks(d, step, res["N"], B) if training else None
        frep, bad = flip_report(sd, graph, feat, d, training, masks, res["dec"])
        dp = None if mode == "mse" else dprob
        p64, g64, x64 = oracle_grads(sd, graph, feat, d, training, masks, res["dec"], dp, tt, torch.float64)
        _, g32, x32 = oracle_grads(sd, graph, feat, d, training, masks, res["dec"], dp, tt, torch.float32)
        grep, gbad = compare(res, g64, x64, g32, x32, L)
        spectra = rel_err(res["prob"], p64.numpy())
        if not spectra < REL:
            gbad.append("spectra")
        if not bool((res["canary"] == 7.0).all()):
            gbad.append("dfeat rows past N were written")
        report[mode] = dict(flips=frep, grads=grep, spectra=spectra)
        if bad + gbad:
            failures[mode] = bad + gbad
        del plan
    with open(tmp_path / f"feature_grads_{name}_{path}.json", "w") as fh:
        json.dump(report, fh, indent=1)
    assert not failures, (failures, report)


# ------------------------------------------------------------------------------------------------ plan level
def _small(path="tcgen05", name="dropin_defaults"):
    d, table, targets, caps, sd = setup(name)
    return d, table, targets, make_plan(d, *caps, path), sd


@pytest.mark.parametrize("backend", BACKENDS)
def test_eval_backward_has_no_side_effects_and_finite_outputs(backend):
    """An eval forward + backward on a NaN-poisoned plan: parameters and running statistics bit-unchanged, every output
    finite (the head data gradients must not rely on a zeroing only a training forward does)."""
    d, table, targets, plan, sd = _small(backend)
    ds = DeviceDataset(table, targets, DEV)
    fp = FlatParams(d, DEV)
    fp.load_state_dict(sd)
    p0, r0 = fp.params.clone(), fp.bn_running.clone()
    dprob = torch.randn(table.num_mols, d.max_mz, device=DEV)
    res = gpu_backward(plan, ds, fp, "eval", make_step(step=1, seed=3), dprob)
    assert torch.equal(fp.params, p0) and torch.equal(fp.bn_running, r0)
    assert fp.num_batches_tracked == [0] * d.num_gcn_layers
    assert np.isfinite(res["dfeat"]).all() and all(np.isfinite(g).all() for g in res["grads"].values())
    assert np.isfinite(res["prob"]).all()


@pytest.mark.parametrize("backend", BACKENDS)
def test_backward_feat_without_dfeat_equals_backward(backend):
    """Training mode: eims_backward_feat(dfeat=NULL) and eims_backward give the same parameter gradients."""
    d, table, targets, caps, sd = setup("dropin_defaults")
    ds = DeviceDataset(table, targets, DEV)
    out = []
    for feat_call in (False, True):
        plan = make_plan(d, *caps, backend)
        fp = FlatParams(d, DEV)
        fp.load_state_dict(sd)
        plan.batch_build(ds, None, ds.num_mols)
        plan.forward(fp, True, make_step(step=2, seed=5))
        plan.loss(ds.targets, None, "mse", True)
        fp.grads.zero_()
        plan.backward_feat(fp) if feat_call else plan.backward(fp)
        out.append({k: v.cpu().numpy().copy() for k, v in fp.named_grads().items()})
    a, b = out
    gmax = max(float(np.abs(g).max()) for g in a.values())
    worst = max(float(np.abs(a[k] - b[k]).max()) for k in a) / gmax
    assert worst <= ORDER_REL, worst


def test_state_errors_and_canary():
    """eims_backward keeps refusing eval forwards; eims_backward_feat refuses an eval backward without dprob and a
    second training backward; dfeat rows past N keep their canary."""
    d, table, targets, plan, sd = _small()
    ds = DeviceDataset(table, targets, DEV)
    fp = FlatParams(d, DEV)
    fp.load_state_dict(sd)
    lib = _lib.load()
    plan.batch_build(ds, None, ds.num_mols)
    N, _ = plan.check()
    plan.forward(fp, False)
    assert lib.eims_backward(plan.h, _lib.ptr(fp.params), None, _lib.ptr(fp.grads), plan.stream) == _lib.ERR_STATE
    dprob = torch.randn(ds.num_mols, d.max_mz, device=DEV)
    assert lib.eims_backward(plan.h, _lib.ptr(fp.params), _lib.ptr(dprob), _lib.ptr(fp.grads), plan.stream) == _lib.ERR_STATE
    assert lib.eims_backward_feat(plan.h, _lib.ptr(fp.params), None, _lib.ptr(fp.grads), None, plan.stream) == _lib.ERR_ARG
    dfeat = torch.full((N + 64, d.node_feat_dim), 7.0, device=DEV)
    plan.backward_feat(fp, dprob, dfeat)
    torch.cuda.synchronize()
    assert bool((dfeat[N:] == 7.0).all()) and bool(torch.isfinite(dfeat[:N]).all()) and not bool((dfeat[:N] == 7.0).all())
    plan.forward(fp, True, make_step(step=1, seed=1))
    plan.loss(ds.targets, None, "mse", True)
    plan.backward_feat(fp, None, dfeat)
    with pytest.raises(_lib.EimsError):
        plan.backward_feat(fp, None, dfeat)


def test_launches_under_the_profiler():
    """backward_feat with dfeat launches the new kernels (and the eval statistics kernel in eval mode); without dfeat
    layer 0 stays the fused apply pass; a training step (eims_train_step) launches none of them."""
    d, table, targets, plan, sd = _small()
    ds = DeviceDataset(table, targets, DEV)
    fp = FlatParams(d, DEV)
    fp.load_state_dict(sd)
    dprob = torch.randn(ds.num_mols, d.max_mz, device=DEV)
    acts = [torch.profiler.ProfilerActivity.CPU, torch.profiler.ProfilerActivity.CUDA]
    runs = {}
    for key in ("eval_dfeat", "train_dfeat", "eval_nodfeat", "train_step"):
        with torch.profiler.profile(activities=acts) as prof:
            if key == "train_step":
                plan.train_step(ds, None, fp, make_step(step=4, seed=2))
            else:
                plan.batch_build(ds, None, ds.num_mols)
                N, _ = plan.check()
                plan.forward(fp, key.startswith("train"), make_step(step=3, seed=2))
                plan.sigmoid()
                dfeat = torch.empty(N, d.node_feat_dim, device=DEV) if key.endswith("_dfeat") else None
                plan.backward_feat(fp, dprob, dfeat)
            torch.cuda.synchronize()
        runs[key] = kernel_names(prof)
    has = lambda key, k: any(k in n for n in runs[key])
    for k in NEW_KERNELS:
        assert has("eval_dfeat", k), (k, runs["eval_dfeat"])
        assert not has("train_step", k), (k, runs["train_step"])
    for k in NEW_KERNELS[:3]:
        assert has("train_dfeat", k), (k, runs["train_dfeat"])
    assert not has("train_dfeat", "bn_eval_zstat_kernel")
    for key in ("eval_nodfeat", "train_step"):
        assert has(key, "bn_bwd_apply_kernel<true>") and not any(has(key, k) for k in NEW_KERNELS[:3]), runs[key]


# ------------------------------------------------------------------------------------------------ the module
def small_cfg(dropout=0.0):
    c = S.Config()
    c.hidden_dim, c.max_mz, c.dropout = 64, 100, dropout
    return c


def molgraphs(n, seed, max_atoms=14):
    t = synth_molecules(n, max_atoms=max_atoms, seed=seed)
    return t, [S.MolGraph(*t.mol(i)) for i in range(n)]


def make_model(sd, cfg, seed=1234):
    m = S.GCNSpectrum(6, cfg).to(DEV)
    m.load_state_dict(sd)
    m._seed = seed
    return m


def test_node_features_are_honoured():
    """ndata['feat'] after .to(device) is a CUDA tensor of the host features; None, the graph's own tensor and a copy
    of it give bit-identical spectra in both modes; perturbed features give the oracle's spectra on them."""
    cfg = small_cfg()
    d = O.Dims(hidden_dim=64, max_mz=100, dropout=0.0)
    sd = random_running_stats(O.init_params(d, 21), d, 22)
    table, graphs = molgraphs(12, 23)
    g = S.batch(graphs).to(DEV)
    feat = g.ndata["feat"]
    assert feat.is_cuda and feat.dtype == torch.float32 and tuple(feat.shape) == (g.num_nodes(), 6)
    assert torch.equal(feat.cpu(), torch.from_numpy(table.feat))
    graph, hfeat = O.Graph.from_mols([table.mol(i) for i in range(12)])
    pert = feat.clone()
    pert[::3, 0] += 0.5
    pert[1::4, 5] -= 1.0
    for training in (False, True):
        outs = []
        for arg in (None, "own", "clone", "pert"):
            m = make_model(sd, cfg)
            m.train(training)
            x = {None: None, "own": feat, "clone": feat.clone(), "pert": pert}[arg]
            with torch.no_grad():
                outs.append(m(g, x).cpu().numpy())
        if training:   # a training forward's head GEMMs split K over float atomics: equal to summation order
            assert max(rel_err(outs[1], outs[0]), rel_err(outs[2], outs[0])) <= ORDER_REL
        else:
            assert np.array_equal(outs[0], outs[1]) and np.array_equal(outs[0], outs[2])
        work = OrderedDict((n, t.clone()) for n, t in sd.items())
        ref, _ = O.forward(work, graph, pert.cpu(), d, training, update_running=False, dtype=torch.float64)
        assert rel_err(outs[3], ref.numpy()) < REL, training
        assert not np.array_equal(outs[3], outs[0])


def attribution(model, graphs, m):
    g = S.batch(graphs).to(DEV)
    x = g.ndata["feat"].clone().requires_grad_()
    prob = model(g, x)
    prob[:, m].sum().backward()
    return (x.grad * x).sum(1).detach().cpu().numpy(), prob.detach()


def test_eval_attribution_batched_equals_looped():
    """Eval mode couples nothing across molecules: the attribution of one batched backward equals one-molecule calls;
    parameters, running statistics and num_batches_tracked are left as they were."""
    cfg = small_cfg(dropout=0.2)
    d = O.Dims(hidden_dim=64, max_mz=100, dropout=0.2)
    sd = random_running_stats(O.init_params(d, 31), d, 32)
    _, graphs = molgraphs(16, 33)
    model = make_model(sd, cfg).eval()
    before = {k: v.clone() for k, v in model.state_dict().items()}
    m = 40
    batched, prob = attribution(model, graphs, m)
    assert np.isfinite(batched).all() and np.abs(batched).max() > 0
    looped = np.concatenate([attribution(model, [gr], m)[0] for gr in graphs])
    assert rel_err(batched, looped) < 1e-5
    after = model.state_dict()
    assert all(torch.equal(before[k], after[k]) for k in before)


def test_eval_forward_is_differentiable_and_frozen_models_give_feature_grads():
    cfg = small_cfg()
    d = O.Dims(hidden_dim=64, max_mz=100)
    sd = random_running_stats(O.init_params(d, 41), d, 42)
    _, graphs = molgraphs(6, 43)
    g = S.batch(graphs).to(DEV)
    model = make_model(sd, cfg).eval()
    out = model(g, None)
    assert out.grad_fn is not None
    out.sum().backward()
    assert model.flat.grad is not None and float(model.flat.grad.abs().max()) > 0
    model.flat.requires_grad_(False)
    x = g.ndata["feat"].clone().requires_grad_()
    model(g, x).sum().backward()
    assert x.grad is not None and bool(torch.isfinite(x.grad).all())
    with torch.no_grad():
        assert model(g, None).grad_fn is None


def test_module_errors_raise_before_any_launch():
    cfg = small_cfg()
    sd = O.init_params(O.Dims(hidden_dim=64, max_mz=100), 51)
    _, graphs = molgraphs(5, 52)
    g = S.batch(graphs).to(DEV)
    model = make_model(sd, cfg).eval()
    feat = g.ndata["feat"]
    model(g, None)   # builds the plan
    seq = model._fwd_seq
    for bad in (feat[:-1].clone(), feat.double(), feat.cpu(), feat[:, :5].clone()):
        with pytest.raises(RuntimeError):
            model(g, bad.requires_grad_())
        assert model._fwd_seq == seq
    # a backward after a newer forward
    x1, x2 = feat.clone().requires_grad_(), feat.clone().requires_grad_()
    p1 = model(g, x1)
    model(g, x2)
    with pytest.raises(RuntimeError, match="another forward"):
        p1.sum().backward()
    # the same forward differentiated twice, and a double backward
    p = model(g, x1)
    p.sum().backward(retain_graph=True)
    with pytest.raises(RuntimeError):
        p.sum().backward()
    p = model(g, x2)
    gx, = torch.autograd.grad(p.sum(), x2, create_graph=True)
    with pytest.raises(RuntimeError):
        gx.sum().backward()
