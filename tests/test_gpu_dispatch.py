"""Whole-step parity at the shapes the plan and the launchers dispatch on, on a poisoned workspace.

The C ABI takes hidden 64..1024, 1..16 layers, 1..8 atom features and 4..4096 bins, and the plan picks kernels and
template instances from those sizes, from its capacities and from the live batch.  Each row below exists for a set of
variants that no other test reaches (one-layer network, hidden widths that leave a partial 128-column tile, SpMM rows
split over two warps, LayerNorm at widths that are not a power-of-two multiple of 128, the shortest and longest
spectra, atom feature widths other than 6, the persistent GEMM with BatchNorm statistics in its epilogue, the
molecule-tile SpMM of large plans, the BatchNorm-backward statistics pass over a materialised dh that only widths
above 256 take, ...); `test_rows_launch_their_kernels` proves under the profiler that they are reached, so that a
later change of a dispatch threshold cannot silently turn a row into a copy of another.

Every plan here is poisoned before its first use: each float workspace buffer is filled with NaN, so a kernel that
reads what no producer wrote this batch (rows past the live size, the padding of a partial tile, a stale plane)
turns the result into NaN instead of passing on the zeros a fresh allocation happens to hold.

Comparison protocol (as in test_gpu_e2e.test_full_size_flip_aware_gradients, for any depth and pooling): the GPU's
discrete decisions (ReLU masks, max-pool arg-max) are checked to be near-ties of the free-running fp64 oracle and then
injected into it, so both differentiate the same branch; spectra, loss, every gradient tensor and the BatchNorm
running statistics are then held to 1e-4 of that oracle.  Two-dimensional gradients are also held column by column
(and row by row) against their own scale, which a wrong tail tile cannot hide under."""
import ctypes as C
import json
import os

import numpy as np
import pytest
import torch

from eims_b200 import _lib
from eims_b200._lib import check, ptr
from eims_b200.engine import DeviceDataset, FlatParams, ModelDims, Plan, make_step
from eims_b200.synth import MolTable, dense_spectra, synth_molecules, synth_peaks
from oracle import gcn_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
REL = 1e-4
COL_REL = 1e-3      # column-scaled bound (columns down to 1e-3 of the tensor's scale), or 16 x the fp32 oracle's own
COL_MIN_SCALE = 1e-3
ORDER_REL = 2e-5    # same maths, other summation order (test_gpu_dp.test_two_part_indirect_step_equals_whole_step)
BACKENDS = os.environ.get("EIMS_TEST_BACKENDS", "tcgen05,simt").split(",")


def _dims(H, L, F, M, pooling, p):
    return ModelDims(node_feat_dim=F, hidden_dim=H, num_gcn_layers=L, max_mz=M, pooling=pooling, dropout=p)


def _defaults():
    from eims_b200 import script
    return ModelDims.from_config(script.Config())


# name -> model dims, live batch (molecules, atoms per molecule <= max_atoms), plan capacity (None: exact), GEMM paths,
# the kernels the row exists for (tensor-core backend) and kernels whose absence is the point
ROWS = {
    "one_layer": dict(d=_dims(64, 1, 6, 100, "max", 0.0), B=24, atoms=20, paths=["tcgen05", "simt"],
                      expect=["bn_bwd_apply_kernel<true>", "layer0_fwd_kernel"],
                      absent=["spmm_norm_kernel", "spmm_mol_kernel", "bn_bwd_apply_kernel<false>"]),
    "odd_width": dict(d=_dims(192, 2, 3, 12, "mean", 0.2), B=33, atoms=40, paths=["tcgen05", "simt"],
                      expect=["spmm_norm_kernel<2, 2, false>", "spmm_norm_kernel<2, 1, true>", "ln_relu_drop_bwd_kernel<4>",
                              "ln_relu_drop_bwd_kernel<2>", "bn_bwd_stats_top_kernel"],
                      absent=["bn_bwd_stats_kernel"]),
    "wide_odd": dict(d=_dims(320, 4, 8, 4, "sum", 0.0), B=40, atoms=40, paths=["tcgen05", "simt"],
                     expect=["spmm_norm_kernel<4, 1, false>", "bn_bwd_stats_kernel", "ln_relu_drop_bwd_kernel<8>",
                             "ln_relu_drop_bwd_kernel<4>"],
                     absent=["spmm_norm_kernel<4, 1, true>"]),
    "two_part_rows": dict(d=_dims(768, 2, 6, 500, "combined", 0.2), B=24, atoms=64, paths=["tcgen05", "tcgen05+planes"],
                          expect=["spmm_norm_kernel<4, 1, false>", "ln_relu_drop_bwd_kernel<16>", "bn_bwd_stats_kernel"]),
    "longest_spectrum": dict(d=_dims(512, 3, 1, 4096, "combined", 0.0), B=48, atoms=40, paths=["tcgen05", "simt"],
                             expect=["loss_kernel<false>", "spmm_norm_kernel<4, 1, false>", "ln_relu_drop_bwd_kernel<8>",
                                     "bn_bwd_stats_kernel"]),
    "dropin_defaults": dict(d=_defaults(), B=64, atoms=64, paths=["tcgen05", "simt"],
                            expect=["spmm_norm_kernel<2, 2, false>", "spmm_norm_kernel<2, 1, true>", "bn_bwd_stats_top_kernel"]),
    "persistent_fused_bn": dict(d=_dims(512, 3, 6, 1000, "combined", 0.0), B=24, atoms=64, cap=(24, 40960),
                                paths=["tcgen05+noplanes"], expect=["gemm_3xtf32_persistent_kernel"],
                                absent=["gemm_planes_kernel"]),
    "wide": dict(d=_dims(1024, 3, 6, 1000, "combined", 0.0), B=24, atoms=128, paths=["tcgen05"],
                 expect=["spmm_norm_kernel<4, 1, false>", "ln_relu_drop_bwd_kernel<16>"], absent=["gemm_planes_kernel"]),
    "big_batch": dict(d=_dims(256, 3, 6, 1000, "combined", 0.2), B=4096, atoms=6, cap=(4096, 4096 * 48), paths=["tcgen05"],
                      expect=["spmm_mol_kernel<2, false, 256>", "k1_scan_kernel", "gemm_planes_kernel",
                              "spmm_norm_kernel<2, 1, true>", "bn_bwd_stats_top_kernel"]),
    "tiles_128": dict(d=_dims(512, 3, 6, 1000, "combined", 0.0), B=64, atoms=160, cap=(2048, 2048 * 100), paths=["tcgen05"],
                      expect=["spmm_mol_kernel<1, false, 128>", "gemm_planes_kernel"]),
}
SEEDS = {name: 100 + 7 * k for k, name in enumerate(ROWS)}


def row_cases():
    out = []
    for name, r in ROWS.items():
        for path in r["paths"]:
            if path.split("+")[0] in BACKENDS:
                out.append(pytest.param(name, path, id=f"{name}-{path}"))
    return out


# ------------------------------------------------------------------------------------------------ helpers
def rel_err(got, ref):
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    return float(np.abs(got - ref).max() / max(np.abs(ref).max(), 1e-30))


def col_err(got, ref, axis):
    """Worst error of a 2-D tensor relative to each column's (axis=0) or row's (axis=1) own max-abs, over the
    columns whose scale is at least COL_MIN_SCALE of the tensor's."""
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    scale = np.abs(ref).max(axis=axis)
    keep = scale >= COL_MIN_SCALE * max(scale.max(), 1e-30)
    if not keep.any():
        return 0.0
    err = np.abs(got - ref).max(axis=axis)
    return float((err[keep] / scale[keep]).max())


def odims(d: ModelDims):
    return O.Dims(d.node_feat_dim, d.hidden_dim, d.num_gcn_layers, d.max_mz, d.pooling, d.dropout)


def make_table(n, max_atoms, seed, F):
    """Synthetic molecules; for F != 6 the atom features are random normal (the synthetic descriptors take 1 to 6
    distinct values per column, which makes narrow feature widths degenerate)."""
    t = synth_molecules(n, max_atoms=max_atoms, seed=seed)
    if F == 6:
        return t
    feat = np.random.default_rng(seed + 1).standard_normal((t.feat.shape[0], F)).astype(np.float32)
    return MolTable(t.node_ptr, t.bond_ptr, feat, t.bond_begin, t.bond_end)


def float_buffer_names(plan):
    """Every float buffer eims_plan_create carves (both sets of the double-buffered batch tables, a_l / q / wplanes at
    their full two-plane size); not the integer tables, nor dims / flags / bn_partials, which the bind zeroes."""
    L = plan.d.num_gcn_layers
    names = [f"{n}#{s}" for n in ("norm", "x", "a0") for s in (0, 1)]
    names += [f"a{l}" for l in range(1, L)] + ["wplanes"]
    for l in range(L):
        names += [f"z{l}", f"bn_mean{l}", f"bn_invstd{l}", f"bn_scale{l}", f"bn_shift{l}"]
    names += ["bn_means2", "readout", "zstat", "u1", "u2", "logits", "dy2", "dy1", "dG", "y1", "ln1", "y2", "ln2",
              "prob", "dlogits", "row_loss", "row_cos", "dh", "q", "da"]
    return names


def poison(plan):
    for n in float_buffer_names(plan):
        try:
            buf = plan.buffer(n)
        except _lib.EimsError:
            assert n == "wplanes", n          # only plans that may take the planes path have it
            continue
        buf.fill_(float("nan"))
    torch.cuda.synchronize()


def make_plan(d, Bc, Nc, Ec, path):
    plan = Plan(d, Bc, Nc, Ec, DEV, gemm_backend=path.split("+")[0])
    if path.endswith("+planes"):
        plan.set_gemm_planes("on")
    elif path.endswith("+noplanes"):
        plan.set_gemm_planes("off")
    poison(plan)
    return plan


def random_running_stats(sd, d, seed):
    """Random BatchNorm running statistics, and nonzero GraphConv biases and BatchNorm affines: with the reference's
    zero biases a GEMM row past the live size (zero-filled operands, zero bias, ReLU) evaluates to 0 and a statistic
    that wrongly counts it would not change."""
    g = torch.Generator().manual_seed(seed)
    for l in range(d.num_gcn_layers):
        sd[f"gcn_layers.{l}.bias"] = torch.randn(d.hidden_dim, generator=g) * 0.1
        sd[f"batch_norms.{l}.weight"] = 1.0 + torch.randn(d.hidden_dim, generator=g) * 0.1
        sd[f"batch_norms.{l}.bias"] = torch.randn(d.hidden_dim, generator=g) * 0.1
        sd[f"batch_norms.{l}.running_mean"] = torch.randn(d.hidden_dim, generator=g) * 0.3
        sd[f"batch_norms.{l}.running_var"] = torch.rand(d.hidden_dim, generator=g) * 1.5 + 0.5
    return sd


def kernel_names(prof):
    out = set()
    for e in prof.key_averages():
        k = e.key
        if "eims::" in k:
            k = k[5:] if k.startswith("void ") else k
            out.add(k.split("(")[0])
    return sorted(out)


def gpu_step(plan, ds, fp, step):
    """Batch build + training forward + MSE loss + backward (no optimiser): spectra, loss, gradients, decisions,
    BatchNorm running statistics after the step."""
    B, d = ds.num_mols, plan.d
    plan.batch_build(ds, None, B)
    plan.forward(fp, True, step)
    plan.loss(ds.targets, None, "mse", True)
    fp.grads.zero_()
    plan.backward(fp)
    N, _ = plan.check()
    H, L = d.hidden_dim, d.num_gcn_layers
    dec = {("relu", l): (plan.buffer(f"z{l}", torch.float32, (N, H)) > 0).cpu() for l in range(L)}
    dec[("head_relu", 0)] = (plan.buffer("y1", torch.float32, (B, 2 * H)) > 0).cpu()
    dec[("head_relu", 1)] = (plan.buffer("y2", torch.float32, (B, H)) > 0).cpu()
    if d.pooling in ("max", "combined"):
        dec["argmax"] = plan.buffer("argmax", torch.int32, (B, H)).cpu().to(torch.int64)
    return dict(prob=plan.buffer("prob", torch.float32, (B, d.max_mz)).cpu().numpy().copy(),
                loss=plan.buffer("row_loss")[:B].double().sum().item() / (B * d.max_mz),
                grads={k: v.cpu().numpy().copy() for k, v in fp.named_grads().items()},
                running=fp.bn_running.cpu().numpy().copy(), dec=dec, N=N)


def dropout_masks(d, step, N, B):
    """The Philox masks of the step: GCN site l (< L-1) is oracle key ("gcn", l), the head sites are L and L+1."""
    if d.dropout == 0.0:
        return None
    lib, H, L = _lib.load(), d.hidden_dim, d.num_gcn_layers
    sites = [(("gcn", l), l, N, H) for l in range(L - 1)] + [(("head", 0), L, B, 2 * H), (("head", 1), L + 1, B, H)]
    masks = {}
    for key, site, rows, width in sites:
        m = torch.empty(rows, width, device=DEV)
        check(lib.eims_dropout_mask(float(d.dropout), int(step.seed), int(step.step), site, rows, width, ptr(m),
                                    C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        masks[key] = m.cpu()
    return masks


def setup_row(name, path, extra_cap=None):
    r = ROWS[name]
    d, B, seed = r["d"], r["B"], SEEDS[name]
    table = make_table(B, r["atoms"], seed, d.node_feat_dim)
    targets = dense_spectra(*synth_peaks(B, d.max_mz, seed=seed + 2), d.max_mz)
    N, E = int(table.node_ptr[-1]), int(2 * table.bond_ptr[-1])
    Bc, Nc = r.get("cap") or (B, N)
    Ec = E if "cap" not in r else 2 * (Nc + 3 * Bc)
    sd = random_running_stats(O.init_params(odims(d), seed + 3), d, seed + 4)
    return d, table, targets, (Bc, Nc, Ec), sd


def run_gpu(d, table, targets, caps, sd, path, step, profile=False):
    """One poisoned plan: a training step, then (re-poisoned) an eval forward with the running statistics the step
    left.  Returns the step's results, the eval spectra and (profile=True) the kernels launched."""
    plan = make_plan(d, *caps, path)
    ds = DeviceDataset(table, targets, DEV)
    fp = FlatParams(d, DEV)
    fp.load_state_dict(sd)
    prof = None
    if profile:
        prof = torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU, torch.profiler.ProfilerActivity.CUDA])
        prof.__enter__()
    res = gpu_step(plan, ds, fp, step)
    poison(plan)
    res["eval"] = plan.infer_batch(ds, None, fp).clone().cpu().numpy()
    res["eval_sd"] = {k: v.cpu() for k, v in fp.state_dict().items()}
    torch.cuda.synchronize()
    if profile:
        prof.__exit__(None, None, None)
        res["kernels"] = kernel_names(prof)
    res["masks"] = dropout_masks(d, step, res["N"], table.num_mols)
    return res


def oracle_check(d, table, targets, sd, res):
    """Flip-aware comparison of one GPU step with the fp64 oracle.  Returns (report, failures)."""
    B, L, H = table.num_mols, d.num_gcn_layers, d.hidden_dim
    graph, feat = O.Graph.from_mols([table.mol(i) for i in range(B)])
    tt = torch.from_numpy(targets)
    od, masks, dec = odims(d), res["masks"], res["dec"]
    rep, bad = {"flips": {}}, []
    # 1. every decision on which the GPU and the free-running fp64 oracle disagree is a near-tie
    _, _, _, aux = O.loss_and_grads(sd, graph, feat, tt, od, dtype=torch.float64, keep=True, dropout_masks=masks)
    for l in range(L):
        r = aux[f"r{l}"].detach()
        diff = dec[("relu", l)] != (r > 0)
        scale = r.abs().amax(dim=0, keepdim=True).clamp_min(1e-30)
        worst = float((r.abs() / scale)[diff].max()) if diff.any() else 0.0
        rep["flips"][f"relu{l}"] = {"count": int(diff.sum()), "of": diff.numel(), "max_abs_r_over_col_scale": worst}
        if int(diff.sum()) > 4096 or worst >= 1e-4:
            bad.append(f"relu{l} flips")
    sp = "spectrum_predictor"
    for i, (u, k) in enumerate([("u1", 1), ("u2", 5)]):
        x = aux[u].detach()
        ln = torch.nn.functional.layer_norm(x, (x.shape[1],), sd[f"{sp}.{k}.weight"].double(), sd[f"{sp}.{k}.bias"].double(), 1e-5)
        live = masks[("head", i)].bool() if masks is not None else torch.ones_like(ln, dtype=torch.bool)
        diff = (dec[("head_relu", i)] != (ln > 0)) & live      # a dropped position is 0 on both sides whatever its sign
        scale = ln.abs().amax(dim=0, keepdim=True).clamp_min(1e-30)
        worst = float((ln.abs() / scale)[diff].max()) if diff.any() else 0.0
        rep["flips"][f"head_relu{i}"] = {"count": int(diff.sum()), "of": diff.numel(), "max_abs_over_col_scale": worst}
        if worst >= 1e-4:
            bad.append(f"head_relu{i} flips")
    if "argmax" in dec:
        hbn = aux[f"bn{L - 1}"].detach()
        adiff = dec["argmax"] != aux["argmax"]
        gap = (hbn.gather(0, aux["argmax"]) - hbn.gather(0, dec["argmax"])).abs() / hbn.abs().amax(dim=0, keepdim=True).clamp_min(1e-30)
        rep["flips"]["argmax"] = {"count": int(adiff.sum()), "of": adiff.numel(), "max_gap_over_col_scale": float(gap.max())}
        if float(gap.max()) >= 1e-4:
            bad.append("argmax flips")
    # 2. same branch on both sides: spectra, loss, gradients, running statistics
    p64, l64, g64, a64 = O.loss_and_grads(sd, graph, feat, tt, od, dtype=torch.float64, keep=True, dropout_masks=masks, decisions=dec)
    _, _, g32, _ = O.loss_and_grads(sd, graph, feat, tt, od, dropout_masks=masks, decisions=dec)
    rep["spectra"] = rel_err(res["prob"], p64.numpy())
    rep["loss"] = abs(res["loss"] - float(l64)) / float(l64)
    gmax = max(float(g.abs().max()) for g in g64.values())
    rep["grads"], rep["grads_abs"], rep["cols"], rep["floors"] = {}, {}, {}, {}
    for n, g in res["grads"].items():
        ref, own = g64[n].numpy(), g32[n].numpy()
        if np.abs(ref).max() < 1e-6 * gmax:
            # zero in exact arithmetic (BatchNorm makes the loss invariant to it): what is left is rounding noise on
            # both sides, bounded against the largest gradient scale of the step
            rep["grads_abs"][n] = float(np.abs(g - ref).max() / gmax)
            if rep["grads_abs"][n] >= REL:
                bad.append(f"grad {n} (abs)")
            continue
        rep["grads"][n] = rel_err(g, ref)
        if rep["grads"][n] >= REL:
            bad.append(f"grad {n}")
        if g.ndim == 2:
            e = max(col_err(g, ref, 0), col_err(g, ref, 1))
            floor = max(col_err(own, ref, 0), col_err(own, ref, 1))
            rep["cols"][n], rep["floors"][n] = e, floor
            if e >= max(COL_REL, 16 * floor):
                bad.append(f"grad {n} (column-scaled)")
    if len(res["grads"]) != 4 * L + 10:
        bad.append("gradient count")
    rep["running"] = 0.0
    for l in range(L):
        z = a64[f"z{l}"].detach()
        rm0, rv0 = sd[f"batch_norms.{l}.running_mean"].double(), sd[f"batch_norms.{l}.running_var"].double()
        rm = 0.9 * rm0 + 0.1 * z.mean(0)
        rv = 0.9 * rv0 + 0.1 * z.var(0, unbiased=True)
        rep["running"] = max(rep["running"], rel_err(res["running"][l, 0], rm.numpy()), rel_err(res["running"][l, 1], rv.numpy()))
    # 3. eval forward with the running statistics the step left
    ref_eval, _ = O.forward(res["eval_sd"], graph, feat, od, False, dtype=torch.float64)
    rep["eval"] = rel_err(res["eval"], ref_eval.numpy())
    for k in ("spectra", "loss", "running", "eval"):
        if not rep[k] < REL:
            bad.append(k)
    finite = np.isfinite(res["prob"]).all() and np.isfinite(res["eval"]).all() and np.isfinite(res["running"]).all()
    finite = finite and all(np.isfinite(g).all() for g in res["grads"].values())
    if not finite:
        bad.append("NaN / Inf in an output")
    return rep, bad


def check_kernels(name, path, kernels):
    r = ROWS[name]
    if path.startswith("simt"):
        expect, absent = ["sgemm_simt_kernel"], ["gemm_3xtf32", "gemm_planes_kernel"]
        expect += [k for k in r["expect"] if "gemm" not in k]
    else:
        expect, absent = list(r["expect"]), []
        if path.endswith("+planes"):
            expect.append("gemm_planes_kernel")
    absent += r.get("absent", [])
    missing = [k for k in expect if not any(k in n for n in kernels)]
    present = [k for k in absent if any(k in n for n in kernels)]
    return missing, present


# ------------------------------------------------------------------------------------------------ rows
@pytest.mark.parametrize("name,path", row_cases())
def test_rows_launch_their_kernels(name, path, tmp_path):
    """One training step + one eval forward of the row on a poisoned plan, under the profiler: the kernels the row
    exists for are launched (and those whose absence is the point are not), and the results meet the fp64 oracle."""
    d, table, targets, caps, sd = setup_row(name, path)
    step = make_step(step=3, seed=11)
    res = run_gpu(d, table, targets, caps, sd, path, step, profile=True)
    rep, bad = oracle_check(d, table, targets, sd, res)
    missing, present = check_kernels(name, path, res["kernels"])
    rep.update(row=name, path=path, kernels=res["kernels"], missing=missing, unexpected=present)
    with open(tmp_path / f"dispatch_{name}_{path}.json", "w") as fh:   # kept under pytest's --basetemp
        json.dump(rep, fh, indent=1)
    assert not missing and not present, (missing, present, res["kernels"])
    assert not bad, (bad, rep)


# ------------------------------------------------------------------------------------------------ live sizes
@pytest.mark.parametrize("backend", BACKENDS)
def test_shrinking_and_growing_live_sizes(backend):
    """One poisoned plan runs batches of decreasing, then increasing, molecule and atom counts; each must give what a
    fresh plan sized exactly for it gives (eval spectra bit for bit - no atomics -, gradients and running statistics
    to summation order).  A stale read of an earlier, larger batch would show here."""
    d = ROWS["odd_width"]["d"]
    sizes = [(40, 40), (24, 30), (7, 12), (1, 5), (16, 25), (40, 40), (33, 36)]
    Bc, Nc = 40, 40 * 40
    long_plan = make_plan(d, Bc, Nc, 2 * (Nc + 3 * Bc), backend)
    for k, (n, atoms) in enumerate(sizes):
        table = make_table(n, atoms, 300 + k, d.node_feat_dim)
        targets = dense_spectra(*synth_peaks(n, d.max_mz, seed=400 + k), d.max_mz)
        ds = DeviceDataset(table, targets, DEV)
        sd = random_running_stats(O.init_params(odims(d), k), d, 500 + k)
        N, E = int(table.node_ptr[-1]), int(2 * table.bond_ptr[-1])
        out = []
        for plan in (long_plan, make_plan(d, n, N, E, backend)):
            fp = FlatParams(d, DEV)
            fp.load_state_dict(sd)
            res = gpu_step(plan, ds, fp, make_step(step=k + 1, seed=17))
            res["eval"] = plan.infer_batch(ds, None, fp).clone().cpu().numpy()
            out.append(res)
        a, b = out
        assert np.isfinite(a["eval"]).all() and np.isfinite(a["prob"]).all(), (n, atoms)
        assert np.array_equal(a["eval"], b["eval"]), (n, atoms)
        assert rel_err(a["prob"], b["prob"]) <= 1e-6, (n, atoms)
        gmax = max(float(np.abs(g).max()) for g in b["grads"].values())
        worst = max(float(np.abs(a["grads"][x] - b["grads"][x]).max()) for x in b["grads"]) / gmax
        assert worst <= ORDER_REL, (n, atoms, worst)
        assert rel_err(a["running"], b["running"]) <= ORDER_REL, (n, atoms)


# ------------------------------------------------------------------------------------------------ GEMM edges
def _gemm_case(backend, M, N, K, b_mn, acc, live=None, seed=0):
    """eims_gemm on A[M,K] (row-major) x B ([K,N] when b_mn else [N,K]) into C with 16 canary rows past M; live
    rows on the device when `live` is given.  accumulate 2: C starts as NaN (the split-K memset must clear it);
    accumulate 3: the caller has zeroed C."""
    g = torch.Generator().manual_seed(seed + M + N + K)
    A = torch.randn(M, K, generator=g, dtype=torch.float64)
    Bm = torch.randn(K, N, generator=g, dtype=torch.float64)
    Ad = A.float().to(DEV)
    Bd = (Bm if b_mn else Bm.t()).contiguous().float().to(DEV)
    Cd = torch.full((M + 16, N), 7.0, device=DEV)
    Cd[:M] = float("nan") if acc == 2 else 0.0
    m_dev = torch.tensor([live], dtype=torch.int32, device=DEV) if live is not None else None
    check(_lib.load().eims_gemm(backend, ptr(Ad), K, 0, ptr(Bd), Bd.stride(0), b_mn, ptr(Cd), N, M, N, K, ptr(m_dev), None,
                                None, None, 0, acc, C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    m = M if live is None else live
    ref = Ad[:m].double().cpu() @ (Bd.double().cpu() if b_mn else Bd.double().cpu().t())
    out = Cd.cpu()
    return out, ref, m


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("acc", [2, 3])
@pytest.mark.parametrize("b_mn", [0, 1])
@pytest.mark.parametrize("N,K", [(192, 1000), (256, 1000), (192, 4096), (256, 4096)])
def test_gemm_split_k_store(backend, acc, b_mn, N, K):
    """Head data-gradient shapes (M = a batch, K up to 4096): the split-K store forms accumulate 2 (C zeroed by the
    launcher) and 3 (zeroed by the caller) against fp64; the canary rows past M stay untouched."""
    be = {"tcgen05": _lib.GEMM_TCGEN05, "simt": _lib.GEMM_FP32_SIMT}[backend]
    out, ref, m = _gemm_case(be, 64, N, K, b_mn, acc, live=57)
    err = float((out[:m].double() - ref).abs().max() / ref.abs().max())
    assert err < (2e-5 if backend == "tcgen05" else 5e-6), err
    assert bool((out[64:] == 7.0).all())


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("acc", [0, 2])
@pytest.mark.parametrize("N", [4, 12])
@pytest.mark.parametrize("K", [4, 12, 31])
def test_gemm_tiny(backend, acc, N, K):
    """M = 1, K below one k-block, N = the shortest spectra: one partial tile in every direction."""
    be = {"tcgen05": _lib.GEMM_TCGEN05, "simt": _lib.GEMM_FP32_SIMT}[backend]
    for b_mn in (0, 1):
        out, ref, m = _gemm_case(be, 1, N, K, b_mn, acc)
        err = float((out[:1].double() - ref).abs().max() / ref.abs().max())
        assert err < (2e-5 if backend == "tcgen05" else 2e-6), (b_mn, err)
        assert bool((out[1:] == 7.0).all())
