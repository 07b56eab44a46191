"""Integrated-gradients attribution of predicted peaks (eims_attribute_peaks, script.attribute_peaks) on poisoned plans.

1. Against the fp64 oracle (oracle/ig_oracle.py) with the flip-aware protocol of test_gpu_feature_grads: the GPU's ReLU
   and arg-max decisions at every path point are read by running that point through the existing entry points (batch
   build, K1's aggregate a0 scaled by alpha exactly as the attribution scales it, eval eims_forward), every disagreement
   with the free-running fp64 oracle must be a near-tie, and the oracle then takes the GPU's decisions.
2. Against the same integrated gradients computed through eims_backward_feat with a dense one-hot dprob per path point.
3. Contracts: the peaks are eims_topk_peaks of eims_infer_batch's spectra bit for bit; a molecule's outputs do not
   depend on its batch; parameters and running statistics are untouched and a backward is refused afterwards; argument
   errors launch nothing; the profiler sees only data-gradient work.

The checks that read kernels under a profiler (torch.profiler, eims_plan_profile) run in a child process
(test_profiled_contracts): they leave profiler state and timing events behind in the process that opens them, and the
tests after this file read kernel names under torch.profiler in the pytest process.
"""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from eims_b200 import _lib
from eims_b200 import script as S
from eims_b200.engine import DeviceDataset, FlatParams, topk_peaks
from eims_b200.synth import MolTable, synth_molecules
from oracle import gcn_oracle as O
from oracle import ig_oracle as IG
from test_gpu_dispatch import BACKENDS, _dims, kernel_names, make_plan, make_table, odims, random_running_stats
from test_gpu_feature_grads import flip_report, gpu_decisions

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
REL = 1e-4

# name -> model dims, molecules, replicas k, path points S, max atoms, plan capacity (None: exact), GEMM paths
AROWS = {
    "small": dict(d=_dims(64, 3, 6, 100, "combined", 0.0), n=8, k=3, S=6, atoms=20, paths=["tcgen05", "simt"]),
    "one_layer": dict(d=_dims(64, 1, 6, 100, "max", 0.0), n=8, k=2, S=4, atoms=20, paths=["tcgen05"]),
    "hidden192_f3": dict(d=_dims(192, 2, 3, 40, "mean", 0.0), n=10, k=3, S=4, atoms=30, paths=["tcgen05"]),
    "sum_pool": dict(d=_dims(128, 2, 6, 64, "sum", 0.0), n=10, k=2, S=4, atoms=30, paths=["tcgen05"]),
    "dropout": dict(d=_dims(256, 3, 6, 1000, "combined", 0.2), n=12, k=5, S=4, atoms=40, paths=["tcgen05", "simt"]),
    # a plan of 4096 replica graphs (the capacity picks the planes GEMM and the molecule tiles), 1000 of them live
    "replicas_4096": dict(d=_dims(256, 3, 6, 1000, "combined", 0.0), n=200, k=5, S=2, atoms=6, cap=(4096, 4096 * 48),
                          paths=["tcgen05"]),
}
ASEEDS = {name: 900 + 13 * j for j, name in enumerate(AROWS)}


def acases():
    return [pytest.param(n, p, id=f"{n}-{p}") for n, r in AROWS.items() for p in r["paths"] if p in BACKENDS]


def replicate(table: MolTable, k: int) -> MolTable:
    """Each molecule k times in a row: replica j of molecule g is graph g*k + j."""
    mols = [table.mol(g) for g in range(table.num_mols) for _ in range(k)]
    na = np.array([len(m[0]) for m in mols])
    nb = np.array([len(m[1]) for m in mols])
    node_ptr = np.concatenate([[0], np.cumsum(na)]).astype(np.int64)
    bond_ptr = np.concatenate([[0], np.cumsum(nb)]).astype(np.int64)
    feat = np.concatenate([m[0] for m in mols]).astype(np.float32)
    return MolTable(node_ptr, bond_ptr, feat, np.concatenate([m[1] for m in mols]).astype(np.int32),
                    np.concatenate([m[2] for m in mols]).astype(np.int32))


def setup(name):
    r = AROWS[name]
    d, seed = r["d"], ASEEDS[name]
    base = make_table(r["n"], r["atoms"], seed, d.node_feat_dim)
    table = replicate(base, r["k"])
    N, E = int(table.node_ptr[-1]), int(2 * table.bond_ptr[-1])
    caps = r.get("cap") or (table.num_mols, N, E)
    if "cap" in r:
        caps = (caps[0], caps[1], 2 * (caps[1] + 3 * caps[0]))
    sd = random_running_stats(O.init_params(odims(d), seed + 3), d, seed + 4)
    return d, table, caps, sd


def attribute(plan, fp, k, steps, B, N, canary_rows=3):
    """eims_attribute_peaks on NaN-filled outputs and scratch; ig has canary rows past N filled with 7."""
    lib = _lib.load()
    F = plan.d.node_feat_dim
    bins = torch.full((B,), -7, dtype=torch.int32, device=DEV)
    pk, p0 = torch.full((B,), float("nan"), device=DEV), torch.full((B,), float("nan"), device=DEV)
    ig = torch.full((N + canary_rows, F), float("nan"), device=DEV)
    ig[N:] = 7.0
    scratch = torch.full((plan.attribute_scratch_bytes(k) // 4 + 64,), float("nan"), device=DEV)
    base = (scratch.data_ptr() + 255) // 256 * 256
    rc = lib.eims_attribute_peaks(plan.h, _lib.ptr(fp.params), _lib.ptr(fp.bn_running), k, steps, _lib.ptr(bins),
                                  _lib.ptr(pk), _lib.ptr(p0), _lib.ptr(ig), C.c_void_p(base), plan.stream)
    _lib.check(rc)
    torch.cuda.synchronize()
    assert bool((ig[N:] == 7.0).all()), "ig rows past N were written"
    return dict(bins=bins.cpu().numpy(), peak_prob=pk.cpu().numpy(), base_prob=p0.cpu().numpy(), ig=ig[:N].cpu().numpy())


def forward_at(plan, ds, fp, alpha, B):
    """The eval forward at alpha X through the existing entry points: K1, a0 scaled by alpha (a0 is linear in x; the
    attribution scales it the same way), eims_forward.  Returns N."""
    plan.batch_build(ds, None, B)
    N, _ = plan.check()
    a0 = plan.buffer("a0")[: N * plan.d.node_feat_dim]
    if alpha != 1.0:
        a0.mul_(alpha)
    plan.forward(fp, False)
    return N


def per_graph_err(got, ref, gptr):
    """max over graphs of max|got - ref| / max|ref| on the graph's rows."""
    worst = 0.0
    for r in range(len(gptr) - 1):
        a, b = got[gptr[r]:gptr[r + 1]], ref[gptr[r]:gptr[r + 1]]
        scale = max(float(np.abs(b).max()), 1e-30)
        worst = max(worst, float(np.abs(a - b).max()) / scale)
    return worst


def loop_reference(plan, ds, fp, bins, steps, B):
    """The same integrated gradients through today's API: per path point an eval forward and eims_backward_feat with a
    dense one-hot dprob."""
    M = plan.d.max_mz
    dprob = torch.zeros(B, M, device=DEV)
    dprob[torch.arange(B, device=DEV), torch.as_tensor(bins, device=DEV).long()] = 1.0
    acc = None
    for a in IG.path_alphas(steps):
        N = forward_at(plan, ds, fp, a, B)
        dfeat = torch.empty(N, plan.d.node_feat_dim, device=DEV)
        plan.backward_feat(fp, dprob, dfeat)
        acc = dfeat / steps if acc is None else acc + dfeat / steps
    x = ds.feat[: N * plan.d.node_feat_dim].view(N, -1)
    torch.cuda.synchronize()
    return (acc * x).cpu().numpy()


@pytest.mark.parametrize("name,path", acases())
def test_attribution_matches_the_oracle_and_the_backward_loop(name, path, tmp_path):
    r = AROWS[name]
    d, table, caps, sd = setup(name)
    k, steps, B = r["k"], r["S"], table.num_mols
    ds = DeviceDataset(table, None, DEV)
    plan = make_plan(d, *caps, path)
    fp = FlatParams(d, DEV)
    fp.load_state_dict(sd)
    plan.batch_build(ds, None, B)
    N, _ = plan.check()
    res = attribute(plan, fp, k, steps, B, N)

    # the GPU's decisions at every point, each checked against the free-running fp64 oracle
    graph, feat = O.Graph.from_mols([table.mol(i) for i in range(B)])
    decs, flips, bad = {}, {}, []
    for a in [1.0, 0.0] + IG.path_alphas(steps):
        forward_at(plan, ds, fp, a, B)
        torch.cuda.synchronize()
        decs[a] = gpu_decisions(plan, d, B, N)
        rep, b = flip_report(sd, graph, feat.double() * a, d, False, None, decs[a])
        flips[str(a)] = rep
        bad += [f"alpha {a}: {x}" for x in b]
    ref = IG.integrated_gradients(sd, graph, feat, odims(d), k, steps, decisions=decs)
    gptr = O.graph_ptr(graph.batch_num_nodes.numpy())
    ig_err = per_graph_err(res["ig"], ref["ig"], gptr)
    prob_err = max(float(np.abs(res["peak_prob"] - ref["peak_prob"]).max()),
                   float(np.abs(res["base_prob"] - ref["base_prob"]).max()))
    if not np.array_equal(res["bins"], ref["bins"]):
        bad.append("bins differ from the oracle's top-k")
    if not ig_err < REL:
        bad.append(f"ig vs oracle {ig_err}")
    if not prob_err < REL:
        bad.append(f"peak / base prob vs oracle {prob_err}")
    if not (np.isfinite(res["ig"]).all() and np.isfinite(res["peak_prob"]).all() and np.isfinite(res["base_prob"]).all()):
        bad.append("NaN / Inf in an output")

    # the same integrated gradients through eims_backward_feat
    loop = loop_reference(plan, ds, fp, res["bins"], steps, B)
    loop_err = per_graph_err(res["ig"], loop, gptr)
    if not loop_err < 1e-5:
        bad.append(f"ig vs the eims_backward_feat loop {loop_err}")
    report = dict(flips=flips, ig_vs_oracle=ig_err, prob_vs_oracle=prob_err, ig_vs_loop=loop_err)
    with open(tmp_path / f"attribution_{name}_{path}.json", "w") as fh:
        json.dump(report, fh, indent=1)
    assert not bad, (bad, report)


def _replica_pass_kernels():
    """A pass in a plan of 4096 replica graphs takes the planes GEMM and the molecule-tile SpMM (both chosen by the
    plan's capacity) and launches the data-only kernels, none of the parameter-gradient ones."""
    d, table, caps, sd = setup("replicas_4096")
    r = AROWS["replicas_4096"]
    plan = make_plan(d, *caps, "tcgen05")
    fp = FlatParams(d, DEV)
    fp.load_state_dict(sd)
    ds = DeviceDataset(table, None, DEV)
    plan.batch_build(ds, None, table.num_mols)
    N, _ = plan.check()
    acts = [torch.profiler.ProfilerActivity.CPU, torch.profiler.ProfilerActivity.CUDA]
    with torch.profiler.profile(activities=acts) as prof:
        torch.ones(1, device=DEV).add_(1)
        torch.cuda.synchronize()
        plan.attribute_peaks(fp, r["k"], r["S"], table.num_mols, N)
        torch.cuda.synchronize()
    names = kernel_names(prof)
    for k in ("gemm_planes_kernel", "spmm_mol_kernel", "peak_head_dgrad_kernel", "ln_relu_dgrad_kernel",
              "bn_apply_dgrad_kernel", "ig_feat_accum_kernel", "layer0_dgrad_kernel", "topk_peaks_kernel"):
        assert any(k in n for n in names), (k, names)
    for k in ("colsum_kernel", "bn_bwd_stats", "bn_bwd_apply_kernel", "ln_relu_drop_bwd_kernel", "feat_grad_kernel",
              "bn_eval_zstat_kernel", "dprob_to_dlogits_kernel"):
        assert not any(k in n for n in names), (k, names)


# ------------------------------------------------------------------------------------------------ contracts
def _contract_setup(n=9, k=3, cap=None, seed=5):
    d = _dims(128, 3, 6, 200, "combined", 0.0)
    base = make_table(n, 24, seed, 6)
    table = replicate(base, k)
    N, E = int(table.node_ptr[-1]), int(2 * table.bond_ptr[-1])
    caps = cap or (table.num_mols, N, E)
    sd = random_running_stats(O.init_params(odims(d), seed + 1), d, seed + 2)
    fp = FlatParams(d, DEV)
    fp.load_state_dict(sd)
    return d, base, table, caps, fp


@pytest.mark.parametrize("backend", BACKENDS)
def test_peaks_are_the_topk_report_of_infer_batch(backend):
    """On a batch that is NOT replicated, graph r attributes its own (r mod k)-th peak: bins and peak_prob are
    eims_topk_peaks of eims_infer_batch's spectra, bit for bit."""
    d, base, _, _, fp = _contract_setup()
    k, B = 4, base.num_mols
    N, E = int(base.node_ptr[-1]), int(2 * base.bond_ptr[-1])
    plan = make_plan(d, B, N, E, backend)
    ds = DeviceDataset(base, None, DEV)
    prob = plan.infer_batch(ds, None, fp).clone()
    idx, val = topk_peaks(prob, k)
    plan.batch_build(ds, None, B)
    res = attribute(plan, fp, k, 3, B, N)
    rows = np.arange(B)
    assert np.array_equal(res["bins"], idx.cpu().numpy()[rows, rows % k])
    assert np.array_equal(res["peak_prob"].view(np.uint32), val.cpu().numpy()[rows, rows % k].view(np.uint32))


def test_a_molecule_alone_equals_it_inside_a_full_batch():
    """No float atomics on the data-only path: a molecule's k replicas give the same bits alone and inside a full
    replicated batch, on plans of the same capacity."""
    k, steps = 3, 4
    d, base, table, caps, fp = _contract_setup(n=9, k=k, cap=(64, 64 * 24, 2 * (64 * 24 + 3 * 64)))
    full = attribute_ds(d, caps, fp, table, k, steps)
    gptr = np.asarray(table.node_ptr)
    for g in (0, 4, 8):
        alone = attribute_ds(d, caps, fp, replicate(MolTable(*[np.asarray(a) for a in _one(base, g)]), k), k, steps)
        lo, hi = gptr[g * k], gptr[(g + 1) * k]
        assert np.array_equal(alone["ig"].view(np.uint32), full["ig"][lo:hi].view(np.uint32)), g
        for key in ("bins", "peak_prob", "base_prob"):
            assert np.array_equal(alone[key].view(np.uint32), full[key][g * k:(g + 1) * k].view(np.uint32)), (g, key)


def _one(t: MolTable, g):
    f, b, e = t.mol(g)
    return (np.array([0, len(f)], np.int64), np.array([0, len(b)], np.int64), np.asarray(f, np.float32),
            np.asarray(b, np.int32), np.asarray(e, np.int32))


def attribute_ds(d, caps, fp, table, k, steps):
    plan = make_plan(d, *caps, "tcgen05")
    ds = DeviceDataset(table, None, DEV)
    plan.batch_build(ds, None, table.num_mols)
    N, _ = plan.check()
    return attribute(plan, fp, k, steps, table.num_mols, N)


def test_no_side_effects_and_backward_refused_afterwards():
    d, _, table, caps, fp = _contract_setup()
    plan = make_plan(d, *caps, "tcgen05")
    ds = DeviceDataset(table, None, DEV)
    B = table.num_mols
    prob0 = plan.infer_batch(ds, None, fp).clone()
    p0, r0 = fp.params.clone(), fp.bn_running.clone()
    plan.batch_build(ds, None, B)
    N, _ = plan.check()
    attribute(plan, fp, 3, 3, B, N)
    assert torch.equal(fp.params, p0) and torch.equal(fp.bn_running, r0)
    lib = _lib.load()
    dprob = torch.randn(B, d.max_mz, device=DEV)
    dfeat = torch.empty(N, d.node_feat_dim, device=DEV)
    assert lib.eims_backward_feat(plan.h, _lib.ptr(fp.params), _lib.ptr(dprob), _lib.ptr(fp.grads), _lib.ptr(dfeat),
                                  plan.stream) == _lib.ERR_STATE
    assert lib.eims_backward(plan.h, _lib.ptr(fp.params), _lib.ptr(dprob), _lib.ptr(fp.grads), plan.stream) == _lib.ERR_STATE
    # the batch tables are as K1 left them: a forward on them gives the spectra of before, bit for bit
    plan.forward(fp, False)
    plan.sigmoid()
    assert torch.equal(plan.buffer("prob", torch.float32, (B, d.max_mz)), prob0)


def _argument_errors_launch_nothing():
    d, _, table, caps, fp = _contract_setup()
    lib = _lib.load()
    plan = make_plan(d, *caps, "tcgen05")
    B = table.num_mols
    F = d.node_feat_dim
    bins = torch.empty(B, dtype=torch.int32, device=DEV)
    pk, p0 = torch.empty(B, device=DEV), torch.empty(B, device=DEV)
    ig = torch.empty(caps[1], F, device=DEV)
    scratch = torch.empty(plan.attribute_scratch_bytes(d.max_mz) + 256, dtype=torch.uint8, device=DEV)
    sbase = (scratch.data_ptr() + 255) // 256 * 256
    P = _lib.ptr
    good = [plan.h, P(fp.params), P(fp.bn_running), 3, 4, P(bins), P(pk), P(p0), P(ig), C.c_void_p(sbase), plan.stream]

    def call(**over):
        a = list(good)
        for i, v in over.items():
            a[int(i[1:])] = v
        return lib.eims_attribute_peaks(*a)
    plan.profile(True)
    assert call() == _lib.ERR_STATE                      # no batch built yet
    ds = DeviceDataset(table, None, DEV)
    plan.batch_build(ds, None, B)
    plan.check()
    plan.profile(True)
    for i in (1, 2, 5, 6, 7, 8, 9):
        assert call(**{f"a{i}": None}) == _lib.ERR_ARG, i
    for kk, ss in ((0, 4), (-1, 4), (d.max_mz + 1, 4), (3, 0), (3, -2)):
        assert call(a3=kk, a4=ss) == _lib.ERR_ARG, (kk, ss)
    assert call(a9=C.c_void_p(sbase + 16)) == _lib.ERR_ARG
    _, launches = plan.profile_read()
    assert launches == 0
    assert call(a0=None) == _lib.ERR_STATE
    assert call(a3=d.max_mz) == 0      # k = max_mz is allowed
    torch.cuda.synchronize()


def _profiler_sees_data_gradients_only():
    """An attribution pass launches no colsum and no BatchNorm-backward statistics; its head GEMMs are two data-gradient
    launches per path point (gemm_head_dgrad), its GraphConv GEMMs gemm_gcn_dgrad only; eims_backward_feat makes three
    grouped gemm_head_bwd launches."""
    d, _, table, caps, fp = _contract_setup()
    plan = make_plan(d, *caps, "tcgen05")
    ds = DeviceDataset(table, None, DEV)
    B, L, steps = table.num_mols, d.num_gcn_layers, 5
    plan.batch_build(ds, None, B)
    N, _ = plan.check()
    plan.profile(True)
    attribute(plan, fp, 3, steps, B, N)
    st, _ = plan.profile_read()
    assert st["colsum"][1] == 0 and st["bn_bwd_stats"][1] == 0, st
    assert st["gemm_head_dgrad"][1] == 2 * steps and st["gemm_head_bwd"][1] == 0, st
    assert st["gemm_gcn_dgrad"][1] == L * steps and st["gemm_gcn_bwd"][1] == 0 and st["gemm_gcn_wgrad"][1] == 0, st
    assert st["gemm_head_fwd"][1] == 3 * (steps + 2), st
    plan.profile(False)
    plan.batch_build(ds, None, B)
    plan.forward(fp, False)
    plan.profile(True)
    plan.backward_feat(fp, torch.randn(B, d.max_mz, device=DEV), torch.empty(N, d.node_feat_dim, device=DEV))
    st, _ = plan.profile_read()
    assert st["gemm_head_bwd"][1] == 3 and st["gemm_head_dgrad"][1] == 0, st


def test_profiled_contracts():
    """_replica_pass_kernels, _argument_errors_launch_nothing and _profiler_sees_data_gradients_only, in a child
    process."""
    here = os.path.dirname(os.path.abspath(__file__))
    root = os.path.dirname(here)
    code = ("import sys; sys.path[:0] = sys.argv[1:4]\n"
            "import test_gpu_attribution as T\n"
            "for f in (T._replica_pass_kernels, T._argument_errors_launch_nothing, T._profiler_sees_data_gradients_only):\n"
            "    f()\n"
            "    print('passed', f.__name__, flush=True)\n")
    out = subprocess.run([sys.executable, "-c", code, here, os.path.join(root, "computational-chemistry-ai_b200"), root],
                         capture_output=True, text=True, timeout=900, cwd=root)
    assert out.returncode == 0, (out.stdout[-2000:], out.stderr[-6000:])
    assert out.stdout.count("passed ") == 3, out.stdout


# ------------------------------------------------------------------------------------------------ the module
def test_script_attribute_peaks():
    """script.attribute_peaks: the model's peaks (predict_graphs' report), the per-molecule ig of the replicated plan
    call, chunking by batch_size, and ZeroInDegreeError for an isolated atom."""
    cfg = S.Config()
    cfg.hidden_dim, cfg.max_mz, cfg.dropout = 64, 100, 0.0
    d = O.Dims(hidden_dim=64, max_mz=100, dropout=0.0)
    sd = random_running_stats(O.init_params(d, 61), d, 62)
    t = synth_molecules(7, max_atoms=14, seed=63)
    graphs = [S.MolGraph(*t.mol(i)) for i in range(7)]
    model = S.GCNSpectrum(6, cfg).to(DEV)
    model.load_state_dict(sd)
    k, steps = 3, 4
    bins, prob, delta, ig = S.attribute_peaks(model, graphs, k=k, steps=steps, batch_size=6)   # 2 molecules per pass
    _, rb, rv = S.predict_graphs(model, graphs, top_k=k)
    assert np.array_equal(bins, rb) and np.array_equal(prob.view(np.uint32), rv.view(np.uint32))
    assert len(ig) == 7 and all(ig[g].shape == (k, graphs[g].num_nodes(), 6) for g in range(7))
    graph, feat = O.Graph.from_mols([t.mol(i) for i in range(7) for _ in range(k)])
    ref = IG.integrated_gradients(sd, graph, feat, d, k, steps)
    assert np.abs(delta.reshape(-1) - (ref["peak_prob"] - ref["base_prob"])).max() < 1e-4
    big = np.concatenate([ig[g].transpose(1, 0, 2).reshape(-1, 6) for g in range(7)])
    assert np.isfinite(big).all() and np.abs(big).max() > 0
    bad = MolTable(np.array([0, 3], np.int64), np.array([0, 1], np.int64), np.ones((3, 6), np.float32),
                   np.array([0], np.int32), np.array([1], np.int32))
    with pytest.raises(_lib.ZeroInDegreeError):
        S.attribute_peaks(model, [S.MolGraph(*bad.mol(0))], k=2, steps=2)
