"""The training loops the benchmark times, step by step against eager `Plan.train_step`, at bench.py's training shape
(batch 512, hidden 256, 3 GCN layers, 1000 bins, combined pooling, dropout 0.2, molecules of <= 64 atoms).

The loops wrap the same kernels in CUDA graphs, step blocks, ping-pong batch tables, copy streams and pinned rings:
`GraphedTrainStep` (device-resident set), `Plan.train_step_prefetch` (K1 of the next batch on a side stream),
`HostBatchRunner` with `HostPacker` (host-resident set, with and without K1 on the copy stream) and
`GraphedHostTrainer` (fixed-layout pinned ring, H2D copy and K1 inside the graph).  A plumbing error there - a step
that trains on the neighbouring batch, dropout keys or AdamW scalars read from the wrong step block, a K1 racing
the step that still reads the other table set, a stale slot - gives plausible losses, so it is checked here.

Protocol.  Phase 1 runs every loop with lr = 0 in every `Step` (beta1 from the OneCycle table, weight decay 1e-4,
dropout, step = k + 1): AdamW then leaves the parameters exactly unchanged, every step's loss is a pure function of
(initial weights, the step's batch, the step's dropout keys), and the Adam moments and BatchNorm running statistics
are sums over the steps in order.  Only a ReLU or max-pool decision that rounding flips amplifies the atomics'
noise, so a loop must agree with the eager reference to summation order at every step.  The graphs are captured with a `Step` of lr 1e-3, so parameters
bit-identical to the initial ones prove that replays read lr from the step blocks.  Phase 2 runs a short OneCycle
schedule (max lr 1e-3) and compares the parameters, which checks lr, bias correction and weight decay.

The reference runs twice; the spread between the two runs is each quantity's noise floor, and every comparison is
held to max(8 x that spread, a small fixed floor); Adam moments and trained parameters per tensor, by their median
element to that bound and by their worst element to a loose one (see FLIP_FLOOR).  Negative controls (two
neighbouring `Step`s swapped; a step fed its neighbour's batch) must fail the same comparison by at least 100 x, which proves that it can see such errors.
The losses of step 0 and of the first step whose batch reuses a pinned ring buffer are also tied to the fp64
oracle with the GPU's own dropout masks.

Every plan, device slot and pinned buffer is filled with 0xFF bytes (NaN / -1) before first use, and the batches
come in order of non-increasing atom count, so every slot, ring buffer and table set holds a larger stale batch
behind the live one.  Each test writes its error-to-bound ratios as JSON under its tmp_path."""
import ctypes as C
import json

import numpy as np
import pytest
import torch

from eims_b200 import _lib
from eims_b200.engine import (DeviceDataset, DevicePeaks, FlatParams, GraphedTrainStep, ModelDims, Plan, make_step,
                              onecycle_schedule, param_offsets, param_spec)
from eims_b200.hostpath import GraphedHostTrainer, HostBatchRunner, HostDataset, HostPacker, PackedHostBatch
from eims_b200.synth import MolTable, dense_spectra, synth_molecules, synth_peaks
from oracle import gcn_oracle as O
from test_gpu_dispatch import dropout_masks, odims, poison, random_running_stats

DEV = "cuda:0"
BATCH, MAX_ATOMS, N_MOLS, SEED = 512, 64, 4096, 2024
D = ModelDims(6, 256, 3, 1000, "combined", 0.2)
M = D.max_mz
S1, S2 = 60, 12                    # frozen steps (every pinned buffer of the G = 10 ring reused twice), trained steps
CAPTURE = make_step(lr=1e-3, step=1, seed=SEED)
LOSS_FLOOR, STATE_FLOOR, ORACLE_REL = 2e-6, 1e-6, 1e-4
# A ReLU or max-pool decision that rounding noise flips moves one atom's share of a gradient: a few elements of the
# Adam moments (and, through Adam, of the trained parameters and later losses) differ by far more than the summation
# order, in either run.  So tensors are held twice: the bulk (median element error) to the tight bound, the worst
# element to a loose one - 1e-3 of the largest moment, Adam's reach 2.5 x sum(lr) for a parameter, and the oracle's
# 1e-4 for a loss after trained steps.
FLIP_FLOOR, TRAINED_LOSS_FLOOR = 1e-3, 1e-4
# The one-call eager step and the steps on tables built ahead sum some gradients in another, fixed order: their Adam
# moments differ by a few 1e-6 of the largest moment in the bulk of a tensor (2.7e-6 measured on a B200), in every run,
# and the trained parameters by up to 1e-6 of the tensor's largest element.  A wrong lr or bias correction moves the
# bulk by 1e-3 of a parameter or more.
ORDER_FLOOR = 1e-5


def frozen_steps(n):
    sched = onecycle_schedule(4096)   # bench.py's table: beta1 of its first steps
    return [make_step(lr=0.0, beta1=sched[k][1], weight_decay=1e-4, step=k + 1, seed=SEED) for k in range(n)]


def trained_steps(n):
    sched = onecycle_schedule(20)     # the longest trained run; lr reaches its 1e-3 peak at step 6
    return [make_step(lr=sched[k][0], beta1=sched[k][1], weight_decay=1e-4, step=k + 1, seed=SEED) for k in range(n)]


def swapped(seq, k):
    seq = list(seq)
    seq[k], seq[k + 1] = seq[k + 1], seq[k]
    return seq


# ------------------------------------------------------------------------------------------------ data and plans
def select_peaks(pk, ids):
    ptr_, mz, inten = pk
    cnt = np.diff(ptr_)[ids]
    out = np.zeros(len(ids) + 1, np.int64)
    np.cumsum(cnt, out=out[1:])
    idx = np.concatenate([np.arange(ptr_[i], ptr_[i + 1]) for i in ids]) if len(ids) else np.zeros(0, np.int64)
    return out, mz[idx], inten[idx]


def peak_arrays(data, kind):
    ptr_, mz, inten = data["peaks"]
    return ptr_, mz.astype(np.float64 if kind == "f64" else np.float32), inten


@pytest.fixture(scope="module")
def data():
    table = synth_molecules(N_MOLS, max_atoms=MAX_ATOMS, seed=1234)
    pk = synth_peaks(N_MOLS, M, seed=4321)
    rng = np.random.default_rng(5)
    batches = np.stack([rng.choice(N_MOLS, BATCH, replace=False) for _ in range(S1 + 1)]).astype(np.int32)
    atoms = np.diff(table.node_ptr)
    batches = batches[np.argsort(-atoms[batches].sum(1), kind="stable")]
    sd = random_running_stats(O.init_params(odims(D), 3), D, 4)
    return dict(table=table, peaks=pk, dense=dense_spectra(*pk, M), batches=batches, sd=sd)


def device_set(data, kind):
    if kind == "dense":
        return DeviceDataset(data["table"], data["dense"], DEV)
    return DeviceDataset(data["table"], None, DEV, peaks=DevicePeaks(*peak_arrays(data, kind), DEV))


def host_set(data, kind):
    if kind == "dense":
        return HostDataset(data["table"], data["dense"])
    return HostDataset(data["table"], None, peaks=peak_arrays(data, kind))


def caps_of(data, batches):
    """Exact maxima of (atoms, bonds, peaks) over the batches: the fixed layout is as tight as it can be."""
    t, pk = data["table"], data["peaks"]
    cnt = lambda p: np.diff(p)[batches].sum(1).max()
    return int(cnt(t.node_ptr)), int(cnt(t.bond_ptr)), int(cnt(pk[0]))


def fresh_params(data):
    fp = FlatParams(D, DEV)
    fp.load_state_dict(data["sd"])
    return fp


def warm_plan(data, dense_ds, max_nodes=BATCH * MAX_ATOMS, max_edges=None):
    """bench.py's plan, warmed up by one eager step on scratch parameters (modules loaded before any capture), then
    poisoned."""
    plan = Plan(D, BATCH, max_nodes, max_edges or 2 * (max_nodes + 3 * BATCH), DEV)
    scratch = fresh_params(data)
    ids = torch.from_numpy(data["batches"][-1]).to(DEV)
    plan.train_step(dense_ds, ids, scratch, frozen_steps(1)[0], torch.zeros(8, device=DEV))
    torch.cuda.synchronize()
    poison(plan)
    return plan


def snapshot(fp):
    return dict(params=fp.params.cpu().numpy().copy(), bn_running=fp.bn_running.cpu().numpy().copy(),
                adam_m=fp.adam_m.cpu().numpy().copy(), adam_v=fp.adam_v.cpu().numpy().copy(),
                nbt=list(fp.num_batches_tracked))


def fill_ff(tensors):
    for t in tensors:
        t.view(torch.uint8).fill_(0xFF)


# ------------------------------------------------------------------------------------------------ eager reference
class Reference:
    """Eager `Plan.train_step` on a device-resident set, run twice per (targets, phase): cumulative metrics after
    every step and the state after the step counts the loops stop at."""

    SNAPS = {"frozen": (39, S1), "trained": (S2, 20)}

    def __init__(self, data):
        self.data, self.cache = data, {}

    def __call__(self, kind="dense", phase="frozen"):
        key = (kind, phase)
        if key not in self.cache:
            self.cache[key] = [self._run(kind, phase) for _ in range(2)]
        return self.cache[key]

    def _run(self, kind, phase):
        data = self.data
        n = max(self.SNAPS[phase])
        steps = frozen_steps(n) if phase == "frozen" else trained_steps(n)
        dense_ds = device_set(data, "dense")
        ds = dense_ds if kind == "dense" else device_set(data, kind)
        plan = warm_plan(data, dense_ds)
        fp = fresh_params(data)
        metrics = torch.zeros(8, device=DEV)
        ids = torch.from_numpy(data["batches"]).to(DEV)
        per, snaps = [], {}
        for k in range(n):
            plan.train_step(ds, ids[k], fp, steps[k], metrics)
            per.append(metrics.clone())
            if k + 1 in self.SNAPS[phase]:
                snaps[k + 1] = snapshot(fp)
        return dict(metrics=torch.stack(per).cpu().double().numpy(), snaps=snaps)


@pytest.fixture(scope="module")
def ref(data):
    return Reference(data)


# ------------------------------------------------------------------------------------------------ comparison
def _segments():
    spec, offs = param_spec(D), param_offsets(D)
    return [(name, slice(o, o + int(np.prod(shape)))) for (name, shape), o in zip(spec, offs)]


def compare(got, refs, n, phase, lr_sum=0.0):
    """(ratios of error to bound, exact mismatches) of one loop's run of n steps against the two reference runs."""
    A, B = refs
    r, bad = {}, []
    rel = lambda x, a: np.abs(np.asarray(x, np.float64) - a) / np.abs(a)

    def put(name, v):       # a NaN (a read of poisoned bytes) counts as an infinite error
        r[name] = max(r.get(name, 0.0), float(v) if np.isfinite(v) else float("inf"))

    def ratio(name, x, a, b, floor, stat=np.max):
        bound = max(8 * float(stat(np.abs(np.asarray(b, np.float64) - a))), floor)
        put(name, float(stat(np.abs(np.asarray(x, np.float64) - a))) / bound)

    loss_floor = LOSS_FLOOR if phase == "frozen" else TRAINED_LOSS_FLOOR

    if got.get("per_step") is not None:             # per-step (loss, cosine)
        ps = np.asarray(got["per_step"], np.float64)
        for j, name in ((4, "loss"), (5, "cosine")):
            a, b = A["metrics"][:n, j], B["metrics"][:n, j]
            put(name, float(rel(ps[:, j - 4], a).max()) / max(8 * float(rel(b, a).max()), loss_floor))
    for c, m in sorted(got["checkpoints"].items()):  # cumulative loss / cosine sums, step count, non-finite count
        for j, name in ((0, "loss_sum"), (1, "cosine_sum"), (4, "loss"), (5, "cosine")):
            a, b = A["metrics"][c - 1, j], B["metrics"][c - 1, j]
            put(f"checkpoint_{name}", float(rel(m[j], a)) / max(8 * float(rel(b, a)), loss_floor))
        if m[2] != A["metrics"][c - 1, 2] or m[6] != 0:
            bad.append(f"metrics after {c} steps: count {m[2]}, non-finite {m[6]}")
    sa, sb, sg = A["snaps"][n], B["snaps"][n], got["state"]
    if sg["nbt"] != sa["nbt"]:
        bad.append(f"num_batches_tracked {sg['nbt']} != {sa['nbt']}")
    if phase == "frozen":
        p0 = got["initial_params"]
        if not np.array_equal(sg["params"], p0):
            bad.append(f"parameters moved under lr = 0 ({int((sg['params'] != p0).sum())} elements)")
        for q in ("adam_m", "adam_v"):
            top = float(np.abs(sa[q]).max())
            for name, sl in _segments():
                ratio(q, sg[q][sl], sa[q][sl], sb[q][sl], ORDER_FLOOR * top, np.median)
                ratio(f"{q}_worst", sg[q][sl], sa[q][sl], sb[q][sl], FLIP_FLOOR * top)
        floor = STATE_FLOOR * float(np.abs(sa["bn_running"]).max())
        for l in range(D.num_gcn_layers):
            for s in range(2):
                ratio("bn_running", sg["bn_running"][l, s], sa["bn_running"][l, s], sb["bn_running"][l, s], floor)
    else:
        for name, sl in _segments():
            a, b, x = sa["params"][sl], sb["params"][sl], sg["params"][sl]
            # a GraphConv bias feeds BatchNorm: its exact gradient is 0, and Adam turns rounding noise into steps
            if name.startswith("gcn_layers") and name.endswith("bias"):
                ratio("params_worst", x, a, b, 2.5 * lr_sum)
            else:
                ratio("params", x, a, b, ORDER_FLOOR * float(np.abs(a).max()), np.median)
                ratio("params_worst", x, a, b, 2.5 * lr_sum)
    return r, bad


def report(tmp_path, name, payload):
    with open(tmp_path / f"{name}.json", "w") as f:
        json.dump(payload, f, indent=1, sort_keys=True, default=float)


def check_run(tmp_path, name, got, refs, n, phase, lr_sum=0.0, controls=None):
    """Writes the ratios (and the negative controls' ratios), then asserts: every ratio <= 1, nothing exact differs,
    and every control fails by at least 100 x."""
    r, bad = compare(got, refs, n, phase, lr_sum)
    ctl = {k: compare(g, refs, n, phase, lr_sum)[0] for k, g in (controls or {}).items()}
    report(tmp_path, name, dict(ratios=r, exact=bad, controls={k: max(v.values()) for k, v in ctl.items()},
                                control_ratios=ctl, oracle=got.get("oracle", {})))
    assert not bad, bad
    assert max(r.values()) <= 1.0, r
    for k, v in ctl.items():
        assert max(v.values()) >= 100.0, (k, v)
    for step, e in got.get("oracle", {}).items():
        assert e < ORACLE_REL, (step, e)


def oracle_errors(data, batches, steps, losses, which):
    """Relative error of the looped path's loss of step k against the fp64 oracle on that batch, with the GPU's
    dropout masks of that step (dense targets)."""
    out = {}
    for k in which:
        ids = batches[k]
        sub = data["table"].select(ids)
        graph, feat = O.Graph.from_mols([sub.mol(i) for i in range(len(ids))])
        masks = dropout_masks(D, steps[k], int(sub.node_ptr[-1]), len(ids))
        _, loss, _, _ = O.loss_and_grads(data["sd"], graph, feat, torch.from_numpy(data["dense"][ids]), odims(D),
                                         dtype=torch.float64, dropout_masks=masks)
        out[k] = abs(losses[k] - float(loss)) / float(loss)
    return out


# ------------------------------------------------------------------------------------------------ the loops
GRAPH_SCHEDULE = {"frozen": [("flush", 3), ("step", 1), ("hold", 10), ("step", 10), ("step", 10), ("flush", 5)],
                  "trained": [("flush", 2), ("step", 10)]}


def run_graphed(data, steps, batches, schedule):
    """GraphedTrainStep at group 10; metrics read at every flush / release / full-group point."""
    ds = device_set(data, "dense")
    plan = warm_plan(data, ds)
    fp = fresh_params(data)
    p0 = fp.params.cpu().numpy().copy()
    metrics = torch.zeros(8, device=DEV)
    ids = torch.from_numpy(batches).to(DEV)
    gs = GraphedTrainStep(plan, ds, fp, BATCH, metrics, group=10)
    assert gs.group == 10
    gs.capture(ids[0], CAPTURE)
    assert gs.multi is not None and len(gs.singles) == 2
    k, marks = 0, {}
    for op, n in schedule:
        if op == "hold":
            assert gs.can_hold(n)
            gs.hold_next = True
            while gs.held is None:
                gs.step(steps[k], ids[k + 1])
                k += 1
            gs.release()
        else:
            for _ in range(n):
                gs.step(steps[k], ids[k + 1])
                k += 1
            if op == "flush":
                gs.flush()
        assert not gs.pending and (op != "step" or n != 1 or gs.k == 0)   # the lone step went out as a single
        marks[k] = metrics.clone()
    torch.cuda.synchronize()
    return dict(checkpoints={c: m.cpu().double().numpy() for c, m in marks.items()}, state=snapshot(fp), initial_params=p0)


def run_prefetch(data, steps, batches):
    ds = device_set(data, "dense")
    plan = warm_plan(data, ds)
    fp = fresh_params(data)
    p0 = fp.params.cpu().numpy().copy()
    metrics = torch.zeros(8, device=DEV)
    ids = torch.from_numpy(batches).to(DEV)
    n, per = len(steps), []
    for k in range(n):
        plan.train_step_prefetch(ds, ids[k], ids[k + 1] if k + 1 < n else None, fp, steps[k], metrics)
        per.append(metrics.clone())
    torch.cuda.synchronize()
    m = torch.stack(per).cpu().double().numpy()
    return dict(per_step=m[:, 4:6], checkpoints={n: m[-1]}, state=snapshot(fp), initial_params=p0)


def run_host_runner(data, steps, batches, build):
    """bench.py's eager e2e loop: pack, upload (build=True: K1 on the copy stream), step; losses read two behind."""
    plan = warm_plan(data, device_set(data, "dense"))
    fp = fresh_params(data)
    p0 = fp.params.cpu().numpy().copy()
    metrics = torch.zeros(8, device=DEV)
    cap = BATCH * (MAX_ATOMS * (6 * 4 + 8 + 10) + 4 * M + 64) + (1 << 16)
    packer = HostPacker(host_set(data, "dense"), M, cap, n_buffers=4)
    runner = HostBatchRunner(plan, fp, cap, metrics=metrics)
    fill_ff(packer.bufs + runner.slots + runner.host_ring)
    n, per = len(steps), [None] * len(steps)
    hb = packer.pack(batches[0])
    slot = runner.upload(hb, build=build)
    for k in range(n):
        runner.train_step(slot, hb, steps[k])
        if k + 1 < n:
            hb = packer.pack(batches[k + 1])
            slot = runner.upload(hb, build=build)
        if k >= 2:
            per[k - 2] = runner.read(2)
    per[n - 2], per[n - 1] = runner.read(1), runner.read(0)
    torch.cuda.synchronize()
    return dict(per_step=per, checkpoints={n: metrics.cpu().double().numpy()}, state=snapshot(fp), initial_params=p0)


def run_host_trainer(data, steps, batches, kind, G, pack_order=None):
    """GraphedHostTrainer with bench.py's packing discipline: the next group is packed right after each launch, and
    the results of launch l - 1 are read after launching l.  pack_order[n]: the batch packed as batch n."""
    order = list(range(len(batches))) if pack_order is None else pack_order
    plan = warm_plan(data, device_set(data, "dense"))
    fp = fresh_params(data)
    p0 = fp.params.cpu().numpy().copy()
    metrics = torch.zeros(8, device=DEV)
    tr = GraphedHostTrainer(plan, fp, host_set(data, kind), BATCH, M, *caps_of(data, batches), metrics=metrics, group=G)
    try:
        fill_ff(tr.pinned + tr.slots + [tr.out_host])
        n = len(steps)
        futs = {j: tr.pack_async(j, batches[order[j]]) for j in range(G + 1)}
        tr.prime(futs.pop(0))
        tr.capture(CAPTURE)
        assert len(tr.graphs) == 2
        per = []
        for l in range(n // G):
            assert tr.launch(steps[l * G:(l + 1) * G], [futs.pop(j) for j in range(l * G + 1, l * G + G + 1)]) == l
            for j in range((l + 1) * G + 1, min((l + 2) * G, n) + 1):
                futs[j] = tr.pack_async(j, batches[order[j]])
            if l:
                per += tr.results(l - 1)
        per += tr.results(n // G - 1)
        torch.cuda.synchronize()
        return dict(per_step=per, checkpoints={n: metrics.cpu().double().numpy()}, state=snapshot(fp), initial_params=p0)
    finally:
        tr.close()


# ------------------------------------------------------------------------------------------------ tests
@pytest.mark.gpu
def test_graphed_train_step_equals_eager(data, ref, tmp_path):
    """Every launch form of GraphedTrainStep: singles to table parity 1, a lone single, a group through hold_next /
    release, two groups through step(), a flushed tail."""
    b = data["batches"]
    steps = frozen_steps(39)
    got = run_graphed(data, steps, b[:40], GRAPH_SCHEDULE["frozen"])
    controls = {"steps_swapped": run_graphed(data, swapped(steps, 20), b[:40], GRAPH_SCHEDULE["frozen"]),
                "batch_shifted": run_graphed(data, steps, np.array(swapped(b[:40], 20)), GRAPH_SCHEDULE["frozen"])}
    check_run(tmp_path, "graphed_frozen", got, ref("dense", "frozen"), 39, "frozen", controls=controls)
    tsteps = trained_steps(S2)
    got = run_graphed(data, tsteps, b[:S2 + 1], GRAPH_SCHEDULE["trained"])
    check_run(tmp_path, "graphed_trained", got, ref("dense", "trained"), S2, "trained", sum(s.lr for s in tsteps))


@pytest.mark.gpu
def test_prefetch_loop_equals_eager(data, ref, tmp_path):
    b = data["batches"]
    got = run_prefetch(data, frozen_steps(S1), b)
    check_run(tmp_path, "prefetch_frozen", got, ref("dense", "frozen"), S1, "frozen")
    tsteps = trained_steps(S2)
    got = run_prefetch(data, tsteps, b[:S2 + 1])
    check_run(tmp_path, "prefetch_trained", got, ref("dense", "trained"), S2, "trained", sum(s.lr for s in tsteps))


@pytest.mark.gpu
@pytest.mark.parametrize("build", [False, True])
def test_host_batch_runner_equals_eager(data, ref, tmp_path, build):
    b = data["batches"]
    steps = frozen_steps(S1)
    got = run_host_runner(data, steps, b, build)
    got["oracle"] = oracle_errors(data, b, steps, [p[0] for p in got["per_step"]], [0])
    check_run(tmp_path, f"runner_build{int(build)}_frozen", got, ref("dense", "frozen"), S1, "frozen")
    tsteps = trained_steps(S2)
    got = run_host_runner(data, tsteps, b[:S2 + 1], build)
    check_run(tmp_path, f"runner_build{int(build)}_trained", got, ref("dense", "trained"), S2, "trained", sum(s.lr for s in tsteps))


@pytest.mark.gpu
@pytest.mark.parametrize("G", [10, 2])
@pytest.mark.parametrize("kind", ["dense", "f32", "f64"])
def test_graphed_host_trainer_equals_eager(data, ref, tmp_path, kind, G):
    """Dense targets and peak lists with float32 / float64 m/z; G = 10 as bench.py, G = 2 wraps the ring most often."""
    b = data["batches"]
    steps = frozen_steps(S1)
    got = run_host_trainer(data, steps, b, kind, G)
    controls = None
    if kind == "dense":
        got["oracle"] = oracle_errors(data, b, steps, [p[0] for p in got["per_step"]], [0, 2 * G])
        if G == 10:
            controls = {"steps_swapped": run_host_trainer(data, swapped(steps, 24), b, kind, G),
                        "pack_order_swapped": run_host_trainer(data, steps, b, kind, G, pack_order=swapped(range(S1 + 1), 24))}
    check_run(tmp_path, f"host_trainer_{kind}_G{G}_frozen", got, ref(kind, "frozen"), S1, "frozen", controls=controls)
    n2 = 20 if G == 10 else S2
    tsteps = trained_steps(n2)
    got = run_host_trainer(data, tsteps, b[:n2 + 1], kind, G)
    check_run(tmp_path, f"host_trainer_{kind}_G{G}_trained", got, ref(kind, "trained"), n2, "trained", sum(s.lr for s in tsteps))


def with_isolated_atom(data):
    """The set plus one molecule of a single atom (id N_MOLS): an atom without bonds, which DGL's GraphConv refuses."""
    t, (ptr_, mz, inten) = data["table"], data["peaks"]
    table = MolTable(np.append(t.node_ptr, t.node_ptr[-1] + 1), np.append(t.bond_ptr, t.bond_ptr[-1]),
                     np.concatenate([t.feat, t.feat[:1]]), t.bond_begin, t.bond_end)
    return dict(data, table=table, dense=np.concatenate([data["dense"], data["dense"][:1]]),
                peaks=(np.append(ptr_, ptr_[-1]), mz, inten))


@pytest.mark.gpu
def test_host_trainer_zero_degree_flag_follows_the_replays(data):
    """K1 inside the host trainer's graphs tags an isolated atom with the step's own sequence number: `check()` raises
    after the launch whose last batch has one, not after later launches of clean batches that replay the same graph,
    and again after a later isolated atom."""
    G = 2
    iso = with_isolated_atom(data)
    b = data["batches"][:5 * G + 1].copy()
    b[G, 0] = b[4 * G, 0] = N_MOLS          # the last batch built by launch 0, and by launch 3
    plan = warm_plan(iso, device_set(iso, "dense"))
    tr = GraphedHostTrainer(plan, fresh_params(iso), host_set(iso, "dense"), BATCH, M, *caps_of(iso, b), group=G)
    try:
        futs = {j: tr.pack_async(j, b[j]) for j in range(G + 1)}
        tr.prime(futs.pop(0))
        tr.capture(CAPTURE)
        plan.check()
        steps = frozen_steps(5 * G)
        for l, isolated in enumerate((True, False, False, True)):
            tr.launch(steps[l * G:(l + 1) * G], [futs.pop(j) for j in range(l * G + 1, l * G + G + 1)])
            for j in range((l + 1) * G + 1, (l + 2) * G + 1):
                futs[j] = tr.pack_async(j, b[j])
            torch.cuda.synchronize()
            if isolated:
                with pytest.raises(_lib.ZeroInDegreeError):
                    plan.check()
            else:
                plan.check()
    finally:
        tr.close()


@pytest.mark.gpu
def test_host_trainer_capacity_overflow_enqueues_nothing(data):
    """A batch over the fixed layout's caps makes `launch` raise ERR_CAPACITY before anything is enqueued."""
    G = 2
    b = data["batches"][:2 * G + 1]
    plan = warm_plan(data, device_set(data, "dense"))
    fp = fresh_params(data)
    metrics = torch.zeros(8, device=DEV)
    tr = GraphedHostTrainer(plan, fp, host_set(data, "dense"), BATCH, M, *caps_of(data, b), metrics=metrics, group=G)
    try:
        futs = {j: tr.pack_async(j, b[j]) for j in range(G + 1)}
        tr.prime(futs.pop(0))
        tr.capture(CAPTURE)
        steps = trained_steps(2 * G)
        tr.launch(steps[:G], [futs.pop(j) for j in range(1, G + 1)])
        largest = np.argsort(np.diff(data["table"].node_ptr))[-BATCH:].astype(np.int32)
        futs[G + 1] = tr.pack_async(G + 1, largest)
        futs[G + 2] = tr.pack_async(G + 2, b[G + 2])
        torch.cuda.synchronize()
        before = (snapshot(fp), metrics.clone(), tr.launches)
        with pytest.raises(_lib.EimsError) as exc:
            tr.launch(steps[G:], [futs.pop(j) for j in range(G + 1, 2 * G + 1)])
        assert exc.value.code == _lib.ERR_CAPACITY
        torch.cuda.synchronize()
        after = snapshot(fp)
        assert tr.launches == before[2] and torch.equal(metrics, before[1])
        for q in ("params", "adam_m", "adam_v", "bn_running"):
            assert np.array_equal(after[q], before[0][q]), q
    finally:
        tr.close()


@pytest.mark.gpu
def test_host_batch_runner_infer_equals_device_resident(data):
    """Eval forward from pinned host batches == `Plan.infer_batch` on the device-resident set, bit for bit (no
    atomics in the eval forward): one molecule, a partial batch, full batches, one exactly at the plan's and the
    staging slot's capacity."""
    t, b = data["table"], data["batches"]
    sets = [b[5][:1], b[7][:100], b[0], b[30], b[60][::-1].copy()]    # b[0]: the most atoms of all batches
    subs = [t.select(ids) for ids in sets]
    max_edges = max(int(2 * s.bond_ptr[-1]) for s in subs)
    plan = Plan(D, BATCH, int(subs[2].node_ptr[-1]), max_edges, DEV)
    ds = device_set(data, "dense")
    fp = fresh_params(data)
    need = [PackedHostBatch.bytes_needed(s, M) for s in subs]
    packer = HostPacker(host_set(data, "dense"), M, max(need), n_buffers=2)
    runner = HostBatchRunner(plan, fp, max(need))
    fill_ff(packer.bufs + runner.slots)
    out = torch.empty(BATCH, M, dtype=torch.float32, pin_memory=True)
    for ids, nbytes in zip(sets, need):
        poison(plan)
        want = plan.infer_batch(ds, torch.from_numpy(ids).to(DEV), fp).cpu().clone()
        poison(plan)
        fill_ff([out])
        hb = packer.pack(ids)
        assert hb.nbytes == nbytes
        runner.infer(runner.upload(hb), hb, out)
        torch.cuda.synchronize()
        assert torch.equal(out[:len(ids)], want), len(ids)


# ------------------------------------------------------------------------------------------------ CPU: the packer
def pack_fixed(hds, ids, caps, out):
    lay = _lib.HostBatchLayout()
    ids = np.ascontiguousarray(ids, np.int32)
    rc = _lib.load().eims_host_pack_batch_fixed(C.byref(hds.struct), C.c_void_p(ids.ctypes.data), len(ids), hds.feat_dim, M, *caps,
                                                None if out is None else C.c_void_p(out.ctypes.data),
                                                0 if out is None else out.size, C.byref(lay))
    return rc, lay


SECTIONS = ("node_ptr", "bond_ptr", "bond_begin", "bond_end", "feat", "targets", "peak_ptr", "peak_mz", "peak_inten", "nbytes")


@pytest.mark.parametrize("kind", ["dense", "f32", "f64"])
def test_fixed_layout_packer(kind):
    """`eims_host_pack_batch_fixed`: one layout for every batch of n molecules, equal to the layout query's whatever
    molecules the query names; live bytes equal to the variable-layout packing of the same molecules; batches
    exactly at each cap pack, one atom, bond or peak more is refused with the true sizes; cap_bonds = 0 works."""
    n, n_mols = 16, 400
    table = synth_molecules(n_mols, max_atoms=24, seed=21)
    ptr_, mz, inten = synth_peaks(n_mols, M, seed=22)
    mz = mz + np.float32(0.25) if kind == "f32" else mz.astype(np.float64) + 1.0 / 3 if kind == "f64" else mz
    pk = (ptr_, mz, inten)
    dense = dense_spectra(ptr_, mz.astype(np.float32), inten, M)
    hds = HostDataset(table, dense) if kind == "dense" else HostDataset(table, None, peaks=pk)
    rng = np.random.default_rng(23)
    batches = np.stack([rng.choice(n_mols, n, replace=False) for _ in range(40)]).astype(np.int32)
    count = lambda p, ids: int(np.diff(p)[ids].sum())
    sizes = np.array([[count(table.node_ptr, i), count(table.bond_ptr, i), count(ptr_, i)] for i in batches])
    caps = tuple(int(c) for c in sizes.max(0))

    # the layout query names the n largest molecules, which exceed every cap: the fixed layout comes back anyway
    largest = np.argsort(np.diff(table.node_ptr))[-n:].astype(np.int32)
    rc, query = pack_fixed(hds, largest, caps, None)
    assert rc == _lib.ERR_CAPACITY and query.nbytes > 0
    assert query.num_nodes == count(table.node_ptr, largest) > caps[0]
    layout = {s: getattr(query, s) for s in SECTIONS}
    assert (layout["targets"] >= 0) == (kind == "dense") and (layout["peak_ptr"] >= 0) == (kind != "dense")

    buf = np.empty(query.nbytes, np.uint8)
    mzsz = 8 if kind == "f64" else 4
    for ids, (na, nb, npk) in zip(batches, sizes):
        buf.fill(0xFF)
        rc, lay = pack_fixed(hds, ids, caps, buf)
        assert rc == 0 and {s: getattr(lay, s) for s in SECTIONS} == layout
        assert (lay.num_graphs, lay.num_nodes, lay.num_edges, lay.mz_is_f64) == (n, na, 2 * nb, int(kind == "f64"))
        want = PackedHostBatch(table.select(ids), dense[ids] if kind == "dense" else None, pin=False,
                               peaks=None if kind == "dense" else select_peaks(pk, ids))
        live = dict(node_ptr=8 * (n + 1), bond_ptr=8 * (n + 1), bond_begin=4 * nb, bond_end=4 * nb, feat=4 * 6 * na,
                    targets=4 * n * M, peak_ptr=8 * (n + 1), peak_mz=mzsz * npk, peak_inten=4 * npk)
        raw = want.buf.numpy()
        for s, o in want.offsets.items():
            assert np.array_equal(buf[layout[s]:layout[s] + live[s]], raw[o:o + live[s]]), s

    # exactly at each cap packs; one more atom / bond / peak is refused with the batch's true sizes in the layout
    for j in range(3 if kind != "dense" else 2):
        ids = batches[int(np.argmax(sizes[:, j]))]
        na, nb = count(table.node_ptr, ids), count(table.bond_ptr, ids)
        assert pack_fixed(hds, ids, caps, buf)[0] == 0
        tight = list(caps)
        tight[j] -= 1
        rc, lay = pack_fixed(hds, ids, tuple(tight), buf)
        assert rc == _lib.ERR_CAPACITY and (lay.num_nodes, lay.num_edges) == (na, 2 * nb) and lay.nbytes > 0

    # cap_bonds = 0: molecules of one atom pack; a molecule with a bond does not
    single = MolTable(np.arange(n + 1, dtype=np.int64), np.zeros(n + 1, np.int64), table.feat[:n].copy(),
                      np.zeros(0, np.int32), np.zeros(0, np.int32))
    hs = HostDataset(single, dense[:n]) if kind == "dense" else HostDataset(single, None, peaks=(ptr_[:n + 1], mz, inten))
    rc, lay = pack_fixed(hs, np.arange(n), (n, 0, caps[2]), buf)
    assert rc == 0 and lay.num_edges == 0 and lay.num_nodes == n
    assert pack_fixed(hds, batches[0], (caps[0], 0, caps[2]), buf)[0] == _lib.ERR_CAPACITY
