"""The plan's call order and its workspace layout, through the public ABI.

Call order: a small plan is driven into each phase of a batch (unbuilt, built, training forward done, loss gradient
ready, head backward done, eval forward done) and every call whose acceptance depends on the phase is made there.  A
refused call returns before it enqueues anything.

Layout: at the benchmark's shapes and at a few edge shapes every workspace buffer name resolves to a 256-aligned range
inside the workspace, the ranges tile the workspace without overlapping, the split-K head outputs u1 .. dG (which a
training forward zeroes as one range) follow one another, the tf32 weight planes exist only on plans that can take the
planes GEMM, and an unknown name is refused without changing what the known names resolve to."""
import ctypes as C

import pytest
import torch

from eims_b200 import _lib
from eims_b200.engine import DeviceDataset, FlatParams, ModelDims, Plan, make_step
from eims_b200.synth import dense_spectra, synth_molecules, synth_peaks
from oracle import gcn_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
OK, ARG, STATE = 0, _lib.ERR_ARG, _lib.ERR_STATE

# ------------------------------------------------------------------------------------------------------------ call order
PHASES = ["unbuilt", "built", "train_fwd", "loss_grad", "head_bwd", "eval_fwd"]
# return code of each call in each phase, in PHASES order
EXPECT = {
    "forward":             [STATE, OK, OK, OK, OK, OK],
    "loss":                [OK, OK, OK, OK, OK, OK],
    "backward":            [STATE, STATE, STATE, OK, STATE, STATE],
    "backward_dprob":      [STATE, STATE, OK, OK, OK, STATE],
    "backward_part_head":  [STATE, STATE, STATE, OK, STATE, STATE],
    "backward_part_gcn":   [STATE, STATE, STATE, STATE, OK, STATE],
    "backward_feat":       [STATE, STATE, STATE, OK, STATE, ARG],
    "backward_feat_dprob": [STATE, STATE, OK, OK, STATE, OK],
}
SMALL = ModelDims(hidden_dim=64, max_mz=100, dropout=0.2)
N_MOLS = 12


def small_setup():
    table = synth_molecules(N_MOLS, max_atoms=16, seed=7)
    targets = dense_spectra(*synth_peaks(N_MOLS, SMALL.max_mz, seed=8), SMALL.max_mz)
    ds = DeviceDataset(table, targets, DEV)
    fp = FlatParams(SMALL, DEV)
    fp.load_state_dict(O.init_params(O.Dims(6, 64, 3, SMALL.max_mz, "combined", SMALL.dropout), 0))
    caps = (N_MOLS, int(table.node_ptr[-1]), int(2 * table.bond_ptr[-1]))
    dprob = torch.randn(N_MOLS, SMALL.max_mz, device=DEV)
    return ds, fp, caps, dprob


def enter(phase, plan, ds, fp):
    """Drive `plan` (fresh when `phase` is "unbuilt") into `phase` with calls that must all be accepted."""
    if phase == "unbuilt":
        return
    plan.batch_build(ds, None, N_MOLS)
    if phase == "eval_fwd":
        plan.forward(fp, False)
    if phase in ("train_fwd", "loss_grad", "head_bwd"):
        plan.forward(fp, True, make_step(step=1, seed=1))
    if phase in ("loss_grad", "head_bwd"):
        plan.loss(ds.targets, None, "mse", True)
    if phase == "head_bwd":
        assert plan.lib.eims_backward_part(plan.h, _lib.ptr(fp.params), None, _lib.ptr(fp.grads), _lib.BWD_HEAD,
                                           plan.stream) == OK


def call(name, plan, ds, fp, dprob):
    lib, h, st = plan.lib, plan.h, plan.stream
    prm, grd = _lib.ptr(fp.params), _lib.ptr(fp.grads)
    if name == "forward":
        step = make_step(step=1, seed=1)
        return lib.eims_forward(h, prm, _lib.ptr(fp.bn_running), 1, C.byref(step), st)
    if name == "loss":
        return lib.eims_loss(h, _lib.ptr(ds.targets), None, _lib.LOSS["mse"], 1, st)
    if name == "backward":
        return lib.eims_backward(h, prm, None, grd, st)
    if name == "backward_dprob":
        return lib.eims_backward(h, prm, _lib.ptr(dprob), grd, st)
    if name == "backward_part_head":
        return lib.eims_backward_part(h, prm, None, grd, _lib.BWD_HEAD, st)
    if name == "backward_part_gcn":
        return lib.eims_backward_part(h, prm, None, grd, _lib.BWD_GCN, st)
    if name == "backward_feat":
        return lib.eims_backward_feat(h, prm, None, grd, None, st)
    if name == "backward_feat_dprob":
        return lib.eims_backward_feat(h, prm, _lib.ptr(dprob), grd, None, st)
    raise KeyError(name)


@pytest.mark.parametrize("phase", PHASES)
def test_calls_accepted_and_refused_in_each_phase(phase):
    ds, fp, caps, dprob = small_setup()
    plan = Plan(SMALL, *caps, DEV)
    k = PHASES.index(phase)
    got = {}
    for name, codes in EXPECT.items():
        if phase == "unbuilt":
            plan = Plan(SMALL, *caps, DEV)
        enter(phase, plan, ds, fp)
        got[name] = call(name, plan, ds, fp, dprob)
    torch.cuda.synchronize()
    plan.check()
    assert got == {name: codes[k] for name, codes in EXPECT.items()}


def test_buffer_lookup_needs_a_bound_plan():
    lib = _lib.load()
    cd = SMALL.c()
    h = C.c_void_p()
    assert lib.eims_plan_create(C.byref(cd), 4, 64, 64, C.byref(h)) == OK
    for name in (b"dims", b"dims#0", b"z0", b"nope"):
        assert lib.eims_plan_buffer(h, name, None, None) == STATE
    assert lib.eims_plan_destroy(h) == OK


def test_bare_table_names_follow_the_current_set():
    """eims_batch_build fills the other set of batch tables and makes it current."""
    ds, fp, caps, _ = small_setup()
    plan = Plan(SMALL, *caps, DEV)
    for cur in (0, 1, 0):
        for t in TABLES:
            assert resolve(plan.lib, plan.h, t) == resolve(plan.lib, plan.h, f"{t}#{cur}")
        plan.batch_build(ds, None, N_MOLS)
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------------------- layout
SHAPES = {  # name: (dims, max_graphs, atoms per molecule); node and edge capacities as bench.py sizes them
    "cfg2": (ModelDims(6, 256, 3, 1000), 512, 64),
    "infer_4096": (ModelDims(6, 256, 3, 1000), 4096, 64),
    "cfg5": (ModelDims(6, 1024, 6, 1000), 512, 128),
    "hidden_192": (ModelDims(6, 192, 3, 1000), 512, 64),
    "one_layer": (ModelDims(6, 256, 1, 1000), 512, 64),
    "sum_pooling": (ModelDims(6, 256, 3, 1000, "sum"), 512, 64),
    "three_features": (ModelDims(3, 256, 3, 1000), 512, 64),
}
TABLES = ["dims", "gptr", "eptr", "gid", "bids", "src", "dst", "rowptr", "col", "norm", "x", "a0"]
SINGLE = ["flags", "argmax", "bn_means2", "bn_partials", "readout", "zstat", "u1", "u2", "logits", "dy2", "dy1", "dG",
          "y1", "ln1", "y2", "ln2", "prob", "dlogits", "row_loss", "row_cos", "dh", "q", "da"]
HEAD_ZEROED = ["u1", "u2", "logits", "dy2", "dy1", "dG"]
PER_LAYER = ["z", "bn_mean", "bn_invstd", "bn_scale", "bn_shift"]


def buffer_names(d: ModelDims):
    """Every name eims_plan_buffer accepts, bare batch-table names and "wplanes" aside."""
    L = d.num_gcn_layers
    return ([f"{t}#{k}" for t in TABLES for k in (0, 1)] + SINGLE + [f"a{l}" for l in range(1, L)]
            + [f"{n}{l}" for n in PER_LAYER for l in range(L)])


def resolve(lib, h, name):
    p, n = C.c_void_p(), C.c_int64()
    rc = lib.eims_plan_buffer(h, name.encode(), C.byref(p), C.byref(n))
    return rc, p.value, n.value


def layout(plan):
    """{name: (offset from the workspace base, bytes)} of every buffer of a bound plan, "wplanes" when it exists."""
    out = {}
    for name in buffer_names(plan.d) + ["wplanes"]:
        rc, ptr, n = resolve(plan.lib, plan.h, name)
        if name == "wplanes" and rc == ARG:
            continue
        assert rc == OK, name
        out[name] = (ptr - plan._base, n)
    return out


def shape_plan(shape):
    d, B, atoms = SHAPES[shape]
    return Plan(d, B, B * atoms, 2 * (B * atoms + 3 * B), DEV)


@pytest.mark.parametrize("shape", list(SHAPES))
def test_workspace_layout(shape):
    plan = shape_plan(shape)
    lib, d = plan.lib, plan.d
    total = lib.eims_plan_workspace_bytes(plan.h)
    lay = layout(plan)
    for name, (off, n) in lay.items():
        assert off % 256 == 0 and n > 0 and 0 <= off and off + n <= total, (name, off, n, total)
    spans = sorted(lay.values())
    assert all(a_off + a_n <= b_off for (a_off, a_n), (b_off, _) in zip(spans, spans[1:]))
    assert sum(n for _, n in spans) == total
    for a, b in zip(HEAD_ZEROED, HEAD_ZEROED[1:]):
        assert lay[a][0] + lay[a][1] == lay[b][0], (a, b)
    # the weight planes exist exactly where the planes GEMM can be selected
    planes_shape = d.hidden_dim % 256 == 0 and d.num_gcn_layers > 1
    assert ("wplanes" in lay) == planes_shape
    assert (lib.eims_plan_set_gemm_planes(plan.h, 1) == OK) == planes_shape
    assert lib.eims_plan_set_gemm_planes(plan.h, -1) == OK
    L = d.num_gcn_layers
    unknown = ["", "nope", "dims#2", "dims#", "a0#2", "u1#0", "a00", "z01", f"z{L}", f"a{L}", f"bn_mean{L}", "bn_mean", "a",
               "Dims"] + ([] if planes_shape else ["wplanes"])
    for name in unknown:
        assert resolve(lib, plan.h, name)[0] == ARG, name
    assert layout(plan) == lay
