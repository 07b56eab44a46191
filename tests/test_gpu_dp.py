"""Parity of the data-parallel optimiser kernel (`eims_dp_adamw_fused`, csrc/dp_fused.cu) and of the
CUDA-graph replay of a step, through the C ABI.  Needs a B200 (`-m gpu`).

  * world = 1 (runs on a one-GPU box): the fused all-reduce + AdamW + broadcast kernel degenerates to
    AdamW on the own slice and must equal `eims_adamw_flat` bit for bit, step after step;
  * world = 2 (skipped with fewer than two GPUs): `tools/dp_parity.py` under torchrun - five
    optimiser steps of the fused path (NVSwitch multicast branch and peer-load branch) against the
    shard-sequential oracle `Trainer.step(world_shards=...)` (SURVEY 4 T4), parameters bit-identical
    across ranks;
  * a step replayed from the captured CUDA graphs equals the eagerly launched step.
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from eims_b200 import _lib
from eims_b200._lib import check, ptr
from eims_b200.engine import DeviceDataset, FlatParams, GraphedTrainStep, ModelDims, Plan, make_step, onecycle_schedule
from eims_b200.synth import dense_spectra, synth_molecules, synth_peaks
from oracle import gcn_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_world1_fused_equals_adamw_flat_bitwise():
    lib = _lib.load()
    n = 4 * 50_021  # not a multiple of the grid: exercises the strided tail
    g = torch.Generator(device="cpu").manual_seed(0)
    p0 = torch.randn(n, generator=g)
    a = {k: t.to(DEV) for k, t in dict(p=p0.clone(), m=torch.zeros(n), v=torch.zeros(n)).items()}
    b = {k: t.clone() for k, t in a.items()}
    grads_b = [torch.zeros(n, device=DEV), torch.full((n,), 7.0, device=DEV)]  # the "other" buffer must come back zeroed
    pad = torch.zeros(1024, dtype=torch.int32, device=DEV)
    ticket = torch.zeros(16, dtype=torch.int32, device=DEV)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    sched = onecycle_schedule(8)
    one = lambda t: (C.c_uint64 * 1)(t.data_ptr())
    for k in range(8):
        grad = torch.randn(n, generator=g).to(DEV) * (10.0 ** (k - 4))
        step = make_step(lr=sched[k][0], beta1=sched[k][1], grad_scale=1.0, step=k + 1)
        ga = grad.clone()
        check(lib.eims_adamw_flat(ptr(a["p"]), ptr(ga), ptr(a["m"]), ptr(a["v"]), n, C.byref(step), st))
        cur = k % 2
        grads_b[cur].copy_(grad)
        check(lib.eims_dp_adamw_fused(0, 1, one(grads_b[cur]), one(b["p"]), one(pad), C.c_uint64(0), C.c_uint64(0), ptr(b["m"]),
                                      ptr(b["v"]), ptr(grads_b[1 - cur]), 0, n, C.byref(step), C.c_uint32(k + 1), 0, ptr(ticket), st))
        torch.cuda.synchronize()
        for key in ("p", "m", "v"):
            assert torch.equal(a[key], b[key]), (k, key)
        assert not ga.any() and not grads_b[1 - cur].any()   # zero_grad of GCN:414 on both paths
    assert int(ticket[1]) == 0  # no peer was waited for in vain


def test_lost_peer_is_reported_not_trapped():
    """A rank whose peer never arrives must come back with the status word set (ADVICE r1: no __trap)."""
    env = dict(os.environ, EIMS_DP_TIMEOUT_S="0.05")
    code = (
        "import ctypes as C, torch, sys\n"
        f"sys.path[:0] = [{ROOT!r}, {os.path.join(ROOT, 'computational-chemistry-ai_b200')!r}]\n"
        "from eims_b200 import _lib\n"
        "from eims_b200._lib import check, ptr\n"
        "from eims_b200.engine import make_step\n"
        "lib = _lib.load(); n = 4096\n"
        "z = lambda: torch.zeros(n, device='cuda')\n"
        "p, m, v, g0, g1 = z(), z(), z(), z(), z()\n"
        "pad = torch.zeros(1024, dtype=torch.int32, device='cuda'); ticket = torch.zeros(16, dtype=torch.int32, device='cuda')\n"
        "two = lambda t: (C.c_uint64 * 2)(t.data_ptr(), t.data_ptr())\n"  # 'rank 1' is this GPU too, but nobody ever signals for it
        "step = make_step(step=1)\n"
        "check(lib.eims_dp_adamw_fused(0, 2, two(g0), two(p), two(pad), C.c_uint64(0), C.c_uint64(0), ptr(m), ptr(v), ptr(g1), 0, n,\n"
        "      C.byref(step), C.c_uint32(5), 0, ptr(ticket), C.c_void_p(torch.cuda.current_stream().cuda_stream)))\n"
        "torch.cuda.synchronize()\n"
        "print('STATUS', int(ticket[1]))\n")
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "STATUS 5" in r.stdout, r.stdout


@pytest.mark.parametrize("dropout", [0.0, 0.2])
def test_graph_replay_equals_eager_steps(dropout):
    """6 optimiser steps replayed from the two captured graphs == the same 6 steps launched eagerly: same ids,
    same dropout keys and AdamW scalars (read from the device step block instead of kernel parameters)."""
    d = ModelDims(hidden_dim=128, max_mz=200, dropout=dropout)
    n_mols, batch, steps = 512, 32, 6
    table = synth_molecules(n_mols, max_atoms=40, seed=11)
    targets = dense_spectra(*synth_peaks(n_mols, d.max_mz, seed=12), d.max_mz)
    ds = DeviceDataset(table, targets, DEV)
    od = O.Dims(6, 128, 3, 200, "combined", dropout)
    ids = torch.from_numpy(np.random.default_rng(3).permutation(n_mols).astype(np.int32)).to(DEV).view(-1, batch)
    sched = onecycle_schedule(steps)
    mk = lambda k: make_step(lr=sched[k][0], beta1=sched[k][1], step=k + 1, seed=77)
    out = {}
    for mode in ("eager", "graph", "group4"):
        plan = Plan(d, batch, batch * 40, 2 * (batch * 40 + 3 * batch), DEV)
        fp = FlatParams(d, DEV)
        fp.load_state_dict(O.init_params(od, 0))
        metrics = torch.zeros(8, device=DEV)
        losses = []
        if mode == "eager":
            for k in range(steps):
                plan.train_step(ds, ids[k], fp, mk(k), metrics)
                losses.append(float(metrics[4]))
        else:
            # "graph": single-step graphs, flushed after every step; "group4": 4 steps per graph + 2 single steps
            gs = GraphedTrainStep(plan, ds, fp, batch, metrics, group=0 if mode == "graph" else 4)
            gs.capture(ids[0], mk(0))
            for k in range(steps):
                gs.step(mk(k), ids[min(k + 1, steps - 1)])
                if mode == "graph":
                    gs.flush()
                    losses.append(float(metrics[4]))
            gs.flush()
            if mode != "graph":
                assert gs.multi is not None and gs.k == 0
                losses = out["eager"][2][:-1] + [float(metrics[4])]   # only the last step's loss is visible
        plan.check()
        out[mode] = (fp.params.clone(), fp.bn_running.clone(), losses, metrics.clone())
    for mode in ("graph", "group4"):
        pe, pg = out["eager"][0], out[mode][0]
        # training sums with atomics (BatchNorm, split-K): equal up to summation order, and AdamW's sign-like
        # first steps amplify last-bit gradient noise on elements whose gradient is ~0
        np.testing.assert_allclose(out[mode][2], out["eager"][2], rtol=2e-5)
        assert float((out["eager"][1] - out[mode][1]).abs().max() / out["eager"][1].abs().max()) < 2e-4
        close = ((pe - pg).abs() <= 1e-5 * pe.abs().max()).float().mean()
        assert close > 0.995, (mode, float(close))
        assert float(out[mode][3][2]) == steps and float(out[mode][3][6]) == 0.0
        np.testing.assert_allclose(float(out[mode][3][0]), float(out["eager"][3][0]), rtol=2e-5)   # the epoch's loss sum


def test_two_part_indirect_step_equals_whole_step():
    """eims_train_step_built_indirect_part (part 1: forward + loss + head backward, part 2: GraphConv backward - what a
    data-parallel caller runs around its early head-bucket exchange) leaves the gradients of the one-call step."""
    d = ModelDims(hidden_dim=128, max_mz=200, dropout=0.2)
    n_mols, batch = 256, 32
    table = synth_molecules(n_mols, max_atoms=40, seed=21)
    targets = dense_spectra(*synth_peaks(n_mols, d.max_mz, seed=22), d.max_mz)
    ds = DeviceDataset(table, targets, DEV)
    ids = torch.arange(batch, dtype=torch.int32, device=DEV)
    step = make_step(step=3, seed=5)
    res = []
    for parts in (False, True):
        plan = Plan(d, batch, batch * 40, 2 * (batch * 40 + 3 * batch), DEV)
        fp = FlatParams(d, DEV)
        fp.load_state_dict(O.init_params(O.Dims(6, 128, 3, 200, "combined", 0.2), 0))
        metrics = torch.zeros(8, device=DEV)
        plan.enable_step_block(1)
        plan.select_step_block(0)
        plan.step_block_upload(step, ids, 0)
        plan.batch_build(ds, ids, batch)
        fp.grads.zero_()
        if parts:
            plan.train_step_built_indirect_part(ds, fp, 1, metrics)
            plan.train_step_built_indirect_part(ds, fp, 2, metrics)
        else:
            plan.train_step_built_indirect(ds, fp, metrics, optimizer=False)
        plan.check()
        res.append((fp.grads.clone(), float(metrics[4]), plan.buffer("prob", torch.float32, (batch, d.max_mz)).clone()))
    (ga, la, pa), (gb, lb, pb) = res
    assert la == pytest.approx(lb, rel=1e-6)
    assert float((pa - pb).abs().max()) <= 1e-6 * float(pa.abs().max())
    # atomics (BatchNorm sums, split-K) fix the gradients up to summation order
    assert float((ga - gb).abs().max()) <= 2e-5 * float(ga.abs().max())


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
@pytest.mark.parametrize("branch", ["multicast", "peer"])
def test_two_rank_fused_step_vs_shard_sequential_oracle(branch, tmp_path):
    out = tmp_path / "dp_parity.json"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29533", os.path.join(ROOT, "tools", "dp_parity.py"), "--branch", branch, "--out", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    assert "DP PARITY OK" in r.stdout


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_rank_train_model_through_the_drop_in(tmp_path):
    """`script.train_model(..., world_size=2)` under torchrun: bit-identical weights on both ranks, history and
    validation against the shard-sequential oracle, reference-format checkpoint round trip (tools/dp_dropin.py)."""
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29534", os.path.join(ROOT, "tools", "dp_dropin.py"), "--out", str(tmp_path / "dropin.json")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    assert "DP DROP-IN OK" in r.stdout
