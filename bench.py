#!/usr/bin/env python
"""bench.py - GCN EI-MS training throughput (molecules/s) on N B200s of one node.

    python bench.py --gpus 1 --steps 200 --warmup 20          # our arm (default N=1)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference --steps 10 --warmup 1    # the reference path on host cores

A "step" is one optimiser step of the reference's hot path (GCN:410-431) over one batch of
512 synthetic molecules: batch build (K1) -> GCNSpectrum forward -> MSE loss + cosine metric
-> backward -> AdamW, with H=256, L=3, 1000 m/z bins, dropout 0.2, fp32 (BASELINE.json
configs[1]; at N>1 configs[3]: 1 M molecules, batch 512 per GPU, one gradient exchange per
step).  One JSON line is printed by rank 0.

Timing protocol (the driver's): W warm-up steps, then exactly K steps between two CUDA events,
bracketed by a barrier + synchronize on both sides; max over ranks.  At N>1 the clock sampler is
started BEFORE the barrier and a device-side all-reduce sits immediately in front of the first
event, so every rank's timed region starts within microseconds of the others'.
"""
import argparse
import json
import os
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "computational-chemistry-ai_b200"))

METRIC = "gcn_eims_train_molecules_per_sec"
UNIT = "molecules/s"
BATCH, H, L, M, F0, DROPOUT, MAX_ATOMS = 512, 256, 3, 1000, 6, 0.2, 64
# the two training workloads of BASELINE.json: configs[1]/[3] ("train") and configs[4] ("wide")
WORKLOADS = {
    "train": dict(batch=BATCH, hid=H, layers=L, atoms=MAX_ATOMS, mols1=100_000, molsN=1_000_000),
    "wide": dict(batch=BATCH, hid=1024, layers=6, atoms=128, mols1=20_000, molsN=160_000),
}
SAMPLINGS = ("global_uniform_balanced", "rank_strided_uniform", "stratified")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps (default 200); --workload infer: timed batches (default one pass over the resident set)")
    ap.add_argument("--warmup", type=int, default=None, help="warm-up steps (default 20); --workload infer: warm-up batches (default 3)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--molecules", type=int, default=0, help="molecules in the resident set (0 = BASELINE config)")
    ap.add_argument("--gemm", default="tcgen05", choices=["tcgen05", "simt"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="N=1: skip the configs[2] / configs[4] measurements (extra_workloads)")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel of a step from the host instead of replaying the captured CUDA graphs")
    ap.add_argument("--sampling", default=SAMPLINGS[0], choices=SAMPLINGS,
                    help="N>1: which molecules a rank's batch holds. global_uniform_balanced (default): the global batch is the "
                         "reference's uniform shuffle (GCN:561-568) at batch world*512, dealt to the ranks so that atom counts are equal; "
                         "rank_strided_uniform: the same global batch, every world-th molecule per rank (DistributedSampler); "
                         "stratified: size-stratified batches (every batch the same work). The other two are timed as sampling_variants")
    ap.add_argument("--no-variants", action="store_true")
    ap.add_argument("--step-events", default="auto", choices=["auto", "on", "off"],
                    help="one CUDA event per timed step (per-rank step_times); auto = only at N>1, where the diagnosis matters: the "
                         "event between two steps costs the eager path its kernel-to-kernel launch overlap across the step boundary")
    ap.add_argument("--no-prefetch", action="store_true", help="eager N=1: build each batch inside its own step instead of one step ahead")
    ap.add_argument("--dp", default="fused", choices=["fused", "nccl"], help="N>1: gradient exchange implementation")
    ap.add_argument("--dp-overlap", action="store_true", help="fused path: exchange the head bucket early on a side stream / graph branch (measured slower, see TrainBench)")
    ap.add_argument("--no-overlap", action="store_true", help="nccl path: one-shot all-reduce after backward instead of two overlapped buckets")
    ap.add_argument("--targets", default="dense", choices=["dense", "peaks"],
                    help="target spectra as dense rows (what the reference's dataset holds, GCN:256) or as the peak lists they are "
                         "binned from, binned inside the loss kernel (~0.9 KB instead of 4 KB per molecule in HBM and over PCIe)")
    ap.add_argument("--profile-steps", type=int, default=20)
    ap.add_argument("--workload", default="train", choices=["train", "infer", "wide"],
                    help="train = BASELINE configs[1]/[3] (the metric); wide = configs[4] (6 layers, hidden 1024, <=128 atoms; "
                         "data-parallel under torchrun like train); infer = configs[2] (batch 4096 eval forward, 1 GPU)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (rank 0); the inputs "
                         "are seeded, so two builds run with the same arguments can be compared output for output "
                         "(tools/compare_dumps.py). Training sums with atomics, so repeated runs agree up to summation order, not "
                         "bit for bit; profiles/r3_dump_repeatability.json records how far apart two runs of one build were")
    a = ap.parse_args()
    if a.steps is not None and a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.warmup is not None and a.warmup < 0:
        ap.error("--warmup must not be negative")
    if a.impl == "reference" or a.workload != "infer":
        a.steps = 200 if a.steps is None else a.steps
        a.warmup = 20 if a.warmup is None else a.warmup
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return a


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """Writes every array as path/<name>.npy in the dtype it was computed in (float32 / float64)."""
    arrays = {k: v.detach().cpu().numpy() for k, v in arrays.items()}
    for k, v in arrays.items():
        if v.dtype not in (np.float32, np.float64):
            raise TypeError(f"output {k}: {v.dtype}, expected float32 or float64")
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes of outputs, more than {DUMP_LIMIT_BYTES}")
    os.makedirs(path, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(path, k + ".npy"), v)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return dict(hbm_gbs=float(j["hbm_gbs"]), bf16_tflops=float(j["bf16_tflops"]),
                    bf16_tflops_sustained=float(j.get("bf16_tflops_sustained", j["bf16_tflops"])), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons during the timed region (NVML)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self._halt = index, [], set(), None, threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                 "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                 "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.002)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------
# algorithmic bytes / flops per stage and step (SURVEY 8d; fp32 values, int32 indices)
# ------------------------------------------------------------------------------------------
def stage_work(N, E, B, P, H=H, L=L):
    pd = 2 * H
    nb = E // 2
    gemm_head = 2 * B * (pd * 2 * H + 2 * H * H + H * M)
    return {
        # name: (bound, work per STEP in bytes or flops)
        "k1_batch_build": ("hbm", 3 * N * F0 * 4 + nb * 8 + B * 16 + 3 * E * 4 + 3 * N * 4 + 2 * B * 4),
        "layer0_fwd": ("hbm", N * F0 * 4 + 4 * N + 4 * N * H),
        "bn_stats": ("hbm", L * 4 * N * H),
        "spmm_fwd": ("hbm", (L - 1) * (8 * N * H + 4 * E + 8 * N)),
        "gemm_gcn_fwd": ("tensor", (L - 1) * 2 * N * H * H),
        "readout": ("hbm", 4 * N * H + 12 * B * H),
        "gemm_head_fwd": ("tensor", gemm_head),
        "ln_fwd": ("hbm", 8 * B * (2 * H + H)),
        "loss": ("hbm", 16 * B * M),
        "metrics": ("hbm", 8 * B),
        "gemm_head_wgrad": ("tensor", gemm_head),
        "colsum": ("hbm", 4 * B * M),
        "gemm_head_dgrad": ("tensor", gemm_head),
        "ln_bwd": ("hbm", 16 * B * (2 * H + H)),
        # top layer from per-graph quantities (dG [B,2H] + zstat [B,2H]); the layers below ride on K2 when H <= 256,
        # else they are node passes over dh and z
        "bn_bwd_stats": ("hbm", 4 * B * (pd + 2 * H) + (0 if H <= 256 else (L - 1) * 8 * N * H)),
        "bn_bwd_apply": ("hbm", L * 12 * N * H - 8 * N * H),     # dh + z read, q written (layer 0 writes no q)
        "gemm_gcn_wgrad": ("tensor", (L - 1) * 2 * N * H * H),
        "gemm_gcn_dgrad": ("tensor", (L - 1) * 2 * N * H * H),
        "spmm_bwd": ("hbm", (L - 1) * ((12 if H <= 256 else 8) * N * H + 4 * E + 8 * N)),  # H <= 256: + the z row of the BatchNorm below (fused backward statistics)
        "layer0_wgrad": ("hbm", 4 * N * H + 4 * N * F0),
        "adamw": ("hbm", 28 * P),
        "elementwise": ("hbm", 0),
        # weight gradient + data gradient of a layer in one launch (the default)
        "gemm_head_bwd": ("tensor", 2 * gemm_head),
        "gemm_gcn_bwd": ("tensor", 2 * (L - 1) * 2 * N * H * H),
    }


def stage_report(prof, work, n_steps, pk_):
    """Per-stage timing (CUDA events around every launch) -> achieved GB/s or TFLOP/s."""
    tot_ms = sum(v[0] for v in prof.values())
    out = {}
    for name, (tms, cnt) in prof.items():
        if cnt == 0 or name not in work:
            continue
        bound, w = work[name]
        per_step_ms = tms / n_steps
        ach = w / (per_step_ms * 1e-3) / (1e9 if bound == "hbm" else 1e12) if per_step_ms > 0 else 0.0
        peak = pk_["hbm_gbs"] if bound == "hbm" else pk_["bf16_tflops"]
        out[name] = {"ms_per_step": round(per_step_ms, 5), "share": round(tms / tot_ms, 4), "launches_per_step": cnt / n_steps,
                     "bound": bound, "achieved": round(ach, 3), "unit": "GB/s" if bound == "hbm" else "TFLOP/s",
                     "frac": round(ach / peak, 4)}
    return out


# ------------------------------------------------------------------------------------------
# the reference path on host cores (oracle port of the script's train step)
# ------------------------------------------------------------------------------------------
def cpu_reference_run(steps, warmup, batch, n_mols=4096, time_budget=None):
    import torch
    from eims_b200.synth import dense_spectra, synth_molecules, synth_peaks
    from oracle import gcn_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    d = O.Dims(F0, H, L, M, "combined", DROPOUT)
    n_mols = max(n_mols, batch)
    table = synth_molecules(n_mols, max_atoms=MAX_ATOMS, seed=1234)
    spectra = torch.from_numpy(dense_spectra(*synth_peaks(n_mols, M, seed=4321), M))
    tr = O.Trainer(O.init_params(d, 0), d, total_steps=max(steps + warmup, 4))
    rng = np.random.default_rng(0)

    def one():
        ids = rng.choice(n_mols, size=batch, replace=False)
        sub = table.select(ids)  # host-side collate (dgl.batch equivalent, vectorised)
        src, dst = O.mol_edges(sub.bond_begin.astype(np.int64), sub.bond_end.astype(np.int64))
        off = np.repeat(sub.node_ptr[:-1], 2 * np.diff(sub.bond_ptr))
        g = O.Graph(src + off, dst + off, np.diff(sub.node_ptr))
        pred, loss = tr.step(g, torch.from_numpy(sub.feat), spectra[ids])
        O.cosine_similarity_batch(pred, spectra[ids], "cupy")  # the per-step metric (GCN:435)
        return loss

    for _ in range(warmup):
        one()
    t0 = time.perf_counter()
    done = 0
    for _ in range(steps):
        one()
        done += 1
        if time_budget and time.perf_counter() - t0 > time_budget and done >= 3:
            break
    dt = time.perf_counter() - t0
    return dict(value=done * batch / dt, steps=done, seconds=dt, cores=torch.get_num_threads(), batch=batch)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # always the configured batch of 512; a long --steps request is bounded by time (180 s), never by a smaller batch
    r = cpu_reference_run(args.steps, max(args.warmup, 1), BATCH, time_budget=180.0)
    sample = (f"{r['steps']} optimiser steps of batch {BATCH} drawn from 4096 synthetic molecules (same generator, H={H}, L={L}, M={M}, "
              f"dropout {DROPOUT})" + ("" if r["steps"] == args.steps else f"; stopped at the 180 s budget, {args.steps} were asked for"))
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": r["steps"], "warmup": max(args.warmup, 1), "ms_per_step": 1e3 * r["seconds"] / r["steps"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.gpus, "train"),
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": sample},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "oracle/gcn_oracle.py (torch-CPU restatement of the reference script; dgl/cupy/rdkit are not installable offline) on the box's host cores; host collate inside the timed loop",
    }
    print(json.dumps(line), flush=True)


def workload_config(n_gpus, workload="train", sampling=None):
    c = WORKLOADS[workload]
    if workload == "wide":
        wl = (f"BASELINE configs[4]: wide/deep variant, 6 GCN layers, hidden 1024, molecules up to 128 heavy atoms, batch 512/GPU, "
              f"training on {n_gpus} B200" + (" (data-parallel, fused NVLink gradient exchange)" if n_gpus > 1 else ""))
    elif n_gpus == 1:
        wl = "BASELINE configs[1]: GCN EI-MS training, 100k synthetic molecules (<=64 heavy atoms), batch 512, 3 GCN layers, hidden 256, 1000 m/z bins, fp32, single B200"
    else:
        wl = f"BASELINE configs[3]: data-parallel GCN EI-MS training, 1M synthetic molecules on {n_gpus} B200, batch 512/GPU, one gradient all-reduce per step over NVLink"
    out = {"workload": wl, "batch_per_gpu": c["batch"], "hidden_dim": c["hid"], "num_gcn_layers": c["layers"], "max_mz": M,
           "dropout": DROPOUT, "loss": "mse", "optimizer": "AdamW+OneCycleLR",
           "l2_policy": "no explicit flush: every step reads a fresh batch from a device-resident set (graph tables + 4 KB/molecule targets, >= 0.5 GB) larger than the 126 MB L2; activations are produced and consumed inside the step",
           "parallelism": f"dp{n_gpus}"}
    if sampling and n_gpus > 1:
        out["sampling"] = sampling
    return out


# ------------------------------------------------------------------------------------------
# data: the resident molecule set
# ------------------------------------------------------------------------------------------
def build_dataset(cfg, n_mols, world, rank, dev, targets_mode):
    """Returns (device data set holding ALL n_mols molecules, atoms per molecule [n_mols] (host), this rank's own
    host shard (table, peak lists) for the host-buffer e2e path).

    N=1: the set is generated on the host and uploaded.  N>1: every rank generates 1/world of the molecules (its own
    seed), the flat arrays are all-gathered over NCCL so that each rank holds the whole set in HBM (1 M molecules
    ~ 1 GB of graph tables + 4 GB of dense targets: 3 % of a B200) - which lets any rank process any molecule of the
    global batch (see --sampling) - and the dense target rows are binned on the device from the gathered peak lists by
    the product's own `eims_peaks_to_spectrum` kernel (bit-exact with the reference's peaks_to_spectrum_batch)."""
    import torch
    import torch.distributed as dist
    from eims_b200.engine import DeviceDataset, DevicePeaks
    from eims_b200.synth import dense_spectra, synth_molecules, synth_peaks
    n_local = n_mols // world
    table = synth_molecules(n_local, max_atoms=cfg["atoms"], seed=1234 + 7919 * rank)
    pk = synth_peaks(n_local, M, seed=4321 + 7919 * rank)
    if world == 1:
        if targets_mode == "peaks":
            ds = DeviceDataset(table, None, dev, peaks=DevicePeaks(*pk, dev))
        else:
            ds = DeviceDataset(table, dense_spectra(*pk, M), dev)
        return ds, np.diff(table.node_ptr), (table, pk)

    def gather_cat(a, dt):
        t = torch.from_numpy(np.ascontiguousarray(a)).to(dt).to(dev)
        n = torch.tensor([t.numel()], device=dev, dtype=torch.int64)
        ns = [torch.zeros_like(n) for _ in range(world)]
        dist.all_gather(ns, n)
        ns = [int(x.item()) for x in ns]
        pad = torch.zeros(max(ns), dtype=dt, device=dev)
        pad[: t.numel()] = t
        out = [torch.empty_like(pad) for _ in range(world)]
        dist.all_gather(out, pad)
        return torch.cat([o[:k] for o, k in zip(out, ns)])

    ptr_of = lambda counts: torch.cat([torch.zeros(1, dtype=torch.int64, device=dev), torch.cumsum(counts, 0)])
    node_ptr = ptr_of(gather_cat(np.diff(table.node_ptr), torch.int64))
    bond_ptr = ptr_of(gather_cat(np.diff(table.bond_ptr), torch.int64))
    feat = gather_cat(table.feat.reshape(-1), torch.float32)
    bb, be = gather_cat(table.bond_begin, torch.int32), gather_cat(table.bond_end, torch.int32)
    peak_ptr = ptr_of(gather_cat(np.diff(pk[0]), torch.int64))
    mz, inten = gather_cat(pk[1], torch.float64), gather_cat(pk[2], torch.float32)
    dpk = DevicePeaks.from_device(peak_ptr, mz, inten)
    dense = None if targets_mode == "peaks" else dpk.to_spectrum(M)
    ds = DeviceDataset.from_device(node_ptr, bond_ptr, feat, bb, be, targets=dense, peaks=dpk if dense is None else None)
    torch.cuda.synchronize()
    return ds, ds.host_num_atoms, (table, pk)


def make_ids(sampling, sizes, world, rank, batch, n_steps, seed):
    """int32 [n_steps + 1, batch] molecule ids of this rank (one spare batch: the graph replay builds one ahead)."""
    from eims_b200.dist import global_batches, stratified_epoch
    out, ep = [], 0
    need = n_steps + 1
    while sum(len(o) for o in out) < need:
        if sampling == "stratified":
            # size-stratified batches over this rank's strided share of the set: every batch carries the same work
            mine = np.arange(rank, len(sizes), world)
            out.append(mine[stratified_epoch(sizes[mine], batch, ep, seed=seed + rank)].astype(np.int32))
        else:
            out.append(global_batches(sizes, world, rank, batch, ep, seed=seed, balance=(sampling == "global_uniform_balanced")))
        ep += 1
    return np.concatenate(out)[:need]


# ------------------------------------------------------------------------------------------
# one training workload, timed
# ------------------------------------------------------------------------------------------
class TrainBench:
    def __init__(self, args, workload, world, rank, dev, n_mols=None):
        import torch
        from eims_b200.dist import FusedP2PAdamW, GradReducer, broadcast_params
        from eims_b200.engine import FlatParams, ModelDims, Plan, onecycle_schedule
        self.args, self.world, self.rank, self.dev, self.workload = args, world, rank, dev, workload
        cfg = self.cfg = WORKLOADS[workload]
        self.batch = cfg["batch"]
        n_mols = n_mols or args.molecules or (cfg["mols1"] if world == 1 else cfg["molsN"])
        n_mols = max(n_mols // world, self.batch) * world
        self.ds, self.sizes, self.host_shard = build_dataset(cfg, n_mols, world, rank, dev, args.targets)
        self.n_mols = n_mols
        self.d = ModelDims(F0, cfg["hid"], cfg["layers"], M, "combined", DROPOUT)
        cap_nodes = self.batch * cfg["atoms"]
        self.plan = Plan(self.d, self.batch, cap_nodes, 2 * (cap_nodes + 3 * self.batch), dev, gemm_backend=args.gemm)
        self.fp = FlatParams(self.d, dev)
        init_weights(self.fp, self.d)
        broadcast_params(self.fp)
        self.reducer = GradReducer(self.fp.offsets, cfg["layers"], overlap=not args.no_overlap)
        self.fused, self.dp_note = None, "single GPU"
        if world > 1:
            self.dp_note = "NCCL all-reduce (two buckets) + AdamW kernel"
            if args.dp == "fused":
                try:
                    # --dp-overlap: two buckets, the head's exchange on a side branch under the GraphConv backward.  Measured
                    # at N=2 under graph replay (same box each): 0.3558 vs 0.3473 ms/step with a block of the early kernel
                    # spinning on every SM, 0.3490 vs 0.3480 with 16 blocks (the default now) - the exchange costs its
                    # barriers, not its bytes, so hiding 84 % of the bytes buys nothing; one exchange kernel per step stays.
                    self.fused = FusedP2PAdamW(self.fp, cfg["layers"], overlap=args.dp_overlap)
                    self.dp_note = ("one fused kernel: all-reduce + AdamW + parameter broadcast over NVLink peer memory ("
                                    + ("NVSwitch multimem" if self.fused.multicast else "peer loads/stores") + ")")
                except Exception as exc:  # symmetric memory unavailable: say so, use the NCCL path
                    self.dp_note += f" [fused path unavailable: {type(exc).__name__}: {exc}]"
        self.metrics = torch.zeros(8, device=dev)
        self.gscale = 1.0 / world
        self.k = 0            # optimiser steps taken
        self.graphed = None
        self.graph_note = "eager launches"
        self.sched = onecycle_schedule(4096)
        self.launches_per_step = None
        self.sampler = ClockSampler(dev.index or 0)   # nvmlInit + handle lookup now, sampling thread later

    def step_scalars(self, k=None):
        from eims_b200.engine import make_step
        k = self.k if k is None else k
        lr, b1 = self.sched[min(k, len(self.sched) - 1)]
        return make_step(lr=lr, beta1=b1, grad_scale=self.gscale, step=k + 1, seed=2024 + self.rank)

    def eager_step(self, ids, next_ids):
        from eims_b200.dist import train_step_dp, train_step_fused
        st = self.step_scalars()
        if self.world == 1:
            if self.args.no_prefetch:
                self.plan.train_step(self.ds, ids, self.fp, st, self.metrics)
            else:  # K1 of the next batch is built on a side stream while this step runs
                self.plan.train_step_prefetch(self.ds, ids, next_ids, self.fp, st, self.metrics)
        elif self.fused is not None:
            train_step_fused(self.plan, self.ds, ids, self.fp, st, self.fused, self.metrics, next_ids=next_ids)
        else:
            train_step_dp(self.plan, self.ds, ids, self.fp, st, self.reducer, self.metrics)
        self.k += 1

    def try_capture(self, first_ids):
        """Two eager steps have run (modules loaded, one-time attributes set): capture the step graphs."""
        from eims_b200.engine import GraphedTrainStep
        if self.args.no_graph or (self.world > 1 and self.fused is None):
            return
        try:
            self.plan.profile(False)
            g = GraphedTrainStep(self.plan, self.ds, self.fp, self.batch, self.metrics, fused=self.fused)
            g.capture(first_ids, self.step_scalars())
            _, n = self.plan.profile_read()
            per = n // (2 + g.group)                                  # launches the plan counted per captured step
            self.launches_per_step = per + (1 if self.fused is not None else 0) + 1.0 / max(g.group, 1)   # (+ exchange kernel) + upload per group
            self.graphed = g
            self.graph_note = (f"captured CUDA graphs: {g.group} consecutive steps per graph (step || next batch build || head optimiser), one "
                               "step-block upload + one graph launch per group; single-step graphs for the remainder")
        except Exception as exc:
            self.graph_note = f"eager launches [graph capture failed: {type(exc).__name__}: {str(exc)[:200]}]"
            self.graphed = None

    def step(self, ids, next_ids):
        """Returns True when work was actually enqueued (graph groups are launched when full)."""
        if self.graphed is not None:
            self.graphed.step(self.step_scalars(), next_ids)
            self.k += 1
            return not self.graphed.pending
        self.eager_step(ids, next_ids)
        return True

    def flush(self):
        if self.graphed is not None:
            self.graphed.flush()

    def outputs(self):
        """What a caller of the last step receives: the model after its optimiser update (flat parameters in
        param_spec order, BatchNorm running statistics [L, 2, H]), the step's predicted spectra [batch, M] and its
        loss and mean cosine."""
        import torch
        return {"params": self.fp.params, "bn_running": self.fp.bn_running,
                "spectra": self.plan.buffer("prob", torch.float32, (self.batch, M)),
                "loss": self.metrics[4:5], "cosine": self.metrics[5:6]}

    def device_barrier(self):
        """All ranks leave together, ON THE DEVICE: a tiny all-reduce on the compute stream; what is enqueued next
        (the first timing event) executes only after every rank has arrived."""
        import torch
        import torch.distributed as dist
        if self.world > 1:
            t = torch.zeros(1, device=self.dev)
            dist.all_reduce(t)

    def timed(self, ids_dev, i0, n_steps, with_sampler=False):
        """Times steps i0 .. i0+n_steps-1 of ids_dev (device int32 [*, batch]); the batch of step i0 must be the one
        built last.  Returns (total ms (max over ranks), per-step ms of this rank, clocks)."""
        import torch
        import torch.distributed as dist
        torch.cuda.synchronize()
        # NVML was initialised when the bench object was built (tens of ms, 8 processes at once): here only the sampling
        # thread starts, BEFORE the barrier, so the GPU is idle for microseconds, not milliseconds, ahead of the timed steps
        sampler = self.sampler if with_sampler else None
        if sampler:
            self.sampler = None
            sampler.start()
        per_step = self.args.step_events == "on" or (self.args.step_events == "auto" and self.world > 1)
        # Graph replay: the host side of the FIRST group (step scalars, sequence numbers, argument arrays: ~0.1-0.2 ms of
        # Python) is done before the start barrier, so that after it only the upload kernel + one graph launch remain.
        # Otherwise the ranks leave the barrier together but submit their first graph at different times, and in a
        # 20-step window everyone pays the slowest rank's Python once (first step 0.53 ms against 0.355 at N=8).  All
        # device work of the K steps stays between the two events.
        j0 = 0
        held = self.graphed is not None and self.graphed.can_hold(n_steps)
        if held:
            self.graphed.hold_next = True
            while self.graphed.held is None:
                self.step(ids_dev[i0 + j0], ids_dev[i0 + j0 + 1])
                j0 += 1
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        self.device_barrier()
        ev0 = torch.cuda.Event(enable_timing=True)
        ev0.record()
        marks = []   # (event, steps enqueued since the previous mark): one per launch (a graph group, or an eager step)
        since = 0
        if held:
            self.graphed.release()
            since = j0
            if per_step or j0 == n_steps:
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                marks.append((e, since))
                since = 0
        for j in range(j0, n_steps):
            launched = self.step(ids_dev[i0 + j], ids_dev[i0 + j + 1])
            since += 1
            if j == n_steps - 1:
                self.flush()
                launched = True
            if launched and (per_step or j == n_steps - 1):
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                marks.append((e, since))
                since = 0
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        clocks = sampler.stop() if sampler else None
        ms = ev0.elapsed_time(marks[-1][0])
        per, prev = [], ev0
        for e, cnt in marks:   # a group's time is spread evenly over its steps
            per += [prev.elapsed_time(e) / cnt] * cnt
            prev = e
        per = np.array(per)
        if self.world > 1:
            t = torch.tensor([ms], device=self.dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, per, clocks


def run_ours(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    tb = TrainBench(args, args.workload, world, rank, dev)
    K, W_req = args.steps, max(args.warmup, 3)
    # Graph replay: the multi-step graph must have been replayed ONCE before the timed region - its first launch
    # uploads the instantiated graph to the device (measured at N=2: the first group of 10 steps 5.06 ms, every later one
    # 3.55 ms), which is set-up, not a training step.  Two eager steps + capture + one full group = 12 untimed steps at
    # least; the line reports the requested warm-up and what was run.
    W = W_req if args.no_graph else max(W_req, 2 + int(os.environ.get("EIMS_GRAPH_GROUP", 10)))
    variants = [s for s in SAMPLINGS if s != args.sampling] if (world > 1 and not args.no_variants) else []
    Kv = min(K, 50)
    ids_main = make_ids(args.sampling, tb.sizes, world, rank, tb.batch, W + K, seed=99)
    segs = [ids_main[:-1]] + [make_ids(s, tb.sizes, world, rank, tb.batch, Kv, seed=199)[:-1] for s in variants]
    ids_host = np.concatenate(segs + [ids_main[-1:]])
    ids_dev = torch.from_numpy(ids_host).to(dev)

    # The step runs on a high-priority stream, so that its kernels win over the batch build of the NEXT
    # step (default-priority side stream) whenever both have blocks to place.
    torch.cuda.synchronize()
    if os.environ.get("EIMS_BENCH_DEFAULT_STREAM", "0") != "1":
        torch.cuda.set_stream(torch.cuda.Stream(dev, priority=-1))
    # ---- warm-up: two eager steps, graph capture, the rest replayed
    for i in range(2):
        tb.eager_step(ids_dev[i], ids_dev[i + 1])
    tb.plan.check()
    tb.try_capture(ids_dev[2])
    if tb.graphed is None and world == 1 and not args.no_prefetch:
        pass  # the eager prefetch path already built batch 2
    for i in range(2, W):
        tb.step(ids_dev[i], ids_dev[i + 1])
    tb.flush()
    tb.plan.check()
    # ---- the timed region
    tb.plan.profile(False)  # resets the launch counter
    ms, per_step, clocks = tb.timed(ids_dev, W, K, with_sampler=True)
    if args.dump_outputs and rank == 0:   # before the passes below run more steps on the same model
        dump_outputs(args.dump_outputs, tb.outputs())
    _, launches = tb.plan.profile_read()
    if tb.graphed is not None:
        launches = int(round(K * tb.launches_per_step))
    tb.plan.check()
    if tb.fused is not None and tb.fused.lost_peer():
        raise SystemExit(f"rank {rank}: a peer did not arrive at the gradient exchange (sequence {tb.fused.lost_peer()})")
    value = K * tb.batch * world / (ms * 1e-3)
    final_loss = float(tb.metrics[4].item())
    nonfinite_steps = int(tb.metrics[6].item())

    # ---- per-rank step times (who is the straggler?)
    step_times = None
    if world > 1:
        allp = [torch.zeros(K, device=dev) for _ in range(world)]
        dist.all_gather(allp, torch.from_numpy(per_step).float().to(dev))
        allp = torch.stack(allp).cpu().numpy()
        wr, ws = np.unravel_index(np.argmax(allp), allp.shape)
        atoms = [int(tb.sizes[ids_host[W + j]].sum()) for j in range(K)]
        step_times = {"note": "graph groups are timed as a whole and spread evenly over their steps",
                      "median_ms_per_rank": [round(float(np.median(r)), 4) for r in allp],
                      "max_ms_per_rank": [round(float(r.max()), 4) for r in allp],
                      "worst": {"rank": int(wr), "step": int(ws), "ms": round(float(allp[wr, ws]), 4)},
                      "rank0_atoms_per_batch_min_max": [min(atoms), max(atoms)]}
    else:
        step_times = {"median_ms": round(float(np.median(per_step)), 4), "max_ms": round(float(per_step.max()), 4)}

    # ---- the other sampling policies, same protocol, shorter (N>1)
    sampling_variants = None
    if variants:
        sampling_variants = {args.sampling: {"value": value, "ms_per_step": ms / K, "steps": K}}
        off = W + K
        for s in variants:
            # the batch built last belongs to the previous segment's successor row = first row of this segment
            vms, _, _ = tb.timed(ids_dev, off, Kv)
            sampling_variants[s] = {"value": Kv * tb.batch * world / (vms * 1e-3), "ms_per_step": vms / Kv, "steps": Kv}
            off += Kv

    # ---- per-stage pass (same steps launched eagerly with CUDA events around every launch; not used for `value`)
    roofline, stages_out = None, None
    if rank == 0 and args.profile_steps > 0:
        roofline, stages_out = stage_pass(tb, ids_host, ids_dev, args.profile_steps)

    # ---- e2e: the same step through the host-buffer call (collate + H2D of inputs + D2H of loss inside)
    e2e = None if args.no_e2e else e2e_pass(tb, min(K, 100))

    extra = None
    if world == 1 and args.workload == "train" and not args.no_extra:
        del tb.graphed
        extra = extra_workloads(args, dev)

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    cpu = None
    if world == 1 and not args.no_cpu_baseline and args.workload == "train":
        r = cpu_reference_run(120, 1, BATCH, time_budget=20.0)  # ~15 s of host work
        cpu = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port",
               "sample": f"{r['steps']} optimiser steps of batch {BATCH} from 4096 synthetic molecules in {r['seconds']:.1f} s (oracle/gcn_oracle.py, torch-CPU fp32, all host threads)"}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W_req, "warmup_run": W,
        "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": workload_config(world, args.workload, args.sampling), "gemm": args.gemm,
        "targets": args.targets, "gpu_launches": int(launches), "launch_mode": tb.graph_note, "data_parallel": tb.dp_note,
        "clocks": clocks, "final_loss": final_loss, "nonfinite_loss_steps": nonfinite_steps, "resident_molecules": tb.n_mols,
        "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "step_times": step_times, "sampling_variants": sampling_variants,
        "extra_workloads": extra, "stages": stages_out,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def stage_pass(tb, ids_host, ids_dev, n_prof):
    pk_ = peaks()
    plan, ds, fp = tb.plan, tb.ds, tb.fp
    plan.profile(True)
    Ns, Es = [], []
    for j in range(n_prof):
        i = j % (len(ids_host) - 1)
        n_, e_ = ds.batch_counts(ids_host[i])
        Ns.append(n_)
        Es.append(e_)
        plan.train_step(ds, ids_dev[i], fp, tb.step_scalars(), tb.metrics)
        tb.k += 1
    prof, _ = plan.profile_read()
    plan.profile(False)
    work = stage_work(float(np.mean(Ns)), float(np.mean(Es)), tb.batch, fp.numel, tb.cfg["hid"], tb.cfg["layers"])
    stages_out = stage_report(prof, work, n_prof, pk_)
    dom = max(stages_out, key=lambda n: stages_out[n]["ms_per_step"])
    s = stages_out[dom]
    traffic, l2_traffic = None, None
    tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tp) and tb.workload == "train":
        tj = json.load(open(tp))
        traffic = tj.get(dom)  # bytes per launch, ncu dram__bytes_read + dram__bytes_write (cold-cache capture of the same launch, see profiles/)
        l2_traffic = tj.get("_l2_bytes_per_launch", {}).get(dom)  # lts__t_bytes.sum of that capture
    roofline = {"kernel": dom, "bound": s["bound"], "achieved": s["achieved"], "peak": pk_["hbm_gbs"] if s["bound"] == "hbm" else pk_["bf16_tflops"],
                "unit": s["unit"], "frac": s["frac"], "traffic": traffic, "l2_traffic": l2_traffic,
                "traffic_source": "profiles/ncu_traffic.json: one `ncu --set full` capture of this launch (round 2, cold cache), not measured by this run",
                "peak_source": f"{pk_['source']} ({'copy bandwidth' if s['bound'] == 'hbm' else 'cuBLAS bf16 burst; tf32 is half of it and the kernel runs 3 tf32 passes, so 1/6 is the ceiling'})",
                "launch_ms": round(s["ms_per_step"] / s["launches_per_step"], 5)}
    if s["bound"] == "tensor":  # the arithmetic is 3xTF32: what fraction of THAT ceiling (peak / 6) the kernel reaches
        roofline["ceiling_3xtf32"] = round(pk_["bf16_tflops"] / 6.0, 1)
        roofline["frac_of_3xtf32_ceiling"] = round(s["achieved"] / (pk_["bf16_tflops"] / 6.0), 4)
    return roofline, stages_out


def e2e_pass(tb, n_e2e):
    """The reference-facing path with HOST buffers.  Default: `GraphedHostTrainer` - the copies, K1 and the steps replayed
    as CUDA graphs of 10 steps, the host collating into a pinned ring.  Falls back to the eagerly launched
    `HostBatchRunner` loop (and says so) if the graphs cannot be captured or with --no-graph."""
    if not tb.args.no_graph and (tb.world == 1 or tb.fused is not None):
        try:
            return e2e_graph_pass(tb, n_e2e)
        except Exception as exc:
            note = f"graph e2e path failed ({type(exc).__name__}: {str(exc)[:160]}); eager host-buffer loop instead"
            out = e2e_eager_pass(tb, n_e2e)
            out["note"] = note
            return out
    return e2e_eager_pass(tb, n_e2e)


def e2e_graph_pass(tb, n_e2e):
    import torch
    import torch.distributed as dist
    from eims_b200.hostpath import GraphedHostTrainer, HostDataset
    from eims_b200.synth import dense_spectra
    table, pk = tb.host_shard
    n_local = table.num_mols
    peaks_mode = tb.args.targets == "peaks"
    hds = HostDataset(table, None, peaks=pk) if peaks_mode else HostDataset(table, dense_spectra(*pk, M))
    G = 10
    groups = max(1, n_e2e // G)
    workers = max(1, min(4, (os.cpu_count() or 4) // tb.world - 1))   # the ranks share the box's host cores
    cap_nodes = tb.batch * tb.cfg["atoms"]
    tr = GraphedHostTrainer(tb.plan, tb.fp, hds, tb.batch, M, cap_nodes, cap_nodes + 3 * tb.batch, tb.batch * 150 if peaks_mode else 0,
                            metrics=tb.metrics, fused=tb.fused, group=G, workers=workers)
    rng = np.random.default_rng(7 + tb.rank)
    n_batches = (groups + 2) * G + 2
    order = np.concatenate([rng.permutation(n_local) for _ in range(n_batches * tb.batch // n_local + 2)]).astype(np.int32)
    ids_of = lambda n: order[n * tb.batch:(n + 1) * tb.batch]
    futs = {n: tr.pack_async(n, ids_of(n)) for n in range(G + 1)}
    tr.prime(futs.pop(0))
    tr.capture(tb.step_scalars())

    def run_group(l):
        steps = [tb.step_scalars(tb.k + j) for j in range(G)]
        tb.k += G
        li = tr.launch(steps, [futs.pop(n) for n in range(l * G + 1, l * G + G + 1)])
        for n in range((l + 1) * G + 1, (l + 2) * G + 1):     # collate the next group's batches while this one runs
            futs[n] = tr.pack_async(n, ids_of(n))
        return li

    run_group(0)                                              # untimed warm-up group
    torch.cuda.synchronize()
    if tb.world > 1:
        dist.barrier()
    tr.h2d_bytes = tr.d2h_bytes = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tb.device_barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e0.record()
    last = None
    for l in range(1, groups + 1):
        run_group(l)
        if l > 1:
            last = tr.results(l - 1)[-1]                      # the host reads a group's losses while the next group runs
    last = tr.results(groups)[-1]
    e1.record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    if tb.world > 1:
        t = torch.tensor([wall], device=tb.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        wall = float(t.item())
    tr.close()
    n_steps = groups * G
    return {"value": n_steps * tb.batch * tb.world / wall, "unit": UNIT, "h2d_bytes_per_step": int(tr.h2d_bytes / n_steps),
            "d2h_bytes_per_step": int(tr.d2h_bytes / n_steps), "steps": n_steps,
            "timing": ("host wall clock around the loop, max over ranks (device events: %.1f ms); INSIDE the timed region per step: host collate "
                       "of the batch from the host-resident set into a pinned ring (C, %d worker threads, one group of %d batches ahead), "
                       "H2D copy of the batch (fixed-layout buffer), K1 + step%s, D2H of the step's loss/cosine; copies, K1 and steps are "
                       "replayed from captured CUDA graphs of %d steps, the host reads each group's losses while the next group runs"
                       % (e0.elapsed_time(e1), workers, G, " + fused gradient exchange" if tb.world > 1 else "", G)),
            "last_loss": last[0]}


def e2e_eager_pass(tb, n_e2e):
    """The reference-facing call with HOST buffers, per step and inside the timed region: collate of the batch from the
    host-resident set into pinned memory (`eims_host_pack_batch`, C, on 4 worker threads - the reference's DataLoader
    uses num_workers=4, GCN:100 - prefetching 4 batches ahead), ONE H2D copy, K1 + step, D2H of the step's loss / cosine,
    which the host reads two steps behind.  N>1: every rank feeds from its own host shard (uniform shuffle) and the
    gradients go through the same fused exchange kernel."""
    import torch
    import torch.distributed as dist
    from eims_b200.dist import train_step_fused  # noqa: F401
    from eims_b200.hostpath import HostBatchRunner, HostDataset, HostPacker
    from eims_b200.synth import dense_spectra
    if tb.world > 1 and tb.fused is None:
        return {"value": None, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "note": "e2e needs the fused exchange path at N>1"}
    table, pk = tb.host_shard
    n_local = table.num_mols
    if tb.args.targets == "peaks":
        hds = HostDataset(table, None, peaks=pk)
    else:
        hds = HostDataset(table, dense_spectra(*pk, M))
    depth = 4
    workers = max(1, min(4, (os.cpu_count() or 4) // tb.world - 1))   # the ranks share the box's host cores
    cap = tb.batch * (tb.cfg["atoms"] * (F0 * 4 + 8 + 10) + 4 * M + 64) + (1 << 16)
    packer = HostPacker(hds, M, cap, n_buffers=depth + 3)
    runner = HostBatchRunner(tb.plan, tb.fp, cap)
    rng = np.random.default_rng(7 + tb.rank)
    n_total = n_e2e + 3
    order = np.concatenate([rng.permutation(n_local) for _ in range(n_total * tb.batch // n_local + 2)]).astype(np.int32)
    pool = ThreadPoolExecutor(workers)
    lock = threading.Lock()

    def submit(j):
        with lock:   # ring-slot assignment is serial; the gather itself (ctypes releases the GIL) runs in parallel
            k = packer._i % len(packer.bufs)
            packer._i += 1
        ids = order[j * tb.batch:(j + 1) * tb.batch]

        def work():
            packer2 = packer
            if packer2.events[k] is not None:
                packer2.events[k].synchronize()
            return pack_into(packer2, k, ids)
        return pool.submit(work)

    futs = {j: submit(j) for j in range(min(depth, n_total))}

    def one(j, slot):
        st = tb.step_scalars()
        hb_next = None
        if tb.world == 1:
            runner.train_step(slot, cur_hb[0], st)
        else:
            tb.fused.begin_step()
            runner.train_step(slot, cur_hb[0], st, optimizer=False)
            tb.fused.finish(st, tb.plan.stream)
        tb.k += 1
        if j + depth < n_total:
            futs[j + depth] = submit(j + depth)
        if j + 1 < n_total:
            hb_next = futs.pop(j + 1).result()
            nslot = runner.upload(hb_next, build=not tb.args.no_prefetch)
            cur_hb[0] = hb_next
            return nslot
        return None

    cur_hb = [futs.pop(0).result()]
    slot = runner.upload(cur_hb[0], build=not tb.args.no_prefetch)
    for j in range(3):
        slot = one(j, slot)
    torch.cuda.synchronize()
    if tb.world > 1:
        dist.barrier()
    runner.h2d_bytes = runner.d2h_bytes = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tb.device_barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e0.record()
    last = None
    for j in range(3, 3 + n_e2e):
        slot = one(j, slot)
        last = runner.read(2) or last   # a finished step's loss on the host, two steps behind the GPU (waits for ITS copy only)
    loss_e2e, _ = runner.result()
    e1.record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    if tb.world > 1:
        t = torch.tensor([wall], device=tb.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        wall = float(t.item())
    pool.shutdown(wait=True)
    return {"value": n_e2e * tb.batch * tb.world / wall, "unit": UNIT, "h2d_bytes_per_step": int(runner.h2d_bytes / n_e2e),
            "d2h_bytes_per_step": int(runner.d2h_bytes / n_e2e), "steps": n_e2e,
            "timing": ("host wall clock around the loop, max over ranks (device events: %.1f ms); INSIDE the timed region per step: host collate of "
                       "the batch into pinned memory (C, %d worker threads, %d batches ahead), one H2D copy, K1 + step%s, D2H of loss/cosine "
                       "read by the host two steps behind" % (e0.elapsed_time(e1), workers, depth, " + fused gradient exchange" if tb.world > 1 else "")),
            "last_loss": loss_e2e}


def pack_into(packer, k, ids):
    """HostPacker.pack with the ring slot chosen by the caller (worker threads)."""
    import ctypes as C
    from eims_b200 import _lib
    from eims_b200.hostpath import PackedHostBatch
    import torch
    ids = np.ascontiguousarray(ids, np.int32)
    lay = _lib.HostBatchLayout()
    buf = packer.bufs[k]
    _lib.check(packer.lib.eims_host_pack_batch(C.byref(packer.hds.struct), C.c_void_p(ids.ctypes.data), len(ids), packer.hds.feat_dim,
                                               packer.max_mz, C.c_void_p(buf.data_ptr()), buf.numel(), C.byref(lay)))
    hb = PackedHostBatch.__new__(PackedHostBatch)
    hb.offsets = {n: getattr(lay, n) for n in ("node_ptr", "bond_ptr", "bond_begin", "bond_end", "feat", "targets", "peak_ptr",
                                               "peak_mz", "peak_inten") if getattr(lay, n) >= 0}
    hb.nbytes, hb.buf, hb.mz_is_f64 = int(lay.nbytes), buf, int(lay.mz_is_f64)
    hb.num_graphs, hb.num_nodes, hb.num_edges, hb.feat_dim = lay.num_graphs, lay.num_nodes, lay.num_edges, lay.feat_dim
    hb.has_targets, hb.has_peaks = lay.targets >= 0, lay.peak_ptr >= 0
    if packer.events[k] is None:
        packer.events[k] = torch.cuda.Event()
    hb._ring_event = packer.events[k]
    return hb


# ------------------------------------------------------------------------------------------
# configs[2] and configs[4] on one GPU: secondary numbers carried by the N=1 line
# ------------------------------------------------------------------------------------------
def infer_bench(args, dev, n_mols, batch=4096, with_stages=True, dump=None, steps=None, warmup=None):
    """BASELINE configs[2]: batched eval-mode prediction over n_mols resident molecules, by default one pass (steps=None)
    after 3 warm-up batches; `steps` batches run through a seeded permutation of the set, wrapping around it.
    dump: directory for the spectra of the last timed batch (dump_outputs)."""
    import torch
    from eims_b200.engine import DeviceDataset, FlatParams, ModelDims, Plan
    from eims_b200.synth import synth_molecules
    table = synth_molecules(n_mols, max_atoms=MAX_ATOMS, seed=1234)
    ds = DeviceDataset(table, None, dev)
    d = ModelDims(F0, H, L, M, "combined", DROPOUT)
    plan = Plan(d, batch, batch * MAX_ATOMS, 2 * (batch * MAX_ATOMS + 3 * batch), dev)
    fp = FlatParams(d, dev)
    init_weights(fp, d)
    per_pass = n_mols // batch
    if per_pass == 0:
        raise SystemExit(f"--workload infer: {n_mols} molecules are fewer than one batch of {batch}")
    n_batches = per_pass if steps is None else steps
    warmup = 3 if warmup is None else warmup
    ids = lambda i: perm[i % per_pass * batch:(i % per_pass + 1) * batch]
    perm_h = np.random.default_rng(5).permutation(n_mols).astype(np.int32)
    perm = torch.from_numpy(perm_h).to(dev)
    out = torch.empty(batch, M, device=dev)
    for i in range(warmup):
        plan.infer_batch(ds, ids(i), fp, out)
    plan.check()
    torch.cuda.synchronize()
    sampler = ClockSampler(dev.index or 0)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n_batches):
        plan.infer_batch(ds, ids(i), fp, out)
    e1.record()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1)
    if dump:
        dump_outputs(dump, {"spectra": out})
    res = {"metric": "gcn_eims_infer_molecules_per_sec", "value": n_batches * batch / (ms * 1e-3), "unit": UNIT, "ms_per_batch": ms / n_batches,
           "batches": n_batches, "warmup": warmup, "batch": batch, "resident_molecules": n_mols, "clocks": clocks,
           "workload": f"BASELINE configs[2]: inference-only spectrum prediction for {n_mols} synthetic molecules (<=64 heavy atoms), batch {batch}, single B200; "
                       + ("one pass over the resident set" if steps is None else f"{n_batches} batches through a seeded permutation of the resident set")
                       + ", spectra written to HBM"}
    if with_stages:
        plan.profile(True)
        n_prof = 5
        Ns, Es = [], []
        for j in range(n_prof):
            n_, e_ = ds.batch_counts(perm_h[j * batch:(j + 1) * batch])
            Ns.append(n_)
            Es.append(e_)
            plan.infer_batch(ds, perm[j * batch:(j + 1) * batch], fp, out)
        prof, _ = plan.profile_read()
        plan.profile(False)
        work = stage_work(float(np.mean(Ns)), float(np.mean(Es)), batch, fp.numel, H, L)
        work["bn_stats"] = ("hbm", L * 6 * H * 4)   # eval mode: running buffers -> scale / shift
        work["elementwise"] = ("hbm", 8 * batch * M)  # the sigmoid
        st = stage_report(prof, work, n_prof, peaks())
        res["top_stages"] = {k: st[k] for k in sorted(st, key=lambda n: -st[n]["ms_per_step"])[:3]}
        res["stages"] = st
    return res


def extra_workloads(args, dev):
    """Time-capped secondary measurements for the driver-visible N=1 line (VERDICT r1 item 7)."""
    import torch
    out = {}
    t0 = time.perf_counter()
    try:
        r = infer_bench(args, dev, 1_000_000)
        r.pop("stages", None)
        out["infer"] = r
    except Exception as exc:
        out["infer"] = {"error": f"{type(exc).__name__}: {str(exc)[:200]}"}
    torch.cuda.empty_cache()
    try:
        sub = argparse.Namespace(**vars(args))
        sub.molecules, sub.targets = 0, "dense"
        tb = TrainBench(sub, "wide", 1, 0, dev)
        Kw, Ww = 20, 3
        ids_h = make_ids("rank_strided_uniform", tb.sizes, 1, 0, tb.batch, Ww + Kw, seed=5)
        ids_d = torch.from_numpy(ids_h).to(dev)
        for i in range(2):
            tb.eager_step(ids_d[i], ids_d[i + 1])
        tb.try_capture(ids_d[2])
        for i in range(2, Ww):
            tb.step(ids_d[i], ids_d[i + 1])
        tb.flush()
        ms, per, clocks = tb.timed(ids_d, Ww, Kw, with_sampler=True)
        _, st = stage_pass(tb, ids_h, ids_d, 5)
        out["wide"] = {"metric": METRIC, "value": Kw * tb.batch / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / Kw, "steps": Kw,
                       "clocks": clocks, "launch_mode": tb.graph_note, "workload": workload_config(1, "wide")["workload"],
                       "top_stages": {k: st[k] for k in sorted(st, key=lambda n: -st[n]["ms_per_step"])[:3]}}
        del tb
    except Exception as exc:
        out["wide"] = {"error": f"{type(exc).__name__}: {str(exc)[:200]}"}
    out["seconds"] = round(time.perf_counter() - t0, 1)
    return out


def init_weights(fp, d):
    """Reference initial distributions (GraphConv xavier-uniform / zero bias; nn.Linear
    U(+-1/sqrt(fan_in)); norm layers 1/0) from a NumPy stream - same on every rank."""
    import math
    import torch
    rng = np.random.Generator(np.random.PCG64(0))
    with torch.no_grad():
        for name, t in fp.named_params().items():
            if name.startswith("gcn_layers") and name.endswith("weight"):
                b = math.sqrt(6.0 / (t.shape[0] + t.shape[1]))
                t.copy_(torch.from_numpy(rng.uniform(-b, b, size=tuple(t.shape)).astype(np.float32)))
            elif name.startswith("spectrum_predictor") and int(name.split(".")[1]) in (0, 4, 8):
                fan_in = dict(fp.spec)[name.rsplit(".", 1)[0] + ".weight"][1]
                b = 1.0 / math.sqrt(fan_in)
                t.copy_(torch.from_numpy(rng.uniform(-b, b, size=tuple(t.shape)).astype(np.float32)))
            elif name.endswith("weight"):
                t.fill_(1.0)
            else:
                t.zero_()


def _claim_stdout():
    """Route everything libraries print on fd 1 (NCCL's version banner, ...) to stderr and keep
    the real stdout for the ONE JSON line the driver parses."""
    global print
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    import builtins

    def _print(*args, **kw):
        kw.setdefault("file", real)
        kw["flush"] = True
        builtins.print(*args, **kw)

    print = _print


def run_infer(args):
    import torch
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    r = infer_bench(args, dev, args.molecules or 1_000_000, dump=args.dump_outputs, steps=args.steps, warmup=args.warmup)
    print(json.dumps({"metric": r["metric"], "value": r["value"], "unit": UNIT, "n_gpus": 1, "steps": r["batches"], "warmup": r["warmup"],
                      "ms_per_step": r["ms_per_batch"], "higher_is_better": True, "dtype": "f32", "data": "synthetic", "clocks": r["clocks"],
                      "config": {"workload": r["workload"], "batch_per_gpu": r["batch"], "hidden_dim": H, "num_gcn_layers": L, "max_mz": M,
                                 "resident_molecules": r["resident_molecules"]}, "stages": r.get("stages")}))


if __name__ == "__main__":
    _claim_stdout()
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    elif a.workload == "infer":
        run_infer(a)
    else:
        run_ours(a)
