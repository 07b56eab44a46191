"""Cost of integrated-gradients attribution of every molecule's top-k peaks at the inference shape: hidden 256, 3 layers,
1000 bins, combined pooling, synthetic molecules of <= 64 atoms, k = 5 peaks and S = 32 path points, 4096 replica graphs
(819 molecules x 5) per pass.  Times on the same molecules, with CUDA events,
    new:  one eims_attribute_peaks call per pass (data-only eval backward)
    loop: the same integrated gradients through the earlier API - per path point a batch build, a0 scaled by alpha,
          an eval eims_forward and eims_backward_feat with a dense one-hot dprob
checks that the two agree, and prints one JSON line: (molecule, peak) pairs/s and ms per pass of both, the ratio,
per-stage device time of one pass of each (eims_plan_profile), the GPU's name and power limit.

    python tools/attribution_time.py [--passes 3] [--warmup 1] [--out DIR]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "computational-chemistry-ai_b200"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from eims_b200.engine import DeviceDataset, FlatParams, ModelDims, Plan  # noqa: E402
from eims_b200.synth import MolTable, synth_molecules  # noqa: E402
from feature_grad_time import gpu_info  # noqa: E402


def replicate(t: MolTable, k: int) -> MolTable:
    mols = [t.mol(g) for g in range(t.num_mols) for _ in range(k)]
    ptr = lambda v: np.concatenate([[0], np.cumsum(v)]).astype(np.int64)
    return MolTable(ptr([len(m[0]) for m in mols]), ptr([len(m[1]) for m in mols]),
                    np.concatenate([m[0] for m in mols]).astype(np.float32),
                    np.concatenate([m[1] for m in mols]).astype(np.int32), np.concatenate([m[2] for m in mols]).astype(np.int32))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--passes", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--k", type=int, default=5)
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--replicas", type=int, default=4096)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = "cuda:0"
    k, S = args.k, args.steps
    n = args.replicas // k
    d = ModelDims(6, 256, 3, 1000, "combined", 0.2)
    fp = FlatParams(d, dev)
    torch.manual_seed(0)
    with torch.no_grad():
        fp.params.normal_(0, 0.05)
        for name, t in fp.named_params().items():
            if name.startswith("batch_norms") and name.endswith("weight"):
                t.fill_(1.0)
        fp.bn_running[:, 0].normal_(0, 0.3)
        fp.bn_running[:, 1].uniform_(0.5, 2.0)
    tables = [replicate(synth_molecules(n, max_atoms=64, seed=100 + p), k) for p in range(args.passes)]
    B = tables[0].num_mols
    Nc = max(int(t.node_ptr[-1]) for t in tables)
    Ec = max(int(2 * t.bond_ptr[-1]) for t in tables)
    plan = Plan(d, B, Nc, Ec, dev)
    sets = [DeviceDataset(t, None, dev) for t in tables]
    F = d.node_feat_dim
    alphas = [float(np.float32(np.float32(s + 0.5) / np.float32(S))) for s in range(S)]

    def new_pass(ds):
        plan.batch_build(ds, None, B)
        N = int(ds.host_num_atoms.sum())
        return plan.attribute_peaks(fp, k, S, B, N)

    def loop_pass(ds, bins):
        N = int(ds.host_num_atoms.sum())
        dprob = torch.zeros(B, d.max_mz, device=dev)
        dprob[torch.arange(B, device=dev), bins.long()] = 1.0
        acc = torch.zeros(N, F, device=dev)
        dfeat = torch.empty(N, F, device=dev)
        for a in alphas:
            plan.batch_build(ds, None, B)
            plan.buffer("a0")[: N * F].mul_(a)
            plan.forward(fp, False)
            plan.backward_feat(fp, dprob, dfeat)
            acc.add_(dfeat, alpha=1.0 / S)
        return acc * ds.feat[: N * F].view(N, F)

    # warm-up, and the agreement check on every pass's molecules
    worst = 0.0
    for ds in sets[: max(1, args.warmup)] + sets:
        bins, _, _, ig = new_pass(ds)
        ref = loop_pass(ds, bins)
        scale = torch.segment_reduce(ref.abs().amax(1).cpu(), "max", lengths=torch.as_tensor(ds.host_num_atoms))
        err = torch.segment_reduce((ig - ref).abs().amax(1).cpu(), "max", lengths=torch.as_tensor(ds.host_num_atoms))
        worst = max(worst, float((err / scale.clamp_min(1e-30)).max()))
    torch.cuda.synchronize()

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for ds in sets:
            fn(ds)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / len(sets)

    bins_of = [new_pass(ds)[0].clone() for ds in sets]
    times = {"new": [], "loop": []}
    for _ in range(2):   # alternate the two, twice
        times["new"].append(timed(new_pass))
        it = iter(bins_of)
        times["loop"].append(timed(lambda ds: loop_pass(ds, next(it))))
    ms_new, ms_loop = min(times["new"]), min(times["loop"])

    def stages(fn):
        plan.profile(True)
        fn()
        st, launches = plan.profile_read()
        plan.profile(False)
        return {kk: round(v[0], 4) for kk, v in st.items() if v[1]}, launches
    st_new, l_new = stages(lambda: new_pass(sets[0]))
    st_loop, l_loop = stages(lambda: loop_pass(sets[0], bins_of[0]))
    pairs = n * k
    rec = dict(workload=dict(hidden=256, layers=3, max_mz=1000, pooling="combined", max_atoms=64, k=k, steps=S,
                             replicas_per_pass=B, molecules_per_pass=n, passes=len(sets)),
               ms_per_pass=dict(new=round(ms_new, 3), loop=round(ms_loop, 3)),
               pairs_per_s=dict(new=round(pairs / ms_new * 1e3, 1), loop=round(pairs / ms_loop * 1e3, 1)),
               speedup=round(ms_loop / ms_new, 3), all_times_ms=times, ig_max_rel_err_vs_loop=worst,
               stage_ms_one_pass=dict(new=st_new, loop=st_loop), launches_one_pass=dict(new=l_new, loop=l_loop), **gpu_info())
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "attribution_time.json"), "w") as fh:
            fh.write(line + "\n")
    assert worst < 1e-5, worst


if __name__ == "__main__":
    main()
