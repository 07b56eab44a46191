"""Cost of per-atom attribution at the inference shape: batches of 4096 molecules, hidden 256, 3 layers, 1000 bins
(BASELINE configs[2]).  Times, with CUDA events over many batches of one resident data set,
    A: eval forward + sigmoid                                   (eims_forward + eims_sigmoid)
    B: A + eims_backward_feat with the atom-feature gradient    (one backward over the whole batch)
after the batch build, and prints one JSON line: ms per batch, molecules/s, the GPU's name and power limit.

    python tools/feature_grad_time.py [--batches 50] [--warmup 5]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "computational-chemistry-ai_b200"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from eims_b200.engine import DeviceDataset, FlatParams, ModelDims, Plan  # noqa: E402
from eims_b200.synth import synth_molecules  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return dict(gpu=name, power_limit=power, sm_max_clock=clock)
    except Exception:
        return dict(gpu=torch.cuda.get_device_name(0), power_limit="unknown", sm_max_clock="unknown")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=4096)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device (B200)")
    dev = "cuda:0"
    d = ModelDims(node_feat_dim=6, hidden_dim=256, num_gcn_layers=3, max_mz=1000, pooling="combined", dropout=0.2)
    B, n_sets = args.batch, 8
    table = synth_molecules(B * n_sets, seed=5)
    ds = DeviceDataset(table, None, dev)
    ids = [torch.arange(k * B, (k + 1) * B, dtype=torch.int32, device=dev) for k in range(n_sets)]
    counts = [ds.batch_counts(np.arange(k * B, (k + 1) * B)) for k in range(n_sets)]
    plan = Plan(d, B, max(c[0] for c in counts), max(c[1] for c in counts), dev)
    fp = FlatParams(d, dev)
    g = torch.Generator(device="cpu").manual_seed(1)
    fp.params.copy_((torch.rand(fp.numel, generator=g) - 0.5).mul_(0.1))
    fp.bn_running[:, 1].uniform_(0.5, 2.0)
    dprob = torch.zeros(B, d.max_mz, device=dev)
    dprob[:, 41] = 1.0                                        # attribution of one bin
    dfeat = torch.empty(max(c[0] for c in counts), d.node_feat_dim, device=dev)

    def run(k, backward):
        plan.batch_build(ds, ids[k % n_sets], B)
        plan.forward(fp, False)
        plan.sigmoid()
        if backward:
            plan.backward_feat(fp, dprob, dfeat)

    res = {}
    for backward in (False, True, False, True):              # alternated: A, B, A, B; the second pair is reported
        for k in range(args.warmup):
            run(k, backward)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for k in range(args.batches):
            run(k, backward)
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / args.batches
        res["forward_sigmoid_backward_feat" if backward else "forward_sigmoid"] = dict(
            ms_per_batch=round(ms, 4), molecules_per_s=round(B / ms * 1e3, 1))
    plan.check()
    assert bool(torch.isfinite(dfeat[:counts[(args.batches - 1) % n_sets][0]]).all())
    res["backward_over_forward"] = round(res["forward_sigmoid_backward_feat"]["ms_per_batch"] / res["forward_sigmoid"]["ms_per_batch"], 3)
    res.update(batch=B, hidden=256, layers=3, max_mz=1000, batches=args.batches, **gpu_info(),
               note="batch build (K1) included in both; same resident set, cycled over 8 batches")
    print(json.dumps(res))


if __name__ == "__main__":
    main()
