#!/usr/bin/env python
"""Pipeline timeline of the planes GEMM (diagnostic, on a B200): -DEIMS_GEMM_TRACE build, one launch of each GraphConv
product of BASELINE configs[1], SM-clock stamps of the roles of CTAs 0, 1 and 7.   python tools/gemm_planes_trace.py [--no-build]"""
import ctypes as C
import importlib.util
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "computational-chemistry-ai_b200"))
spec = importlib.util.spec_from_file_location("b", os.path.join(ROOT, "computational-chemistry-ai_b200", "build.py"))
b = importlib.util.module_from_spec(spec)
spec.loader.exec_module(b)
path = b.OUT.replace(".so", "_trace.so") if "--no-build" in sys.argv else b.build_variant("trace", ["-DEIMS_GEMM_TRACE"])
from eims_b200 import _lib  # noqa: E402
_lib.LIB_PATH = path
import torch  # noqa: E402
sys.path.insert(0, os.path.join(ROOT, "tools"))
from gemm_planes_check import Runner, problem  # noqa: E402


def main():
    dev = "cuda"
    Nl, Nc, H = 16900, 32768, 256
    R = Runner()
    rd = R.lib.eims_debug_trace_read_planes
    rd.restype, rd.argtypes = C.c_int, [C.c_void_p, C.c_int]
    X = torch.randn(Nc, H, device=dev)
    Q = torch.randn(Nc, H, device=dev)
    X[Nl:] = 0
    Q[Nl:] = 0
    W = torch.randn(H, H, device=dev)
    nd = torch.tensor([Nl], dtype=torch.int32, device=dev)
    Z = torch.zeros(Nc, H, device=dev)
    DW = torch.zeros(H, H, device=dev)
    pf = problem(X, 0, W, 1, Z, Nc, H, H, m_dev=nd)
    pd = problem(Q, 0, W, 0, Z, Nc, H, H, m_dev=nd)
    pw = problem(X, 1, Q, 1, DW, H, H, Nc, k_dev=nd, acc=1)
    names = {0: "start", 1: "prologue done", 2: "pdl wait done", 3: "roles done", 4: "end"}
    inames = ["copy: item begins", "mma: accumulator free", "mma: first k-block landed", "mma: last k-block landed",
              "epi: waits", "epi: accumulator complete", "epi: tile stored"]
    buf = (C.c_ulonglong * 512)()
    for title, p0, p1 in (("forward", pf, None), ("wgrad", pw, None), ("dgrad + wgrad", pd, pw)):
        for _ in range(3):
            R.run(p0, p1)
            torch.cuda.synchronize()
        assert rd(buf, 512) == 0   # reset
        R.run(p0, p1)
        torch.cuda.synchronize()
        assert rd(buf, 512) == 0
        t = np.array(buf[:], dtype=np.int64).reshape(8, 64)
        print(f"==== {title}")
        for c in (0, 1, 7):
            base = t[c, 0]
            ev = [(t[c, k] - base, names[k]) for k in names if t[c, k]]
            for i in range(6):
                for k, nm in enumerate(inames):
                    v = t[c, 8 + i * 8 + k]
                    if v:
                        ev.append((v - base, f"item {i} {nm}"))
            for cb in range(4):
                for k, nm in enumerate(("before tcgen05.ld", "after tcgen05.ld", "patch written", "block stored")):
                    v = t[c, 40 + cb * 4 + k]
                    if v:
                        ev.append((v - base, f"item 0 epi block {cb}: {nm}"))
            print(f"--- CTA {c} (cycles since its start)")
            for v, nm in sorted(ev):
                print(f"{v:8d}  {nm}")


if __name__ == "__main__":
    main()
