#!/usr/bin/env python
"""Parity and back-to-back timing of the planes GEMM (csrc/gemm_tma.cu) through the C ABI (diagnostic, on a B200):
every GraphConv product of BASELINE configs[1] - forward, data gradient, weight gradient, and the grouped
data + weight gradient launch - against an fp64 matmul and against eims_gemm.
    python tools/gemm_planes_check.py [--atoms 16900] [--hidden 256] [--no-time]"""
import argparse
import ctypes as C
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "computational-chemistry-ai_b200"))
from eims_b200 import _lib  # noqa: E402
from eims_b200._lib import GemmProblem, check, ptr  # noqa: E402


def problem(A, a_mn, B, b_mn, Cm, M, N, K, m_dev=None, k_dev=None, rs=None, bias=None, relu=0, acc=0):
    return GemmProblem(A.data_ptr(), A.shape[1], a_mn, B.data_ptr(), B.shape[1], b_mn, Cm.data_ptr(), Cm.shape[1], M, N, K,
                       m_dev.data_ptr() if m_dev is not None else None, k_dev.data_ptr() if k_dev is not None else None,
                       rs.data_ptr() if rs is not None else None, bias.data_ptr() if bias is not None else None, relu, acc)


class Runner:
    def __init__(self):
        self.lib = _lib.load()
        self.st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        self.scratch = None

    def run(self, p0, p1=None):
        need = self.lib.eims_gemm_planes_scratch_bytes(C.byref(p0), C.byref(p1) if p1 is not None else None)
        if self.scratch is None or self.scratch.numel() < need:
            self.scratch = torch.empty(need, dtype=torch.uint8, device="cuda")
        check(self.lib.eims_gemm_planes(C.byref(p0), C.byref(p1) if p1 is not None else None, ptr(self.scratch), self.scratch.numel(), self.st))

    def old(self, p):
        check(self.lib.eims_gemm(0, C.c_void_p(p.A), p.lda, p.a_mn_major, C.c_void_p(p.B), p.ldb, p.b_mn_major, C.c_void_p(p.C), p.ldc,
                                 p.M, p.N, p.K, C.c_void_p(p.m_dev) if p.m_dev else None, C.c_void_p(p.k_dev) if p.k_dev else None,
                                 C.c_void_p(p.row_scale) if p.row_scale else None, C.c_void_p(p.bias) if p.bias else None, p.relu,
                                 p.accumulate, self.st))


def rel(a, b):
    return float((a.double() - b).abs().max() / b.abs().max().clamp_min(1e-30))


def timeit(fn, n=200):
    for _ in range(20):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1e3


def planes_kernel_us(fn, n=200):
    """Mean time of the gemm_planes_kernel launches of one call of fn, from the profiler's kernel records: the GEMM alone,
    without the split kernels eims_gemm_planes launches in front of it."""
    for _ in range(20):
        fn()
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            fn()
        torch.cuda.synchronize()
    return sum(e.device_time_total for e in prof.key_averages() if "gemm_planes_kernel" in e.key) / n


def sweep(R, Nl, Nc, H):
    dev = "cuda"
    nd = torch.tensor([Nl], dtype=torch.int32, device=dev)
    for K in (32, 64, 128, 256, 512):
        X = torch.randn(Nc, K, device=dev)
        W = torch.randn(K, H, device=dev)
        Z = torch.zeros(Nc, H, device=dev)
        p = problem(X, 0, W, 1, Z, Nc, H, K, m_dev=nd)
        us = planes_kernel_us(lambda: R.run(p))
        old = timeit(lambda: R.old(p))
        print(f"K={K:4d}  planes {us:7.2f} us   in-kernel split {old:7.2f} us")
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--atoms", type=int, default=16900)
    ap.add_argument("--cap", type=int, default=32768)
    ap.add_argument("--hidden", type=int, default=256)
    ap.add_argument("--no-time", action="store_true")
    ap.add_argument("--sweep", action="store_true", help="forward product at K = 32 .. 512: slope per k-block and fixed cost")
    a = ap.parse_args()
    torch.manual_seed(0)
    dev = "cuda"
    Nl, Nc, H = a.atoms, a.cap, a.hidden
    R = Runner()
    if a.sweep:
        return sweep(R, Nl, Nc, H)
    ok = True
    X = torch.randn(Nc, H, device=dev)                 # activations (a_l)
    Q = torch.randn(Nc, H, device=dev) * 0.01          # output gradient (q)
    X[Nl:] = 0                                         # the producers zero the rows behind the live range up to a multiple of 32
    Q[Nl:] = 0
    W = torch.randn(H, H, device=dev) / H ** 0.5       # GraphConv weight [in, out]
    rs = torch.rand(Nc, device=dev) + 0.5
    bias = torch.randn(H, device=dev)
    nd = torch.tensor([Nl], dtype=torch.int32, device=dev)
    canary = 777.0
    # forward: z = relu((a W) * c + b)
    Z = torch.full((Nc, H), canary, device=dev)
    pf = problem(X, 0, W, 1, Z, Nc, H, H, m_dev=nd, rs=rs, bias=bias, relu=1)
    R.run(pf)
    torch.cuda.synchronize()
    ref = torch.relu((X[:Nl].double() @ W.double()) * rs[:Nl, None].double() + bias.double())
    e = rel(Z[:Nl], ref)
    intact = bool((Z[Nl:] == canary).all())
    print(f"forward  rel err {e:.2e}  rows behind the live range untouched: {intact}")
    ok &= e < 2e-5 and intact
    # data gradient: da = q W^T
    DA = torch.full((Nc, H), canary, device=dev)
    pd = problem(Q, 0, W, 0, DA, Nc, H, H, m_dev=nd)
    R.run(pd)
    torch.cuda.synchronize()
    ref = Q[:Nl].double() @ W.double().T
    e = rel(DA[:Nl], ref)
    print(f"dgrad    rel err {e:.2e}  untouched: {bool((DA[Nl:] == canary).all())}")
    ok &= e < 2e-5
    # weight gradient: dW = a^T q (split-K over the atoms, added into dW)
    DW = torch.zeros(H, H, device=dev)
    pw = problem(X, 1, Q, 1, DW, H, H, Nc, k_dev=nd, acc=1)
    R.run(pw)
    torch.cuda.synchronize()
    refw = X[:Nl].double().T @ Q[:Nl].double()
    e = rel(DW, refw)
    print(f"wgrad    rel err {e:.2e}")
    ok &= e < 2e-5
    # grouped launch
    DA.fill_(canary)
    DW.zero_()
    R.run(pd, pw)
    torch.cuda.synchronize()
    e1, e2 = rel(DA[:Nl], ref), rel(DW, refw)
    print(f"grouped  dgrad {e1:.2e}  wgrad {e2:.2e}  untouched: {bool((DA[Nl:] == canary).all())}")
    ok &= e1 < 2e-5 and e2 < 2e-5
    # against the in-kernel split of gemm_tc.cu
    Z2 = torch.zeros(Nc, H, device=dev)
    po = problem(X, 0, W, 1, Z2, Nc, H, H, m_dev=nd, rs=rs, bias=bias, relu=1)
    R.old(po)
    torch.cuda.synchronize()
    print(f"forward  planes vs in-kernel split: max abs diff {float((Z[:Nl] - Z2[:Nl]).abs().max()):.2e}")
    print("PARITY", "OK" if ok else "FAILED")
    if a.no_time or not ok:
        return 0 if ok else 1

    lib, st = R.lib, R.st
    # time the GEMM launch alone (profiler kernel time) and back to back with the split kernels in front of it
    for name, p0, p1, flops in (("forward", pf, None, 2.0 * Nl * H * H), ("dgrad", pd, None, 2.0 * Nl * H * H),
                                ("wgrad", pw, None, 2.0 * Nl * H * H), ("dgrad+wgrad", pd, pw, 4.0 * Nl * H * H)):
        call = lambda: check(lib.eims_gemm_planes(C.byref(p0), C.byref(p1) if p1 is not None else None, ptr(R.scratch), R.scratch.numel(), st))  # noqa: E731
        split = timeit(call, 50)
        us = planes_kernel_us(call)
        if p1 is None:
            old = timeit(lambda: R.old(p0))
        else:
            old = float("nan")
        print(f"{name:12s} planes {us:7.2f} us ({flops / us * 1e-6:6.1f} TFLOP/s)   with the splits {split:7.2f} us   in-kernel split {old:7.2f} us")
    return 0


if __name__ == "__main__":
    sys.exit(main())
