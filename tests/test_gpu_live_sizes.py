"""The GEMMs and the training step at every live size a capacity-sized plan can be handed.

A plan picks its GEMM kernels from its capacity, and every kernel then reads the live sizes from the device: the
persistent kernels deal tiles and split-K k-blocks out from them (`pg::make_sched`, gemm_persist.cuh), the
in-kernel-split kernel kills the split-K slices and tiles past them, and the fused BatchNorm statistics count only
live tiles.  So the last batch of an epoch, or of a prediction, runs through the big-plan kernels at a small, ragged
size.

1. GEMMs through the C ABI, bit for bit: operands are integers in [-2, 2], row scales 0.5 / 1 / 2, biases integers,
   so every product and partial sum is an integer far below 2^24 - the 3xTF32 split leaves lo = 0 and fp32
   accumulation and atomics are exact - and every path must equal a float64 matmul after the cast to fp32, whatever
   its summation order.  An all-ones probe turns each output into the count of live k-rows; a mismatch is reported
   in k-blocks.  Rows past the live M of a store problem are NaN; the k-rows of a split-K problem are zero up to the
   next multiple of 32 past the live K (what the producers guarantee) and NaN beyond, so one k-block read too many
   shows as NaN; C has canary rows behind the live rows and integer start values where it is accumulated into.
   The live sizes are derived from the tile constants of the sources, and the host probe of test_gemm_schedule shows
   that they reach every branch of the planes kernel's deal.

2. Whole training steps (forward, MSE loss, backward) and eval forwards on one capacity-sized plan per row of
   test_gpu_dispatch (planes, molecule tiles, K1 prescan, persistent GEMM with fused BatchNorm statistics, forced deep
   planes) and the benchmark's training shape, over a descending then ascending sequence of live batches, held to the
   fp64 oracle with test_gpu_dispatch.oracle_check.  The plan is poisoned at creation and before every second batch,
   so half the batches meet NaN where nothing was written and half meet a stale batch."""
import ctypes as C
import json
import os
import re

import pytest
import torch

from eims_b200 import _lib
from eims_b200._lib import GemmProblem, check, ptr
from eims_b200.engine import DeviceDataset, FlatParams, ModelDims, make_step
from eims_b200.synth import dense_spectra, synth_peaks
from oracle import gcn_oracle as O
from test_gemm_schedule import build_probe, probe_flags, source_constants
from test_gpu_dispatch import (ROWS, dropout_masks, gpu_step, make_plan, odims, oracle_check, poison,
                               random_running_stats, rel_err)
from test_gpu_graph_shapes import K1_SCAN_CHUNK, chain, mol_table, profiled, ring, worst_ratio

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "computational-chemistry-ai_b200", "csrc")

CONST = source_constants()
BM, BN, BK, KMAX = CONST["BM"], CONST["BN"], CONST["BK"], CONST["kMaxKbPerItem"]
SMS = 148


def _grep(path, pattern):
    m = re.search(pattern, open(os.path.join(CSRC, path)).read())
    assert m, (path, pattern)
    return int(m.group(1))


PAIR = _grep("gemm_tma.cu", r"constexpr int PAIR = (\d+);")
ITEM_OVH = _grep("gemm_tma.cu", r"constexpr int kItemOverhead = (\d+);")
MAX_KB_DEEP = _grep("gemm_tma.cu", r"constexpr int kMaxKbDeep = (\d+);")
G_PAIRS = SMS // PAIR
assert _grep("gemm_tc.cu", r"launch_pdl\(gemm_3xtf32_persistent_kernel, dim3\((\d+)\)") == SMS


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ceil_div(a, b):
    return -(-a // b)


def around(*xs):
    return [x + e for x in xs for e in (-1, 0, 1)]


def clip(sizes, cap):
    return sorted({s for s in sizes if 1 <= s <= cap})


def m_sizes(TM, cap, tiles_per_row=1, G=None):
    """Live rows of a store problem: the smallest, the warp edges, one and two output tiles, where the store tiles
    number G - 1, G, G + 1 and 2G + 1, and the capacity."""
    s = [1, 2, 31, 32, 33] + around(TM, 2 * TM) + [cap - 1, cap]
    if G is not None:
        for tiles in (G - 1, G, G + 1, 2 * G + 1):
            if tiles % tiles_per_row == 0:
                s += around(tiles // tiles_per_row * TM)
    return clip(s, cap)


def k_sizes(cap, G=None, units_per_kb=1):
    """Live K of a split-K problem: the warp and k-block edges, one item's limit of k-blocks, where the split-K units
    number G - 1, G and G + 1, and the capacity."""
    s = [1, 2, 31, 32, 33] + around(KMAX * BK, 2 * KMAX * BK) + [cap - 1, cap]
    if G is not None:
        for units in (G - 1, G, G + 1):
            if units % units_per_kb == 0:
                s += around(units // units_per_kb * BK)
    return clip(s, cap)


# ------------------------------------------------------------------------------------------------ exact operands
def int_values(shape, gen, kind):
    if kind == "ones":
        return torch.ones(shape, dtype=torch.float64, device=DEV)
    return torch.randint(-2, 3, shape, generator=gen, device=DEV).double()


class Operands:
    """A logical [M, K] and B [K, N] (float64, exact integers) at capacity, stored in the requested orders with the
    poison of the problem's live sizes."""

    def __init__(self, Mc, N, Kc, a_mn, b_mn, gen, kind):
        self.A = int_values((Mc, Kc), gen, kind)
        self.B = int_values((Kc, N), gen, kind)
        self.a_mn, self.b_mn = a_mn, b_mn

    def stored(self, live_m=None, live_k=None):
        A, B = self.A.clone(), self.B.clone()
        if live_m is not None:
            A[live_m:] = float("nan")                  # rows past the live M
        if live_k is not None:
            pad = ceil_div(live_k, BK) * BK
            A[:, live_k:pad] = 0.0                     # zero up to the next k-block edge, as the producers leave it
            B[live_k:pad] = 0.0
            A[:, pad:] = float("nan")
            B[pad:] = float("nan")
        As = (A.t() if self.a_mn else A).contiguous().float()
        Bs = (B if self.b_mn else B.t()).contiguous().float()
        return As, Bs

    def reference(self, m, k):
        return self.A[:m, :k] @ self.B[:k]


def epilogue_inputs(M, N, gen, rs_on, bias_on):
    rs = (torch.tensor([0.5, 1.0, 2.0], device=DEV)[torch.randint(0, 3, (M,), generator=gen, device=DEV)] if rs_on else None)
    bias = torch.randint(-3, 4, (N,), generator=gen, device=DEV).float() if bias_on else None
    return rs, bias


def expected(ref, rs, bias, relu, m):
    out = ref.clone()
    if rs is not None:
        out = out * rs[:m, None].double()
    if bias is not None:
        out = out + bias.double()
    if relu:
        out = out.clamp_min(0.0)
    return out.float()


def compare(tag, got, want, kind, k_live=None):
    """Bit-for-bit comparison; on a mismatch, where and (all-ones probe) by how many k-blocks."""
    bad = ~((got == want) | (torch.isnan(got) & torch.isnan(want)))
    if not bool(bad.any()):
        return None
    idx = bad.nonzero()[0].tolist()
    msg = (f"{tag}: {int(bad.sum())} of {bad.numel()} elements differ, first at {idx}: got {float(got[tuple(idx)])}, "
           f"want {float(want[tuple(idx)])}, NaN {int(torch.isnan(got).sum())}")
    if kind == "ones" and k_live:
        d = (got.double() - want.double())[bad]
        d = d[torch.isfinite(d)]
        if d.numel():
            msg += f"; off by {float(d.min()) / BK:+.3f} .. {float(d.max()) / BK:+.3f} k-blocks"
    return msg


# ------------------------------------------------------------------------------------------------ eims_gemm
FORMS = {0: "store", 1: "split-K", 2: "store, K split, launcher zeroes C", 3: "store, K split, caller zeroes C"}


def gemm_case(backend, Mc, N, Kc, a_mn, b_mn, form, live, kind, seed):
    """One eims_gemm launch at one live size: store forms (0, 2, 3) take the live M from m_dev, the split-K form (1)
    the live K from k_dev.  Returns the failures found."""
    gen = torch.Generator(device=DEV).manual_seed(seed)
    ops = Operands(Mc, N, Kc, a_mn, b_mn, gen, kind)
    split = form == 1
    live_m, live_k = (None, live) if split else (live, None)
    As, Bs = ops.stored(live_m, live_k)
    # forms 2 / 3 split K only without ReLU or row scale (a split-K partial must stay linear); form 1 likewise
    relu = form == 0
    rs, bias = epilogue_inputs(Mc, N, gen, rs_on=form in (0, 1), bias_on=True)
    canary = 777.0
    Cd = torch.full((Mc + 16, N), canary, device=DEV)
    if form == 1:
        Cd[:Mc] = torch.randint(-5, 6, (Mc, N), generator=gen, device=DEV).float()   # added into
    elif form == 3:
        Cd[:Mc] = 0.0
    start = Cd.clone()
    dev_size = torch.tensor([live], dtype=torch.int32, device=DEV)
    check(_lib.load().eims_gemm(backend, ptr(As), As.shape[1], a_mn, ptr(Bs), Bs.shape[1], b_mn, ptr(Cd), N, Mc, N, Kc,
                                None if split else ptr(dev_size), ptr(dev_size) if split else None,
                                ptr(rs) if rs is not None else None, ptr(bias) if bias is not None else None,
                                int(relu), form, stream()))
    torch.cuda.synchronize()
    m = Mc if split else live
    k = live if split else Kc
    want = expected(ops.reference(m, k), rs, bias, relu, m)
    if form == 1:
        want = (want.double() + start[:m].double()).float()
    tag = f"M {Mc} N {N} K {Kc} a_mn {a_mn} b_mn {b_mn} form {form} live {live} {kind}"
    bad = []
    e = compare(tag, Cd[:m], want, kind, k if kind == "ones" else None)
    if e:
        bad.append(e)
    rest = Cd[m:Mc]
    if form == 2:
        if not bool((rest == 0).all()):
            bad.append(f"{tag}: rows past the live M are not the zeroes of the launcher")
    elif not torch.equal(rest, start[m:Mc]):
        bad.append(f"{tag}: rows past the live M were written")
    if not bool((Cd[Mc:] == canary).all()):
        bad.append(f"{tag}: canary rows past the capacity were written")
    return bad


def run_gemm_sweep(backend, Mc, N, Kc, orders, forms, sizes_of, tmp_path, name, kinds=("int", "ones")):
    bad, n = [], 0
    for a_mn, b_mn in orders:
        for form in forms:
            for live in sizes_of(form):
                for kind in kinds:
                    bad += gemm_case(backend, Mc, N, Kc, a_mn, b_mn, form, live, kind, seed=live * 7 + form + 2 * a_mn + b_mn)
                    n += 1
    with open(tmp_path / f"live_sizes_{name}.json", "w") as fh:
        json.dump({"launches": n, "failures": bad}, fh, indent=1)
    assert not bad, bad[:8]


ALL_ORDERS = [(0, 0), (0, 1), (1, 0), (1, 1)]
TC, SIMT = _lib.GEMM_TCGEN05, _lib.GEMM_FP32_SIMT


def test_full_capacity_bit_exact():
    """First of all: tcgen05's tf32 products and fp32 accumulation are exact on these operands at full capacity."""
    bad = gemm_case(TC, 8192, 256, 512, 0, 1, 0, 8192, "int", seed=1)        # 128 x 256 in-kernel split, 64 tiles
    bad += gemm_case(TC, 512, 256, 16384, 1, 1, 1, 16384, "int", seed=2)     # split-K over 512 k-blocks
    bad += gemm_case(TC, 40960, 512, 512, 0, 1, 0, 40960, "int", seed=3)     # persistent, 640 tiles
    assert not bad, bad


def test_in_kernel_split_128_columns(tmp_path):
    """gemm_3xtf32_kernel<128, 3>: 16 x 2 tiles at capacity (too few for the 256-wide tile); all four operand
    orders; stores with the live M, split-K over a capacity-sized split count with the live K, and the split store
    forms 2 and 3 of the head's data gradients."""
    Mc, N, Kc = 2048, 256, 2048
    sizes = lambda form: k_sizes(Kc) if form == 1 else m_sizes(BM, Mc)   # noqa: E731
    run_gemm_sweep(TC, Mc, N, Kc, ALL_ORDERS, [0, 1], sizes, tmp_path, "tc128")
    # forms 2 / 3: a grid small enough to split K (<= 37 tiles, no ReLU / row scale)
    run_gemm_sweep(TC, 512, 256, 1024, [(0, 1), (1, 0)], [2, 3], lambda f: m_sizes(BM, 512), tmp_path, "tc128_split_store")


def test_in_kernel_split_256_columns(tmp_path):
    """gemm_3xtf32_kernel<256, 2>: 64 row tiles (store), and the split-K form at K >= 4096 with 74 slices from the
    capacity of which most are dead at a small live K."""
    Mc, N, Kc = 8192, 256, 512
    run_gemm_sweep(TC, Mc, N, Kc, ALL_ORDERS, [0], lambda f: m_sizes(BM, Mc), tmp_path, "tc256_store")
    Kc = 8192
    run_gemm_sweep(TC, 256, 256, Kc, ALL_ORDERS, [1], lambda f: k_sizes(Kc, G=SMS // 2), tmp_path, "tc256_splitk")


def test_persistent_kernel(tmp_path):
    """gemm_3xtf32_persistent_kernel: 320 x 2 tiles at capacity (>= 4 per SM), 148 CTAs; live M around the store
    tiles numbering G - 1 .. 2G + 1 (74 * 128 = 9472 rows at N = 512)."""
    Mc, N, Kc = 40960, 512, KMAX * BK
    sizes = m_sizes(BM, Mc, tiles_per_row=N // BN, G=SMS)
    assert 9472 in sizes and 9473 in sizes
    run_gemm_sweep(TC, Mc, N, Kc, [(0, 1), (1, 0)], [0], lambda f: sizes, tmp_path, "persistent")


def test_simt(tmp_path):
    """The fp32 SIMT GEMM at the same edges (store and split-K)."""
    Mc, N, Kc = 2048, 256, 2048
    sizes = lambda form: k_sizes(Kc) if form == 1 else m_sizes(BM, Mc)   # noqa: E731
    run_gemm_sweep(SIMT, Mc, N, Kc, [(0, 1), (1, 1)], [0, 1], sizes, tmp_path, "simt", kinds=("int",))


# ------------------------------------------------------------------------------------------------ eims_gemm_planes
def planes_problem(As, a_mn, Bs, b_mn, Cd, M, N, K, m_dev=None, k_dev=None, rs=None, bias=None, relu=0, acc=0):
    return GemmProblem(As.data_ptr(), As.shape[1], a_mn, Bs.data_ptr(), Bs.shape[1], b_mn, Cd.data_ptr(), Cd.shape[1], M, N, K,
                       m_dev.data_ptr() if m_dev is not None else None, k_dev.data_ptr() if k_dev is not None else None,
                       rs.data_ptr() if rs is not None else None, bias.data_ptr() if bias is not None else None, relu, acc)


def planes_run(p0, p1=None):
    lib = _lib.load()
    b1 = C.byref(p1) if p1 is not None else None
    need = lib.eims_gemm_planes_scratch_bytes(C.byref(p0), b1)
    scratch = torch.empty(need, dtype=torch.uint8, device=DEV)
    check(lib.eims_gemm_planes(C.byref(p0), b1, ptr(scratch), scratch.numel(), stream()))
    torch.cuda.synchronize()


def planes_grid(problems):
    """Pairs of the launch (gemm_tma.cu launch_gemm_tma): one per item at capacity, at most 148 / PAIR."""
    items = sum(ceil_div(M, BM * PAIR) * (N // BN) * (SMS if red else 1) for (red, N, M, K) in problems)
    return max(1, min(items, G_PAIRS))


def planes_case(Mc, N, Kc, live, kind, seed, grouped, store_k=None):
    """Planes kernel at one live atom count: the store problem q W^T (live rows = atoms; K = store_k or N), alone or
    grouped with the split-K weight gradient a^T q (K = atoms).  Returns (failures, probe case)."""
    gen = torch.Generator(device=DEV).manual_seed(seed)
    Ks = store_k or N
    st = Operands(Mc, N, Ks, 0, 0, gen, kind)                  # q [atoms, Ks] K-major, W as [N, Ks] (b_mn = 0)
    As, Bs = st.stored(live_m=live)
    rs, bias = epilogue_inputs(Mc, N, gen, rs_on=True, bias_on=True)
    canary = 777.0
    Cs = torch.full((Mc + 16, N), canary, device=DEV)
    nd = torch.tensor([live], dtype=torch.int32, device=DEV)
    p0 = planes_problem(As, 0, Bs, 0, Cs, Mc, N, Ks, m_dev=nd, rs=rs, bias=bias, relu=1)
    probs = [(0, N, Mc, Ks)]
    tag = f"planes M {Mc} N {N} K {Ks} live {live} {kind} {'grouped' if grouped else 'alone'}"
    bad = []
    if grouped:
        wk = Operands(N, N, Kc, 1, 1, gen, kind)                 # a^T [N, atoms] stored as a [atoms, N]; q [atoms, N]
        Aw, Bw = wk.stored(live_k=live)
        Cw = torch.full((N + 16, N), canary, device=DEV)
        Cw[:N] = torch.randint(-5, 6, (N, N), generator=gen, device=DEV).float()
        start = Cw.clone()
        wbias = torch.randint(-3, 4, (N,), generator=gen, device=DEV).float()
        p1 = planes_problem(Aw, 1, Bw, 1, Cw, N, N, Kc, k_dev=nd, bias=wbias, acc=1)
        probs.append((1, N, N, Kc))
        planes_run(p0, p1)
        want = (wk.reference(N, live) + wbias.double() + start[:N].double()).float()
        e = compare(tag + " weight gradient", Cw[:N], want, kind, live)
        if e:
            bad.append(e)
        if not bool((Cw[N:] == canary).all()):
            bad.append(f"{tag}: weight-gradient canary rows written")
    else:
        planes_run(p0)
    want = expected(st.reference(live, Ks), rs, bias, True, live)
    e = compare(tag + " store", Cs[:live], want, kind)
    if e:
        bad.append(e)
    if not bool((Cs[live:] == canary).all()):
        bad.append(f"{tag}: store rows past the live M written")
    G = planes_grid(probs)
    case = [PAIR, G, len(probs), ITEM_OVH, 0, N, live, Ks] + ([1, N, N, live] if grouped else [0, N, 0, 0])
    return bad, case


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    return build_probe(tmp_path_factory.mktemp("sched_probe_gpu"))


def planes_sweep(cases, tmp_path, name):
    bad, probe_cases = [], []
    for (Mc, N, Kc, live, grouped, store_k) in cases:
        for kind in ("int", "ones"):
            b, case = planes_case(Mc, N, Kc, live, kind, seed=live * 3 + N, grouped=grouped, store_k=store_k)
            bad += b
        probe_cases.append(case)
    with open(tmp_path / f"live_sizes_{name}.json", "w") as fh:
        json.dump({"launches": 2 * len(cases), "failures": bad}, fh, indent=1)
    assert not bad, bad[:8]
    return probe_cases


def test_planes_alone(tmp_path):
    """The store problem alone at H = 256: one 256-row tile per pair-item, 74 pairs; live rows around 74 * 256 =
    18944 and 2 * 74 + 1 tiles."""
    Mc, N = 40960, 256
    sizes = m_sizes(BM * PAIR, Mc, tiles_per_row=1, G=G_PAIRS)
    assert {18943, 18944, 18945} <= set(sizes)
    planes_sweep([(Mc, N, None, s, False, None) for s in sizes], tmp_path, "planes_alone")


def test_planes_deep_k(tmp_path):
    """Deep mode: store K = 2048 (main + correction accumulators)."""
    Mc, N, Ks = 4096, 256, MAX_KB_DEEP * BK
    planes_sweep([(Mc, N, None, s, False, Ks) for s in m_sizes(BM * PAIR, Mc)], tmp_path, "planes_deep")


def test_planes_grouped_reaches_every_branch(tmp_path, probe):
    """The grouped data + weight gradient (G = 74 pairs): the atom count is the store problem's live M and the
    split-K problem's live K.  The live sizes cover the tile and k-block edges, the store tiles at G - 1 .. 2G + 1, the
    split-K units at G - 1 .. G + 1 and 16 k-blocks; the schedule probe shows they take every branch of make_sched."""
    cases = []
    for Mc, N in ((40960, 256), (8192, 512)):
        TM = BM * PAIR
        sizes = set(m_sizes(TM, Mc, tiles_per_row=N // BN, G=G_PAIRS))
        sizes |= set(k_sizes(Mc, G=G_PAIRS, units_per_kb=ceil_div(N, TM) * (N // BN)))
        cases += [(Mc, N, Mc, s, True, None) for s in sorted(sizes)]
    probe_cases = planes_sweep(cases, tmp_path, "planes_grouped")
    flags = probe_flags(probe, probe_cases)
    assert all(f["error"] == "" and f["recompute_ok"] for f in flags), [f for f in flags if f["error"]][:4]
    assert all(f["case"][1] == G_PAIRS for f in flags)
    reached = {k: sum(f[k] for f in flags) for k in ("r_zero", "r_pos", "xhi_clamped", "u_lt_g", "multi_item", "clamp_u")}
    with open(tmp_path / "live_sizes_branches.json", "w") as fh:
        json.dump(reached, fh, indent=1)
    for k in ("r_zero", "r_pos", "xhi_clamped", "u_lt_g", "multi_item"):
        assert reached[k] > 0, (k, reached)


# ------------------------------------------------------------------------------------------------ whole steps
BENCH_D = ModelDims(6, 256, 3, 1000, "combined", 0.2)
STEP_ROWS = {
    "big_batch": dict(d=ROWS["big_batch"]["d"], cap=ROWS["big_batch"]["cap"], path="tcgen05",
                      expect=["gemm_planes_kernel", "spmm_mol_kernel"]),
    "tiles_128": dict(d=ROWS["tiles_128"]["d"], cap=ROWS["tiles_128"]["cap"], path="tcgen05",
                      expect=["gemm_planes_kernel", "spmm_mol_kernel"]),
    "persistent_fused_bn": dict(d=ROWS["persistent_fused_bn"]["d"], cap=ROWS["persistent_fused_bn"]["cap"],
                                path="tcgen05+noplanes", expect=["gemm_3xtf32_persistent_kernel"],
                                absent=["gemm_planes_kernel"]),
    "wide_planes": dict(d=ROWS["wide"]["d"], cap=(ROWS["wide"]["B"], ROWS["wide"]["B"] * ROWS["wide"]["atoms"]),
                        path="tcgen05+planes", expect=["gemm_planes_kernel"]),
    # the benchmark's training plan: neither planes nor persistent kernels at this capacity, the GraphConv backward
    # takes the grouped in-kernel-split launch with split counts from the capacity
    "bench_train": dict(d=BENCH_D, cap=(512, 512 * 64), path="tcgen05", expect=["gemm_3xtf32_kernel"],
                        absent=["gemm_planes_kernel", "gemm_3xtf32_persistent_kernel"]),
}


def step_sizes(d, Bc, Nc, planes, persistent):
    """(molecules, atoms) of the live batches of a row, largest first."""
    H = d.hidden_dim
    s = [(1, 2), (1, 31), (1, 32), (1, 33), (2, 129), (3, 257), (Bc, Nc - 1), (Bc, Nc)]
    if planes:   # data-gradient store tiles = the deal width, and one more
        TM = BM * PAIR
        rows = G_PAIRS // (H // BN) * TM if G_PAIRS % (H // BN) == 0 else None
        if rows:
            s += [(None, rows), (None, rows + 1)]
    if persistent:
        rows = SMS // (H // BN) * BM
        s += [(None, rows), (None, rows + 1)]
    if Bc >= 2 * K1_SCAN_CHUNK:
        s += [(K1_SCAN_CHUNK, None), (K1_SCAN_CHUNK + 1, None)]
    out = set()
    for B, N in s:
        if N is None:
            N = B * min(48, Nc // Bc)
        if B is None:
            B = min(Bc, max(1, ceil_div(N, min(64, max(2, Nc // Bc)))))
        if N <= Nc and B <= Bc and N >= 2 * B:
            out.add((B, N))
    return sorted(out, key=lambda x: (x[1], x[0]), reverse=True)


def exact_table(B, N, seed):
    """B molecules (chains and rings) of N atoms in all."""
    base, rem = divmod(N, B)
    mols = [(chain if (i % 2 or base + (i < rem) < 3) else ring)(base + (1 if i < rem else 0)) for i in range(B)]
    t = mol_table(mols, 6, seed)
    assert t.num_mols == B and int(t.node_ptr[-1]) == N
    return t


def two_atom_floor(d, table, targets, sd, res, rep, bad):
    """Two atoms: even with small GraphConv weights, the two rows of a layer's input differ little while the two rows
    of its BatchNorm-backward output sum to zero, so a weight gradient a^T q is a difference of nearly equal terms
    (measured: the top layer's off by 6e-4 on the GPU, its columns by as much in the fp32 oracle).  There a whole-tensor
    gradient error is held to 16 x the fp32 oracle's own error, as the column-scaled errors always are; everything
    else keeps its bound."""
    graph, feat = O.Graph.from_mols([table.mol(i) for i in range(table.num_mols)])
    tt, od = torch.from_numpy(targets), odims(d)
    kw = dict(dropout_masks=res["masks"], decisions=res["dec"])
    _, _, g64, _ = O.loss_and_grads(sd, graph, feat, tt, od, dtype=torch.float64, keep=True, **kw)
    _, _, g32, _ = O.loss_and_grads(sd, graph, feat, tt, od, **kw)
    rep["grad_floors_two_atoms"] = {}
    keep = []
    for b in bad:
        n = b[len("grad "):] if b.startswith("grad ") else None
        if n in rep["grads"]:
            floor = rel_err(g32[n].numpy(), g64[n].numpy())
            rep["grad_floors_two_atoms"][n] = floor
            if rep["grads"][n] < 16 * floor:
                continue
        keep.append(b)
    return keep


@pytest.mark.parametrize("name", list(STEP_ROWS))
def test_step_at_ragged_live_sizes(name, tmp_path):
    r = STEP_ROWS[name]
    d, (Bc, Nc), path = r["d"], r["cap"], r["path"]
    planes = "planes" in " ".join(r["expect"])
    persistent = "persistent" in " ".join(r["expect"])
    sizes = step_sizes(d, Bc, Nc, planes, persistent)
    order = sizes + sizes[-2::-1]                 # descending, then ascending
    plan = make_plan(d, Bc, Nc, 2 * (Nc + 3 * Bc), path)   # poisoned at creation
    report, failures = [], []
    for k, (B, N) in enumerate(order):
        if k % 2 == 0 and k > 0:
            poison(plan)
        table = exact_table(B, N, 1000 + k)
        targets = dense_spectra(*synth_peaks(B, d.max_mz, seed=2000 + k), d.max_mz)
        ds = DeviceDataset(table, targets, DEV)
        sd = random_running_stats(O.init_params(odims(d), 3000 + k), d, 4000 + k)
        if N == 2:
            # BatchNorm over two atoms maps every column whose two values differ by much more than sqrt(eps) to +-1,
            # and its backward then cancels to rounding noise (measured: the GPU and the fp32 oracle alike miss the
            # fp64 gradients by 1e-3 .. 1e-1).  Small GraphConv weights and biases keep the two atoms' pre-BatchNorm
            # values within sqrt(eps) of each other, where BatchNorm is nearly linear and the step well conditioned.
            for l in range(d.num_gcn_layers):
                for p in ("weight", "bias"):
                    sd[f"gcn_layers.{l}.{p}"] = sd[f"gcn_layers.{l}.{p}"] * 1e-4
        fp = FlatParams(d, DEV)
        fp.load_state_dict(sd)
        step = make_step(step=k + 1, seed=23)

        def run():
            res = gpu_step(plan, ds, fp, step)
            res["eval"] = plan.infer_batch(ds, None, fp).clone().cpu().numpy()
            res["eval_sd"] = {kk: v.cpu() for kk, v in fp.state_dict().items()}
            return res

        profile = (B, N) in (sizes[0], sizes[-1]) and k < len(sizes)
        if profile:
            res, kernels = profiled(run)
            missing = [x for x in r["expect"] if not any(x in kn for kn in kernels)]
            present = [x for x in r.get("absent", []) if any(x in kn for kn in kernels)]
            if missing or present:
                failures.append(dict(B=B, N=N, missing=missing, unexpected=present, kernels=kernels))
        else:
            res = run()
        assert res["N"] == N
        res["masks"] = dropout_masks(d, step, N, B)
        rep, bad = oracle_check(d, table, targets, sd, res)
        if N == 2:
            bad = two_atom_floor(d, table, targets, sd, res, rep, bad)
        report.append(dict(molecules=B, atoms=N, poisoned=k % 2 == 0, worst_error_over_bound=worst_ratio(rep), bad=bad))
        if bad:
            failures.append(dict(B=B, N=N, bad=bad, rep=rep))
        with open(tmp_path / f"live_sizes_step_{name}.json", "w") as fh:
            json.dump(dict(row=name, path=path, capacity=[Bc, Nc], batches=report, failures=failures), fh, indent=1, default=str)
        assert not failures, failures   # stop at the first batch that fails: the later ones start from its state
