"""The graph kernels on molecules large and dense enough to take their fallback paths.

Three kernels pick one of two code paths per molecule from that molecule's size, and the synthetic generator
(`synth.synth_molecules`: a tree plus <= 3 ring bonds, degree <= 4) never leaves the fast one at the sizes the other
tests use.  The shapes below are built explicitly - chains and rings across the warp and tile boundaries, 3-regular
cages at and just past K1's bond limit, hubs of degree 6 and 64, small edge-dense molecules, exactly symmetric atoms,
an isolated atom inside an oversized molecule - and each kernel is held to a plain high-precision reference on both of
its paths:

  * K1 (`k1_build_kernel`): staged in shared memory, or the O(n * bonds) scans over global memory when a molecule has
    more than K1_MAX_N atoms or K1_MAX_B bonds.  Every batch table bit for bit, `a0` against a sequential fp32 loop.
  * `readout_kernel`: the graph's [n, H] tile bulk-copied into READOUT_TILE_BYTES of shared memory, or rows read from
    global memory.  Max and DGL's first arg-max bit for bit on a value grid where BatchNorm apply is exact and ties
    are abundant; sum / mean to the fp32 summation bound; `zstat` of a training forward against fp64.
  * `spmm_mol_kernel`: the molecule tile, or a per-row gather when a molecule has more than `tile_rows` atoms or more
    than 4 * tile_rows + 64 directed edges.  Bit for bit against `spmm_norm_kernel`.

Whole training steps and an inference forward that reach the fallbacks inside a plan are held to the fp64 oracle with
the protocol of test_gpu_dispatch, and eval spectra are held bit for bit wherever a molecule sits in a batch.

`test_shapes_lie_where_they_claim` (no GPU) reads the thresholds from the CUDA sources and checks that every shape
lies on the side of each threshold that the tests rely on."""
import json
import os
import re
from dataclasses import dataclass, field

import numpy as np
import pytest
import torch

from eims_b200 import _lib
from eims_b200.engine import DeviceDataset, FlatParams, ModelDims, Plan, make_step
from eims_b200.synth import MolTable, dense_spectra, synth_molecules, synth_peaks
from oracle import gcn_oracle as O
from test_gpu_dispatch import (COL_REL, REL, kernel_names, make_plan, make_table, odims, oracle_check, poison,
                               random_running_stats, rel_err, run_gpu)
from test_gpu_kernels import dev, make_dims, stream

DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "computational-chemistry-ai_b200", "csrc")

# ------------------------------------------------------------------------------------------------ thresholds
K1_MAX_N, K1_MAX_B = 128, 192          # graph.cu:86 kK1MaxN / kK1MaxB: larger molecules skip K1's shared-memory staging
READOUT_TILE_BYTES = 64 * 1024         # graph.cu:1048 kTileBytes: graphs with n * H * 4 above it read z from global
K1_SCAN_CHUNK = 1024                   # graph.cu:27,319: k1_scan_kernel's block size; batches above it are prescanned
MOL_TILE_MIN_GRAPHS = 2048             # graph.cu:898: plans of >= 2048 molecules aggregate with spmm_mol_kernel


def tile_cap_edges(tile_rows):
    """graph.cu:862: directed edges a molecule tile stages."""
    return 4 * tile_rows + 64


def plan_tile_rows(Bc, Nc):
    """plan.cu:132: the tile of a plan of Bc molecules and Nc atoms."""
    return 64 if (Nc + Bc - 1) // Bc <= 64 else 128


def k1_oversized(n, nb):
    return n > K1_MAX_N or nb > K1_MAX_B


def readout_unstaged(n, H):
    return n * H * 4 > READOUT_TILE_BYTES


def tile_fallback(n, nb, tile_rows):
    return n > tile_rows or 2 * nb > tile_cap_edges(tile_rows)


# ------------------------------------------------------------------------------------------------ shapes
@dataclass
class Mol:
    name: str
    n: int
    bonds: list = field(default_factory=list)   # (begin, end), molecule-local: no self-bonds, no duplicates
    sym: bool = False                           # every atom gets the same raw features (exactly symmetric atoms)


def chain(n, sym=False):
    return Mol(f"chain_{n}", n, [(i, i + 1) for i in range(n - 1)], sym)


def ring(n, sym=False):
    return Mol(f"{'sym_' if sym else ''}ring_{n}", n, chain(n).bonds + ([(n - 1, 0)] if n >= 3 else []), sym)


def cage(k=64, extra=0, sym=False):
    """Prism over two k-rings: 2k atoms, 3k bonds, every atom of degree 3 (at k = 64: 128 atoms, 192 bonds, exactly
    K1's limits).  `extra` bonds (i, i + 2) across the outer ring go past the bond limit at the same atom count."""
    outer = [(i, (i + 1) % k) for i in range(k)]
    inner = [(k + i, k + (i + 1) % k) for i in range(k)]
    rungs = [(i, k + i) for i in range(k)]
    return Mol(f"cage_{2 * k}_{3 * k + extra}", 2 * k, outer + inner + rungs + [(i, i + 2) for i in range(extra)], sym)


def hub(deg, arm, sym=False):
    """Atom 0 bonded to `deg` arms of `arm` atoms each (hypervalent S / P at deg = 6)."""
    bonds = []
    for a in range(deg):
        first = 1 + a * arm
        bonds.append((0, first))
        bonds += [(first + t, first + t + 1) for t in range(arm - 1)]
    return Mol(f"hub_{deg}x{arm}", 1 + deg * arm, bonds, sym)


def dense(n, nb, seed=0):
    """A ring of n atoms plus random chords up to nb bonds (nb <= n(n-1)/2)."""
    have = set(tuple(sorted(b)) for b in ring(n).bonds)
    rest = [(i, j) for i in range(n) for j in range(i + 1, n) if (i, j) not in have]
    rng = np.random.default_rng(seed + 1000 * n + nb)
    extra = [rest[k] for k in rng.permutation(len(rest))[: nb - len(have)]]
    assert len(have) + len(extra) == nb, (n, nb)
    return Mol(f"dense_{n}_{nb}", n, sorted(have) + extra)


def with_isolated(n):
    """A chain of n atoms whose middle atom has no bond (DGL's GraphConv refuses it)."""
    m = n // 2
    bonds = [(i, i + 1) for i in range(n - 1) if m not in (i, i + 1)] + [(m - 1, m + 1)]
    return Mol(f"isolated_in_{n}", n, bonds)


CHAIN_SIZES = [2, 31, 32, 33, 64, 65, 127, 128, 129, 200, 300, 1000]


def catalogue():
    """Every explicit shape, by name."""
    mols = [chain(n) for n in CHAIN_SIZES] + [ring(n) for n in CHAIN_SIZES if n >= 3]
    mols += [cage(), cage(extra=1), cage(sym=True), hub(6, 1), hub(6, 4), hub(6, 1, sym=True), hub(6, 3, sym=True), hub(64, 3),
             ring(40, sym=True), ring(66, sym=True), dense(97, 193), dense(16, 64), dense(16, 65), dense(16, 120),
             dense(12, 66), dense(14, 80), dense(64, 160), dense(64, 161), dense(19, 171), dense(40, 200),
             with_isolated(201)]
    for m in mols[:]:
        if m.sym and not m.name.startswith("sym_"):
            m.name = "sym_" + m.name
    return {m.name: m for m in mols}


SHAPES = catalogue()


def shapes(*names):
    return [SHAPES[n] for n in names]


# the molecules each test mixes into its batches, and which side of which threshold they stand for
K1_SPECIALS = ["chain_129", "ring_129", "chain_1000", "cage_128_193", "hub_64x3", "dense_97_193", "chain_300",
               "chain_200", "ring_200", "ring_300", "ring_1000",                   # oversized: at the K1_POS positions
               "ring_127", "ring_128", "cage_128_192", "hub_6x1", "hub_6x4", "chain_2", "ring_33", "ring_64", "ring_65",
               "sym_ring_40"]
BIG_TRAIN_SPECIALS = ["chain_65", "ring_65", "sym_ring_66", "chain_127", "ring_128", "chain_129", "ring_129",
                      "chain_200", "ring_200", "chain_300", "ring_300", "hub_64x3", "hub_6x4", "cage_128_192",
                      "cage_128_193", "sym_cage_128_192", "dense_64_161", "dense_19_171", "dense_97_193", "ring_127"]
WIDE_SPECIALS = ["sym_ring_40", "sym_cage_128_192", "ring_128", "chain_33", "sym_hub_6x3", "hub_6x4", "ring_65",
                 "cage_128_193"]
PREDICT_SPECIALS = ["chain_1000", "ring_1000", "hub_64x3", "chain_300", "ring_200", "cage_128_192", "cage_128_193",
                    "dense_97_193", "ring_129", "chain_65", "sym_ring_66", "dense_64_161"]
TILE_SPECIALS = {16: ["dense_16_64", "dense_16_65", "dense_16_120", "dense_12_66", "dense_14_80", "ring_32",
                      "hub_6x1", "chain_2", "ring_33", "chain_65"],
                 64: ["dense_64_160", "dense_64_161", "dense_19_171", "dense_40_200", "ring_64", "ring_65",
                      "hub_6x4", "chain_129"]}
BIG_TRAIN_CAP = (4096, 4096 * 48)
BIG_TRAIN_H = 256
WIDE_H = 1024


def claims():
    """(shape, predicate, expected): the side of each threshold a shape is used for."""
    out = [("cage_128_192", lambda m: (m.n, len(m.bonds)) == (K1_MAX_N, K1_MAX_B) and not k1_oversized(m.n, len(m.bonds)), True),
           ("cage_128_193", lambda m: m.n <= K1_MAX_N and len(m.bonds) == K1_MAX_B + 1, True),
           ("dense_97_193", lambda m: m.n <= K1_MAX_N and k1_oversized(m.n, len(m.bonds)), True),
           ("ring_128", lambda m: k1_oversized(m.n, len(m.bonds)), False),
           ("ring_129", lambda m: m.n == K1_MAX_N + 1 and len(m.bonds) <= K1_MAX_B, True),
           ("hub_64x3", lambda m: m.n > K1_MAX_N and max(np.bincount(np.ravel(m.bonds))) == 64, True),
           ("hub_6x1", lambda m: max(np.bincount(np.ravel(m.bonds))) == 6, True),
           ("isolated_in_201", lambda m: m.n > K1_MAX_N and int((np.bincount(np.ravel(m.bonds), minlength=m.n) == 0).sum()) == 1, True),
           ("sym_ring_66", lambda m: readout_unstaged(m.n, BIG_TRAIN_H) and m.n > plan_tile_rows(*BIG_TRAIN_CAP), True),
           ("ring_64", lambda m: readout_unstaged(m.n, 256), False),
           ("ring_65", lambda m: readout_unstaged(m.n, 256), True),
           ("ring_33", lambda m: readout_unstaged(m.n, 512), True),
           ("ring_32", lambda m: readout_unstaged(m.n, 512), False),
           ("sym_ring_40", lambda m: readout_unstaged(m.n, WIDE_H) and m.n <= K1_MAX_N, True)]
    for tr in (16, 64):
        for name in TILE_SPECIALS[tr]:
            m = SHAPES[name]
            if name.startswith("dense") and m.n <= tr:
                at_limit = 2 * len(m.bonds) == tile_cap_edges(tr)
                out.append((name, lambda m, tr=tr: tile_fallback(m.n, len(m.bonds), tr), not at_limit))
    return out


def atom_features(deg, F, rng, sym):
    """Raw descriptor columns in the layout of synth.py (atomic number, degree, formal charge, hybridisation,
    aromatic, hydrogens); for F != 6 random normal as in test_gpu_dispatch.make_table.  `sym`: the same row for
    every atom of the same degree."""
    n = len(deg)
    if F != 6:
        f = rng.standard_normal((1 if sym else n, F)).astype(np.float32)
        return np.repeat(f, n, axis=0) if sym else f
    f = np.zeros((n, 6), np.float32)
    f[:, 0] = 6.0 if sym else rng.choice(np.array([6, 7, 8, 9, 16, 17], np.float32), size=n,
                                           p=[0.72, 0.08, 0.12, 0.03, 0.02, 0.03])
    f[:, 1] = deg
    f[:, 3] = 3.0 if sym else rng.integers(2, 5, size=n)
    f[:, 4] = 0.0 if sym else rng.integers(0, 2, size=n)
    f[:, 5] = np.clip(4 - deg, 0, 3)
    return f


def mol_table(mols, F=6, seed=0, shuffle_bonds=True):
    """MolTable of explicit molecules.  Bond order is arbitrary, as from RDKit: shuffled, each bond's ends swapped
    at random (symmetric molecules keep their symmetry: every neighbour of a symmetric atom is alike)."""
    rng = np.random.default_rng(seed)
    feats, bb, be, nn, nbs = [], [], [], [], []
    for m in mols:
        b = np.array(m.bonds, np.int32).reshape(-1, 2)
        if shuffle_bonds and len(b):
            b = b[rng.permutation(len(b))]
            flip = rng.random(len(b)) < 0.5
            b[flip] = b[flip][:, ::-1]
        deg = np.bincount(b.ravel(), minlength=m.n)
        feats.append(atom_features(deg, F, rng, m.sym))
        bb.append(b[:, 0])
        be.append(b[:, 1])
        nn.append(m.n)
        nbs.append(len(b))
    return MolTable(np.concatenate([[0], np.cumsum(nn)]).astype(np.int64), np.concatenate([[0], np.cumsum(nbs)]).astype(np.int64),
                    np.concatenate(feats), np.concatenate(bb).astype(np.int32), np.concatenate(be).astype(np.int32))


def concat(*tables):
    nn = np.concatenate([np.diff(t.node_ptr) for t in tables])
    nb = np.concatenate([np.diff(t.bond_ptr) for t in tables])
    return MolTable(np.concatenate([[0], np.cumsum(nn)]).astype(np.int64), np.concatenate([[0], np.cumsum(nb)]).astype(np.int64),
                    np.concatenate([t.feat for t in tables]), np.concatenate([t.bond_begin for t in tables]),
                    np.concatenate([t.bond_end for t in tables]))


def sizes(table):
    return np.diff(table.node_ptr), np.diff(table.bond_ptr)


def arrange(B, n_fill, specials, positions, rng):
    """Batch order of B molecules: special k (table ids n_fill + k, cycled) at positions[k] (those < B; the last
    position is always one of them), further specials at random positions, fillers 0.. everywhere else."""
    pos = list(dict.fromkeys([p for p in positions if p < B] + [B - 1]))
    free = [p for p in rng.permutation(B) if p not in set(pos)]
    pos += free[: max(0, len(specials) - len(pos))]
    order = np.full(B, -1, np.int64)
    for k, p in enumerate(pos):
        order[p] = n_fill + k % len(specials)
    rest = order < 0
    assert rest.sum() <= n_fill
    order[rest] = np.arange(int(rest.sum()))
    return order


# ------------------------------------------------------------------------------------------------ references
def a0_reference(rowptr, col, norm, x):
    """K1's layer-0 aggregate as a plain sequential fp32 loop: a0_i = fl(...fl(fl(0 + p_e0) + p_e1)...) over the
    row's edges in ascending edge id, p_e = fl(x_j * c_j) (numpy float32 arithmetic rounds every operation)."""
    p = x[col] * norm[col][:, None]
    deg = np.diff(rowptr)
    acc = np.zeros_like(x)
    for k in range(int(deg.max()) if len(deg) else 0):
        rows = np.nonzero(deg > k)[0]
        acc[rows] = acc[rows] + p[rowptr[rows] + k]
    return acc


def gamma(n):
    """Higham's gamma_n = n u / (1 - n u), u = 2^-24: any-order fp32 summation of n terms is within gamma_{n-1} of
    the sum of their magnitudes."""
    u = 2.0 ** -24
    return n * u / (1 - n * u)


def bits(a):
    return np.ascontiguousarray(a).view(np.int32)


def check_batch_tables(plan, mols, F):
    """Every table K1 wrote for the batch `mols` against the oracle, raw bits.  Returns the mismatching names."""
    b = O.batch_graphs(mols)
    rowptr, col, deg = O.csr_by_dst(b["src"], b["dst"], b["num_nodes"])
    norm = O.degree_norm(deg)
    N, E, B = b["num_nodes"], len(b["src"]), len(mols)
    assert plan.check() == (N, E)
    i32 = torch.int32
    x = b["feat"].astype(np.float32).reshape(N, F)
    ref = dict(src=b["src"], dst=b["dst"], rowptr=rowptr, col=col, gptr=O.graph_ptr(b["batch_num_nodes"]),
               eptr=O.graph_ptr(b["batch_num_edges"]), gid=np.repeat(np.arange(B), b["batch_num_nodes"]))
    size = dict(src=E, dst=E, rowptr=N + 1, col=E, gptr=B + 1, eptr=B + 1, gid=N)
    bad = [k for k, v in ref.items() if not np.array_equal(plan.buffer(k, i32)[:size[k]].cpu().numpy(), v.astype(np.int32))]
    got_f = {k: plan.buffer(k)[:n].cpu().numpy() for k, n in (("norm", N), ("x", N * F), ("a0", N * F))}
    ref_f = dict(norm=norm, x=x.reshape(-1), a0=a0_reference(rowptr, col, norm, x).reshape(-1))
    bad += [k for k in ref_f if not np.array_equal(bits(got_f[k]), bits(ref_f[k]))]
    return bad


# ------------------------------------------------------------------------------------------------ CPU: the shapes
def test_shapes_lie_where_they_claim():
    """The thresholds named above are the ones in the CUDA sources, every shape is a valid molecule (connected
    bonds, no self-bond, no duplicate), and every shape lies on the side of the threshold its test relies on - so a
    moved threshold fails here instead of silently testing the fast path twice."""
    graph_cu = open(os.path.join(CSRC, "graph.cu")).read()
    plan_cu = open(os.path.join(CSRC, "plan.cu")).read()
    m = re.search(r"constexpr int kK1MaxN = (\d+), kK1MaxB = (\d+);", graph_cu)
    assert m and (int(m.group(1)), int(m.group(2))) == (K1_MAX_N, K1_MAX_B)
    m = re.search(r"constexpr int kTileBytes = (\d+) \* 1024;", graph_cu)
    assert m and int(m.group(1)) * 1024 == READOUT_TILE_BYTES
    assert re.search(r"const int cap_edges = 4 \* tile_rows \+ 64;", graph_cu)
    assert re.search(r"const bool big_batch = max_graphs >= %d && !bf;" % MOL_TILE_MIN_GRAPHS, graph_cu)
    assert re.search(r"const int prescanned = B > %d;" % K1_SCAN_CHUNK, graph_cu)
    assert re.search(r"int tile_rows\(\) const \{ return \(Nc \+ Bc - 1\) / Bc <= 64 \? 64 : 128; \}", plan_cu)
    for name, mol in SHAPES.items():
        b = np.array(mol.bonds).reshape(-1, 2)
        assert (b[:, 0] != b[:, 1]).all(), name
        assert len(set(map(tuple, np.sort(b, axis=1)))) == len(b), name
        assert b.min() >= 0 and b.max() < mol.n, name
    assert [len(SHAPES[f"chain_{n}"].bonds) for n in CHAIN_SIZES] == [n - 1 for n in CHAIN_SIZES]
    for name, pred, want in claims():
        assert pred(SHAPES[name]) == want, name
    for names in (K1_SPECIALS, BIG_TRAIN_SPECIALS, WIDE_SPECIALS, PREDICT_SPECIALS, *TILE_SPECIALS.values()):
        assert all(n in SHAPES for n in names)
    # the mixes reach both sides of every threshold they are for
    k1 = [(m.n, len(m.bonds)) for m in shapes(*K1_SPECIALS)]
    assert any(n > K1_MAX_N for n, nb in k1) and any(n <= K1_MAX_N and nb > K1_MAX_B for n, nb in k1)
    assert any((n, nb) == (K1_MAX_N, K1_MAX_B) for n, nb in k1)
    big = shapes(*BIG_TRAIN_SPECIALS)
    tr = plan_tile_rows(*BIG_TRAIN_CAP)
    assert tr == 64
    assert any(m.n > tr for m in big) and any(m.n <= tr and tile_fallback(m.n, len(m.bonds), tr) for m in big)
    assert any(readout_unstaged(m.n, BIG_TRAIN_H) for m in big)
    assert any(m.n > K1_MAX_N for m in big) and any(m.n <= K1_MAX_N and len(m.bonds) > K1_MAX_B for m in big)
    assert all(readout_unstaged(m.n, WIDE_H) for m in shapes(*WIDE_SPECIALS))
    for tr, names in TILE_SPECIALS.items():
        ms = shapes(*names)
        assert any(m.n <= tr and 2 * len(m.bonds) > tile_cap_edges(tr) for m in ms)     # edge-count fallback
        assert any(m.n <= tr and 2 * len(m.bonds) == tile_cap_edges(tr) for m in ms)    # staged at the limit
        assert any(m.n > tr for m in ms)                                                 # atom-count fallback
    # a0 reference: a hand-checked row (x_j * c_j summed in edge order)
    rowptr, col = np.array([0, 3, 4, 5, 6]), np.array([1, 2, 3, 0, 0, 0])
    norm = np.array([3.0 ** -0.5, 1.0, 1.0, 1.0], np.float32)
    x = np.array([[1.0], [2.0], [3.0], [4.0]], np.float32)
    a0 = a0_reference(rowptr, col, norm, x)
    assert a0[0, 0] == np.float32(np.float32(2.0 + 3.0) + 4.0) and a0[1, 0] == np.float32(norm[0])


# ------------------------------------------------------------------------------------------------ K1
K1_POS = [0, 511, 1022, 1023, 1024, 1025, 2046, 2047, 2048, 2049]


def k1_batch(B, F, shuffle, seed):
    """(dataset table, ids or None, molecules in batch order) of a batch of B molecules: small synthetic fillers and
    the K1 specials at and around the scan's chunk boundaries."""
    rng = np.random.default_rng(seed)
    specials = shapes(*K1_SPECIALS)
    fill = make_table(B, 12, seed, F)
    src = concat(fill, mol_table(specials, F, seed + 1))
    order = arrange(B, B, specials, K1_POS, rng)
    if shuffle:
        perm = rng.permutation(src.num_mols)           # the data set holds the molecules in another order ...
        table = src.select(perm)
        inv = np.empty_like(perm)
        inv[perm] = np.arange(len(perm))
        ids = inv[order]                               # ... and the ids pick the batch out of it
    else:
        table, ids = src.select(order), None
    mols = [src.mol(int(g)) for g in order]
    return table, ids, mols


@pytest.mark.gpu
@pytest.mark.parametrize("B,shuffle,F", [(700, False, 6), (700, True, 1), (1024, True, 8), (1024, False, 6), (1025, True, 6),
                                         (1025, False, 1), (2049, True, 8), (2049, False, 6), (2600, True, 6), (2600, False, 8)])
def test_k1_both_branches_bit_exact(B, shuffle, F):
    """Batches that mix staged molecules with ones over K1's atom limit and over its bond limit alone, in the fused
    (B <= 1024) and the prescanned form (the scan carries once past 1024 molecules, twice past 2048), with the
    oversized molecules at and around positions 1023 / 1024 / 2047 / 2048 and last: every batch table, `a0`
    included, bit for bit."""
    table, ids, mols = k1_batch(B, F, shuffle, seed=B + F)
    n, nb = np.array([len(m[0]) for m in mols]), np.array([len(m[1]) for m in mols])
    assert (n > K1_MAX_N).any() and ((n <= K1_MAX_N) & (nb > K1_MAX_B)).any() and (~((n > K1_MAX_N) | (nb > K1_MAX_B))).any()
    b = O.batch_graphs(mols)
    N, E = b["num_nodes"], len(b["src"])
    plan = Plan(ModelDims(node_feat_dim=F, hidden_dim=64, max_mz=100), B, N + 7, E + 5, DEV)
    ds = DeviceDataset(table, None, DEV)
    plan.batch_build(ds, None if ids is None else dev(ids, torch.int32), B)
    assert not check_batch_tables(plan, mols, F)


@pytest.mark.gpu
@pytest.mark.parametrize("B", [50, 1100])
def test_k1_isolated_atom_in_oversized_molecule(B):
    """An isolated atom inside a molecule over K1's atom limit raises the zero-degree error (DGL's GraphConv refuses
    such a graph) in the fused and the prescanned form; the next, clean batch of the same plan builds correctly."""
    rng = np.random.default_rng(B)
    fill = make_table(B, 12, B, 6)
    src = concat(fill, mol_table(shapes("isolated_in_201"), 6, 3))
    bad = arrange(B, B, shapes("isolated_in_201"), [B // 2], rng)
    clean = np.arange(B)
    nodes, bonds = sizes(src)
    plan = Plan(ModelDims(hidden_dim=64, max_mz=100), B, int(nodes[bad].sum()) + 7, 2 * int(bonds[bad].sum()) + 5, DEV)
    ds = DeviceDataset(src, None, DEV)
    plan.batch_build(ds, dev(bad, torch.int32), B)
    with pytest.raises(_lib.ZeroInDegreeError):
        plan.check()
    plan.batch_build(ds, dev(clean, torch.int32), B)
    assert not check_batch_tables(plan, [src.mol(int(g)) for g in clean], 6)


@pytest.mark.gpu
def test_k1_capacity_overflow_mid_prescanned_batch():
    """A 1000-atom molecule in the middle of a prescanned batch pushes it past the plan's atom capacity: the build
    reports ERR_CAPACITY, and a clean batch in the same plan then builds correctly."""
    B = 1500
    fill = make_table(B, 12, 21, 6)
    src = concat(fill, mol_table(shapes("chain_1000"), 6, 22))
    clean = np.arange(B)
    over = clean.copy()
    over[750] = B
    nodes, bonds = sizes(src)
    N, E = int(nodes[clean].sum()), 2 * int(bonds[clean].sum())
    assert int(nodes[over].sum()) > N + 500
    plan = Plan(ModelDims(hidden_dim=64, max_mz=100), B, N + 500, 2 * E, DEV)
    ds = DeviceDataset(src, None, DEV)
    plan.batch_build(ds, dev(over, torch.int32), B)
    with pytest.raises(_lib.EimsError) as e:
        plan.check()
    assert e.value.code == _lib.ERR_CAPACITY
    plan.batch_build(ds, dev(clean, torch.int32), B)
    assert not check_batch_tables(plan, [src.mol(int(g)) for g in clean], 6)


# ------------------------------------------------------------------------------------------------ readout
def grid_values(shape, rng):
    """relu(k / 8) for k in [-8, 24]: with the BatchNorm coefficients below every fmaf(z, scale, shift) is exact."""
    return (np.maximum(rng.integers(-8, 25, size=shape), 0) / 8.0).astype(np.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("bn", [False, True], ids=["plain", "bn_negative"])
@pytest.mark.parametrize("H", [64, 128, 192, 256, 320, 512, 768, 1024])
def test_readout_both_paths(H, bn):
    """`eims_readout` on graphs on both sides of the shared-memory tile in one launch (H = 64 ... 1024: 16 ... 1 row
    lanes, 192 and 320 leave lanes idle), every pooling, without BatchNorm apply and with it at negative and positive
    power-of-two scales.  Max and DGL's first arg-max bit for bit, with exact ties at nonzero values on the unstaged
    path; sum and mean within the fp32 summation bound of fp64; rows past the batch untouched."""
    lim = READOUT_TILE_BYTES // (4 * H)                 # most atoms a staged graph has
    ns = [1, 2, 3, 7, lim - 1, lim, lim + 1, lim + 2, 2 * lim + 1, 65, 129, 300]
    ns = [k for k in ns if k >= 1]
    rng = np.random.default_rng(H + bn)
    ns = list(rng.permutation(ns))
    B, N = len(ns), int(sum(ns))
    z = grid_values((N, H), rng)
    if bn:
        sc = (rng.choice([-1.0, 1.0], H) * 2.0 ** rng.integers(-1, 2, H)).astype(np.float32)
        sc[: H // 2] = -np.abs(sc[: H // 2])
        sh = (rng.integers(-16, 17, H) / 8.0).astype(np.float32)
        h = z.astype(np.float64) * sc + sh
    else:
        sc = sh = None
        h = z.astype(np.float64)
    assert np.array_equal(h.astype(np.float32).astype(np.float64), h)   # the grid keeps BatchNorm apply exact
    gptr = O.graph_ptr(np.array(ns))
    g = O.Graph(np.zeros(0), np.zeros(0), np.array(ns))
    ref_mx, ref_arg = O.segment_max_first(torch.from_numpy(h), g)
    S = torch.zeros(B, H, dtype=torch.float64).index_add_(0, g.gid, torch.from_numpy(h))
    A = torch.zeros(B, H, dtype=torch.float64).index_add_(0, g.gid, torch.from_numpy(np.abs(h)))
    nn = torch.tensor(ns, dtype=torch.float64)[:, None]
    unstaged = np.array([readout_unstaged(k, H) for k in ns])
    assert unstaged.any() and (~unstaged).any()
    ties = (torch.from_numpy(h) == ref_mx[g.gid]).double()
    ties = torch.zeros(B, H, dtype=torch.float64).index_add_(0, g.gid, ties)
    nonzero_ties = ((ties > 1) & (ref_mx != 0)).numpy()
    assert nonzero_ties[unstaged].sum() > 0 and nonzero_ties[~unstaged].sum() > 0
    keep = (make_dims(B, N, 0), dev(gptr, torch.int32), dev(z), dev(sc) if bn else None, dev(sh) if bn else None)
    for pooling in ("sum", "mean", "max", "combined"):
        pd = 2 * H if pooling == "combined" else H
        out = torch.full((B + 2, pd), 7.0, device=DEV)
        arg = torch.full((B + 2, H), -1, dtype=torch.int32, device=DEV)
        _lib.check(_lib.load().eims_readout(_lib.ptr(keep[0]), _lib.ptr(keep[1]), _lib.ptr(keep[2]), H, _lib.ptr(keep[3]),
                                            _lib.ptr(keep[4]), _lib.POOLING[pooling], _lib.ptr(out), _lib.ptr(arg), B, stream()))
        out, arg = out.cpu(), arg.cpu()
        assert bool((out[B:] == 7.0).all()) and bool((arg[B:] == -1).all()), pooling
        if pooling in ("max", "combined"):
            for part, rows in (("unstaged", unstaged), ("staged", ~unstaged)):
                rows = torch.from_numpy(rows)
                assert torch.equal(out[:B, -H:][rows].double(), ref_mx[rows]), (pooling, part, "max")
                assert torch.equal(arg[:B][rows].long(), ref_arg[rows]), (pooling, part, "arg-max")
        if pooling in ("sum", "mean", "combined"):
            ref, bound = (S, gamma(nn + 1) * A) if pooling != "mean" else (S / nn, gamma(nn + 2) * A / nn)
            err = (out[:B, :H].double() - ref).abs()
            assert bool((err <= bound).all()), (pooling, float((err / bound.clamp_min(1e-300)).max()))


def zstat_check(d, table, caps, sd, path, step):
    """`zstat` after a training forward in a poisoned plan, from the plan's own z_{L-1}, bn_mean_{L-1} and arg-max:
    per graph the column sums of z - mean (fp32 summation bound of fp64) and z - mean at the arg-max node (exact).
    Returns (worst error over bound of the sums, graphs over the readout tile, exact nonzero ties at the arg-max)."""
    B, H, L = table.num_mols, d.hidden_dim, d.num_gcn_layers
    plan = make_plan(d, *caps, path)
    ds = DeviceDataset(table, None, DEV)
    fp = FlatParams(d, DEV)
    fp.load_state_dict(sd)
    plan.batch_build(ds, None, B)
    plan.forward(fp, True, step)
    N, _ = plan.check()
    z = plan.buffer(f"z{L - 1}", torch.float32, (N, H)).cpu().numpy()
    mu = plan.buffer(f"bn_mean{L - 1}", torch.float32, (H,)).cpu().numpy()
    am = plan.buffer("argmax", torch.int32, (B, H)).cpu().numpy().astype(np.int64)
    zs = plan.buffer("zstat", torch.float32, (B, 2 * H)).cpu().numpy()
    ns = np.diff(table.node_ptr)
    cent = z.astype(np.float64) - mu
    ref = np.add.reduceat(cent, table.node_ptr[:-1], axis=0)
    bound = gamma(ns[:, None] + 1) * np.add.reduceat(np.abs(cent), table.node_ptr[:-1], axis=0) + 1e-30
    worst = float((np.abs(zs[:, :H] - ref) / bound).max())
    assert np.isfinite(zs).all()
    gid = np.repeat(np.arange(B), ns)
    assert (gid[am] == np.arange(B)[:, None]).all()           # every arg-max is a node of its own graph
    at_max = z[am, np.arange(H)[None, :]] - mu[None, :]       # float32 arithmetic: one rounding, as in the kernel
    assert np.array_equal(bits(zs[:, H:]), bits(at_max))
    # exact ties at the arg-max among nonzero BatchNorm-applied values (symmetric atoms)
    sc = plan.buffer(f"bn_scale{L - 1}", torch.float32, (H,)).cpu().numpy().astype(np.float64)
    sh = plan.buffer(f"bn_shift{L - 1}", torch.float32, (H,)).cpu().numpy().astype(np.float64)
    h = (z * sc + sh).astype(np.float32)
    hmax = h[am, np.arange(H)[None, :]]
    ties = np.add.reduceat((h == hmax[gid]).astype(np.int64), table.node_ptr[:-1], axis=0)
    return worst, int(sum(readout_unstaged(k, H) for k in ns)), int(((ties > 1) & (hmax != 0)).sum())


# ------------------------------------------------------------------------------------------------ molecule-tile SpMM
@pytest.mark.gpu
@pytest.mark.parametrize("H,tile_rows", [(128, 16), (256, 16), (384, 16), (256, 64)])
def test_spmm_molecule_tiles_edge_fallback(H, tile_rows):
    """Edge-dense molecules that fit the tile by atom count but not by directed edges (4 * tile_rows + 64) take the
    per-row gather inside spmm_mol_kernel, next to molecules staged at exactly that edge count and ones over the atom
    count: bit-identical with `eims_spmm_norm` in all five forms (plain, BatchNorm apply, BatchNorm + dropout,
    backward, backward + dropout), rows past the batch untouched."""
    rng = np.random.default_rng(H + tile_rows)
    specials = shapes(*TILE_SPECIALS[tile_rows])
    fill = synth_molecules(30, max_atoms=tile_rows, seed=H + tile_rows)
    src = concat(fill, mol_table(specials, 6, tile_rows))
    order = rng.permutation(src.num_mols)
    table = src.select(order)
    n, nb = sizes(table)
    cap = tile_cap_edges(tile_rows)
    assert ((n <= tile_rows) & (2 * nb > cap)).any() and ((n <= tile_rows) & (2 * nb == cap)).any() and (n > tile_rows).any()
    G = table.num_mols
    b = O.batch_graphs([table.mol(i) for i in range(G)])
    rowptr, col, deg = O.csr_by_dst(b["src"], b["dst"], b["num_nodes"])
    norm = O.degree_norm(deg)
    N, E = b["num_nodes"], len(b["src"])
    gp = dev(O.graph_ptr(b["batch_num_nodes"]), torch.int32)
    hd = dev(rng.standard_normal((N, H)).astype(np.float32))
    scale_d, shift_d = dev(rng.standard_normal(H).astype(np.float32)), dev(rng.standard_normal(H).astype(np.float32))
    dims = make_dims(G, N, E)
    args = (dims, dev(rowptr, torch.int32), dev(col, torch.int32), dev(norm))
    lib = _lib.load()
    P = _lib.ptr
    cases = [(None, None, 0.0, 0), (scale_d, shift_d, 0.0, 0), (scale_d, shift_d, 0.2, 0), (None, None, 0.0, 1), (None, None, 0.35, 1)]
    for sc, sh, p, mode in cases:
        ref = torch.full((N + 3, H), 7.0, device=DEV)
        got = torch.full((N + 3, H), 7.0, device=DEV)
        _lib.check(lib.eims_spmm_norm(*map(P, args), P(hd), H, P(sc), P(sh), p, 99, 5, 1, mode, P(ref), N, stream()))
        _lib.check(lib.eims_spmm_norm_mol(P(dims), P(gp), *map(P, args[1:]), P(hd), H, P(sc), P(sh), p, 99, 5, 1, mode, P(got),
                                          N, G + 5, tile_rows, stream()))
        torch.cuda.synchronize()
        assert bool((got[N:] == 7.0).all()), (p, mode)
        assert torch.equal(got.view(torch.int32), ref.view(torch.int32)), (H, tile_rows, p, mode)


# ------------------------------------------------------------------------------------------------ whole steps
def mixed_table(n_fill, max_atoms, specials, seed, min_atoms=2):
    """Synthetic molecules with the specials mixed in at random positions."""
    fill = synth_molecules(n_fill, max_atoms=max_atoms, seed=seed, min_atoms=min_atoms)
    src = concat(fill, mol_table(shapes(*specials), 6, seed + 1))
    return src.select(np.random.default_rng(seed).permutation(src.num_mols))


def worst_ratio(rep):
    """Largest error over its bound among everything oracle_check bounds."""
    r = [rep[k] / REL for k in ("spectra", "loss", "running", "eval")]
    r += [v / REL for v in rep["grads"].values()] + [v / REL for v in rep["grads_abs"].values()]
    r += [rep["cols"][n] / max(COL_REL, 16 * rep["floors"][n]) for n in rep["cols"]]
    return max(r)


STEP_ROWS = {
    # ~600 molecules in a plan of 4096 (tile_rows 64): the molecule-tile SpMM's fallbacks by atom and by edge count
    # with dropout, K1's oversized branch by atom and by bond count, the unstaged readout at H = 256
    "big_mixed_train": dict(d=ModelDims(6, 256, 3, 1000, "combined", 0.2), fill=580, atoms=40, specials=BIG_TRAIN_SPECIALS,
                            cap=BIG_TRAIN_CAP, paths=["tcgen05"],
                            expect=["spmm_mol_kernel<2, false, 256>", "spmm_norm_kernel<2, 1, true>", "bn_bwd_stats_top_kernel",
                                    "readout_kernel", "k1_build_kernel"]),
    # every graph over the readout tile at H = 1024 (> 16 atoms), symmetric molecules for exact arg-max ties, and the
    # top-layer BatchNorm-backward statistics that come from zstat
    "wide_unstaged": dict(d=ModelDims(6, 1024, 3, 1000, "combined", 0.0), fill=24, atoms=128, min_atoms=17, specials=WIDE_SPECIALS,
                          cap=None, paths=["tcgen05", "tcgen05+planes"],
                          expect=["readout_kernel", "bn_bwd_stats_top_kernel", "spmm_norm_kernel<4, 1, false>"]),
}
STEP_SEEDS = {"big_mixed_train": 900, "wide_unstaged": 950}


def step_cases():
    return [pytest.param(name, path, id=f"{name}-{path}") for name, r in STEP_ROWS.items() for path in r["paths"]]


@pytest.mark.gpu
@pytest.mark.parametrize("name,path", step_cases())
def test_step_reaches_fallbacks(name, path, tmp_path):
    """One training step and one eval forward on a poisoned plan, under the profiler, against the flip-aware fp64
    oracle of test_gpu_dispatch (spectra, loss, every gradient and its column-scaled form, running statistics, eval
    spectra), plus `zstat` of the training forward; the batch really holds the shapes the row is for."""
    r = STEP_ROWS[name]
    d, seed = r["d"], STEP_SEEDS[name]
    H = d.hidden_dim
    table = mixed_table(r["fill"], r["atoms"], r["specials"], seed, r.get("min_atoms", 2))
    B = table.num_mols
    n, nb = sizes(table)
    N, E = int(n.sum()), 2 * int(nb.sum())
    if r["cap"]:
        Bc, Nc = r["cap"]
        caps = (Bc, Nc, 2 * (Nc + 3 * Bc))
        tr = plan_tile_rows(Bc, Nc)
        assert Bc >= MOL_TILE_MIN_GRAPHS and tr == 64
        assert (n > tr).any() and ((n <= tr) & (2 * nb > tile_cap_edges(tr))).any()
        assert (n > K1_MAX_N).any() and ((n <= K1_MAX_N) & (nb > K1_MAX_B)).any()
    else:
        caps = (B, N, E)
    assert readout_unstaged(n, H).sum() >= (B if name == "wide_unstaged" else 10)
    targets = dense_spectra(*synth_peaks(B, d.max_mz, seed=seed + 2), d.max_mz)
    sd = random_running_stats(O.init_params(odims(d), seed + 3), d, seed + 4)
    step = make_step(step=3, seed=11)
    res = run_gpu(d, table, targets, caps, sd, path, step, profile=True)
    rep, bad = oracle_check(d, table, targets, sd, res)
    expect = r["expect"] + (["gemm_planes_kernel"] if path.endswith("+planes") else [])
    missing = [k for k in expect if not any(k in kn for kn in res["kernels"])]
    zworst, zunstaged, zties = zstat_check(d, table, caps, sd, path, step)
    rep.update(row=name, path=path, molecules=B, atoms=N, kernels=res["kernels"], missing=missing,
               worst_error_over_bound=worst_ratio(rep), zstat_sum_error_over_bound=zworst, zstat_unstaged_graphs=zunstaged,
               argmax_nonzero_ties=zties)
    with open(tmp_path / f"graph_shapes_{name}_{path}.json", "w") as fh:
        json.dump(rep, fh, indent=1)
    assert not missing, (missing, res["kernels"])
    assert zworst <= 1.0, ("zstat", zworst)        # before the gradients, which zstat feeds
    assert not bad, (bad, rep)
    if d.dropout == 0.0:
        assert zties > 0          # symmetric molecules without dropout keep exact ties up to the readout


def profiled(fn):
    """fn() under the profiler: (result, kernel names).  The window opens with a synchronised op, because the record
    of a window's very first kernel has been seen missing in a long pytest session."""
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU, torch.profiler.ProfilerActivity.CUDA]) as prof:
        torch.ones(1, device=DEV).add_(1)
        torch.cuda.synchronize()
        out = fn()
        torch.cuda.synchronize()
    return out, kernel_names(prof)


def predict_setup(seed):
    d = ModelDims(6, 256, 3, 1000, "combined", 0.0)
    sd = random_running_stats(O.init_params(odims(d), seed), d, seed + 1)
    fp = FlatParams(d, DEV)
    fp.load_state_dict(sd)
    return d, sd, fp


@pytest.mark.gpu
def test_predict_large_molecules():
    """Eval forward in a plan of 4096 molecules (prescanned K1, molecule-tile SpMM with tile_rows 64) on a batch with
    molecules of up to 1000 atoms, the degree-64 hub among them: spectra within 1e-4 of the fp64 oracle."""
    d, sd, fp = predict_setup(61)
    table = mixed_table(1090, 16, PREDICT_SPECIALS, 62)
    B = table.num_mols
    n, nb = sizes(table)
    assert B > K1_SCAN_CHUNK and n.max() == 1000 and (n > K1_MAX_N).sum() >= 6
    Bc, Nc = 4096, 4096 * 48
    plan = make_plan(d, Bc, Nc, 2 * (Nc + 3 * Bc), "tcgen05")
    ds = DeviceDataset(table, None, DEV)
    out, kernels = profiled(lambda: plan.infer_batch(ds, None, fp).clone().cpu().numpy())
    graph, feat = O.Graph.from_mols([table.mol(i) for i in range(B)])
    ref, _ = O.forward(sd, graph, feat, odims(d), False, dtype=torch.float64)
    assert np.isfinite(out).all()
    assert rel_err(out, ref.numpy()) < REL
    for k in ("k1_scan_kernel", "spmm_mol_kernel<2, false, 256>", "readout_kernel"):
        assert any(k in kn for kn in kernels), (k, kernels)


# ------------------------------------------------------------------------------------------------ batch position
def position_batches(pool, big, sizes_, cap, rng):
    """(label, ids) batches: subsets of the given sizes with `big` at positions 0, 1023, 1024, 2048 and last."""
    others = np.array([g for g in pool if g != big])
    out = []
    for s in sizes_:
        for p in sorted({q for q in (0, 1023, 1024, 2048, s - 1, s // 2) if q < s}):
            ids = rng.choice(others, s - 1, replace=False)
            out.append((f"{s}@{p}", np.insert(ids, p, big)))
    return [(lab, ids) for lab, ids in out if len(ids) <= cap]


@pytest.mark.gpu
def test_eval_spectra_independent_of_batch_position():
    """The eval forward couples nothing across molecules and uses no atomics, so a molecule's spectrum is the same
    bits wherever it sits: in a plan of 4096 (prescanned K1 - whose scan carries across 1024-molecule chunks -,
    molecule-tile SpMM, planes GEMM) and in a plan of 512, over full, reversed and permuted batches and over subsets
    of 1 ... 2049 molecules that put a large molecule at and around the chunk boundaries."""
    d, sd, fp = predict_setup(71)
    table = mixed_table(4096 - len(PREDICT_SPECIALS), 24, PREDICT_SPECIALS, 72)
    G = table.num_mols
    n, _ = sizes(table)
    big = int(np.argmax(n == SHAPES["hub_64x3"].n))
    assert n[big] == SHAPES["hub_64x3"].n
    ds = DeviceDataset(table, None, DEV)
    rng = np.random.default_rng(73)
    for Bc in (4096, 512):
        Nc = Bc * 48
        plan = make_plan(d, Bc, Nc, 2 * (Nc + 3 * Bc), "tcgen05")
        full = rng.permutation(G)[:Bc] if Bc < G else rng.permutation(G)
        if big not in full:
            full[rng.integers(Bc)] = big
        assert int(n[full].sum()) <= Nc
        ref, kernels = profiled(lambda: plan.infer_batch(ds, dev(full, torch.int32), fp).clone().cpu().numpy())
        if Bc == 4096:
            for k in ("k1_scan_kernel", "spmm_mol_kernel<2, false, 256>", "gemm_planes_kernel"):
                assert any(k in kn for kn in kernels), (k, kernels)
        assert np.isfinite(ref).all()
        row = {int(g): k for k, g in enumerate(full)}
        batches = [("reversed", full[::-1].copy()), ("permuted", rng.permutation(full))]
        sub = (1, 2, 1023, 1024, 1025, 2049) if Bc == 4096 else (1, 2, 255, 511, 512)
        batches += position_batches(full, big, sub, Bc, rng)
        assert any(len(ids) > K1_SCAN_CHUNK for _, ids in batches) == (Bc == 4096)
        for label, ids in batches:
            poison(plan)
            out = plan.infer_batch(ds, dev(ids, torch.int32), fp).clone().cpu().numpy()
            want = ref[[row[int(g)] for g in ids]]
            same = np.all(bits(out) == bits(want), axis=1)
            assert same.all(), (Bc, label, np.nonzero(~same)[0][:8])
