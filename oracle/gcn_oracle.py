"""CPU oracle for the GCN EI-MS hot path  --  TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Only `tests/`, `__graft_entry__.smoke()` and `bench.py`'s CPU-baseline / `--impl reference`
legs may import this module.  The product (`computational-chemistry-ai_b200/`) never does;
it fails loudly when its CUDA library is missing.

What it restates (GCN:n = /root/reference/templates/ms-pred-gcn-eims-cupy.py:n):

  * `mol_edges`            GCN:139-143   bond k -> directed edges 2k (begin->end), 2k+1 (end->begin)
  * `batch_graphs`         GCN:292-297   `dgl.batch`: node ids offset by the running node count,
                                         edges concatenated in graph order, features row-concatenated
  * `graph_conv`           GCN:316,321,359   DGL `GraphConv(norm='both')`, no self loops
  * `forward`              GCN:354-376   L x [GraphConv, ReLU, BatchNorm1d, dropout(not last)],
                                         readout GCN:325-338/366-371, head GCN:341-352
  * `mse_loss`             GCN:393,427
  * `cosine_similarity_batch`  GCN:207-221 (both the CuPy/NumPy and the torch branch)
  * `peaks_to_spectrum_batch`  GCN:193-205 (the NumPy branch, which `cp = np` aliases to, GCN:59)
  * `peaks_to_spectrum_batch_f32`  GCN:170-191 (the CuPy branch: float32 rounding)
  * `make_optimizer`       GCN:385-391   AdamW + OneCycleLR (torch's own classes)
  * `train_step` / `train_epoch`   GCN:410-431

Parity status: **unpinned at the DGL boundary**.  The reference ships no tests or golden
vectors and `dgl` cannot be imported offline (it is not even pinned by the reference's
Dockerfile), so DGL's semantics (edge order kept, GraphConv normalisation with
clamp(min=1), pooling = segment reduce, max-pool gradient to the first arg-max) are
restated from its published source.  Everything else IS pinned: `tests/golden/make_golden.py`
imports the reference script itself (with `oracle/dgl_shim.py` standing in for `dgl`) and
records its outputs; `tests/test_oracle_golden.py` checks this module against them.
"""
from __future__ import annotations

import math
from collections import OrderedDict
from dataclasses import dataclass

import numpy as np
import torch
import torch.nn.functional as F


# --------------------------------------------------------------------------------------
# dims / parameter inventory (SURVEY Appendix A.6; GCN:306-352)
# --------------------------------------------------------------------------------------
@dataclass(frozen=True)
class Dims:
    node_feat_dim: int = 6
    hidden_dim: int = 256
    num_gcn_layers: int = 3
    max_mz: int = 1000
    pooling: str = "combined"
    dropout: float = 0.0

    @property
    def pool_dim(self) -> int:
        return self.hidden_dim * (2 if self.pooling == "combined" else 1)


def state_dict_spec(d: Dims):
    """(name, shape, dtype) in `GCNSpectrum.state_dict()` order (registration order:
    gcn_layers, batch_norms, spectrum_predictor)."""
    H, L, M = d.hidden_dim, d.num_gcn_layers, d.max_mz
    out = []
    for l in range(L):
        fin = d.node_feat_dim if l == 0 else H
        out += [(f"gcn_layers.{l}.weight", (fin, H), torch.float32), (f"gcn_layers.{l}.bias", (H,), torch.float32)]
    for l in range(L):
        out += [(f"batch_norms.{l}.weight", (H,), torch.float32), (f"batch_norms.{l}.bias", (H,), torch.float32),
                (f"batch_norms.{l}.running_mean", (H,), torch.float32),
                (f"batch_norms.{l}.running_var", (H,), torch.float32),
                (f"batch_norms.{l}.num_batches_tracked", (), torch.int64)]
    P = d.pool_dim
    out += [("spectrum_predictor.0.weight", (2 * H, P), torch.float32), ("spectrum_predictor.0.bias", (2 * H,), torch.float32),
            ("spectrum_predictor.1.weight", (2 * H,), torch.float32), ("spectrum_predictor.1.bias", (2 * H,), torch.float32),
            ("spectrum_predictor.4.weight", (H, 2 * H), torch.float32), ("spectrum_predictor.4.bias", (H,), torch.float32),
            ("spectrum_predictor.5.weight", (H,), torch.float32), ("spectrum_predictor.5.bias", (H,), torch.float32),
            ("spectrum_predictor.8.weight", (M, H), torch.float32), ("spectrum_predictor.8.bias", (M,), torch.float32)]
    return out


def is_buffer(name: str) -> bool:
    return name.endswith(("running_mean", "running_var", "num_batches_tracked"))


def init_params(d: Dims, seed: int = 0) -> "OrderedDict[str, torch.Tensor]":
    """Deterministic, torch-RNG-independent initialisation with the reference's
    distributions: GraphConv xavier-uniform weight / zero bias (DGL `reset_parameters`),
    nn.Linear kaiming-uniform(a=sqrt 5) => U(+-1/sqrt(fan_in)) for weight and bias,
    norm layers ones/zeros, BN running stats 0/1."""
    rng = np.random.Generator(np.random.PCG64(seed))
    sd = OrderedDict()
    for name, shape, dt in state_dict_spec(d):
        if name.startswith("gcn_layers") and name.endswith("weight"):
            bound = math.sqrt(6.0 / (shape[0] + shape[1]))
            t = torch.from_numpy(rng.uniform(-bound, bound, size=shape).astype(np.float32))
        elif name.startswith("gcn_layers"):
            t = torch.zeros(shape)
        elif name.startswith("batch_norms"):
            if name.endswith("num_batches_tracked"):
                t = torch.zeros((), dtype=torch.int64)
            elif name.endswith(("weight", "running_var")):
                t = torch.ones(shape)
            else:
                t = torch.zeros(shape)
        else:
            idx = int(name.split(".")[1])
            if idx in (1, 5):  # LayerNorm
                t = torch.ones(shape) if name.endswith("weight") else torch.zeros(shape)
            else:
                lin_w = [s for n, s, _ in state_dict_spec(d) if n == f"spectrum_predictor.{idx}.weight"][0]
                bound = 1.0 / math.sqrt(lin_w[1])
                t = torch.from_numpy(rng.uniform(-bound, bound, size=shape).astype(np.float32))
        sd[name] = t
    return sd


# --------------------------------------------------------------------------------------
# graph construction / batching  (integer work: bit-exact contract, SURVEY A.1)
# --------------------------------------------------------------------------------------
def mol_edges(begin: np.ndarray, end: np.ndarray):
    """GCN:139-143 - src_list.extend([b, e]); dst_list.extend([e, b])."""
    src = np.empty(2 * len(begin), np.int64)
    dst = np.empty(2 * len(begin), np.int64)
    src[0::2], src[1::2] = begin, end
    dst[0::2], dst[1::2] = end, begin
    return src, dst


def batch_graphs(mols):
    """`dgl.batch` (GCN:295).  `mols` = list of (feat[n,F], bond_begin, bond_end); a 2-D feature array
    keeps its own width F, a flat one is read as rows of 6 (the reference's atom features)."""
    srcs, dsts, feats, nn, ne = [], [], [], [], []
    off, width = 0, 6
    for feat, b, e in mols:
        s, d = mol_edges(np.asarray(b, np.int64), np.asarray(e, np.int64))
        srcs.append(s + off)
        dsts.append(d + off)
        f = np.asarray(feat, np.float32)
        width = f.shape[1] if f.ndim == 2 else 6
        feats.append(f.reshape(-1, width) if len(feat) else np.zeros((0, width), np.float32))
        nn.append(len(feat))
        ne.append(len(s))
        off += len(feat)
    cat = lambda xs, dt: np.concatenate(xs).astype(dt) if xs else np.zeros(0, dt)
    return dict(src=cat(srcs, np.int64), dst=cat(dsts, np.int64),
                feat=np.concatenate(feats) if feats else np.zeros((0, width), np.float32),
                batch_num_nodes=np.asarray(nn, np.int64), batch_num_edges=np.asarray(ne, np.int64),
                num_nodes=off)


def csr_by_dst(src: np.ndarray, dst: np.ndarray, num_nodes: int):
    """CSR by destination; inside a row, sources in ascending edge-id order."""
    order = np.argsort(dst, kind="stable")
    col = src[order]
    deg = np.bincount(dst, minlength=num_nodes).astype(np.int64)
    rowptr = np.zeros(num_nodes + 1, np.int64)
    np.cumsum(deg, out=rowptr[1:])
    return rowptr, col, deg


def degree_norm(deg: np.ndarray) -> np.ndarray:
    """DGL GraphConv: `torch.pow(degs.float().clamp(min=1), -0.5)`; fp32, compared as bits."""
    return torch.pow(torch.from_numpy(np.asarray(deg)).float().clamp(min=1), -0.5).numpy()


def graph_ptr(batch_num_nodes: np.ndarray) -> np.ndarray:
    p = np.zeros(len(batch_num_nodes) + 1, np.int64)
    np.cumsum(batch_num_nodes, out=p[1:])
    return p


# --------------------------------------------------------------------------------------
# spectrum processing (GCN:159-221)
# --------------------------------------------------------------------------------------
def peaks_to_spectrum_batch(peaks_list, max_mz: int) -> np.ndarray:
    """Literal restatement of the NumPy branch GCN:193-205."""
    spectra = np.zeros((len(peaks_list), max_mz), dtype=np.float32)
    for i, peaks in enumerate(peaks_list):
        for mz, intensity in peaks:
            mz_int = int(np.round(mz))
            if 0 <= mz_int < max_mz:
                spectra[i, mz_int] = max(spectra[i, mz_int], intensity)
    max_vals = np.max(spectra, axis=1, keepdims=True)
    max_vals = np.where(max_vals > 0, max_vals, 1.0)
    return spectra / max_vals


def peaks_to_spectrum_batch_f32(peaks_list, max_mz: int) -> np.ndarray:
    """Literal restatement of the CuPy branch GCN:170-191 with `cp` bound to NumPy (the alias
    of GCN:59): m/z and intensities become float32 arrays first, so the rounding (half to even)
    happens in float32 - which can pick a different bin than the NumPy branch for m/z within a
    float32 ulp of a half-integer."""
    spectra = np.zeros((len(peaks_list), max_mz), dtype=np.float32)
    for i, peaks in enumerate(peaks_list):
        if peaks:
            mz_array = np.array([p[0] for p in peaks], dtype=np.float32)
            intensity_array = np.array([p[1] for p in peaks], dtype=np.float32)
            mz_indices = np.round(mz_array).astype(np.int32)
            valid_mask = (mz_indices >= 0) & (mz_indices < max_mz)
            for idx, intensity in zip(mz_indices[valid_mask], intensity_array[valid_mask]):
                spectra[i, idx] = np.maximum(spectra[i, idx], intensity)
    max_vals = np.max(spectra, axis=1, keepdims=True)
    max_vals = np.where(max_vals > 0, max_vals, 1.0)
    return spectra / max_vals


def cosine_similarity_batch(pred, target, variant: str = "cupy"):
    """GCN:207-221.  variant 'cupy': x/(||x||+1e-8) (GCN:213-215, what runs on a GPU with
    CuPy and, through `cp = np`, the documented CPU alias); 'torch': F.normalize (GCN:219-221)."""
    if variant == "cupy":
        p = np.asarray(pred.detach() if torch.is_tensor(pred) else pred)
        t = np.asarray(target.detach() if torch.is_tensor(target) else target)
        pn = p / (np.linalg.norm(p, axis=1, keepdims=True) + 1e-8)
        tn = t / (np.linalg.norm(t, axis=1, keepdims=True) + 1e-8)
        return np.sum(pn * tn, axis=1)
    pn = F.normalize(torch.as_tensor(pred), p=2, dim=1)
    tn = F.normalize(torch.as_tensor(target), p=2, dim=1)
    return (pn * tn).sum(dim=1).numpy()


# --------------------------------------------------------------------------------------
# model forward (GCN:354-376) as a pure function of a state dict
# --------------------------------------------------------------------------------------
class Graph:
    """The batched graph in the form the math needs (all torch, CPU)."""

    def __init__(self, src, dst, batch_num_nodes, num_nodes=None):
        self.src = torch.as_tensor(np.asarray(src), dtype=torch.int64)
        self.dst = torch.as_tensor(np.asarray(dst), dtype=torch.int64)
        self.batch_num_nodes = torch.as_tensor(np.asarray(batch_num_nodes), dtype=torch.int64)
        self.num_nodes = int(self.batch_num_nodes.sum()) if num_nodes is None else int(num_nodes)
        self.batch_size = len(self.batch_num_nodes)
        self.gid = torch.repeat_interleave(torch.arange(self.batch_size), self.batch_num_nodes)
        ones = torch.ones(len(self.src))
        self.out_deg = torch.zeros(self.num_nodes).index_add_(0, self.src, ones)
        self.in_deg = torch.zeros(self.num_nodes).index_add_(0, self.dst, ones)

    @classmethod
    def from_mols(cls, mols):
        b = batch_graphs(mols)
        return cls(b["src"], b["dst"], b["batch_num_nodes"], b["num_nodes"]), torch.from_numpy(b["feat"])


class ZeroInDegreeError(RuntimeError):
    """DGL GraphConv(allow_zero_in_degree=False) raises DGLError for isolated nodes."""


def graph_conv(g: Graph, h, W, b):
    """DGL GraphConv, norm='both', aggregate-then-multiply (in_feats <= out_feats)."""
    if bool((g.in_deg == 0).any()):
        raise ZeroInDegreeError("There are 0-in-degree nodes in the graph")
    c_src = torch.pow(g.out_deg.clamp(min=1), -0.5).to(h.dtype)
    c_dst = torch.pow(g.in_deg.clamp(min=1), -0.5).to(h.dtype)
    s = h * c_src[:, None]
    if W.shape[0] > W.shape[1]:  # never on this path; kept for fidelity
        s = s @ W
        a = torch.zeros(g.num_nodes, s.shape[1], dtype=h.dtype).index_add_(0, g.dst, s[g.src])
        r = a
    else:
        a = torch.zeros(g.num_nodes, s.shape[1], dtype=h.dtype).index_add_(0, g.dst, s[g.src])
        r = a @ W
    return r * c_dst[:, None] + b, a


def segment_max_first(h, g: Graph):
    """MaxPooling with DGL's CPU tie rule: the first node (in segment order) attaining
    the max receives the gradient.  Returns (values[B,H], arg[B,H])."""
    N, H = h.shape
    B = g.batch_size
    gid = g.gid[:, None].expand(N, H)
    mx = torch.full((B, H), -float("inf"), dtype=h.dtype).scatter_reduce(0, gid, h.detach(), "amax", include_self=True)
    node = torch.arange(N)[:, None].expand(N, H)
    cand = torch.where(h.detach() == mx[g.gid], node, torch.full_like(node, N))
    arg = torch.full((B, H), N, dtype=torch.int64).scatter_reduce(0, gid, cand, "amin", include_self=True)
    return h.gather(0, arg), arg


def forward(sd, g: Graph, feat, d: Dims, training: bool, *, dropout_masks=None, update_running=True,
            dtype=torch.float32, keep=False, decisions=None):
    """Returns (spectrum[B,M], aux).  `sd` maps state-dict names to tensors (leaf tensors
    with requires_grad for the trainable ones when gradients are wanted).  In training
    mode BN uses batch statistics and (when `update_running`) updates the running buffers
    in place exactly as nn.BatchNorm1d does.  `dropout_masks`: optional dict
    {('gcn', l): keep[N,H], ('head', i): keep[B,*]} of 0/1 masks; when absent and
    d.dropout > 0 in training, torch's own dropout is used (not reproducible on the GPU).
    `decisions` (SURVEY 7.3-2, the flip-aware protocol): optional dict of DISCRETE choices taken
    from another run of the same network, which replace this run's own - {('relu', l): bool[N,H]}
    (z = r * mask instead of max(r, 0)), {('head_relu', i): bool[B,*]} and {'argmax': int64[B,H]}
    (max-pool gathers that node).  With them two implementations differentiate the same
    piecewise-linear branch, so their gradients are comparable at 1e-4 even when a pre-activation
    within rounding distance of 0 falls on different sides."""
    L, p = d.num_gcn_layers, d.dropout
    dec = decisions or {}

    def relu(x, key):
        if key in dec:
            return x * dec[key].to(x.dtype)
        return F.relu(x)
    aux = {}
    cast = (lambda t: t.to(dtype)) if dtype != torch.float32 else (lambda t: t)
    h = cast(feat)

    def drop(x, key):
        if not training or p == 0.0:
            return x
        if dropout_masks is not None:
            return x * cast(dropout_masks[key]) / (1.0 - p)
        return F.dropout(x, p=p, training=True)

    for l in range(L):
        r, a = graph_conv(g, h, cast(sd[f"gcn_layers.{l}.weight"]), cast(sd[f"gcn_layers.{l}.bias"]))
        z = relu(r, ("relu", l))
        rm, rv = sd[f"batch_norms.{l}.running_mean"], sd[f"batch_norms.{l}.running_var"]
        if training and update_running and dtype == torch.float32:
            sd[f"batch_norms.{l}.num_batches_tracked"] += 1
            h = F.batch_norm(z, rm, rv, sd[f"batch_norms.{l}.weight"], sd[f"batch_norms.{l}.bias"], True, 0.1, 1e-5)
        elif training:
            h = F.batch_norm(z, None, None, cast(sd[f"batch_norms.{l}.weight"]), cast(sd[f"batch_norms.{l}.bias"]), True, 0.1, 1e-5)
        else:
            h = F.batch_norm(z, cast(rm), cast(rv), cast(sd[f"batch_norms.{l}.weight"]), cast(sd[f"batch_norms.{l}.bias"]), False, 0.1, 1e-5)
        if keep:
            aux[f"a{l}"], aux[f"r{l}"], aux[f"z{l}"], aux[f"bn{l}"] = a, r, z, h
        if l < L - 1:
            h = drop(h, ("gcn", l))
    N, H = h.shape
    B = g.batch_size
    if d.pooling in ("sum", "mean", "combined"):
        S = torch.zeros(B, H, dtype=h.dtype).index_add_(0, g.gid, h)
    if d.pooling in ("max", "combined"):
        Mx, arg = segment_max_first(h, g)
        if "argmax" in dec:
            arg = dec["argmax"].to(torch.int64)
            Mx = h.gather(0, arg)
        aux["argmax"] = arg
    if d.pooling == "sum":
        G = S
    elif d.pooling == "mean":
        G = S / g.batch_num_nodes.to(h.dtype)[:, None]
    elif d.pooling == "max":
        G = Mx
    else:
        G = torch.cat([S, Mx], dim=1)
    sp = "spectrum_predictor"
    u1 = F.linear(G, cast(sd[f"{sp}.0.weight"]), cast(sd[f"{sp}.0.bias"]))
    y1 = drop(relu(F.layer_norm(u1, (u1.shape[1],), cast(sd[f"{sp}.1.weight"]), cast(sd[f"{sp}.1.bias"]), 1e-5), ("head_relu", 0)), ("head", 0))
    u2 = F.linear(y1, cast(sd[f"{sp}.4.weight"]), cast(sd[f"{sp}.4.bias"]))
    y2 = drop(relu(F.layer_norm(u2, (u2.shape[1],), cast(sd[f"{sp}.5.weight"]), cast(sd[f"{sp}.5.bias"]), 1e-5), ("head_relu", 1)), ("head", 1))
    u3 = F.linear(y2, cast(sd[f"{sp}.8.weight"]), cast(sd[f"{sp}.8.bias"]))
    P = torch.sigmoid(u3)
    if keep:
        aux.update(G=G, u1=u1, y1=y1, u2=u2, y2=y2, u3=u3)
    return P, aux


def mse_loss(pred, target):
    return F.mse_loss(pred, target)


def cosine_loss(pred, target):
    """North-star variant (`--loss cosine`): 1 - mean cosine (x/(||x||+1e-8) convention)."""
    pn = pred / (pred.norm(dim=1, keepdim=True) + 1e-8)
    tn = target / (target.norm(dim=1, keepdim=True) + 1e-8)
    return 1.0 - (pn * tn).sum(dim=1).mean()


def trainable(sd):
    return [n for n in sd if not is_buffer(n)]


def loss_and_grads(sd, g, feat, target, d: Dims, *, training=True, dropout_masks=None, loss_kind="mse",
                   dtype=torch.float32, update_running=False, keep=False, decisions=None):
    """One forward + autograd backward.  Returns (pred, loss, grads dict, aux)."""
    work = OrderedDict()
    for n, t in sd.items():
        if is_buffer(n):
            work[n] = t if update_running else t.clone()
        else:
            work[n] = t.detach().to(dtype).clone().requires_grad_(True)
    pred, aux = forward(work, g, feat, d, training, dropout_masks=dropout_masks,
                        update_running=update_running, dtype=dtype, keep=keep, decisions=decisions)
    tgt = target.to(dtype)
    loss = mse_loss(pred, tgt) if loss_kind == "mse" else cosine_loss(pred, tgt)
    names = trainable(work)
    gs = torch.autograd.grad(loss, [work[n] for n in names], retain_graph=keep)
    return pred.detach(), loss.detach(), OrderedDict(zip(names, gs)), aux


# --------------------------------------------------------------------------------------
# optimiser (GCN:385-391, 429-431): torch's own AdamW + OneCycleLR
# --------------------------------------------------------------------------------------
def onecycle_table(total_steps: int, max_lr: float = 1e-3):
    """(lr, beta1) that AdamW sees at optimiser step k = 0..total-1 (scheduler.step() is
    called after optimizer.step(), GCN:429-431)."""
    p = torch.nn.Parameter(torch.zeros(1))
    opt = torch.optim.AdamW([p], lr=max_lr)
    sch = torch.optim.lr_scheduler.OneCycleLR(opt, max_lr=max_lr, total_steps=total_steps)
    out = []
    for _ in range(total_steps):
        out.append((opt.param_groups[0]["lr"], opt.param_groups[0]["betas"][0]))
        opt.step()
        sch.step()
    return out


class Trainer:
    """Stateful oracle trainer: parameters as leaf tensors, torch AdamW + OneCycleLR."""

    def __init__(self, sd, d: Dims, total_steps: int, lr: float = 1e-3, weight_decay: float = 1e-4,
                 loss_kind: str = "mse"):
        self.d = d
        self.sd = OrderedDict((n, (t.clone() if is_buffer(n) else t.clone().requires_grad_(True))) for n, t in sd.items())
        self.names = trainable(self.sd)
        self.opt = torch.optim.AdamW([self.sd[n] for n in self.names], lr=lr, weight_decay=weight_decay)
        self.sched = torch.optim.lr_scheduler.OneCycleLR(self.opt, max_lr=lr, total_steps=total_steps)
        self.loss_kind = loss_kind

    def step(self, g, feat, target, dropout_masks=None, world_shards=None):
        """One training step (GCN:414-431).  `world_shards`: optional list of
        (g, feat, target) per emulated rank - gradients are averaged (DDP semantics,
        BN statistics stay shard-local, rank 0's running stats are kept)."""
        self.opt.zero_grad(set_to_none=True)
        shards = world_shards if world_shards is not None else [(g, feat, target)]
        preds, losses = [], []
        for r, (gg, ff, tt) in enumerate(shards):
            sd_r = self.sd if r == 0 else OrderedDict((n, (t.clone() if is_buffer(n) else t)) for n, t in self.sd.items())
            pred, _ = forward(sd_r, gg, ff, self.d, True, dropout_masks=dropout_masks)
            loss = mse_loss(pred, tt) if self.loss_kind == "mse" else cosine_loss(pred, tt)
            (loss / len(shards)).backward()
            preds.append(pred.detach())
            losses.append(float(loss.detach()))
        self.opt.step()
        self.sched.step()
        return preds[0] if world_shards is None else preds, losses[0] if world_shards is None else losses

    @torch.no_grad()
    def predict(self, g, feat):
        return forward(self.sd, g, feat, self.d, False)[0]

    def state_dict(self):
        return OrderedDict((n, t.detach().clone()) for n, t in self.sd.items())
