"""Host-side mirror of the reference script's interface (templates/ms-pred-gcn-eims-cupy.py,
"GCN:n"): same names, arguments and error behaviour, with the GPU work behind the C ABI.

    Config, get_atom_features, mol_to_dgl_graph, CuPySpectrumProcessor, OptimizedEIMSDataset,
    collate_fn, GCNSpectrum, train_model, predict_spectrum, main

RDKit featurisation stays on the host in Python (north star); DGL and CuPy are not used:
`mol_to_dgl_graph` returns a `MolGraph` (the few DGLGraph members the script touches) and
`collate_fn` a `BatchedGraph` whose `.to(device)` is one packed H2D copy.  There is no CPU
fallback: using the model without a B200 raises.
"""
from __future__ import annotations

import argparse
import glob
import os
import sys
from collections import OrderedDict
from dataclasses import dataclass

import numpy as np
import torch
import torch.nn as nn
from torch.autograd.function import once_differentiable

from . import _lib
from .engine import FlatParams, ModelDims, Plan, make_step, onecycle_schedule, state_dict_order
from .hostpath import PackedHostBatch
from .synth import MolTable

device = torch.device("cuda" if torch.cuda.is_available() else "cpu")


# ------------------------------------------------------------------------------ Config (GCN:73-101)
@dataclass
class Config:
    nist_dir: str = "nist17_data"
    output_dir: str = "processed_data"
    model_save_path: str = "gcn_eims_model.pth"
    max_mz: int = 500
    train_ratio: float = 0.8
    hidden_dim: int = 256
    num_gcn_layers: int = 3
    dropout: float = 0.2
    pooling: str = "combined"
    batch_size: int = 64
    num_epochs: int = 100
    learning_rate: float = 1e-3
    weight_decay: float = 1e-4
    use_cupy: bool = True
    use_mixed_precision: bool = True  # accepted for compatibility; this path is fp32 (BASELINE configs)
    num_workers: int = 4
    cache_graphs: bool = True


_EXTRA_KEYS = ("loss",)  # superset fields tolerated in checkpoints written by this package


# ------------------------------------------------------------------------------ featurisation (GCN:113-153)
def get_atom_features(atom):
    """Six raw descriptors, in the reference's order (GCN:113-122)."""
    return np.array([atom.GetAtomicNum(), atom.GetDegree(), atom.GetFormalCharge(), int(atom.GetHybridization()),
                     int(atom.GetIsAromatic()), atom.GetTotalNumHs()], dtype=np.float32)


class MolGraph:
    """What `dgl.graph((src, dst), num_nodes)` + `ndata['feat']` is to the script: node
    features and the bond list; directed edges are bond k -> (2k: begin->end, 2k+1: end->begin)."""

    def __init__(self, feat: np.ndarray, bond_begin, bond_end):
        self._feat = np.ascontiguousarray(feat, np.float32).reshape(-1, 6) if len(feat) else np.zeros((0, 6), np.float32)
        self._bb = np.asarray(bond_begin, np.int32).reshape(-1)
        self._be = np.asarray(bond_end, np.int32).reshape(-1)
        self.ndata = {"feat": torch.from_numpy(self._feat)}

    def num_nodes(self):
        return len(self._feat)

    number_of_nodes = num_nodes

    def num_edges(self):
        return 2 * len(self._bb)

    def edges(self):
        src = np.empty(2 * len(self._bb), np.int64)
        dst = np.empty_like(src)
        src[0::2], src[1::2] = self._bb, self._be
        dst[0::2], dst[1::2] = self._be, self._bb
        return torch.from_numpy(src), torch.from_numpy(dst)

    @property
    def batch_size(self):
        return 1

    def batch_num_nodes(self):
        return torch.tensor([self.num_nodes()])

    def batch_num_edges(self):
        return torch.tensor([self.num_edges()])

    def to(self, dev):
        return batch([self]).to(dev)


def mol_to_dgl_graph(mol):
    """RDKit Mol -> graph (GCN:124-153).  None in, None out."""
    if mol is None:
        return None
    feats = [get_atom_features(a) for a in mol.GetAtoms()]
    bb, be = [], []
    for bond in mol.GetBonds():
        bb.append(bond.GetBeginAtomIdx())
        be.append(bond.GetEndAtomIdx())
    feat = np.array(feats, dtype=np.float32) if feats else np.zeros((0, 6), np.float32)
    if feat.shape[0] != mol.GetNumAtoms():
        feat = feat.reshape(mol.GetNumAtoms(), -1)
    return MolGraph(feat, bb, be)


class BatchedGraph:
    """`dgl.batch(graphs)` (GCN:295): a packed MolTable on the host; `.to(device)` uploads it
    with one copy.  The CSR / offsets / normalisation are built on the GPU by K1."""

    def __init__(self, table: MolTable):
        self.table = table
        self.ndata = {"feat": torch.from_numpy(table.feat)}
        self.device = torch.device("cpu")
        self._packed = None
        self._dev_buf = None

    @property
    def batch_size(self):
        return self.table.num_mols

    def num_nodes(self):
        return int(self.table.node_ptr[-1])

    def num_edges(self):
        return int(2 * self.table.bond_ptr[-1])

    def batch_num_nodes(self):
        return torch.from_numpy(np.diff(self.table.node_ptr))

    def batch_num_edges(self):
        return torch.from_numpy(2 * np.diff(self.table.bond_ptr))

    def edges(self):
        t = self.table
        off = np.repeat(t.node_ptr[:-1], np.diff(t.bond_ptr))
        src = np.empty(2 * len(t.bond_begin), np.int64)
        dst = np.empty_like(src)
        src[0::2], src[1::2] = t.bond_begin + off, t.bond_end + off
        dst[0::2], dst[1::2] = t.bond_end + off, t.bond_begin + off
        return torch.from_numpy(src), torch.from_numpy(dst)

    def packed(self, targets=None) -> PackedHostBatch:
        if self._packed is None or (targets is not None and not self._packed.has_targets):
            self._packed = PackedHostBatch(self.table, targets, pin=torch.cuda.is_available())
        return self._packed

    def to(self, dev):
        dev = torch.device(dev)
        if dev.type != "cuda":
            return self
        g = BatchedGraph(self.table)
        g._packed = self.packed()
        g._dev_buf = g._packed.buf.to(dev, non_blocking=True)
        g.device = dev
        # the features section of the uploaded batch, as a tensor (no copy): what K1 reads when forward() is given
        # this tensor or no features
        hb, n = g._packed, g.num_nodes()
        o = hb.offsets["feat"]
        g.ndata = {"feat": g._dev_buf[o:o + 4 * n * hb.feat_dim].view(torch.float32).view(n, hb.feat_dim)}
        return g


def batch(graphs) -> BatchedGraph:
    n = np.array([g.num_nodes() for g in graphs], np.int64)
    b = np.array([len(g._bb) for g in graphs], np.int64)
    node_ptr = np.zeros(len(graphs) + 1, np.int64)
    bond_ptr = np.zeros(len(graphs) + 1, np.int64)
    np.cumsum(n, out=node_ptr[1:])
    np.cumsum(b, out=bond_ptr[1:])
    feat = np.concatenate([g._feat for g in graphs]) if graphs else np.zeros((0, 6), np.float32)
    bb = np.concatenate([g._bb for g in graphs]) if graphs else np.zeros(0, np.int32)
    be = np.concatenate([g._be for g in graphs]) if graphs else np.zeros(0, np.int32)
    return BatchedGraph(MolTable(node_ptr, bond_ptr, feat, bb.astype(np.int32), be.astype(np.int32)))


def collate_fn(items):
    """GCN:292-297."""
    graphs, spectra = zip(*items)
    return batch(list(graphs)), torch.stack([torch.as_tensor(s) for s in spectra])


# ------------------------------------------------------------------------------ spectra (GCN:159-221)
class CuPySpectrumProcessor:
    def __init__(self, max_mz=500, use_cupy=True):
        self.max_mz = max_mz
        self.use_cupy = use_cupy

    def peaks_to_spectrum_batch(self, peaks_list):
        """Round half-to-even, max-merge duplicates, drop bins outside [0, max_mz), divide by
        the row maximum.  use_cupy (the reference's default on a GPU machine): the device kernel
        eims_peaks_to_spectrum on float32 m/z - the reference's CuPy branch (GCN:170-191);
        otherwise its NumPy branch (GCN:193-205) on the host, vectorised.  Both bit-identical to
        the reference (tests/test_gpu_kernels.py, tests/test_host_logic.py)."""
        n = len(peaks_list)
        if self.use_cupy and n and torch.cuda.is_available():
            from .engine import DevicePeaks
            lens = np.fromiter((len(p) for p in peaks_list), np.int64, n)
            ptr_ = np.zeros(n + 1, np.int64)
            np.cumsum(lens, out=ptr_[1:])
            flat = np.array([q for p in peaks_list for q in p], dtype=np.float32).reshape(-1, 2)
            return DevicePeaks(ptr_, flat[:, 0], flat[:, 1], device).to_spectrum(self.max_mz).cpu().numpy()
        spectra = np.zeros((n, self.max_mz), dtype=np.float32)
        lens = np.fromiter((len(p) for p in peaks_list), np.int64, n)
        if lens.sum():
            flat = np.array([q for p in peaks_list for q in p], dtype=np.float64).reshape(-1, 2)
            row = np.repeat(np.arange(n), lens)
            b = np.round(flat[:, 0]).astype(np.int64)
            ok = (b >= 0) & (b < self.max_mz)
            np.maximum.at(spectra, (row[ok], b[ok]), flat[ok, 1].astype(np.float32))
        mx = spectra.max(axis=1, keepdims=True) if n else np.zeros((0, 1), np.float32)
        mx = np.where(mx > 0, mx, 1.0)
        return spectra / mx

    def cosine_similarity_batch(self, pred, target):
        """x/(||x||+1e-8) convention of the CuPy branch (GCN:213-215) for device tensors,
        F.normalize for host tensors (GCN:219-221).  The training loop does not call this: the
        fused loss kernel already produces the per-spectrum cosine."""
        if pred.is_cuda:
            pn = pred / (pred.norm(dim=1, keepdim=True) + 1e-8)
            tn = target / (target.norm(dim=1, keepdim=True) + 1e-8)
            return (pn * tn).sum(dim=1)
        return (torch.nn.functional.normalize(pred, p=2, dim=1) * torch.nn.functional.normalize(target, p=2, dim=1)).sum(dim=1)


# ------------------------------------------------------------------------------ dataset (GCN:227-290)
class OptimizedEIMSDataset(torch.utils.data.Dataset):
    """GCN:227-290.  Two additions, both off the reference's path unless asked for:
    `cache_path` - a packed binary cache (dataio.save_packed) written after the first load and
    read instead of the MOL / MSP files afterwards (no RDKit needed then); `robust_msp` - read peak
    lines with several `mz intensity;` pairs (real NIST exports), which the reference's reader
    drops (GCN:277-278)."""

    def __init__(self, mol_files, msp_files, config, cache_path=None, robust_msp=False):
        from . import dataio
        self.graphs, self.spectra, self.config = [], [], config
        self.processor = CuPySpectrumProcessor(config.max_mz, config.use_cupy)
        all_peaks = []
        print("Loading molecular data...")
        if cache_path and os.path.exists(cache_path):
            table, (pptr, pmz, pint), _ = dataio.load_packed(cache_path)
            self.graphs = [MolGraph(*table.mol(g)) for g in range(table.num_mols)]
            all_peaks = [list(zip(pmz[pptr[g]:pptr[g + 1]].tolist(), pint[pptr[g]:pptr[g + 1]].tolist())) for g in range(table.num_mols)]
        else:
            from rdkit import Chem  # RDKit stays on the host; imported lazily (absent offline)
            names = []
            for mol_file, msp_file in zip(mol_files, msp_files):
                mol = Chem.MolFromMolFile(mol_file) if os.path.exists(mol_file) else None
                peaks = self.load_peaks(msp_file) if os.path.exists(msp_file) else None
                if peaks is None and robust_msp and os.path.exists(msp_file):
                    recs = dataio.parse_msp(msp_file)
                    peaks = recs[0]["peaks"] if recs and recs[0]["peaks"] else None
                if mol is not None and peaks is not None:
                    graph = mol_to_dgl_graph(mol) if config.cache_graphs else mol
                    if graph is not None:
                        self.graphs.append(graph)
                        all_peaks.append(peaks)
                        names.append(os.path.basename(mol_file))
            if cache_path and self.graphs and config.cache_graphs:
                lens = np.fromiter((len(p) for p in all_peaks), np.int64, len(all_peaks))
                pptr = np.zeros(len(all_peaks) + 1, np.int64)
                np.cumsum(lens, out=pptr[1:])
                flat = np.array([q for p in all_peaks for q in p], np.float64).reshape(-1, 2)
                dataio.save_packed(cache_path, dataio.pack_graphs(self.graphs), pptr, flat[:, 0], flat[:, 1], names)
        if all_peaks:
            print("Processing spectra...")
            self.spectra = self.processor.peaks_to_spectrum_batch(all_peaks)
        print(f"Dataset size: {len(self.graphs)} molecules")

    @staticmethod
    def load_peaks(msp_file):
        """One `mz intensity` pair per line after a `Num Peaks:` line; any parse error drops
        the molecule (GCN:260-278)."""
        from .dataio import load_peaks_reference
        return load_peaks_reference(msp_file)

    def __len__(self):
        return len(self.graphs)

    def __getitem__(self, idx):
        g = self.graphs[idx] if self.config.cache_graphs else mol_to_dgl_graph(self.graphs[idx])
        return g, torch.FloatTensor(self.spectra[idx])


# ------------------------------------------------------------------------------ model (GCN:303-376)
class _ForwardFn(torch.autograd.Function):
    """Differentiable GCNSpectrum.forward for callers that drive their own loop (`loss.backward()` as in GCN:428, or
    per-atom attribution in eval mode): backward goes through eims_backward_feat, to the parameters (flat) and to the
    atom features x (None: the graph's own, not differentiated).  The parameter gradients are always computed into the
    model's scratch buffer and returned only when flat requires them."""

    @staticmethod
    def forward(ctx, flat, x, model, g):
        prob = model._run_forward(g, training=model.training, feat=x)
        ctx.model, ctx.seq, ctx.done = model, model._fwd_seq, False
        ctx.x_shape = None if x is None else tuple(x.shape)
        return prob

    @staticmethod
    @once_differentiable
    def backward(ctx, dprob):
        m = ctx.model
        if ctx.done:
            raise RuntimeError("GCNSpectrum: this forward was differentiated already")
        if m._fwd_seq != ctx.seq:
            raise RuntimeError("GCNSpectrum: the model ran another forward since this one; its activations are gone "
                               "(call backward before the next forward)")
        ctx.done = True
        want_x = ctx.x_shape is not None and ctx.needs_input_grad[1]
        dfeat = torch.empty(ctx.x_shape, dtype=torch.float32, device=dprob.device) if want_x else None
        m._fp.grads.zero_()
        m._plan.backward_feat(m._fp, dprob.contiguous(), dfeat)
        return (m._fp.grads.clone() if ctx.needs_input_grad[0] else None), dfeat, None, None


class GCNSpectrum(nn.Module):
    """Same constructor, `forward(g, node_features)`, `train()/eval()`, `state_dict()` keys and
    shapes as the reference module (SURVEY A.6); parameters live in one flat fp32 buffer."""

    def __init__(self, node_feat_dim, config):
        super().__init__()
        self.config = config
        self.dims = ModelDims.from_config(config, node_feat_dim)
        from .engine import param_offsets
        self.flat = nn.Parameter(torch.zeros(param_offsets(self.dims)[-1]))
        self._fp = None
        self._plan = None
        self._step = 0
        self._fwd_seq = 0  # forwards run so far: a backward must belong to the last one (_ForwardFn)
        self._seed = int(np.random.SeedSequence().entropy % (1 << 62))
        self._init_host()

    # -- parameters ---------------------------------------------------------------------
    def _views(self, flat):
        from .engine import param_offsets, param_spec
        spec, off = param_spec(self.dims), param_offsets(self.dims)
        return OrderedDict((n, flat[o:o + int(np.prod(s))].view(s)) for (n, s), o in zip(spec, off))

    def _init_host(self):
        """Reference initial distributions: GraphConv xavier-uniform / zero bias (DGL),
        nn.Linear kaiming-uniform(a=sqrt 5) => U(+-1/sqrt(fan_in)), norm layers 1 / 0."""
        with torch.no_grad():
            for name, t in self._views(self.flat.data).items():
                if name.startswith("gcn_layers") and name.endswith("weight"):
                    nn.init.xavier_uniform_(t)
                elif name.startswith("spectrum_predictor") and int(name.split(".")[1]) in (0, 4, 8):
                    fan_in = self._views(self.flat.data)[name.rsplit(".", 1)[0] + ".weight"].shape[1]
                    t.uniform_(-1.0 / np.sqrt(fan_in), 1.0 / np.sqrt(fan_in))
                elif name.endswith("weight"):
                    t.fill_(1.0)
                else:
                    t.zero_()
        L, Hd = self.dims.num_gcn_layers, self.dims.hidden_dim
        self.register_buffer("bn_running", torch.stack([torch.zeros(L, Hd), torch.ones(L, Hd)], dim=1).contiguous())
        self.num_batches_tracked = [0] * L

    def named_views(self):
        return self._views(self.flat.data)

    def state_dict(self, *a, **k):
        sd, p = OrderedDict(), self.named_views()
        for name in state_dict_order(self.dims):
            if name in p:
                sd[name] = p[name].detach().clone()
            else:
                l = int(name.split(".")[1])
                sd[name] = (self.bn_running[l, 0].clone() if name.endswith("running_mean") else
                            self.bn_running[l, 1].clone() if name.endswith("running_var") else
                            torch.tensor(self.num_batches_tracked[l], dtype=torch.int64, device=self.flat.device))
        return sd

    def load_state_dict(self, sd, strict=True):
        order, p = state_dict_order(self.dims), self.named_views()
        missing, unexpected = [n for n in order if n not in sd], [n for n in sd if n not in order]
        if strict and (missing or unexpected):
            raise RuntimeError(f"Error(s) in loading state_dict for GCNSpectrum: missing {missing}, unexpected {unexpected}")
        with torch.no_grad():
            for name, t in sd.items():
                if name not in order:
                    continue
                t = torch.as_tensor(t)
                l = int(name.split(".")[1])
                if name in p:
                    if tuple(t.shape) != tuple(p[name].shape):
                        raise RuntimeError(f"size mismatch for {name}: {tuple(t.shape)} vs {tuple(p[name].shape)}")
                    p[name].copy_(t)
                elif name.endswith("running_mean"):
                    self.bn_running[l, 0].copy_(t)
                elif name.endswith("running_var"):
                    self.bn_running[l, 1].copy_(t)
                else:
                    self.num_batches_tracked[l] = int(t)
        return torch.nn.modules.module._IncompatibleKeys(missing, unexpected)

    # -- engine -------------------------------------------------------------------------
    def _engine(self, n_graphs, n_nodes, n_edges):
        dev = self.flat.device
        if dev.type != "cuda":
            raise RuntimeError("GCNSpectrum (eims_b200) runs on a B200 only: move the model with .to('cuda'); there is no CPU path")
        if self._fp is None or self._fp.params.data_ptr() != self.flat.data.data_ptr():
            fp = FlatParams.__new__(FlatParams)
            fp.d, fp.device = self.dims, dev
            from .engine import param_offsets, param_spec
            fp.spec, fp.offsets = param_spec(self.dims), param_offsets(self.dims)
            fp.numel = fp.offsets[-1]
            fp.params = self.flat.data
            fp.grads = torch.zeros_like(self.flat.data)
            fp.adam_m = fp.adam_v = None
            fp.bn_running = self.bn_running
            fp.num_batches_tracked = self.num_batches_tracked
            self._fp = fp
        p = self._plan
        if p is None or n_graphs > p.max_graphs or n_nodes > p.max_nodes or n_edges > p.max_edges:
            up = lambda v, lo: max(lo, 1 << (int(v) - 1).bit_length())
            self._plan = Plan(self.dims, up(n_graphs, 16), up(n_nodes, 256), up(n_edges, 512), dev)
        return self._plan, self._fp

    def _run_forward(self, g, training, targets=None, feat=None):
        """feat: atom features [N, F] (validated by _node_features) read instead of the graph's own."""
        from .engine import PackedDataset
        if isinstance(g, MolGraph):
            g = g.to(self.flat.device)
        if g._dev_buf is None:
            g = g.to(self.flat.device)
        plan, fp = self._engine(g.batch_size, g.num_nodes(), g.num_edges())
        hb = g._packed
        feat = None if feat is None else feat.detach().contiguous()
        self._keep = (g, feat)  # the packed batch and the features must outlive the asynchronous kernels
        self._fwd_seq += 1
        plan.batch_build(PackedDataset(g._dev_buf.data_ptr(), hb.offsets, hb.num_graphs,
                                       feat=None if feat is None else feat.data_ptr()), None, hb.num_graphs)
        if training:
            self._step += 1
            fp.count_steps()
        plan.forward(fp, training, make_step(step=self._step, seed=self._seed))
        plan.sigmoid()
        plan.check()  # raises ZeroInDegreeError like DGL's GraphConv
        return plan.buffer("prob", torch.float32, (hb.num_graphs, self.dims.max_mz)).clone()

    def _node_features(self, g, node_features):
        """None when the graph's own features are to be read (no features given, or the graph's own tensor that needs
        no gradient); otherwise the tensor, checked as the reference's first GraphConv would check its input."""
        own = getattr(g, "ndata", {}).get("feat")
        if node_features is None or (node_features is own and not node_features.requires_grad):
            return None
        x = node_features
        if not isinstance(x, torch.Tensor):
            raise TypeError(f"node_features must be a tensor, not {type(x).__name__}")
        want = (g.num_nodes(), self.dims.node_feat_dim)
        if tuple(x.shape) != want:
            raise RuntimeError(f"node_features has shape {tuple(x.shape)}; this graph and model need {want}")
        if x.dtype != torch.float32:
            raise RuntimeError(f"node_features must be float32 (the model's dtype), got {x.dtype}")
        if x.device != self.flat.device:
            raise RuntimeError(f"node_features is on {x.device}, the model on {self.flat.device}")
        return x

    def forward(self, g, node_features=None):
        if self.flat.device.type != "cuda":
            self._engine(0, 0, 0)  # raises: no CPU path
        x = self._node_features(g, node_features)
        if torch.is_grad_enabled() and (self.flat.requires_grad or (x is not None and x.requires_grad)):
            return _ForwardFn.apply(self.flat, x, self, g)
        return self._run_forward(g, training=self.training, feat=x)


# ------------------------------------------------------------------------------ training (GCN:382-488)
def _zero_in_degree(table: MolTable) -> bool:
    """True when some atom of the batch has no bond: DGL's GraphConv (allow_zero_in_degree=False, the default the
    reference uses, GCN:316,321) raises DGLError on the first forward of such a batch."""
    n = int(table.node_ptr[-1])
    if n == 0:
        return False
    off = np.repeat(table.node_ptr[:-1], np.diff(table.bond_ptr))
    deg = np.bincount(table.bond_begin + off, minlength=n) + np.bincount(table.bond_end + off, minlength=n)
    return bool((deg == 0).any())


def _loader_capacity(loaders, fallback):
    """(graphs, atoms, directed edges, bytes of a dense-target batch) no batch of these loaders can exceed: the
    batch_size largest molecules of the underlying data set.  Sizes the plan and the staging buffers ONCE, before
    the first step.  None when the loaders do not expose a dataset of MolGraphs (then `fallback` grows on demand)."""
    try:
        bs, atoms, bonds, M = 0, [], [], 0
        for ld in loaders:
            ds = ld.dataset
            base, idx = (ds.dataset, ds.indices) if hasattr(ds, "indices") else (ds, range(len(ds)))
            graphs = base.graphs
            if not all(isinstance(graphs[i], MolGraph) for i in list(idx)[:4]):
                return None
            bs = max(bs, int(ld.batch_size))
            atoms += [graphs[i].num_nodes() for i in idx]
            bonds += [len(graphs[i]._bb) for i in idx]
            M = max(M, int(np.asarray(base.spectra).shape[1]))
        top = lambda v: int(np.sort(np.asarray(v))[::-1][:bs].sum())
        n, b = top(atoms), top(bonds)
        nbytes = 16 * (bs + 1) + 8 * b + 24 * n + 4 * bs * M + 8 * 256
        return bs, n, 2 * b, nbytes
    except Exception:
        return fallback


def train_model(model, train_loader, val_loader, config, loss="mse", world_size=1, allreduce=None, verbose=True):
    """AdamW(lr, weight_decay) + OneCycleLR(max_lr=lr, epochs, steps_per_epoch) + MSE loss, the
    cosine metric per step, an eval pass per epoch, the same history dict and prints
    (GCN:382-488).  Differences by construction: one fused call per step (K1, forward, loss +
    metric, backward, AdamW) and the running loss / cosine stay on the device until the end of
    the epoch instead of three `.item()` syncs per step; the device-side flags (isolated atoms, capacity, non-finite
    loss, a lost data-parallel peer) are read with them, once per epoch.

    Data parallel (new: the reference is single-GPU, GCN:63): under torchrun with an initialised process group and
    world_size > 1 every rank calls this with ITS shard's loader (same number of steps on every rank, e.g.
    `dist.shard_epoch`); gradients are exchanged and the optimiser applied by the fused NVLink kernel
    (`dist.FusedP2PAdamW`), all ranks hold bit-identical weights, BatchNorm statistics stay rank-local (DDP without
    SyncBN) and every rank runs the (replicated) validation pass.  `allreduce` (a callable on the flat gradient
    tensor) selects the plain all-reduce + AdamW path instead."""
    import torch.distributed as tdist
    from .hostpath import HostBatchRunner
    dev = model.flat.device
    steps_per_epoch = len(train_loader)
    sched = onecycle_schedule(config.num_epochs * steps_per_epoch, max_lr=config.learning_rate)
    history = {"train_loss": [], "val_loss": [], "train_cosine": [], "val_cosine": []}
    best_val_cosine = 0
    k = 0
    runner, fused = None, None
    metrics = torch.zeros(8, dtype=torch.float32, device=dev)   # epoch sums live here, whatever happens to the runner
    cap = _loader_capacity((train_loader, val_loader), None)
    if cap is not None:   # size the plan and the staging slots once, from the data set's maxima: nothing regrows mid-epoch
        model._engine(cap[0], cap[1], cap[2])
    pinned, pinned_ev = [], [None, None, None]   # ring of pinned staging buffers, reused (a fresh cudaHostAlloc per step costs
                                                 # more than the step); a buffer is repacked only after the copy that read it
    use_fused = world_size > 1 and allreduce is None and tdist.is_available() and tdist.is_initialized()
    try:
        from tqdm import tqdm
    except Exception:  # pragma: no cover - tqdm is optional
        tqdm = None
    for epoch in range(config.num_epochs):
        model.train()
        metrics.zero_()
        # the reference's progress bar (GCN:409) with its loss / cosine postfix (GCN:439) - read one step behind the
        # GPU through the runner's pinned ring, so the display costs no device synchronisation
        bar = tqdm(train_loader, desc=f"Epoch {epoch+1}/{config.num_epochs}", leave=False) if (verbose and tqdm is not None) else None
        for batch_graph, batch_spectra in (bar if bar is not None else train_loader):
            if _zero_in_degree(batch_graph.table):
                raise _lib.ZeroInDegreeError(_lib.ERR_ZERO_DEGREE, "There are 0-in-degree nodes in the graph (DGL GraphConv would raise)")
            ring = k % 3
            if pinned_ev[ring] is not None:
                pinned_ev[ring].synchronize()
            else:
                pinned_ev[ring] = torch.cuda.Event()
            need = PackedHostBatch.bytes_needed(batch_graph.table, batch_spectra.shape[1])
            if len(pinned) <= ring or pinned[ring].numel() < need:
                size = max(need, cap[3] if cap else 0)
                buf = torch.empty(size, dtype=torch.uint8, pin_memory=True)
                pinned[ring:ring + 1] = [buf]
            hb = PackedHostBatch(batch_graph.table, batch_spectra.numpy(), out=pinned[ring])
            hb._ring_event = pinned_ev[ring]   # recorded by runner.upload after the H2D copy
            plan, fp = model._engine(hb.num_graphs, hb.num_nodes, hb.num_edges)
            if runner is None or runner.plan is not plan or runner.slots[0].numel() < hb.nbytes:
                runner = HostBatchRunner(plan, fp, max(2 * hb.nbytes, cap[3] if cap else 0, 1 << 20), metrics=metrics)
            if use_fused and fused is None:
                from .dist import FusedP2PAdamW, broadcast_params
                broadcast_params(fp)
                fused = FusedP2PAdamW(fp, model.dims.num_gcn_layers, overlap=False)
                model.flat.data = fp.params        # the parameters now live in the symmetric (peer-mapped) buffer
            st = make_step(lr=sched[k][0], beta1=sched[k][1], weight_decay=config.weight_decay, step=k + 1,
                           seed=model._seed, grad_scale=1.0 / world_size)
            slot = runner.upload(hb)
            if fused is not None:
                fused.begin_step()
                runner.train_step(slot, hb, st, loss, optimizer=False)
                fused.finish(st, plan.stream)
            elif allreduce is None:
                runner.train_step(slot, hb, st, loss)
            else:
                runner.train_step(slot, hb, st, loss, optimizer=False)
                allreduce(fp.grads)
                plan.adamw(fp, st)
            model._step = k + 1
            k += 1
            if bar is not None and k % 16 == 0:
                last = runner.read(1)
                if last is not None:
                    bar.set_postfix({"loss": f"{last[0]:.4f}", "cos": f"{last[1]:.4f}"})
        m = metrics.cpu().numpy()
        if runner is not None:
            runner.plan.check()    # capacity / isolated-atom flags K1 left on the device (raises like DGL's GraphConv)
        if m[6] > 0:
            raise FloatingPointError(f"the training loss was NaN / Inf in {int(m[6])} step(s) of epoch {epoch + 1}")
        if fused is not None and fused.lost_peer():
            raise RuntimeError(f"a data-parallel peer did not arrive at the gradient exchange (sequence {fused.lost_peer()})")
        train_loss, train_cosine = float(m[0] / max(m[2], 1)), float(m[1] / max(m[2], 1))
        model.eval()
        vm = torch.zeros(8, device=dev)
        n_val = 0
        with torch.no_grad():
            for batch_graph, batch_spectra in val_loader:
                g = batch_graph.to(dev)
                model._run_forward(g, training=False)
                tgt = batch_spectra.to(dev, non_blocking=True).contiguous()
                model._plan.loss(tgt, None, "mse", False)
                model._plan.metrics_accumulate(vm)
                model._keep_t = tgt
                n_val += 1
        vmh = vm.cpu().numpy()
        val_loss, val_cosine = float(vmh[0] / max(vmh[2], 1)), float(vmh[1] / max(vmh[2], 1))
        history["train_loss"].append(train_loss)
        history["val_loss"].append(val_loss)
        history["train_cosine"].append(train_cosine)
        history["val_cosine"].append(val_cosine)
        if verbose:
            print(f"Epoch {epoch+1}: Train Loss={train_loss:.4f}, Train Cos={train_cosine:.4f}, "
                  f"Val Loss={val_loss:.4f}, Val Cos={val_cosine:.4f}")
        if val_cosine > best_val_cosine:
            best_val_cosine = val_cosine
            # the reference keeps a shallow copy that aliases the live parameters (GCN:476), so
            # what it reloads at the end is the last epoch's weights; nothing to restore here
            if verbose:
                print(f"✓ Best model saved (Val Cosine: {val_cosine:.4f})")
    return model, history


# ------------------------------------------------------------------------------ prediction (GCN:494-511)
def predict_spectrum(model, smiles, config):
    from rdkit import Chem
    mol = Chem.MolFromSmiles(smiles)
    if mol is None:
        return None
    graph = mol_to_dgl_graph(mol)
    if graph is None:
        return None
    return predict_graphs(model, [graph])[0]


def predict_spectrum_batch(model, smiles_list, config, batch_size=4096, top_k=0):
    """predict_spectrum for a list of SMILES in batches of `batch_size` (BASELINE configs[2]):
    a list aligned with the input, None where the reference would return None (GCN:497-502).
    top_k > 0: also the top_k bins (value descending) and their intensities per molecule, found
    on the device (GCN:610-613) -> (spectra, bins, intensities)."""
    from rdkit import Chem
    graphs, where = [], []
    for i, smi in enumerate(smiles_list):
        mol = Chem.MolFromSmiles(smi)
        g = mol_to_dgl_graph(mol) if mol is not None else None
        if g is not None:
            graphs.append(g)
            where.append(i)
    res = predict_graphs(model, graphs, batch_size, top_k=top_k)
    spectra = [None] * len(smiles_list)
    if not top_k:
        for j, i in enumerate(where):
            spectra[i] = res[j]
        return spectra
    bins, vals = [None] * len(smiles_list), [None] * len(smiles_list)
    for j, i in enumerate(where):
        spectra[i], bins[i], vals[i] = res[0][j], res[1][j], res[2][j]
    return spectra, bins, vals


def predict_graphs(model, graphs, batch_size=4096, top_k=0):
    """Batched eval-mode prediction (BASELINE configs[2]); equals the looped single-molecule
    result because eval mode couples nothing across molecules."""
    model.eval()
    out, bins, vals = [], [], []
    with torch.no_grad():
        for s in range(0, len(graphs), batch_size):
            prob = model._run_forward(batch(graphs[s:s + batch_size]).to(model.flat.device), training=False)
            if top_k:
                from .engine import topk_peaks
                bi, va = topk_peaks(prob, top_k)
                bins.append(bi.cpu().numpy())
                vals.append(va.cpu().numpy())
            out.append(prob.cpu().numpy())
    spectra = np.concatenate(out) if out else np.zeros((0, model.dims.max_mz), np.float32)
    if not top_k:
        return spectra
    return (spectra, np.concatenate(bins) if bins else np.zeros((0, top_k), np.int32),
            np.concatenate(vals) if vals else np.zeros((0, top_k), np.float32))


def attribute_peaks(model, graphs, k=5, steps=32, batch_size=4096):
    """Per-atom attribution of every molecule's k strongest predicted peaks by integrated gradients (eval mode, zero
    baseline, midpoint rule with `steps` points; eims_attribute_peaks in include/eims_b200.h).  Each molecule is put k
    times in a row, so one pass attributes all its peaks; a pass holds at most `batch_size` replica graphs.
    Returns (bins int32 [n, k], prob [n, k], delta [n, k], ig) with bins / prob the peaks of `--mode predict`'s report
    (value descending), delta = prob - prob at the all-zero baseline, and ig a list of n arrays [k, n_atoms, F]:
    ig[j].sum() ~= delta[:, j] per molecule (completeness), ig[j].sum(1) the per-atom attribution of peak j."""
    from .engine import PackedDataset
    k, steps = int(k), int(steps)
    if k < 1 or k > model.dims.max_mz or steps < 1:
        raise ValueError(f"need 1 <= k <= max_mz ({model.dims.max_mz}) and steps >= 1")
    model.eval()
    per = max(1, int(batch_size) // k)   # molecules per pass
    bins, prob, delta, ig = [], [], [], []
    with torch.no_grad():
        for s in range(0, len(graphs), per):
            chunk = graphs[s:s + per]
            g = batch([gr for gr in chunk for _ in range(k)]).to(model.flat.device)
            plan, fp = model._engine(g.batch_size, g.num_nodes(), g.num_edges())
            hb = g._packed
            model._keep = (g, None)
            model._fwd_seq += 1   # the activations of an earlier forward are overwritten
            plan.batch_build(PackedDataset(g._dev_buf.data_ptr(), hb.offsets, hb.num_graphs), None, hb.num_graphs)
            plan.check()          # raises ZeroInDegreeError like DGL's GraphConv
            b, p, p0, x = plan.attribute_peaks(fp, k, steps, hb.num_graphs, g.num_nodes())
            n = len(chunk)
            bins.append(b.view(n, k).cpu().numpy())
            p = p.view(n, k)
            prob.append(p.cpu().numpy())
            delta.append((p - p0.view(n, k)).cpu().numpy())
            x = x.cpu().numpy()
            start = 0
            for gr in chunk:
                na = gr.num_nodes()
                ig.append(x[start:start + k * na].reshape(k, na, -1))
                start += k * na
    if not bins:
        return (np.zeros((0, k), np.int32), np.zeros((0, k), np.float32), np.zeros((0, k), np.float32), [])
    return np.concatenate(bins), np.concatenate(prob), np.concatenate(delta), ig


# ------------------------------------------------------------------------------ data parallel (new; the reference is single-GPU)
def _init_data_parallel():
    """(world, rank).  Under torchrun (WORLD_SIZE > 1 in the environment) joins the NCCL process group, one process
    per GPU; otherwise (1, 0) and nothing is initialised - the script behaves exactly like the reference."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world <= 1 or not torch.cuda.is_available():
        return 1, 0
    import torch.distributed as tdist
    global device
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if not tdist.is_initialized():
        tdist.init_process_group("nccl", device_id=device)
    return world, tdist.get_rank()


class ShardedLoader:
    """The train loader of one rank of a data-parallel run: every epoch one shuffle shared by all ranks
    (`dist.shard_epoch`: rank r takes every world-th element, the tail that does not fill a batch on every rank is
    dropped so that all ranks take the same number of steps), collated like the reference's DataLoader (GCN:561-568)."""

    def __init__(self, dataset, batch_size, world, rank, seed=0):
        self.dataset, self.batch_size, self.world, self.rank, self.seed, self.epoch = dataset, int(batch_size), world, rank, seed, 0
        from .dist import shard_epoch
        self._shard = shard_epoch

    def __len__(self):
        return len(self.dataset) // (self.world * self.batch_size)

    def __iter__(self):
        ids = self._shard(len(self.dataset), self.world, self.rank, self.batch_size, self.epoch, self.seed)
        self.epoch += 1
        for row in ids:
            yield collate_fn([self.dataset[int(i)] for i in row])


# ------------------------------------------------------------------------------ CLI (GCN:517-633)
def build_parser():
    parser = argparse.ArgumentParser(description="GCN-based EI-MS Spectrum Prediction")
    parser.add_argument("--mode", type=str, default="train", choices=["train", "predict", "preprocess"], help="run mode")
    parser.add_argument("--data_dir", type=str, default="processed_data", help="data directory")
    parser.add_argument("--msp_file", type=str, help="NIST MSP file")
    parser.add_argument("--mol_dir", type=str, help="directory of MOL files")
    parser.add_argument("--batch_size", type=int, default=64)
    parser.add_argument("--num_epochs", type=int, default=100)
    parser.add_argument("--use_cupy", action="store_true", default=True)
    parser.add_argument("--smiles", type=str, help="SMILES to predict")
    return parser


def main(argv=None):
    args = build_parser().parse_args(argv)
    config = Config()
    config.batch_size, config.num_epochs, config.use_cupy = args.batch_size, args.num_epochs, args.use_cupy
    print("=" * 60)
    print("GCN-based EI-MS Spectrum Prediction System")
    print("=" * 60)
    if args.mode == "train":
        from sklearn.model_selection import train_test_split
        mol_files = glob.glob(os.path.join(args.data_dir, "mol_files", "*.mol"))
        msp_files = [f.replace("mol_files", "msp_files").replace(".mol", ".msp") for f in mol_files]
        print(f"Found {len(mol_files)} molecule files")
        dataset = OptimizedEIMSDataset(mol_files, msp_files, config)
        train_idx, val_idx = train_test_split(range(len(dataset)), test_size=0.2, random_state=42)
        world, rank = _init_data_parallel()
        mk = lambda idx, shuffle: torch.utils.data.DataLoader(torch.utils.data.Subset(dataset, idx), batch_size=config.batch_size,
                                                              shuffle=shuffle, collate_fn=collate_fn, num_workers=config.num_workers,
                                                              pin_memory=False)  # the step packs straight into its own pinned ring (GCN:567)
        if world > 1:
            # one process per GPU (torchrun): rank r trains on its shard of every epoch's shuffle, same step count on every rank
            train_loader = ShardedLoader(torch.utils.data.Subset(dataset, train_idx), config.batch_size, world, rank)
        else:
            train_loader = mk(train_idx, True)
        val_loader = mk(val_idx, False)
        sample_graph, _ = dataset[0]
        model = GCNSpectrum(sample_graph.ndata["feat"].shape[1], config).to(device)
        print(f"Model parameters: {sum(p.numel() for p in model.parameters())}")
        model, history = train_model(model, train_loader, val_loader, config, world_size=world, verbose=(rank == 0))
        if rank == 0:   # every rank holds the same weights; rank 0 writes the reference-format checkpoint (GCN:589-593)
            torch.save({"model_state_dict": model.state_dict(), "config": config.__dict__, "history": history}, config.model_save_path)
            print(f"Model saved to {config.model_save_path}")
        if world > 1:
            torch.distributed.barrier()
            torch.distributed.destroy_process_group()
    elif args.mode == "predict":
        if args.smiles:
            checkpoint = torch.load(config.model_save_path)
            saved_config = Config(**{k: v for k, v in checkpoint["config"].items() if k not in _EXTRA_KEYS})
            model = GCNSpectrum(6, saved_config).to(device)
            model.load_state_dict(checkpoint["model_state_dict"])
            spectrum = predict_spectrum(model, args.smiles, saved_config)
            if spectrum is not None:
                print(f"Predicted spectrum for {args.smiles}")
                print(f"Max intensity at m/z: {np.argmax(spectrum)}")
                print(f"Top 5 peaks: {np.argsort(spectrum)[-5:][::-1]}")
            else:
                print("Failed to predict spectrum")
        else:
            print("Please provide SMILES with --smiles option")
    elif args.mode == "preprocess" and args.msp_file and args.mol_dir:
        # the mode the reference advertises (GCN:626-627) but leaves unimplemented (GCN:619-620)
        from .dataio import preprocess
        preprocess(args.msp_file, args.mol_dir, args.data_dir)
    else:
        print("Mode not implemented")


def demo_banner():
    print("Demo mode - showing example usage")
    print("\n1. Preprocess data:")
    print("   python script.py --mode preprocess --msp_file nist.msp")
    print("\n2. Train model:")
    print("   python script.py --mode train --data_dir processed_data")
    print("\n3. Predict spectrum:")
    print("   python script.py --mode predict --smiles 'CC(C)CC1=CC=C(C=C1)C(C)C'")
