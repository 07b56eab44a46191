"""Thin host-side objects over the C ABI: device-resident molecule tables, the workspace
plan and the flat parameter buffer.  torch is used for device memory and streams only."""
from __future__ import annotations

import ctypes as C
import math
from collections import OrderedDict
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib
from ._lib import Dataset, Dims, Step, check, ptr
from .synth import MolTable


@dataclass(frozen=True)
class ModelDims:
    node_feat_dim: int = 6
    hidden_dim: int = 256
    num_gcn_layers: int = 3
    max_mz: int = 500
    pooling: str = "combined"
    dropout: float = 0.2

    @property
    def pool_dim(self):
        return self.hidden_dim * (2 if self.pooling == "combined" else 1)

    def c(self) -> Dims:
        return Dims(self.node_feat_dim, self.hidden_dim, self.num_gcn_layers, self.max_mz,
                    _lib.POOLING[self.pooling], float(self.dropout))

    @classmethod
    def from_config(cls, config, node_feat_dim=6):
        return cls(node_feat_dim, config.hidden_dim, config.num_gcn_layers, config.max_mz, config.pooling, config.dropout)


def param_spec(d: ModelDims):
    """(state-dict name, shape) of the trainable tensors in `model.parameters()` order
    (SURVEY Appendix A.6); offsets come from the library (eims_param_layout)."""
    H, L, M, P = d.hidden_dim, d.num_gcn_layers, d.max_mz, d.pool_dim
    spec = []
    for l in range(L):
        spec += [(f"gcn_layers.{l}.weight", (d.node_feat_dim if l == 0 else H, H)), (f"gcn_layers.{l}.bias", (H,))]
    for l in range(L):
        spec += [(f"batch_norms.{l}.weight", (H,)), (f"batch_norms.{l}.bias", (H,))]
    sp = "spectrum_predictor"
    spec += [(f"{sp}.0.weight", (2 * H, P)), (f"{sp}.0.bias", (2 * H,)), (f"{sp}.1.weight", (2 * H,)), (f"{sp}.1.bias", (2 * H,)),
             (f"{sp}.4.weight", (H, 2 * H)), (f"{sp}.4.bias", (H,)), (f"{sp}.5.weight", (H,)), (f"{sp}.5.bias", (H,)),
             (f"{sp}.8.weight", (M, H)), (f"{sp}.8.bias", (M,))]
    return spec


def param_offsets(d: ModelDims):
    lib = _lib.load()
    cd = d.c()
    n = lib.eims_param_num_tensors(C.byref(cd))
    if n < 0:
        check(_lib.ERR_ARG)
    arr = (C.c_int64 * (n + 1))()
    check(lib.eims_param_layout(C.byref(cd), arr, n + 1))
    return list(arr)


def state_dict_order(d: ModelDims):
    """Full state_dict key order of the reference GCNSpectrum (parameters + BN buffers)."""
    names = []
    for l in range(d.num_gcn_layers):
        names += [f"gcn_layers.{l}.weight", f"gcn_layers.{l}.bias"]
    for l in range(d.num_gcn_layers):
        names += [f"batch_norms.{l}.{k}" for k in ("weight", "bias", "running_mean", "running_var", "num_batches_tracked")]
    names += [n for n, _ in param_spec(d)[4 * d.num_gcn_layers:]]
    return names


class FlatParams:
    """Flat fp32 parameter / gradient / Adam-state buffers with named views, plus the
    BatchNorm buffers [L,2,H] (running_mean, running_var) and num_batches_tracked."""

    def __init__(self, d: ModelDims, device):
        self.d, self.device = d, torch.device(device)
        self.spec = param_spec(d)
        self.offsets = param_offsets(d)
        self.numel = self.offsets[-1]
        self.params = torch.zeros(self.numel, dtype=torch.float32, device=self.device)
        self.grads = torch.zeros_like(self.params)
        self.adam_m = None
        self.adam_v = None
        self.bn_running = torch.zeros(d.num_gcn_layers, 2, d.hidden_dim, dtype=torch.float32, device=self.device)
        self.bn_running[:, 1].fill_(1.0)
        self.num_batches_tracked = [0] * d.num_gcn_layers

    def ensure_adam(self):
        if self.adam_m is None:
            self.adam_m = torch.zeros_like(self.params)
            self.adam_v = torch.zeros_like(self.params)

    def step_ptrs(self, optimizer=True):
        """params, grads, adam_m, adam_v, bn_running as arguments of a training step; without the optimiser the Adam
        state is NULL (the step runs no AdamW)."""
        if optimizer:
            self.ensure_adam()
        return (ptr(self.params), ptr(self.grads), ptr(self.adam_m) if optimizer else None,
                ptr(self.adam_v) if optimizer else None, ptr(self.bn_running))

    def count_steps(self, n=1):
        """n more training-mode forwards: what BatchNorm's num_batches_tracked counts."""
        for l in range(len(self.num_batches_tracked)):
            self.num_batches_tracked[l] += n

    def views(self, flat):
        out = OrderedDict()
        for (name, shape), o in zip(self.spec, self.offsets):
            out[name] = flat[o:o + int(np.prod(shape))].view(shape)
        return out

    def named_params(self):
        return self.views(self.params)

    def named_grads(self):
        return self.views(self.grads)

    def state_dict(self):
        sd = OrderedDict()
        p = self.named_params()
        for name in state_dict_order(self.d):
            if name in p:
                sd[name] = p[name].detach().clone()
            else:
                l = int(name.split(".")[1])
                if name.endswith("running_mean"):
                    sd[name] = self.bn_running[l, 0].clone()
                elif name.endswith("running_var"):
                    sd[name] = self.bn_running[l, 1].clone()
                else:
                    sd[name] = torch.tensor(self.num_batches_tracked[l], dtype=torch.int64, device=self.device)
        return sd

    def load_state_dict(self, sd, strict=True):
        p = self.named_params()
        missing = [n for n in state_dict_order(self.d) if n not in sd]
        unexpected = [n for n in sd if n not in state_dict_order(self.d)]
        if strict and (missing or unexpected):
            raise RuntimeError(f"Error(s) in loading state_dict: missing {missing}, unexpected {unexpected}")
        with torch.no_grad():
            for name, t in sd.items():
                t = torch.as_tensor(t)
                if name in p:
                    if tuple(t.shape) != tuple(p[name].shape):
                        raise RuntimeError(f"size mismatch for {name}: {tuple(t.shape)} vs {tuple(p[name].shape)}")
                    p[name].copy_(t.to(self.device, torch.float32))
                elif name.endswith("running_mean"):
                    self.bn_running[int(name.split(".")[1]), 0].copy_(t.to(self.device, torch.float32))
                elif name.endswith("running_var"):
                    self.bn_running[int(name.split(".")[1]), 1].copy_(t.to(self.device, torch.float32))
                elif name.endswith("num_batches_tracked"):
                    self.num_batches_tracked[int(name.split(".")[1])] = int(t)


class DevicePeaks:
    """Peak lists of a set of spectra resident in HBM (flat: peak_ptr int64[G+1], mz, intensity):
    the `peaks_list` of CuPySpectrumProcessor.peaks_to_spectrum_batch (GCN:166).  m/z is kept in
    float64 (the precision the reference's NumPy branch rounds in, GCN:193-196) unless the arrays
    handed in are float32 (what its CuPy branch rounds, GCN:176-179)."""

    def __init__(self, peak_ptr, mz, intensity, device="cuda"):
        self.device = torch.device(device)
        peak_ptr = np.ascontiguousarray(peak_ptr, np.int64)
        mz = np.ascontiguousarray(mz)
        if mz.dtype != np.float32:
            mz = mz.astype(np.float64)
        self.num_spectra = len(peak_ptr) - 1
        self.num_peaks = int(peak_ptr[-1]) if len(peak_ptr) else 0
        pad = lambda a: a if a.size else np.zeros(1, a.dtype)
        self.peak_ptr = torch.from_numpy(peak_ptr).to(self.device)
        self.mz = torch.from_numpy(pad(mz)).to(self.device)
        self.intensity = torch.from_numpy(pad(np.ascontiguousarray(intensity, np.float32))).to(self.device)
        self._struct = _lib.Peaks(self.peak_ptr.data_ptr(), self.mz.data_ptr(), self.intensity.data_ptr(),
                                  int(mz.dtype == np.float64), self.num_spectra)

    @classmethod
    def from_device(cls, peak_ptr, mz, intensity):
        """Peak lists whose flat arrays are device tensors already (mz float32 or float64)."""
        self = cls.__new__(cls)
        self.device = peak_ptr.device
        self.peak_ptr = peak_ptr.to(torch.int64).contiguous()
        self.num_spectra = self.peak_ptr.numel() - 1
        self.num_peaks = int(self.peak_ptr[-1]) if self.peak_ptr.numel() else 0
        if mz.dtype not in (torch.float32, torch.float64):
            mz = mz.to(torch.float64)
        self.mz = mz.contiguous() if mz.numel() else torch.zeros(1, dtype=mz.dtype, device=self.device)
        self.intensity = intensity.to(torch.float32).contiguous() if intensity.numel() else torch.zeros(1, device=self.device)
        self._struct = _lib.Peaks(self.peak_ptr.data_ptr(), self.mz.data_ptr(), self.intensity.data_ptr(),
                                  int(self.mz.dtype == torch.float64), self.num_spectra)
        return self

    @classmethod
    def from_lists(cls, peaks_list, device="cuda"):
        """From the reference's list-of-lists-of-(mz, intensity) form (GCN:166, 260-278)."""
        lens = np.fromiter((len(p) for p in peaks_list), np.int64, len(peaks_list))
        ptr_ = np.zeros(len(peaks_list) + 1, np.int64)
        np.cumsum(lens, out=ptr_[1:])
        flat = np.array([q for p in peaks_list for q in p], dtype=np.float64).reshape(-1, 2)
        return cls(ptr_, flat[:, 0], flat[:, 1].astype(np.float32), device)

    @property
    def struct(self):
        return self._struct

    @property
    def nbytes(self):
        return self.peak_ptr.numel() * 8 + self.mz.numel() * self.mz.element_size() + self.intensity.numel() * 4

    def to_spectrum(self, max_mz, rows=None, out=None):
        """peaks_to_spectrum_batch on the device: [len(rows) or num_spectra, max_mz] float32."""
        n = self.num_spectra if rows is None else len(rows)
        if out is None:
            out = torch.empty((n, max_mz), dtype=torch.float32, device=self.device)
        check(_lib.load().eims_peaks_to_spectrum(C.byref(self._struct), ptr(rows), n, int(max_mz), ptr(out),
                                                 C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)))
        return out


def topk_peaks(spectra: torch.Tensor, k: int = 5):
    """(bins int32 [n,k], intensities float32 [n,k]) of the k largest bins of every row of a
    device tensor of spectra: the report of `--mode predict` (GCN:610-613) for a whole batch."""
    spectra = spectra.contiguous()
    n, m = spectra.shape
    idx = torch.empty((n, k), dtype=torch.int32, device=spectra.device)
    val = torch.empty((n, k), dtype=torch.float32, device=spectra.device)
    check(_lib.load().eims_topk_peaks(ptr(spectra), n, m, int(k), ptr(idx), ptr(val),
                                      C.c_void_p(torch.cuda.current_stream(spectra.device).cuda_stream)))
    return idx, val


class DeviceDataset:
    """A MolTable (+ target spectra, dense rows or peak lists) resident in HBM: ~1 KB of graph data
    and 4*max_mz bytes of dense targets - or ~12 bytes per peak - per molecule (DESIGN.md §3)."""

    def __init__(self, table: MolTable, targets=None, device="cuda", pinned_stage=False, peaks: "DevicePeaks" = None):
        self.device = torch.device(device)
        self.num_mols = table.num_mols
        self.host_num_atoms = np.diff(table.node_ptr).astype(np.int64)
        self.host_num_bonds = np.diff(table.bond_ptr).astype(np.int64)
        up = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a)).to(dt).to(self.device, non_blocking=False)
        self.node_ptr = up(table.node_ptr, torch.int64)
        self.bond_ptr = up(table.bond_ptr, torch.int64)
        self.feat = up(table.feat.reshape(-1), torch.float32) if table.feat.size else torch.zeros(1, device=self.device)
        self.bond_begin = up(table.bond_begin, torch.int32) if table.bond_begin.size else torch.zeros(1, dtype=torch.int32, device=self.device)
        self.bond_end = up(table.bond_end, torch.int32) if table.bond_end.size else torch.zeros(1, dtype=torch.int32, device=self.device)
        if isinstance(targets, torch.Tensor):     # already resident (e.g. binned on the device from peak lists)
            self.targets = targets.to(self.device, torch.float32).contiguous()
        else:
            self.targets = None if targets is None else up(np.asarray(targets, np.float32), torch.float32)
        self.peaks = peaks
        self._make_struct()

    @classmethod
    def from_device(cls, node_ptr, bond_ptr, feat, bond_begin, bond_end, targets=None, peaks: "DevicePeaks" = None):
        """A data set whose flat arrays are device tensors already (assembled on the GPU, e.g. from the shards the
        ranks of a data-parallel job generated)."""
        self = cls.__new__(cls)
        self.device = node_ptr.device
        self.num_mols = node_ptr.numel() - 1
        self.node_ptr, self.bond_ptr = node_ptr.to(torch.int64).contiguous(), bond_ptr.to(torch.int64).contiguous()
        self.host_num_atoms = torch.diff(self.node_ptr).cpu().numpy().astype(np.int64)
        self.host_num_bonds = torch.diff(self.bond_ptr).cpu().numpy().astype(np.int64)
        self.feat = feat.to(torch.float32).contiguous().view(-1)
        self.bond_begin, self.bond_end = bond_begin.to(torch.int32).contiguous(), bond_end.to(torch.int32).contiguous()
        self.targets = None if targets is None else targets.to(torch.float32).contiguous()
        self.peaks = peaks
        self._make_struct()
        return self

    def _make_struct(self):
        peaks = self.peaks
        self._struct = Dataset(self.node_ptr.data_ptr(), self.bond_ptr.data_ptr(), self.feat.data_ptr(),
                               self.bond_begin.data_ptr(), self.bond_end.data_ptr(),
                               0 if self.targets is None else self.targets.data_ptr(), self.num_mols,
                               C.pointer(peaks.struct) if peaks is not None else None)

    @property
    def struct(self) -> Dataset:
        return self._struct

    def batch_counts(self, ids):
        ids = np.asarray(ids)
        return int(self.host_num_atoms[ids].sum()), int(2 * self.host_num_bonds[ids].sum())


class PackedDataset:
    """One packed batch (the layout of eims_host_pack_batch / PackedHostBatch) at device address `base`, as the data set
    of its `num_graphs` molecules.  offsets: section name -> byte offset from base; a section that is absent has no
    entry.  Duck-types DeviceDataset for the plan: struct, targets (an address), peaks (a Peaks struct).  feat: the
    address of other atom features [N, F] in the batch's order, read instead of the packed ones."""

    def __init__(self, base: int, offsets, num_graphs: int, mz_is_f64: int = 0, feat: int | None = None):
        o = offsets
        self.num_mols = int(num_graphs)
        self.targets = base + o["targets"] if "targets" in o else None
        self.peaks = (_lib.Peaks(base + o["peak_ptr"], base + o["peak_mz"], base + o["peak_inten"], mz_is_f64, self.num_mols)
                      if "peak_ptr" in o else None)
        self.struct = Dataset(base + o["node_ptr"], base + o["bond_ptr"], base + o["feat"] if feat is None else feat, base + o["bond_begin"],
                              base + o["bond_end"], self.targets, self.num_mols,
                              C.pointer(self.peaks) if self.peaks is not None else None)


def make_step(lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=1e-4, grad_scale=1.0, step=1, seed=0) -> Step:
    return Step(lr, beta1, beta2, eps, weight_decay, grad_scale, int(step), int(seed))


def onecycle_schedule(total_steps, max_lr=1e-3, pct_start=0.3, div_factor=25.0, final_div_factor=1e4,
                      base_momentum=0.85, max_momentum=0.95):
    """(lr, beta1) seen by optimiser step k = 0..total-1: torch.optim.lr_scheduler.OneCycleLR
    (cos anneal, two phases) as the reference configures it (GCN:386-391), scheduler stepped
    after the optimiser (GCN:429-431).  Checked against torch in tests/test_host_logic.py."""
    initial_lr = max_lr / div_factor
    min_lr = initial_lr / final_div_factor
    phase1_end = float(pct_start * total_steps) - 1
    phase2_end = float(total_steps) - 1

    def cos(start, end, pct):
        return end + (start - end) / 2.0 * (math.cos(math.pi * pct) + 1)

    out = []
    for k in range(total_steps):
        if k <= phase1_end:
            pct = k / phase1_end if phase1_end != 0 else 0.0
            out.append((cos(initial_lr, max_lr, pct), cos(max_momentum, base_momentum, pct)))
        else:
            pct = (k - phase1_end) / (phase2_end - phase1_end)
            out.append((cos(max_lr, min_lr, pct), cos(base_momentum, max_momentum, pct)))
    return out


class Plan:
    """Workspace plan for batches of up to (max_graphs, max_nodes, max_edges)."""

    def __init__(self, d: ModelDims, max_graphs, max_nodes, max_edges, device="cuda", gemm_backend=None):
        if not torch.cuda.is_available():
            raise RuntimeError("eims_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.lib = _lib.load()
        self.d, self.device = d, torch.device(device)
        with torch.cuda.device(self.device):
            check(self.lib.eims_device_check())
        self.max_graphs, self.max_nodes, self.max_edges = int(max_graphs), int(max_nodes), int(max_edges)
        h = C.c_void_p()
        cd = d.c()
        check(self.lib.eims_plan_create(C.byref(cd), self.max_graphs, self.max_nodes, self.max_edges, C.byref(h)))
        self.h = h
        self._peak_targets = None  # what eims_plan_set_peak_targets was last given (keeps the arrays alive)
        nbytes = self.lib.eims_plan_workspace_bytes(self.h)
        self.workspace = torch.empty(nbytes + 256, dtype=torch.uint8, device=self.device)
        self._base = (self.workspace.data_ptr() + 255) // 256 * 256
        with torch.cuda.device(self.device):
            check(self.lib.eims_plan_bind(self.h, C.c_void_p(self._base), nbytes))
            torch.cuda.synchronize()
        if gemm_backend is not None:
            self.set_gemm_backend(gemm_backend)

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.lib.eims_plan_destroy(self.h)
                self.h = None
        except Exception:
            pass

    def set_gemm_planes(self, mode):
        """'auto' (default) / 'off' / 'on': which kernel runs the GraphConv products (eims_plan_set_gemm_planes)."""
        m = {"auto": -1, "off": 0, "on": 1}.get(mode, mode)
        check(self.lib.eims_plan_set_gemm_planes(self.h, int(m)))

    def set_gemm_backend(self, backend):
        b = {"tcgen05": _lib.GEMM_TCGEN05, "simt": _lib.GEMM_FP32_SIMT}.get(backend, backend)
        check(self.lib.eims_plan_set_gemm_backend(self.h, int(b)))

    @property
    def stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def buffer(self, name, dtype=torch.float32, shape=None):
        p, n = C.c_void_p(), C.c_int64()
        check(self.lib.eims_plan_buffer(self.h, name.encode(), C.byref(p), C.byref(n)))
        off = p.value - self.workspace.data_ptr()
        t = self.workspace[off:off + n.value].view(dtype)
        if shape is not None:
            t = t[: int(np.prod(shape))].view(shape)
        return t

    # -- stages ---------------------------------------------------------------------
    def batch_build(self, ds: DeviceDataset, ids, num_graphs=None):
        n = int(num_graphs if num_graphs is not None else (len(ids) if ids is not None else ds.num_mols))
        check(self.lib.eims_batch_build(self.h, C.byref(ds.struct), ptr(ids), n, self.stream))
        self.num_graphs = n

    def check(self):
        nn, ne = C.c_int32(), C.c_int32()
        check(self.lib.eims_plan_check(self.h, C.byref(nn), C.byref(ne), self.stream))
        return nn.value, ne.value

    def forward(self, fp: FlatParams, training: bool, step: Step | None = None):
        check(self.lib.eims_forward(self.h, ptr(fp.params), ptr(fp.bn_running), int(training),
                                    C.byref(step) if step is not None else None, self.stream))

    def sigmoid(self):
        check(self.lib.eims_sigmoid(self.h, self.stream))

    def set_peak_targets(self, peaks):
        """Targets as peak lists, binned inside the loss kernel (eims_plan_set_peak_targets): a DevicePeaks, the Peaks
        struct of a PackedDataset, or None."""
        s = peaks if peaks is None or isinstance(peaks, _lib.Peaks) else peaks.struct
        check(self.lib.eims_plan_set_peak_targets(self.h, C.byref(s) if s is not None else None))
        self._peak_targets = peaks

    def _targets(self, ds):
        """Dense targets of a DeviceDataset or PackedDataset; without them (None) the plan is pointed at its peak lists."""
        peaks = ds.peaks if ds.targets is None else None
        if peaks is not self._peak_targets:
            self.set_peak_targets(peaks)
        return ds.targets

    def loss(self, targets, target_rows=None, loss_kind="mse", want_grad=True):
        check(self.lib.eims_loss(self.h, ptr(targets), ptr(target_rows), _lib.LOSS[loss_kind], int(want_grad), self.stream))

    def backward(self, fp: FlatParams, dprob=None):
        check(self.lib.eims_backward(self.h, ptr(fp.params), ptr(dprob), ptr(fp.grads), self.stream))

    def backward_feat(self, fp: FlatParams, dprob=None, dfeat=None):
        """The backward of the forward enqueued last, training or eval mode (eims_backward_feat): parameter gradients
        added into fp.grads and, when `dfeat` (a float32 [N, F] device tensor) is given, the gradient w.r.t. the
        batch's atom features written into it.  dprob may be None only after loss(want_grad=True) in training mode."""
        check(self.lib.eims_backward_feat(self.h, ptr(fp.params), ptr(dprob), ptr(fp.grads), ptr(dfeat), self.stream))

    def metrics_accumulate(self, metrics):
        check(self.lib.eims_metrics_accumulate(self.h, ptr(metrics), self.stream))

    def adamw(self, fp: FlatParams, step: Step):
        fp.ensure_adam()
        check(self.lib.eims_adamw_flat(ptr(fp.params), ptr(fp.grads), ptr(fp.adam_m), ptr(fp.adam_v), fp.numel,
                                       C.byref(step), self.stream))

    def train_step(self, ds: DeviceDataset, ids, fp: FlatParams, step: Step, metrics=None, loss_kind="mse",
                   optimizer=True, num_graphs=None):
        """K1 + forward + loss + backward [+ AdamW] of one batch of `ds` (a DeviceDataset or a PackedDataset)."""
        n = int(num_graphs if num_graphs is not None else (len(ids) if ids is not None else ds.num_mols))
        check(self.lib.eims_train_step(self.h, C.byref(ds.struct), ptr(ids), n, *fp.step_ptrs(optimizer),
                                       _lib.LOSS[loss_kind], C.byref(step), ptr(metrics), self.stream))
        self.num_graphs = n
        fp.count_steps()

    def train_step_built(self, ds, ids, fp: FlatParams, step: Step, metrics=None, loss_kind="mse", optimizer=True):
        """Forward + loss + backward [+ AdamW] on the batch built last; ids: its target rows in `ds` (None: in order)."""
        check(self.lib.eims_train_step_built(self.h, ptr(self._targets(ds)), ptr(ids), *fp.step_ptrs(optimizer),
                                             _lib.LOSS[loss_kind], C.byref(step), ptr(metrics), self.stream))
        fp.count_steps()

    def train_step_prefetch(self, ds: DeviceDataset, ids, next_ids, fp: FlatParams, step: Step, metrics=None, loss_kind="mse",
                            optimizer=True, on_head_grads=None):
        """A training step whose batch tables were built ahead of time: K1 of the NEXT batch runs on
        a side stream while this step computes (the plan double-buffers the tables), which takes
        the batch build off the critical path.  Call with next_ids=None for the last step."""
        cur = torch.cuda.current_stream(self.device)
        if getattr(self, "_side", None) is None:
            self._side = torch.cuda.Stream(self.device)
            self._built = None       # (event, ids data_ptr) of the batch waiting in the current table set
            self._step_end = [None, None]
        n = len(ids)
        if self._built is None or self._built[1] != ids.data_ptr():
            self.batch_build(ds, ids, n)             # cold start: build on the compute stream
        else:
            cur.wait_event(self._built[0])
        if on_head_grads is None:
            self.train_step_built(ds, ids, fp, step, metrics, loss_kind, optimizer)
        elif optimizer:
            raise ValueError("on_head_grads is for the data-parallel path, which runs its own optimiser kernel")
        else:
            self._train_split(ds, ids, fp, step, metrics, loss_kind, on_head_grads)
        self.num_graphs = n
        end = torch.cuda.Event()
        end.record(cur)
        prev_end, self._step_end = self._step_end[1], [self._step_end[1], end]
        self._built = None
        if next_ids is not None:
            # the table set the next build overwrites was last read by the PREVIOUS step
            if prev_end is not None:
                self._side.wait_event(prev_end)
            with torch.cuda.stream(self._side):
                self.batch_build(ds, next_ids, len(next_ids))
                ev = torch.cuda.Event()
                ev.record(self._side)
            self._built = (ev, next_ids.data_ptr())
            self._keep_ids = next_ids

    def train_step_split(self, ds: DeviceDataset, ids, fp: FlatParams, step: Step, metrics=None, loss_kind="mse",
                         on_head_grads=None, num_graphs=None):
        """K1 + forward + loss + backward without the optimiser, with a host callback between the
        head and the GCN part of the backward pass (data-parallel bucket overlap, dist.py)."""
        n = int(num_graphs if num_graphs is not None else (len(ids) if ids is not None else ds.num_mols))
        self.batch_build(ds, ids, n)
        self._train_split(ds, ids, fp, step, metrics, loss_kind, on_head_grads)

    def _train_split(self, ds, ids, fp, step, metrics, loss_kind, on_head_grads):
        """train_step_split on the batch built last."""
        self.forward(fp, True, step)
        self.loss(self._targets(ds), ids, loss_kind, True)
        if metrics is not None:
            self.metrics_accumulate(metrics)
        check(self.lib.eims_backward_part(self.h, ptr(fp.params), None, ptr(fp.grads), _lib.BWD_HEAD, self.stream))
        if on_head_grads is not None:
            on_head_grads()
        check(self.lib.eims_backward_part(self.h, ptr(fp.params), None, ptr(fp.grads), _lib.BWD_GCN, self.stream))
        fp.count_steps()

    # -- device step block / CUDA-graph replay (include/eims_b200.h, "one optimiser step as a replayable CUDA graph")
    def enable_step_block(self, count: int = 1):
        """Device array of `count` step blocks (one per step a captured graph holds)."""
        n = int(self.lib.eims_step_block_bytes())
        if getattr(self, "_step_block", None) is None or self._step_block.numel() < n * count:
            self._step_block = torch.zeros(n * count + 16, dtype=torch.uint8, device=self.device)
            check(self.lib.eims_plan_set_step_block(self.h, ptr(self._step_block), n * count))
            self._step_block_bytes = n
        return self._step_block

    def select_step_block(self, index: int):
        check(self.lib.eims_plan_select_step_block(self.h, int(index)))

    def step_block_ptr(self, index: int):
        return C.c_void_p(self._step_block.data_ptr() + int(index) * self._step_block_bytes)

    def step_blocks_args(self, steps, ids_list, dp_seqs):
        """The host-side half of step_blocks_upload: the ctypes arrays of one launch (<= 16 blocks).  An ids entry of
        None makes that step's indirect batch build take molecules 0..n-1 of its dataset."""
        n = len(steps)
        arr = (Step * n)(*steps)
        pid = (C.c_void_p * n)(*[None if t is None else t.data_ptr() for t in ids_list])
        seq = (C.c_uint32 * n)(*[int(x) & 0xffffffff for x in dp_seqs])
        return arr, pid, seq, n

    def step_blocks_upload(self, steps, ids_list, dp_seqs, first: int = 0, prepared=None):
        """Rewrite blocks [first, first + len(steps)) with one launch (<= 16 blocks)."""
        arr, pid, seq, n = prepared if prepared is not None else self.step_blocks_args(steps, ids_list, dp_seqs)
        check(self.lib.eims_step_blocks_upload(self.h, arr, pid, seq, int(first), n, self.stream))

    def step_block_upload(self, step: Step, ids, dp_seq: int = 0):
        """Rewrite the device step block: AdamW scalars + dropout keys of `step`, the ids the next indirect batch
        build reads, the data-parallel sequence number.  One 1-block kernel on the current stream, the one
        step_blocks_upload launches."""
        check(self.lib.eims_step_block_upload(self.h, C.byref(step), ptr(ids), C.c_uint32(int(dp_seq) & 0xffffffff), self.stream))

    def batch_build_indirect(self, ds: DeviceDataset, num_graphs: int):
        check(self.lib.eims_batch_build_indirect(self.h, C.byref(ds.struct), int(num_graphs), self.stream))
        self.num_graphs = int(num_graphs)

    def train_step_built_indirect(self, ds: DeviceDataset, fp: FlatParams, metrics=None, loss_kind="mse", optimizer=True, side=None):
        """side: a torch stream for the step's side branch (output-layer bias gradient, AdamW of the head tensors)."""
        check(self.lib.eims_train_step_built_indirect(self.h, ptr(self._targets(ds)), *fp.step_ptrs(optimizer),
                                                      _lib.LOSS[loss_kind], ptr(metrics), self.stream,
                                                      C.c_void_p(side.cuda_stream) if side is not None else None))

    def train_step_built_indirect_part(self, ds: DeviceDataset, fp: FlatParams, part: int, metrics=None, loss_kind="mse"):
        """part 1: forward + loss + head backward; part 2: GraphConv backward (eims_train_step_built_indirect_part)."""
        check(self.lib.eims_train_step_built_indirect_part(self.h, ptr(self._targets(ds)), ptr(fp.params), ptr(fp.grads),
                                                           ptr(fp.bn_running), _lib.LOSS[loss_kind], ptr(metrics), int(part), self.stream))

    # -- per-stage profiling (bench.py) ------------------------------------------------
    def profile(self, enable: bool):
        check(self.lib.eims_plan_profile(self.h, int(enable)))

    def profile_read(self):
        """{stage: (total ms, brackets)} and the kernel-launch count since profile() was called."""
        n = self.lib.eims_plan_num_stages()
        ms, cnt, tot = (C.c_float * n)(), (C.c_int32 * n)(), C.c_int64()
        check(self.lib.eims_plan_profile_read(self.h, ms, cnt, n, C.byref(tot)))
        names = [self.lib.eims_plan_stage_name(k).decode() for k in range(n)]
        return {names[k]: (float(ms[k]), int(cnt[k])) for k in range(n)}, int(tot.value)

    def infer_batch(self, ds: DeviceDataset, ids, fp: FlatParams, out=None, num_graphs=None):
        n = int(num_graphs if num_graphs is not None else (len(ids) if ids is not None else ds.num_mols))
        check(self.lib.eims_infer_batch(self.h, C.byref(ds.struct), ptr(ids), n, ptr(fp.params), ptr(fp.bn_running),
                                        ptr(out), self.stream))
        self.num_graphs = n
        return out if out is not None else self.buffer("prob", torch.float32, (n, self.d.max_mz))


class StepReplay:
    """What the replayed training loops (GraphedTrainStep, hostpath.GraphedHostTrainer) share: the enqueue of one step
    that reads its scalars from a device step block, the capture bracket and the exchange's sequence numbers.
    Subclasses set plan, fp, metrics, loss_kind, fused (a dist.FusedP2PAdamW or None) and side2."""

    def _enqueue_step(self, ds, block: int, step):
        """One step on the batch built last, with the scalars of step block `block`: forward, loss, backward and AdamW
        (the output layer's bias gradient and the head's AdamW on side2), or the fused exchange as the optimiser."""
        plan, fused = self.plan, self.fused
        plan.select_step_block(block)
        if fused is None:
            plan.train_step_built_indirect(ds, self.fp, self.metrics, self.loss_kind, side=self.side2)
            return
        fused.begin_step()
        blk = plan.step_block_ptr(block)
        if fused.side is not None:
            # two buckets: the head's exchange + AdamW (84 % of the parameters) runs on the exchange's side stream under
            # the GraphConv backward, only the GraphConv bucket is left for the end of the step
            plan.train_step_built_indirect_part(ds, self.fp, 1, self.metrics, self.loss_kind)
            fused.head_ready(step, step_block=blk)
            plan.train_step_built_indirect_part(ds, self.fp, 2, self.metrics, self.loss_kind)
        else:
            plan.train_step_built_indirect(ds, self.fp, self.metrics, self.loss_kind, optimizer=False)
        fused.finish(step, plan.stream, step_block=blk)

    def _capture(self, *bodies):
        """One CUDA graph per callable, captured in turn.  Capture runs nothing, so the exchange's sequence number is
        restored at the end: each graph kept the gradient buffer its place in that sequence selected."""
        seq0 = self.fused.seq if self.fused is not None else 0
        graphs = []
        for body in bodies:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                body()
            graphs.append(g)
        if self.fused is not None:
            self.fused.seq = seq0
        return graphs

    def _seqs(self, n: int):
        """Exchange sequence numbers of the next n replayed steps (0 without the exchange)."""
        return self.fused.next_seqs(n) if self.fused is not None else [0] * n


class GraphedTrainStep(StepReplay):
    """Optimiser steps (GCN:410-431) as replayed CUDA graphs: the host issues one tiny kernel (the step-block upload)
    and one cudaGraphLaunch per GROUP of steps instead of ~30 kernel launches per step, so a descheduled Python thread
    no longer stalls the GPU - which matters most in data-parallel runs, where every rank waits for the slowest one at
    the gradient exchange.

    A captured step holds
        main stream:  forward + loss + backward + AdamW on the current batch tables   [+ fused exchange kernel]
        side stream:  K1 batch build of the NEXT batch into the other set of tables (the plan double-buffers them)
        side stream 2 (single GPU): output-layer bias gradient and the head's AdamW
    and reads everything that changes from step to step from its own device step block.  Two graphs are captured:
    `group` (even, <= 16) consecutive steps in one graph - inside it one step's last kernel chains into the next
    step's first with programmatic dependent launch, as eager launches do, so the ~10 us gap between two graph launches
    is paid once per group (single steps: 0.3436 ms/step, eager 0.3337, measured on one box) - and a pair of single-step
    graphs for what does not fill a group.  `step()` queues, a full group launches at once, `flush()` launches the rest.
    torch is plumbing here (stream capture, graph launch)."""

    def __init__(self, plan: Plan, ds: DeviceDataset, fp: FlatParams, batch: int, metrics=None, loss_kind="mse", fused=None, group: int = 10):
        import os
        self.plan, self.ds, self.fp, self.batch, self.metrics, self.loss_kind, self.fused = plan, ds, fp, int(batch), metrics, loss_kind, fused
        self.group = max(0, min(16, int(os.environ.get("EIMS_GRAPH_GROUP", group)))) // 2 * 2   # even: table parity returns
        self.singles, self.multi, self.k, self.primed = [], None, 0, False
        self.pending = []
        # hold_next: the next full group is prepared on the host (scalars, sequence numbers, argument arrays) but not
        # launched; release() launches it.  Lets a timing harness put a start barrier between the two, so that the ranks'
        # host-side preparation skew is not inside a short timed window (the device work all is).
        self.hold_next, self.held = False, None
        self.side = torch.cuda.Stream(plan.device)
        # second side branch: the bias gradient of the output layer and the head's AdamW run off the chain (single GPU;
        # in data-parallel runs the fused exchange kernel is the optimiser)
        self.side2 = torch.cuda.Stream(plan.device) if fused is None else None
        plan.enable_step_block(max(self.group, 1))
        if fused is None:
            fp.ensure_adam()

    def _enqueue(self, block: int, step):
        cur = torch.cuda.current_stream(self.plan.device)
        self.side.wait_stream(cur)                       # fork: the build may start with the step
        self._enqueue_step(self.ds, block, step)
        with torch.cuda.stream(self.side):
            self.plan.batch_build_indirect(self.ds, self.batch)
        cur.wait_stream(self.side)                       # join

    def capture(self, first_ids, step: Step):
        """Builds batch `first_ids` for real (cold start), then captures the graphs.  Call after a few eager
        warm-up steps (module loading and one-time attribute calls must not happen under capture)."""
        plan = self.plan
        plan.select_step_block(0)
        plan.step_blocks_upload([step], [first_ids], [0], 0)
        plan.batch_build(self.ds, first_ids, self.batch)
        torch.cuda.synchronize(plan.device)
        self.singles = self._capture(lambda: self._enqueue(0, step), lambda: self._enqueue(0, step))   # block 0
        if self.group >= 2:
            self.multi, = self._capture(lambda: [self._enqueue(j, step) for j in range(self.group)])
        plan.select_step_block(0)
        self._keep = [first_ids]
        self.k, self.primed = 0, True

    def _launch(self, items):
        """items: queued (Step, next_ids); a full group goes out as the multi-step graph (only from table parity 0,
        the one it was captured at), anything else step by step through the single-step graphs."""
        seqs = self._seqs(len(items))
        self._keep = [ids for _, ids in items]
        if self.multi is not None and len(items) == self.group and self.k == 0:
            prep = self.plan.step_blocks_args([st for st, _ in items], [ids for _, ids in items], seqs)
            if self.hold_next:      # everything host-side is done; release() issues the upload kernel and the graph launch
                self.hold_next, self.held = False, prep
            else:
                self.plan.step_blocks_upload(None, None, None, 0, prepared=prep)
                self.multi.replay()
        else:
            for (st, ids), q in zip(items, seqs):
                self.plan.step_blocks_upload([st], [ids], [q], 0)
                self.singles[self.k].replay()
                self.k ^= 1
        self.fp.count_steps(len(items))

    def can_hold(self, n_steps: int) -> bool:
        """A full group can be prepared now and launched later with release() (see hold_next)."""
        return self.primed and self.multi is not None and self.k == 0 and not self.pending and n_steps >= self.group and self.held is None

    def release(self):
        """Launch the group that was prepared while hold_next was set: one upload kernel + one graph launch."""
        prep, self.held = self.held, None
        self.plan.step_blocks_upload(None, None, None, 0, prepared=prep)
        self.multi.replay()

    def step(self, step: Step, next_ids):
        """Queues the step on the batch built last (and the build of `next_ids`, same length as every batch, for the
        following one); a full group is launched at once.  Call flush() before reading results."""
        if not self.primed:
            raise RuntimeError("GraphedTrainStep.capture() first")
        self.pending.append((step, next_ids))
        if self.multi is None or self.k != 0 or len(self.pending) >= self.group:
            self.flush()

    def flush(self):
        if self.pending:
            items, self.pending = self.pending, []
            self._launch(items)
