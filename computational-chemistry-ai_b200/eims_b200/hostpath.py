"""The reference-facing call with HOST buffers: a batch of molecules (packed MolTable slice +
target spectra, as dense rows or as the peak lists they are binned from) in pinned host memory -> one H2D copy -> K1 + forward + loss +
backward + AdamW -> loss / cosine read back to the host.

This is what `collate_fn` + `.to(device)` + one `train_model` iteration do in the reference
(GCN:292-297, 411-439); bench.py times it as `e2e`.  Two device slots are used so the
upload of batch i+1 and its K1 batch build (both on the copy stream; the plan double-buffers
the batch tables) overlap the compute of batch i.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import Dataset, check
from .engine import PackedDataset, StepReplay
from .synth import MolTable


def _align(n, a=256):
    return (n + a - 1) // a * a


def _offsets(lay) -> dict:
    """Section offsets of an eims_host_batch_layout (a section at -1 is absent)."""
    return {n: getattr(lay, n) for n in ("node_ptr", "bond_ptr", "bond_begin", "bond_end", "feat", "targets", "peak_ptr",
                                         "peak_mz", "peak_inten") if getattr(lay, n) >= 0}


class PackedHostBatch:
    """One batch packed into a single pinned byte buffer:
    [node_ptr i64 | bond_ptr i64 | bond_begin i32 | bond_end i32 | feat f32 | targets f32]
    or, with peaks=(peak_ptr, mz, intensity) of the batch instead of dense targets,
    [... | feat f32 | peak_ptr i64 | peak_mz f32/f64 | peak_inten f32]  (binned on the device inside
    the loss kernel: ~1 KB instead of 4*max_mz bytes per molecule over PCIe)."""

    @staticmethod
    def bytes_needed(table: MolTable, max_mz: int) -> int:
        """Size of the packed buffer of `table` with dense [B, max_mz] targets."""
        B, N, nb = table.num_mols, int(table.node_ptr[-1]), int(table.bond_ptr[-1])
        F = table.feat.shape[1] if table.feat.ndim == 2 else 6
        return sum(_align(x) for x in (8 * (B + 1), 8 * (B + 1), 4 * nb, 4 * nb, 4 * N * F, 4 * B * int(max_mz)))

    def __init__(self, table: MolTable, targets: np.ndarray | None, pin=True, peaks=None, out=None):
        """out: an existing (pinned) uint8 buffer of at least the packed size to write into instead of allocating."""
        B, N, nb = table.num_mols, int(table.node_ptr[-1]), int(table.bond_ptr[-1])
        F = table.feat.shape[1] if table.feat.ndim == 2 else 6
        parts = [("node_ptr", table.node_ptr.astype(np.int64)), ("bond_ptr", table.bond_ptr.astype(np.int64)),
                 ("bond_begin", table.bond_begin.astype(np.int32)), ("bond_end", table.bond_end.astype(np.int32)),
                 ("feat", np.ascontiguousarray(table.feat, np.float32).reshape(-1))]
        self.mz_is_f64 = 0
        if targets is not None:
            parts.append(("targets", np.ascontiguousarray(targets, np.float32).reshape(-1)))
        elif peaks is not None:
            pptr, mz, inten = peaks
            mz = np.ascontiguousarray(mz)
            if mz.dtype != np.float32:
                mz = mz.astype(np.float64)
            self.mz_is_f64 = int(mz.dtype == np.float64)
            pad = lambda a: a if a.size else np.zeros(1, a.dtype)
            parts += [("peak_ptr", np.ascontiguousarray(pptr, np.int64)), ("peak_mz", pad(mz)),
                      ("peak_inten", pad(np.ascontiguousarray(inten, np.float32)))]
        self.offsets, off = {}, 0
        for name, a in parts:
            self.offsets[name] = off
            off = _align(off + a.nbytes)
        self.nbytes = off
        if out is not None:
            if out.numel() < off:
                raise ValueError(f"staging buffer too small: {out.numel()} < {off}")
            self.buf = out
        else:
            self.buf = torch.empty(off, dtype=torch.uint8, pin_memory=pin)
        view = self.buf.numpy()
        for name, a in parts:
            o = self.offsets[name]
            view[o:o + a.nbytes] = a.view(np.uint8).reshape(-1)
        self.num_graphs, self.num_nodes, self.num_edges, self.feat_dim = B, N, 2 * nb, F
        self.has_targets = targets is not None
        self.has_peaks = targets is None and peaks is not None


class HostDataset:
    """A MolTable (+ dense target rows or peak lists) in HOST memory behind an `eims_dataset` of host pointers:
    what the reference's `OptimizedEIMSDataset` holds (GCN:227-258), packed."""

    def __init__(self, table: MolTable, targets: np.ndarray | None = None, peaks=None):
        c = np.ascontiguousarray
        self.node_ptr, self.bond_ptr = c(table.node_ptr, np.int64), c(table.bond_ptr, np.int64)
        self.feat = c(table.feat, np.float32).reshape(-1, table.feat.shape[1] if table.feat.ndim == 2 else 6)
        self.bond_begin, self.bond_end = c(table.bond_begin, np.int32), c(table.bond_end, np.int32)
        self.feat_dim = self.feat.shape[1]
        self.targets = None if targets is None else c(targets, np.float32)
        self.max_mz = 0 if self.targets is None else self.targets.shape[1]
        self.num_mols = len(self.node_ptr) - 1
        self._peaks = None
        a = lambda x: x.ctypes.data if x is not None and x.size else None
        if targets is None and peaks is not None:
            pptr, mz, inten = peaks
            mz = c(mz)
            if mz.dtype != np.float32:
                mz = mz.astype(np.float64)
            self._pk_arrays = (c(pptr, np.int64), mz if mz.size else np.zeros(1, mz.dtype),
                               c(inten, np.float32) if len(inten) else np.zeros(1, np.float32))
            self._peaks = _lib.Peaks(self._pk_arrays[0].ctypes.data, self._pk_arrays[1].ctypes.data,
                                     self._pk_arrays[2].ctypes.data, int(mz.dtype == np.float64), self.num_mols)
        self.struct = Dataset(self.node_ptr.ctypes.data, self.bond_ptr.ctypes.data, self.feat.ctypes.data,
                              a(self.bond_begin) or self.node_ptr.ctypes.data, a(self.bond_end) or self.node_ptr.ctypes.data,
                              a(self.targets), self.num_mols, C.pointer(self._peaks) if self._peaks is not None else None)


class HostPacker:
    """`collate_fn` (GCN:292-297) + pin_memory (GCN:567) as one C call (`eims_host_pack_batch`): gathers a batch of
    molecule ids from a HostDataset straight into a pinned buffer of a small ring, ready for ONE H2D copy.
    The ring buffer handed out by `pack` is reused `n_buffers` calls later; by then its upload
    (`HostBatchRunner.upload`, which records the buffer's event) has long finished, and `pack` waits if not."""

    def __init__(self, hds: HostDataset, max_mz: int, capacity_bytes: int, n_buffers: int = 4, pin: bool = True):
        self.hds, self.max_mz = hds, int(max_mz or hds.max_mz)
        self.lib = _lib.load()
        self.bufs = [torch.empty(int(capacity_bytes), dtype=torch.uint8, pin_memory=pin) for _ in range(n_buffers)]
        self.events = [None] * n_buffers
        self._i = 0

    def pack(self, ids: np.ndarray) -> PackedHostBatch:
        k = self._i % len(self.bufs)
        self._i += 1
        if self.events[k] is not None:
            self.events[k].synchronize()      # the H2D copy that read this buffer has completed
        ids = np.ascontiguousarray(ids, np.int32)
        lay = _lib.HostBatchLayout()
        buf = self.bufs[k]
        check(self.lib.eims_host_pack_batch(C.byref(self.hds.struct), C.c_void_p(ids.ctypes.data), len(ids), self.hds.feat_dim,
                                            self.max_mz, C.c_void_p(buf.data_ptr()), buf.numel(), C.byref(lay)))
        hb = PackedHostBatch.__new__(PackedHostBatch)
        hb.offsets = _offsets(lay)
        hb.nbytes, hb.buf, hb.mz_is_f64 = int(lay.nbytes), buf, int(lay.mz_is_f64)
        hb.num_graphs, hb.num_nodes, hb.num_edges, hb.feat_dim = lay.num_graphs, lay.num_nodes, lay.num_edges, lay.feat_dim
        hb.has_targets, hb.has_peaks = lay.targets >= 0, lay.peak_ptr >= 0
        if buf.is_pinned() and torch.cuda.is_available():
            if self.events[k] is None:
                self.events[k] = torch.cuda.Event()
            hb._ring_event = self.events[k]
        return hb


class HostBatchRunner:
    """Runs training / inference steps whose inputs start in (pinned) host memory."""

    def __init__(self, plan, fp, capacity_bytes, n_slots=2, metrics=None):
        """metrics: the caller's device tensor [8] the steps accumulate into (kept across runner rebuilds)."""
        self.plan, self.fp = plan, fp
        dev = plan.device
        self.slots = [torch.empty(capacity_bytes, dtype=torch.uint8, device=dev) for _ in range(n_slots)]
        self.copy_stream = torch.cuda.Stream(dev)
        self.copied = [torch.cuda.Event() for _ in range(n_slots)]
        self.consumed = [None] * n_slots
        self.built = [False] * n_slots
        self.metrics = metrics if metrics is not None else torch.zeros(8, dtype=torch.float32, device=dev)
        # the per-step loss / cosine come back through two pinned buffers used in turn, each with the event of its
        # device-to-host copy: the host reads a step's values only after that event (`read`), one step behind the GPU
        self.RING = 4
        self.host_ring = [torch.zeros(8, dtype=torch.float32, pin_memory=True) for _ in range(self.RING)]
        self.d2h_done = [torch.cuda.Event() for _ in range(self.RING)]
        self._n = 0
        self.h2d_bytes = 0
        self.d2h_bytes = 0
        self._i = 0

    def _dataset(self, slot, hb: PackedHostBatch) -> PackedDataset:
        return PackedDataset(self.slots[slot].data_ptr(), hb.offsets, hb.num_graphs, hb.mz_is_f64)

    def upload(self, hb: PackedHostBatch, build: bool = False):
        """Enqueue the H2D copy of `hb` (and, with build=True, its K1 batch build) on the copy
        stream; returns the slot index.  With build=True uploads and steps must alternate."""
        slot = self._i % len(self.slots)
        self._i += 1
        if hb.nbytes > self.slots[slot].numel():
            raise _lib.EimsError(_lib.ERR_CAPACITY, "host batch larger than the staging slot")
        if len(self.slots) != 2 and build:
            raise ValueError("building ahead needs exactly two slots (the plan has two sets of batch tables)")
        with torch.cuda.stream(self.copy_stream):
            if self.consumed[slot] is not None:
                self.copy_stream.wait_event(self.consumed[slot])  # the step that read this slot is done
            self.slots[slot][:hb.nbytes].copy_(self.buf_of(hb), non_blocking=True)
            if build:
                # K1 on the copy stream: the table set it overwrites was last read by the step that
                # consumed this slot, which the wait above already covers
                self.plan.batch_build(self._dataset(slot, hb), None, hb.num_graphs)
            self.built[slot] = build
            self.copied[slot].record(self.copy_stream)
            if getattr(hb, "_ring_event", None) is not None:
                hb._ring_event.record(self.copy_stream)   # the pinned ring buffer may be repacked after this
        self.h2d_bytes += hb.nbytes
        return slot

    @staticmethod
    def buf_of(hb):
        return hb.buf[:hb.nbytes]

    def train_step(self, slot, hb: PackedHostBatch, step, loss_kind="mse", optimizer=True):
        """K1 + forward + loss + backward + AdamW on the uploaded batch; the step's loss and
        cosine are copied back to pinned host memory (asynchronously; read with `result`)."""
        cur = torch.cuda.current_stream(self.plan.device)
        cur.wait_event(self.copied[slot])
        ds = self._dataset(slot, hb)
        if self.built[slot]:
            self.plan.train_step_built(ds, None, self.fp, step, self.metrics, loss_kind, optimizer)
        else:
            self.plan.train_step(ds, None, self.fp, step, self.metrics, loss_kind, optimizer, num_graphs=hb.num_graphs)
        ev = torch.cuda.Event()
        ev.record(cur)
        self.consumed[slot] = ev
        k = self._n % self.RING
        self.host_ring[k].copy_(self.metrics, non_blocking=True)
        self.d2h_done[k].record(cur)
        self._n += 1
        self.d2h_bytes += self.metrics.numel() * 4

    def infer(self, slot, hb: PackedHostBatch, out_host: torch.Tensor):
        cur = torch.cuda.current_stream(self.plan.device)
        cur.wait_event(self.copied[slot])
        prob = self.plan.infer_batch(self._dataset(slot, hb), None, self.fp, num_graphs=hb.num_graphs)
        ev = torch.cuda.Event()
        ev.record(cur)
        self.consumed[slot] = ev
        out_host[:hb.num_graphs].copy_(prob, non_blocking=True)
        self.d2h_bytes += prob.numel() * 4

    def read(self, lag: int = 1):
        """(loss, cosine) of the training step `lag` steps before the one enqueued last (0 <= lag < 4), after waiting
        for THAT step's device-to-host copy only - with lag >= 1 the GPU keeps running the newer steps meanwhile."""
        if self._n - 1 - lag < 0 or lag >= self.RING:
            return None
        k = (self._n - 1 - lag) % self.RING
        self.d2h_done[k].synchronize()
        return float(self.host_ring[k][4]), float(self.host_ring[k][5])

    def result(self):
        """(loss, cosine) of the last enqueued training step (waits for it)."""
        return self.read(0)


class GraphedHostTrainer(StepReplay):
    """Training steps fed from HOST-resident data, replayed as CUDA graphs: per step the graph holds the H2D copy of
    the NEXT batch from a pinned ring buffer into one of two device slots + its K1 batch build (copy stream), the step
    itself on the batch built one step earlier (forward, loss, backward, AdamW or the fused data-parallel exchange),
    and the D2H copy of the step's loss / cosine into a pinned result ring.  The host's part per GROUP of `group` steps:
    collate `group` batches into the pinned ring (`eims_host_pack_batch_fixed`, C, worker threads - the fixed layout
    keeps every device pointer constant, which is what lets the copies and K1 sit inside a graph), one step-block
    upload, one graph launch.  This is what `collate_fn` + `.to(device)` + one `train_model` iteration + `loss.item()`
    are in the reference (GCN:292-297, 411-439), with the launches taken off the host.

    Ring discipline: batch n lives in pinned buffer n % (2*group); launch l runs steps l*group .. l*group+group-1 and
    copies batches l*group+1 .. l*group+group; buffer n % (2*group) may be repacked once the launch that copied batch
    n - 2*group has completed (`done` events)."""

    def __init__(self, plan, fp, hds: HostDataset, batch: int, max_mz: int, cap_nodes: int, cap_bonds: int, cap_peaks: int = 0,
                 metrics=None, loss_kind="mse", fused=None, group: int = 10, workers: int = 4):
        from concurrent.futures import ThreadPoolExecutor
        self.plan, self.fp, self.hds, self.batch, self.max_mz = plan, fp, hds, int(batch), int(max_mz)
        self.caps = (int(cap_nodes), int(cap_bonds), int(cap_peaks))
        self.loss_kind, self.fused = loss_kind, fused
        self.G = max(2, min(16, int(group))) // 2 * 2
        self.lib = _lib.load()
        dev = plan.device
        self.metrics = metrics if metrics is not None else torch.zeros(8, dtype=torch.float32, device=dev)
        # the fixed layout: probe it with the first `batch` molecules
        lay = _lib.HostBatchLayout()
        probe = np.arange(self.batch, dtype=np.int32)
        rc = self.lib.eims_host_pack_batch_fixed(C.byref(hds.struct), C.c_void_p(probe.ctypes.data), self.batch, hds.feat_dim, self.max_mz,
                                                 *self.caps, None, 0, C.byref(lay))
        if rc not in (0, _lib.ERR_CAPACITY) or lay.nbytes <= 0:
            check(rc if rc else _lib.ERR_ARG)
        self.lay, self.nbytes = lay, int(lay.nbytes)
        self.pinned = [torch.empty(self.nbytes, dtype=torch.uint8, pin_memory=True) for _ in range(2 * self.G)]
        self.slots = [torch.empty(self.nbytes, dtype=torch.uint8, device=dev) for _ in range(2)]
        self.out_host = torch.zeros(2 * self.G, 8, dtype=torch.float32, pin_memory=True)
        self.copy_stream = torch.cuda.Stream(dev)
        self.side2 = torch.cuda.Stream(dev) if fused is None else None
        self.pool = ThreadPoolExecutor(max(1, int(workers)))
        self.h2d_bytes = self.d2h_bytes = 0
        self.graphs, self.done, self.launches = [], {}, 0
        self._ds = [PackedDataset(s.data_ptr(), _offsets(lay), self.batch, lay.mz_is_f64) for s in self.slots]
        plan.enable_step_block(self.G)
        if fused is None:
            fp.ensure_adam()

    # -- host side ------------------------------------------------------------------------
    def pack_async(self, n: int, ids: np.ndarray):
        """Collate batch n into its pinned ring buffer on a worker thread (returns a future)."""
        ids = np.ascontiguousarray(ids, np.int32)
        buf = self.pinned[n % (2 * self.G)]
        need = (n - 2 * self.G - 1) // self.G if n - 2 * self.G >= 1 else -1   # the launch that copied this buffer's previous batch
        ev = self.done.get(need)

        def work():
            if ev is not None:
                ev.synchronize()
            lay = _lib.HostBatchLayout()
            check(self.lib.eims_host_pack_batch_fixed(C.byref(self.hds.struct), C.c_void_p(ids.ctypes.data), len(ids), self.hds.feat_dim,
                                                      self.max_mz, *self.caps, C.c_void_p(buf.data_ptr()), buf.numel(), C.byref(lay)))
            return n
        return self.pool.submit(work)

    def prime(self, fut0):
        """Batch 0 (already submitted with pack_async) is uploaded and built eagerly on the current stream."""
        fut0.result()
        self.slots[0].copy_(self.pinned[0], non_blocking=True)
        self.plan.batch_build(self._ds[0], None, self.batch)
        self.h2d_bytes += self.nbytes

    def _enqueue(self, n_local: int, block: int, step):
        cur = torch.cuda.current_stream(self.plan.device)
        slot, nxt = n_local % 2, (n_local + 1) % 2
        self.copy_stream.wait_stream(cur)            # the next batch's slot was last read by the previous step: fork here
        self._enqueue_step(self._ds[slot], block, step)
        self.out_host[n_local].copy_(self.metrics, non_blocking=True)      # the step's loss / cosine back to the host
        with torch.cuda.stream(self.copy_stream):
            self.slots[nxt].copy_(self.pinned[(n_local + 1) % (2 * self.G)], non_blocking=True)
            # indirect: K1 takes its sequence number (the zero-degree tag) from the step block, so every replay tags its
            # batches anew; a number baked in at capture would repeat every other launch
            self.plan.batch_build_indirect(self._ds[nxt], self.batch)
        cur.wait_stream(self.copy_stream)            # join

    def capture(self, step):
        """After prime() and a few eager steps elsewhere (modules loaded): capture the two group graphs."""
        plan = self.plan
        plan.select_step_block(0)
        plan.step_blocks_upload([step], [None], [0], 0)   # loads the upload kernel; ids None: K1 reads the slot in order
        torch.cuda.synchronize(plan.device)

        def group(s):
            for j in range(self.G):
                self._enqueue(s * self.G + j, j, step)
        self.graphs = self._capture(lambda: group(0), lambda: group(1))
        plan.select_step_block(0)

    def launch(self, steps, futures):
        """Run the next group: `steps` = its `group` Step structs, `futures` = the pack futures of the `group` batches it
        uploads (batches l*group+1 .. l*group+group).  Returns the launch index."""
        assert len(steps) == self.G
        for f in futures:
            f.result()
        l = self.launches
        self.plan.step_blocks_upload(list(steps), [None] * self.G, self._seqs(self.G), 0)
        self.graphs[l % 2].replay()
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.plan.device))
        self.done[l] = ev
        self.done.pop(l - 4, None)
        self.launches += 1
        self.h2d_bytes += self.G * self.nbytes
        self.d2h_bytes += self.G * 32
        self.fp.count_steps(self.G)
        return l

    def results(self, l: int):
        """(loss, cosine) of every step of launch l (waits for that launch)."""
        self.done[l].synchronize()
        rows = self.out_host[(l % 2) * self.G:(l % 2 + 1) * self.G]
        return [(float(r[4]), float(r[5])) for r in rows]

    def close(self):
        self.pool.shutdown(wait=True)
