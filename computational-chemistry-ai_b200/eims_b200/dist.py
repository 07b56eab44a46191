"""Data-parallel training of the GCN EI-MS path: one process per GPU, molecules sharded by
rank, one gradient all-reduce per optimiser step (SURVEY.md §8e).

The reference has no multi-GPU code at all (a single process on `cuda:0`,
/root/reference/templates/ms-pred-gcn-eims-cupy.py:63), so the contract is the one
PyTorch DDP would give the script unchanged:

  * every rank starts from rank 0's weights (`broadcast_params`);
  * rank r trains on molecules perm[r::world] of the epoch's shuffled order, `batch` per rank
    (`shard_epoch`), all ranks taking the same number of steps;
  * gradients are summed over ranks in the flat fp32 buffer (NCCL over NVLink on the GPU,
    gloo in the CPU tests) and the 1/world scaling is applied inside the AdamW kernel
    (`eims_step.grad_scale`), so every rank applies the same update to its own copy;
  * BatchNorm batch statistics and running buffers stay rank-local (no SyncBN); rank 0's
    running buffers are the ones a checkpoint keeps.

Nothing here touches the data path of a step: K1 .. backward run on rank-local molecules with
no collective; the all-reduce sits between backward and AdamW.  `GradReducer` splits the flat
buffer into two buckets - the head (whose gradients are final before the GCN layers are
differentiated) and the GCN / BatchNorm tensors - so that the larger bucket's all-reduce
overlaps the rest of the backward pass on a side stream.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.distributed as dist


def shard_epoch(num_mols: int, world: int, rank: int, batch: int, epoch: int, seed: int = 0, drop_last: bool = True):
    """Molecule ids of every step of `rank` in `epoch`: int32 [steps, batch].

    One permutation per epoch, shared by all ranks (same seed), strided by rank; the tail that
    does not fill a batch on every rank is dropped so that all ranks take the same number of
    steps (a rank that ran out of batches would deadlock the all-reduce)."""
    if not (0 <= rank < world):
        raise ValueError(f"rank {rank} outside world of {world}")
    perm = np.random.Generator(np.random.PCG64([seed, epoch])).permutation(num_mols)
    steps = num_mols // (world * batch)
    if steps == 0 or not drop_last:
        raise ValueError(f"{num_mols} molecules do not fill one batch of {batch} on each of {world} ranks")
    mine = perm[rank::world][: steps * batch]
    return mine.astype(np.int32).reshape(steps, batch)


def stratified_epoch(sizes, batch: int, epoch: int, seed: int = 0):
    """One epoch over this rank's molecules in batches of (almost) equal total atom count:
    int32 [steps, batch].

    Synchronous data parallelism runs at the pace of the slowest rank, and a step's cost follows
    the number of atoms in its batch (std ~2.4 % for 512 random molecules of 2..64 atoms - a 3-4 %
    straggler tax at 8 ranks).  Molecules are sorted by size into `batch` strata of equal
    population, each stratum is shuffled, and batch k takes the k-th molecule of every stratum:
    every molecule is still drawn exactly once per epoch in random order, but all batches - on
    all ranks - carry nearly the same work.  (The reference shuffles uniformly, GCN:564; this
    is a sampling-order policy, not a change of the model's arithmetic.)"""
    sizes = np.asarray(sizes)
    n = len(sizes)
    steps = n // batch
    if steps == 0:
        raise ValueError(f"{n} molecules do not fill one batch of {batch}")
    rng = np.random.Generator(np.random.PCG64([seed, epoch]))
    keep = rng.permutation(n)[: steps * batch]                 # drop a random tail, not the largest molecules
    order = keep[np.argsort(sizes[keep], kind="stable")].reshape(batch, steps)   # stratum s = row s
    out = np.empty((steps, batch), np.int32)
    for s in range(batch):
        out[:, s] = order[s, rng.permutation(steps)]
    for k in range(steps):                                      # position inside a batch carries no meaning; shuffle it too
        out[k] = out[k, rng.permutation(batch)]
    return out


def global_batches(sizes, world: int, rank: int, batch: int, epoch: int, seed: int = 0, balance: bool = True, steps: int | None = None):
    """Molecule ids of every step of `rank` in `epoch` when every rank holds the WHOLE data set: int32 [steps, batch].

    The global batch of step k is `perm[k*world*batch : (k+1)*world*batch]` of one uniform permutation per epoch
    shared by all ranks - exactly the batches the reference's `DataLoader(shuffle=True)` (GCN:561-568) draws at batch
    size world*batch.  Only the ASSIGNMENT of those molecules to ranks is free, and the gradient (the mean over the
    global batch, equal counts per rank) does not depend on it:
      balance=False  rank r takes every world-th molecule of the global batch (torch's DistributedSampler);
      balance=True   the global batch is sorted by atom count and dealt out in snake order (r, 2W-1-r, 2W+r, ...),
                     so that every rank gets the same number of molecules AND almost the same number of atoms.
    A synchronous step runs at the pace of the slowest rank and a step's cost follows its atom count (std ~2.4 % for
    512 random molecules of 2..64 atoms: a 3-4 % straggler tax at 8 ranks); the balanced deal removes it without
    touching what is sampled."""
    if not (0 <= rank < world):
        raise ValueError(f"rank {rank} outside world of {world}")
    sizes = np.asarray(sizes)
    n = len(sizes)
    gb = world * batch
    total = n // gb
    if total == 0:
        raise ValueError(f"{n} molecules do not fill one batch of {batch} on each of {world} ranks")
    steps = total if steps is None else min(int(steps), total)
    perm = np.random.Generator(np.random.PCG64([seed, epoch])).permutation(n)[: steps * gb].reshape(steps, gb)
    if not balance or world == 1:
        return np.ascontiguousarray(perm[:, rank::world]).astype(np.int32)
    order = np.argsort(-sizes[perm], axis=1, kind="stable")              # largest first, per global batch
    srt = np.take_along_axis(perm, order, axis=1).reshape(steps, batch, world)
    col = np.where(np.arange(batch) % 2 == 0, rank, world - 1 - rank)    # snake: even rounds forwards, odd rounds backwards
    return np.ascontiguousarray(srt[:, np.arange(batch), col]).astype(np.int32)


def head_split(offsets, num_gcn_layers: int) -> int:
    """Flat-buffer offset where the spectrum_predictor tensors start (parameters() order:
    2L GraphConv tensors, 2L BatchNorm tensors, then the 10 head tensors)."""
    return int(offsets[4 * num_gcn_layers])


class GradReducer:
    """Sum (not mean) of the flat gradient buffer over the ranks of `group`.

    `reduce(grads)` is the plain one-shot form.  With `overlap=True` on CUDA the caller marks
    the point of the backward pass where the head gradients are final (`head_ready()`); that
    bucket is reduced on a side stream while the GCN layers are differentiated, and
    `finish()` reduces the remaining bucket and joins the streams before AdamW."""

    def __init__(self, offsets, num_gcn_layers: int, group=None, overlap: bool = True):
        self.group = group
        self.split = head_split(offsets, num_gcn_layers)
        self.numel = int(offsets[-1])
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.overlap = overlap
        self._side = None
        self._pending = None

    def reduce(self, grads: torch.Tensor):
        if self.world > 1:
            dist.all_reduce(grads, op=dist.ReduceOp.SUM, group=self.group)
        return grads

    # -- two-bucket overlapped form (CUDA) ---------------------------------------------
    def head_ready(self, grads: torch.Tensor):
        if self.world == 1:
            return
        if not (self.overlap and grads.is_cuda):
            return
        if self._side is None:
            self._side = torch.cuda.Stream(grads.device)
        cur = torch.cuda.current_stream(grads.device)
        self._side.wait_stream(cur)
        with torch.cuda.stream(self._side):
            dist.all_reduce(grads[self.split:], op=dist.ReduceOp.SUM, group=self.group)
        self._pending = grads

    def finish(self, grads: torch.Tensor):
        if self.world == 1:
            return grads
        if self._pending is None:
            return self.reduce(grads)
        dist.all_reduce(grads[: self.split], op=dist.ReduceOp.SUM, group=self.group)
        torch.cuda.current_stream(grads.device).wait_stream(self._side)
        self._pending = None
        return grads


class FusedP2PAdamW:
    """Gradient all-reduce + AdamW + parameter broadcast as ONE kernel over NVLink / NVSwitch peer
    memory (`eims_dp_adamw_fused`, csrc/dp_fused.cu) instead of NCCL all-reduce + AdamW.

    The flat parameter buffer and two gradient buffers (double-buffered: peers read this step's
    gradients while the next step's accumulate elsewhere) live in torch symmetric memory, so
    every rank holds peer-mapped addresses of every other rank's buffers and, on an NVSwitch
    box, a multicast address for in-switch reduction (`multimem.ld_reduce`) and multicast stores
    (`multimem.st`).  Rank r owns 1/world of the parameter vector: it keeps Adam state for that
    slice only and is the single writer of those parameters on every rank, so all ranks hold
    bit-identical weights.  Host-side torch is plumbing (allocation, rendezvous); the exchange
    itself is inside the kernel."""

    SIGNAL_OFFSET = 8192  # bytes into torch's signal pad (its own barriers use the front)

    def __init__(self, fp, num_gcn_layers=None, group=None, overlap=True, use_multicast=True):
        import ctypes as C
        import torch.distributed._symmetric_memory as symm
        from . import _lib
        self.C, self.lib = C, _lib.load()
        self.group = group if group is not None else dist.group.WORLD
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        self.fp, dev, n = fp, fp.params.device, fp.numel
        q = 4 * self.world
        self.n_pad = (n + q - 1) // q * q
        self.sym_params = symm.empty(self.n_pad, dtype=torch.float32, device=dev)
        self.sym_params.zero_()
        self.sym_params[:n].copy_(fp.params)
        self.sym_grads = [symm.empty(self.n_pad, dtype=torch.float32, device=dev) for _ in range(2)]
        for g in self.sym_grads:
            g.zero_()
        self.h_params = symm.rendezvous(self.sym_params, self.group)
        self.h_grads = [symm.rendezvous(g, self.group) for g in self.sym_grads]
        if self.h_params.signal_pad_size < self.SIGNAL_OFFSET + 512:
            raise RuntimeError("symmetric-memory signal pad too small")
        pad = self.h_params.get_signal_pad(self.rank, (self.h_params.signal_pad_size // 4,), torch.int32)
        pad[self.SIGNAL_OFFSET // 4: self.SIGNAL_OFFSET // 4 + 128].zero_()
        torch.cuda.synchronize(dev)
        self.h_params.barrier()
        arr = lambda ptrs, off=0: (C.c_uint64 * self.world)(*[int(p) + off for p in ptrs])
        self.param_ptrs = arr(self.h_params.buffer_ptrs)
        self.grad_ptrs = [arr(h.buffer_ptrs) for h in self.h_grads]
        self.signal_ptrs = arr(self.h_params.signal_pad_ptrs, self.SIGNAL_OFFSET)
        mc = lambda h: int(getattr(h, "multicast_ptr", 0) or 0)
        self.params_mc, self.grads_mc = mc(self.h_params), [mc(h) for h in self.h_grads]
        # use_multicast=False forces the peer-load / peer-store branch of the kernel (tests cover both)
        self.multicast = bool(use_multicast and self.params_mc and all(self.grads_mc))
        # buckets: [0, split) = GraphConv + BatchNorm tensors (final at the end of backward),
        # [split, n_pad) = the head (final before the GCN layers are differentiated); the split is
        # rounded UP to the slice granularity so nothing unfinished lands in the early bucket
        self.overlap = bool(overlap and num_gcn_layers is not None)
        split = head_split(fp.offsets, num_gcn_layers) if self.overlap else self.n_pad
        split = min(self.n_pad, (split + q - 1) // q * q)
        self.buckets = [(0, split)] + ([(split, self.n_pad - split)] if split < self.n_pad else [])
        self.m = [torch.zeros(ln // self.world, dtype=torch.float32, device=dev) for _, ln in self.buckets]
        self.v = [torch.zeros_like(t) for t in self.m]
        self.ticket = torch.zeros(16, dtype=torch.int32, device=dev)
        self.side = torch.cuda.Stream(dev) if len(self.buckets) > 1 else None
        self.side_done = None
        self.seq = 0
        # the plan and the checkpoint code see ordinary views of the symmetric buffers
        fp.params = self.sym_params[:n]
        fp.grads = self.sym_grads[0][:n]

    def begin_step(self):
        """Select the gradient buffer of the coming step (call before backward)."""
        self.fp.grads = self.sym_grads[self.seq % 2][: self.fp.numel]
        self.seq += 1

    def next_seqs(self, n: int):
        """Sequence numbers of the next n steps run from captured graphs, which read theirs from the step blocks (the
        gradient buffer each one uses was fixed by begin_step at capture)."""
        self.seq += n
        return list(range(self.seq - n + 1, self.seq + 1))

    def _launch(self, bucket, step, stream, step_block=None):
        from ._lib import check, ptr
        C = self.C
        cur = (self.seq - 1) % 2
        off, ln = self.buckets[bucket]
        check(self.lib.eims_dp_adamw_fused_blk(self.rank, self.world, self.grad_ptrs[cur], self.param_ptrs, self.signal_ptrs,
                                               C.c_uint64(self.grads_mc[cur] if self.multicast else 0),
                                               C.c_uint64(self.params_mc if self.multicast else 0), ptr(self.m[bucket]),
                                               ptr(self.v[bucket]), ptr(self.sym_grads[1 - cur]), off, ln,
                                               C.byref(step) if step is not None else None,
                                               C.c_uint32(self.seq), bucket, C.c_void_p(self.ticket.data_ptr() + 16 * bucket),
                                               step_block if isinstance(step_block, C.c_void_p) else ptr(step_block), stream))

    def lost_peer(self):
        """Sequence number at which this rank gave up waiting for a peer (EIMS_DP_TIMEOUT_S), or 0.  One small
        synchronous read: call it once per epoch, not per step."""
        return int(self.ticket.view(-1, 4)[:, 1].max().item())

    def head_ready(self, step, step_block=None):
        """Call when the head gradients are final (between the two parts of backward): exchanges and
        updates the head bucket on a side stream while the GCN layers are differentiated."""
        if self.side is None:
            return
        dev = self.fp.params.device
        self.side.wait_stream(torch.cuda.current_stream(dev))
        self._launch(1, step, C_stream(self.side), step_block)
        self.side_done = torch.cuda.Event()
        self.side_done.record(self.side)

    def finish(self, step, stream, step_block=None):
        """Exchange + update of the remaining bucket(s) on the compute stream; afterwards the new
        parameters of every bucket are in place for the next forward.  step_block: the device step block
        the kernel reads its scalars and sequence number from (captured graphs) instead of `step`."""
        self._launch(0, step, stream, step_block)
        if self.side is not None:
            if self.side_done is None:      # head_ready was not called: do that bucket here
                self._launch(1, step, stream, step_block)
            else:
                torch.cuda.current_stream(self.fp.params.device).wait_event(self.side_done)
                self.side_done = None

    def step(self, step, stream):
        self.finish(step, stream)


def C_stream(s):
    import ctypes as C
    return C.c_void_p(s.cuda_stream)


def train_step_fused(plan, ds, ids, fp, step, fused: "FusedP2PAdamW", metrics=None, loss_kind="mse", next_ids=None):
    """One data-parallel step with the fused exchange: K1 .. backward on this rank's batch (with
    `next_ids` the next batch is built one step ahead on a side stream), the head bucket exchanged
    and updated while the GCN layers are still being differentiated, the rest at the end."""
    fused.begin_step()
    cb = (lambda: fused.head_ready(step)) if fused.side is not None else None
    plan.train_step_prefetch(ds, ids, next_ids, fp, step, metrics, loss_kind, optimizer=False, on_head_grads=cb)
    fused.finish(step, plan.stream)


def broadcast_params(fp, src: int = 0, group=None):
    """Identical initial weights and BatchNorm buffers on every rank (DDP's constructor)."""
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.broadcast(fp.params, src, group=group)
        dist.broadcast(fp.bn_running, src, group=group)


def train_step_dp(plan, ds, ids, fp, step, reducer: GradReducer, metrics=None, loss_kind="mse"):
    """One data-parallel optimiser step on this rank's batch: K1 + forward + loss + backward,
    gradient all-reduce (head bucket overlapped with the GCN backward), AdamW with
    grad_scale = 1/world."""
    if reducer.world == 1:
        plan.train_step(ds, ids, fp, step, metrics, loss_kind)
        return
    fp.ensure_adam()
    plan.train_step_split(ds, ids, fp, step, metrics, loss_kind, on_head_grads=lambda: reducer.head_ready(fp.grads))
    reducer.finish(fp.grads)
    plan.adamw(fp, step)
