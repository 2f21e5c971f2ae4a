"""Sampled-pair training step: the hot path of BASELINE configs 3 and 5.

The reference only ever trains on all pairs of a node batch (train.py:198-228);
explicit (i, j, hop-count) pair batches are the capability BASELINE.json adds.
One step = zero the gradient, ONE fused kernel (gather, distance, loss term,
gradient, scatter-add), optional NCCL all-reduce of the dense gradient across
ranks, ONE fused optimizer kernel.  The semantics of a step are exactly those of

    loss = objective(targets(hops), softplus(scale) * man.dist(x[I], x[J], squared=True))
    optimizer.zero_grad(); loss.backward(); optimizer.step()

with the reference's manifold / objective / optimizer definitions.
"""
import torch
from torch.nn.functional import softplus

from . import _lib as L
from . import _ops
from . import _torch_ops
from .modules import ManifoldParameter, _softplus_value
from .parallel import (RowShards, ShardedArena, allreduce_step_buffers, cyclic_shard, gather_cyclic,
                       try_peer_arena)


def pack_hops(idx_j, hops):
    """Second-endpoint index and hop count of every pair in ONE int32 word: (hops << 24) | idx_j.  Needs fewer than
    2^24 rows and hop counts < 255 (uint8).  Works on host or device tensors; this is the 4-byte-per-pair upload format
    of `PairTrainer.step*(..., hops=None)` (GM_TGT_HOPS_PACKED)."""
    if idx_j.dtype != torch.int32 or hops.dtype != torch.uint8:
        raise ValueError('pack_hops: int32 indices and uint8 hop counts')
    if idx_j.numel() and int(idx_j.max()) >= (1 << 24):
        raise ValueError('pack_hops: row ids must be below 2^24')
    return (idx_j | (hops.to(torch.int32) << 24)).contiguous()


def pack_hops3(idx_j, hops):
    """(j, hop count) in THREE bytes per pair: little-endian 24-bit words, bits 0-20 = j (fewer than 2^21 rows), bits
    21-23 = hops - 1 (1 <= hops <= 8).  Returns a uint8 tensor of 3*P bytes padded to a multiple of 4; the upload format
    of `PairTrainer.step_host_grouped(..., idx_j=<this>, hops=None)` -- 25 % fewer bytes over PCIe than pack_hops, which
    is what bounds the end-to-end step on one GPU.  Expanded on the device by gm_unpack_pairs3."""
    if idx_j.dtype != torch.int32 or hops.dtype != torch.uint8:
        raise ValueError('pack_hops3: int32 indices and uint8 hop counts')
    if idx_j.numel():
        if int(idx_j.max()) >= (1 << 21) or int(idx_j.min()) < 0:
            raise ValueError('pack_hops3: row ids must be below 2^21')
        if int(hops.min()) < 1 or int(hops.max()) > 8:
            raise ValueError('pack_hops3: hop counts must be in 1..8')
    w = idx_j.to(torch.int64) | ((hops.to(torch.int64) - 1) << 21)
    b = torch.stack([w & 0xFF, (w >> 8) & 0xFF, (w >> 16) & 0xFF], dim=1).to(torch.uint8).reshape(-1)
    pad = (-b.numel()) % 4
    if pad:
        b = torch.cat([b, torch.zeros(pad, dtype=torch.uint8, device=b.device)])
    return b.contiguous()


def pack_hops2(offsets, idx_j, hops):
    """Source-grouped batch -> the TWO-byte-per-pair upload format of gm_unpack_pairs2.  offsets int64 (G + 1,): group
    g is pairs offsets[g] <= k < offsets[g + 1]; idx_j int32 (P,), hops uint8 (P,).  Every group's targets are put in
    ascending row order (the returned permutation `order` says how: pair k of the packed batch is pair order[k] of the
    input) and stored as gaps: word k = (j_k - j_{k-1}) | (hops_k - 1) << 13, the first gap of a group taken from
    bases[g] = the group's smallest row.  Returns (words int16 (P,), bases int32 (G,), order int64 (P,)), or None when
    the batch does not fit (a gap above 8191 rows or a hop count outside 1..8): the caller then uploads 4-byte words."""
    if idx_j.dtype != torch.int32 or hops.dtype != torch.uint8 or offsets.dtype != torch.int64:
        raise ValueError('pack_hops2: int64 offsets, int32 indices, uint8 hop counts')
    P, G = idx_j.numel(), offsets.numel() - 1
    if P == 0:
        return torch.empty(0, dtype=torch.int16), torch.zeros(G, dtype=torch.int32), torch.empty(0, dtype=torch.int64)
    if int(hops.min()) < 1 or int(hops.max()) > 8 or int(idx_j.min()) < 0:
        return None
    counts = offsets[1:] - offsets[:-1]
    group = torch.repeat_interleave(torch.arange(G, dtype=torch.int64), counts)
    # sort by (group, row): one stable sort of the rows, then a stable sort of the groups
    o1 = torch.sort(idx_j.long(), stable=True).indices
    order = o1[torch.sort(group[o1], stable=True).indices]
    j = idx_j.long()[order]
    first = torch.zeros(P, dtype=torch.bool)
    nonempty = counts > 0
    first[offsets[:-1][nonempty]] = True
    gap = torch.zeros(P, dtype=torch.int64)
    gap[1:] = j[1:] - j[:-1]
    gap[first] = 0
    if int(gap.max()) > 0x1FFF:
        return None
    bases = torch.zeros(G, dtype=torch.int32)
    bases[nonempty] = j[offsets[:-1][nonempty]].to(torch.int32)
    words = gap | ((hops.long()[order] - 1) << 13)
    words = torch.where(words >= 0x8000, words - 0x10000, words).to(torch.int16)  # the 16 bits, as torch's signed type
    return words.contiguous(), bases.contiguous(), order


def _named(**tensors):
    return {name: t for name, t in tensors.items() if t is not None}


def _grouped_upload(sources, offsets, idx_j, hops=None, bases=None):
    """The host tensors of a source-grouped batch that go to the device (the bases only with 2-byte words)."""
    two_byte = hops is None and idx_j.dtype == torch.int16
    if two_byte and bases is None:
        raise ValueError('2-byte pair words need the bases vector of pack_hops2')
    return _named(sources=sources, offsets=offsets, j=idx_j, hops=hops, bases=bases if two_byte else None)


class _UploadRing:
    """Device copies of the pinned host tensors of a training step, with the next step's copy overlapped on a second
    stream.  Two slots of grow-only byte buffers, one per tensor name, viewed as each batch's dtypes: while a step reads
    one slot, the next batch is copied into the other.  Each slot keeps the event of its last copy-stream upload, and
    the compute stream waits on it before the slot is rewritten or its buffers are replaced, so a prefetched batch that
    the next step does not take, or a batch larger than any before, never races the copy stream.  All buffers are
    allocated on the compute stream."""

    def __init__(self, device):
        self.device = device
        self.stream = torch.cuda.Stream(device=device)
        self.slots = [{}, {}]
        self.events = [None, None]
        self.current = 0  # slot the current step reads
        self.pending = None  # (batch, slot) of the prefetch the next take() may claim
        self.outputs = {}  # outputs of the expansion kernels: written and read on the compute stream only

    def _buffer(self, bufs, name, numel, dtype):
        n = numel * dtype.itemsize
        if name not in bufs or bufs[name].numel() < n:
            bufs[name] = torch.empty(max(n, 1), dtype=torch.uint8, device=self.device)
        return bufs[name][:n].view(dtype)

    def _claim(self, slot):
        """Views of the slot's buffers may be rewritten or replaced on the compute stream after this."""
        if self.events[slot] is not None:
            torch.cuda.current_stream(self.device).wait_event(self.events[slot])
            self.events[slot] = None

    def _views(self, slot, batch):
        return {name: self._buffer(self.slots[slot], name, t.numel(), t.dtype) for name, t in batch.items()}

    def take(self, batch):
        """Device views of `batch` (name -> pinned host tensor) for a step on the current stream: the prefetched
        slot if prefetch() was given these very tensors, else a copy on the current stream."""
        pending, self.pending = self.pending, None
        if (pending is not None and pending[0].keys() == batch.keys()
                and all(pending[0][name] is t for name, t in batch.items())):
            self.current = pending[1]
            self._claim(self.current)
            return self._views(self.current, batch)
        self.current = 0
        self._claim(0)
        views = self._views(0, batch)
        for name, t in batch.items():
            views[name].copy_(t, non_blocking=True)
        return views

    def prefetch(self, batch):
        """Copy the next step's `batch` on the copy stream into the slot the current step does not read."""
        slot = 1 - self.current
        self._claim(slot)
        views = self._views(slot, batch)
        self.stream.wait_stream(torch.cuda.current_stream(self.device))  # earlier steps are done with the slot
        with torch.cuda.stream(self.stream):
            for name, t in batch.items():
                views[name].copy_(t, non_blocking=True)
        self.events[slot] = self.stream.record_event()
        self.pending = (batch, slot)

    def output(self, name, numel):
        """int32 (numel,) device buffer for the output of an expansion kernel."""
        return self._buffer(self.outputs, name, numel, torch.int32)


def _replace_param(optimizer, old, new):
    """Let the optimizer drive `new` wherever it holds the embedding parameter `old`."""
    replaced = False
    for g in optimizer.param_groups:
        for k, prm in enumerate(g['params']):
            if prm is old:
                g['params'][k] = new
                replaced = True
    if not replaced:
        raise ValueError('optimizer does not hold the embedding parameter')


class PairTrainer:
    """Drives (I, J, hops) pair batches through a single-manifold embedding.

    embedding : ManifoldEmbedding with one factor, on a CUDA device
    optimizer : RiemannianAdam / RiemannianSGD over embedding.xs
    objective : QuotientLoss / StressLoss
    max_hops_sq : max over the graph of hop^2 (GraphDataset normalisation, data/dataset.py:11-12)
    process_group : optional torch.distributed group; gradients (and the loss) are summed over it (pair-sharded data
        parallelism).
    owner_update : with a process group, reduce-scatter the gradient and let every rank update (and keep optimizer
        state for) only the rows it owns, then all-gather the new points; otherwise all-reduce and update replicas.
        Both give the same trajectory up to summation order.  Default: owner update whenever the rows split evenly.
        On GPUs of one NVLink domain the owner update is a single kernel over peer memory (gm_optim_step_peer: pull
        and sum the owned gradient rows from every rank, update, push the new rows to every rank) instead of
        ncclReduceScatter + update + ncclAllGather; it is chosen automatically when CUDA IPC between the ranks works
        (`self.peer` is then the PeerArena; GM_PEER_UPDATE=0 forces the NCCL collectives).
    """

    def __init__(self, embedding, optimizer, objective, max_hops_sq, alpha=1.0, process_group=None, owner_update=None,
                 deterministic=False):
        if embedding.n_components != 1:
            raise ValueError('PairTrainer drives a single-manifold embedding; use BatchedObjective for products')
        self.deterministic = bool(deterministic)
        self.emb, self.opt, self.obj = embedding, optimizer, objective
        self.max_hops_sq, self.alpha, self.pg = float(max_hops_sq), alpha, process_group
        self.x = embedding.xs[0]
        self.n_points = self.x.shape[0]
        self.man = embedding.manifolds[0]
        self.grad = torch.zeros_like(self.x, memory_format=torch.contiguous_format)
        self.x.grad = self.grad
        self.acc = torch.zeros(2, dtype=torch.float64, device=self.x.device)
        self._ring = _UploadRing(self.x.device)
        self.shards = None
        self.peer = None
        if process_group is not None and torch.distributed.get_world_size(process_group) > 1:
            even = self.x.shape[0] % torch.distributed.get_world_size(process_group) == 0
            if owner_update is None:
                owner_update = even
            if owner_update:
                self.peer = try_peer_arena(self.x.data, 2, process_group)
                if self.peer is not None:
                    # points, gradient and step accumulator move into the IPC-mapped arena
                    self.x.data = self.peer.x
                    self.grad = self.peer.grad
                    self.x.grad = self.grad
                    self.acc = self.peer.acc
                    self.shards = self.peer  # same own()/lo/hi/rows interface as RowShards
                else:
                    self.shards = RowShards(self.x.shape[0], process_group)
                # the optimizer now drives a parameter that aliases the owned rows of x
                own = ManifoldParameter(self.shards.own(self.x.data), manifold=self.man)
                if self.peer is not None:
                    own.grad = self.peer.own(self.grad)  # placeholder: the kernel sums every rank's rows itself
                    own._gm_peer_arena = self.peer
                else:
                    own.grad = torch.zeros_like(own.data)
                self._own = own
                _replace_param(optimizer, self.x, own)

    # ---- device-resident inputs ---------------------------------------------------------------------------------
    def step(self, idx_i, idx_j, hops, epoch=1, segments=0):
        """One training step on device tensors; returns the (device, float64) loss of the batch.  `segments`: the
        batch is in window_order(..., segments) (gm_pairs_t.segments: the kernel walks the windows one after another)."""
        pairs = _ops.PairSet.from_lists(idx_i, idx_j, self.x.device, segments=segments)
        if hops is None:  # hop counts packed into the top byte of idx_j (pack_hops)
            if self.n_points > (1 << 24) or pairs.idx64:
                raise ValueError('packed hop counts need int32 indices and fewer than 2^24 points')
            targets = _ops.TargetSpec.hops_packed(self.max_hops_sq)
        else:
            targets = _ops.TargetSpec.hops(hops, self.max_hops_sq)
        return self._step_pairs(pairs, targets, epoch)

    def step_sampled(self, sources, levels, per_src, seed, slots=None, epoch=1):
        """One training step whose pairs are DRAWN INSIDE the pair kernel (GM_PAIRS_SAMPLED): for every BFS source
        sources[g] (int32 device tensor) `per_src` targets j != i come from the counter hash of (seed, pair number) and
        their hop counts from row slots[g] (default g) of the resident uint8 (S, N) matrix `levels`.  Nothing per pair
        is uploaded, stored or read: the step's input is the list of sources.  The draw is stated in include/gm_kernels.h
        and can be reproduced on the host bit for bit, so `step(I, pack_hops(J, H), None)` on such lists is the same step."""
        pairs = _ops.PairSet.sampled(sources, levels, per_src, seed, slots=slots)
        if levels.shape[1] != self.n_points:
            raise ValueError('the level matrix must have one column per embedded point')
        return self._step_pairs(pairs, _ops.TargetSpec.hops_packed(self.max_hops_sq), epoch)

    def step_sampled_host(self, sources, levels, per_src, seed, slots=None, epoch=1, defer_loss=False):
        """step_sampled from PINNED host tensors: `sources` (and `slots`) int32 (G,) are the step's whole upload --
        8 bytes per source instead of 4-9 bytes per pair.  Returns the loss as a Python float (a device->host read), or
        with defer_loss=True the loss of the previous deferred step (see step_host_grouped)."""
        d = self._ring.take(_named(sources=sources, slots=slots))
        loss = self.step_sampled(d['sources'], levels, per_src, seed, slots=d.get('slots'), epoch=epoch)
        if defer_loss:
            return self._queue_loss_read()
        return loss.item()

    def _pairs_deterministic(self, pairs, targets, loss_spec, sp):
        """The fused kernel's job with a fixed summation order: grad (zero on entry) and acc are filled."""
        if pairs.mode != L.GM_PAIRS_LIST:
            raise ValueError('deterministic accumulation takes explicit pair lists')
        x = self.x.detach()
        I = pairs.idx_i
        J = pairs.idx_j
        if targets.mode == L.GM_TGT_HOPS_PACKED:  # split the packed word: row id | hop count << 24
            hops = ((J >> 24) & 0xff).to(torch.uint8)
            J = (J & 0x00ffffff).contiguous()
            targets = _ops.TargetSpec.hops(hops, targets.max_sq)
        plain = _ops.PairSet.from_lists(I, J, x.device)
        d2 = _ops.pairs_dist2(self.man.spec, x, x, plain)
        acc, g = _ops.product_loss([d2], [sp], targets, loss_spec)
        self.acc.copy_(acc[:2])
        xi, xj = x.index_select(0, I.long()), x.index_select(0, J.long())
        gi, gj = torch.empty_like(xi), torch.empty_like(xj)
        _ops.pairs_grad(self.man.spec, xi, xj, _ops.PairSet.elementwise(plain.P), g, gi, gj, coef=sp)
        _ops.scatter_add_rows_deterministic(torch.cat([gi, gj]), torch.cat([I.long(), J.long()]), self.grad)

    def _step_pairs(self, pairs, targets, epoch):
        loss_spec = self.obj.loss_spec(epoch=epoch, alpha=self.alpha)
        # a memset rather than rows handed back zeroed by the optimizer kernel (gm_optim_t.zero_grad): measured on B200
        # (2 M SPD4 points) 1.19 vs 1.28 ms per step, the memset leaves the table L2-resident for the pair kernel
        self.grad.zero_()
        self.acc.zero_()
        if self.deterministic:
            self._pairs_deterministic(pairs, targets, loss_spec, _softplus_value(self.emb.scales[0]))
            if self.peer is not None:
                self.opt.step()
                return self.peer.acc_out[0]
            if self.shards is not None or (self.pg is not None and torch.distributed.get_world_size(self.pg) > 1):
                raise RuntimeError('deterministic accumulation: single GPU, or the peer-memory owner update (which '
                                   'sums the ranks in rank order)')
            self.opt.step()
            return self.acc[0]
        # softplus(scale) is re-read every step (cached on the parameter until somebody steps it or loads a snapshot);
        # the trainer itself does not train the scale: acc[1] (sum l' d2) is there for a caller who does
        sp = _softplus_value(self.emb.scales[0])
        if (pairs.mode == L.GM_PAIRS_LIST and self.man.spec.kind != L.GM_UNIVERSAL
                and targets.mode in (L.GM_TGT_HOPS_PACKED, L.GM_TGT_HOPS_U8, L.GM_TGT_HOPS_U16)):
            # explicit pair lists: through the registered custom op (torch.ops.graphembed_b200.pairs_loss_fused)
            torch.ops.graphembed_b200.pairs_loss_fused(
                self.x.detach(), pairs.idx_i, pairs.idx_j, targets.data, *_torch_ops.manifold_args(self.man.spec),
                loss_spec.kind, bool(loss_spec.inc_l1), bool(loss_spec.inc_l2), float(loss_spec.alpha),
                float(loss_spec.eps), float(targets.max_sq), float(sp), self.grad, self.acc, pairs.segments)
        else:
            _ops.pairs_loss_fused(self.man.spec, self.x.detach(), pairs, targets, loss_spec, sp, self.grad, self.acc)
        if self.peer is not None:
            self.opt.step()  # ONE kernel: cross-GPU barrier, pull+sum gradients, update, push points, sum the loss
            return self.peer.acc_out[0]
        if self.shards is None:
            allreduce_step_buffers(self.grad, self.acc, self.pg)
            self.opt.step()
        else:
            self.shards.reduce_scatter(self.grad, out=self._own.grad)
            torch.distributed.all_reduce(self.acc, group=self.pg)
            self.opt.step()
            self.shards.all_gather(self.x.data)
        return self.acc[0]

    # ---- host-resident inputs (what a data loader hands over) ----------------------------------------------------------
    def step_host(self, idx_i, idx_j, hops, epoch=1, next_batch=None):
        """One step from PINNED host tensors (int32 indices, uint8/int16 hop counts).  Copies the batch to the device,
        runs the step and returns the loss as a Python float (a device->host read).  If `next_batch` (a tuple of
        pinned host tensors) is given its upload is overlapped with this step's kernels on a second stream."""
        d = self._ring.take(_named(i=idx_i, j=idx_j, hops=hops))
        if next_batch is not None:
            self._ring.prefetch(_named(i=next_batch[0], j=next_batch[1], hops=next_batch[2]))
        loss = self.step(d['i'], d['j'], d['hops'], epoch=epoch)
        return loss.item()

    # ---- pipelined loss read-back --------------------------------------------------------------------------------
    def _queue_loss_read(self):
        """Async device->host copy of this step's [loss, d loss/d scale] accumulator into pinned memory; returns the
        loss of the PREVIOUS queued step (None for the first).  The host then runs one step ahead of the GPU."""
        if getattr(self, '_loss_host', None) is None:
            self._loss_host = torch.empty(2, 2, dtype=torch.float64).pin_memory()
            self._loss_events = [torch.cuda.Event(), torch.cuda.Event()]
            self._loss_slot, self._loss_pending = 0, False
        prev = self.flush_loss()
        s = self._loss_slot
        self._loss_host[s].copy_(self.acc if self.peer is None else self.peer.acc_out, non_blocking=True)
        self._loss_events[s].record(torch.cuda.current_stream(self.x.device))
        self._loss_pending = True
        return prev

    def flush_loss(self):
        """Loss of the last step issued with defer_loss=True (waits for it), or None if nothing is pending."""
        if not getattr(self, '_loss_pending', False):
            return None
        s = self._loss_slot
        self._loss_events[s].synchronize()
        self._loss_pending = False
        self._loss_slot = 1 - s
        return float(self._loss_host[s][0])

    def step_host_grouped(self, sources, offsets, idx_j, hops, epoch=1, next_batch=None, defer_loss=False,
                          segments=0, bases=None):
        """One step from PINNED host tensors in source-grouped (CSR-like) form, the natural output of a sampler that
        draws targets per BFS source: pairs offsets[g] <= k < offsets[g+1] are (sources[g], idx_j[k]) with hop count
        hops[k].  sources int32 (G,), offsets int64 (G+1,), idx_j int32 (P,), hops uint8/int16 (P,).  Uploads 5 bytes
        per pair instead of 9 -- or 4 with hops=None and idx_j = pack_hops(j, hops) -- and the first-endpoint index
        vector is expanded on the device (gm_expand_groups).
        `next_batch` = the next step's (sources, offsets, idx_j, hops), uploaded on a second stream meanwhile.
        defer_loss=True returns the loss of the previous deferred step instead of blocking on this one (its own loss
        is copied to pinned host memory asynchronously; `flush_loss()` returns the last one), so that the host can
        enqueue step k+1 while the GPU runs step k.
        Two bytes per pair: idx_j = the int16 words of pack_hops2 (every group's targets sorted by row, stored as
        gaps), hops=None, bases = its int32 (G,) vector; `next_batch` then carries the bases as a fifth entry."""
        batch = _grouped_upload(sources, offsets, idx_j, hops, bases)
        nxt = None if next_batch is None else _grouped_upload(*next_batch)
        packed3 = hops is None and idx_j.dtype == torch.uint8  # pack_hops3: 3 bytes per pair over PCIe
        packed2 = hops is None and idx_j.dtype == torch.int16  # pack_hops2: 2 bytes per pair
        P = int(offsets[-1]) if packed3 else idx_j.numel()
        d = self._ring.take(batch)
        if nxt is not None:
            self._ring.prefetch(nxt)
        di = self._ring.output('i', P)
        if packed2:  # one kernel: gaps -> rows (segmented scan per group) and the group's first endpoint per pair
            dj = self._ring.output('j', P)
            _ops.unpack_pairs2(d['j'], d['bases'], d['offsets'], dj, group_rows=d['sources'], out_i=di)
        else:
            _ops.expand_groups(d['sources'], d['offsets'], di)
            dj = d['j']
        if packed3:  # 3-byte words: staged raw, expanded on the device just before the step
            dj = _ops.unpack_pairs3(d['j'], P, self._ring.output('j', P))
        loss = self.step(di, dj, d.get('hops'), epoch=epoch, segments=segments)
        if defer_loss:  # read this step's loss back asynchronously, hand out the previous step's
            return self._queue_loss_read()
        return loss.item()


class ShardedPairTrainer(PairTrainer):
    """PairTrainer over ROW-SHARDED embeddings (SURVEY 8(e) second scheme, BASELINE config 5 "embeddings row-sharded over
    NVLink"): every rank keeps only the rows v with v % world == rank of the point table, their gradient rows and
    their optimizer state; the pair batch is sharded over the ranks as before (every rank passes ITS pairs, with
    GLOBAL row ids).  One step is

        fused pair kernel   rows gathered from whichever shard holds them (16-byte cp.async over NVLink for remote
                            ones), gradient rows added into the owning shard (red.global.add over NVLink)
        barrier 0           every rank's reductions into my shard are final; loss summed over the ranks
        optimizer kernel    local shard only (gradient rows handed back zeroed)
        barrier 1           every shard updated

    -- no replicated table, no reduce-scatter / all-gather phase, no NCCL call on the step path; the NVLink traffic
    (about 2 x 64 B per remote pair endpoint for SPD 4x4 fp32) rides inside the pair kernel instead of following it.
    Same trajectory as PairTrainer on one GPU up to floating-point summation order.  Needs CUDA IPC between the ranks
    (one NVLink domain), a power-of-two world size dividing the number of points, and an SPD manifold; raises
    otherwise (use PairTrainer's replicated owner update then).

    embedding : every rank passes the same full ManifoldEmbedding (same initial points); after construction the full
        table is released (`keep_full=True` keeps it, stale) and `gather()` rebuilds it from the shards.
    """

    def __init__(self, embedding, optimizer, objective, max_hops_sq, process_group, alpha=1.0, keep_full=False):
        if embedding.n_components != 1:
            raise ValueError('ShardedPairTrainer drives a single-manifold embedding')
        dist = torch.distributed
        self.emb, self.opt, self.obj = embedding, optimizer, objective
        self.max_hops_sq, self.alpha, self.pg = float(max_hops_sq), alpha, process_group
        self.man = embedding.manifolds[0]
        if self.man.spec.kind not in (L.GM_SPD_AI, L.GM_SPD_STEIN):
            raise ValueError('row-sharded training is built for the SPD pair kernels')
        full = embedding.xs[0]
        self.world, self.rank = dist.get_world_size(process_group), dist.get_rank(process_group)
        self.n_points = full.shape[0]
        if self.n_points % self.world:
            raise ValueError(f'{self.n_points} points do not split evenly over {self.world} ranks')
        arena = try_peer_arena(cyclic_shard(full.data, self.rank, self.world), 2, process_group, cls=ShardedArena)
        if arena is None:
            raise RuntimeError('row-sharded training needs CUDA IPC peer memory between all ranks (one NVLink domain, '
                               'NCCL process group, GM_PEER_UPDATE != 0)')
        self.peer = arena
        self.x, self.grad, self.acc = arena.x, arena.grad, arena.acc
        own = ManifoldParameter(arena.x, manifold=self.man)
        own.grad = arena.grad
        own._gm_zero_grad_after_step = True  # the local optimizer kernel hands every gradient row back zeroed
        self._own = own
        _replace_param(optimizer, full, own)
        self._full = full
        if not keep_full:
            full.data = full.data.new_empty((0,) + tuple(full.shape[1:]))
        self._ring = _UploadRing(self.x.device)
        self.shards = None

    def _step_pairs(self, pairs, targets, epoch):
        loss_spec = self.obj.loss_spec(epoch=epoch, alpha=self.alpha)
        self.acc.zero_()
        sp = _softplus_value(self.emb.scales[0])
        a = self.peer
        _ops.pairs_loss_fused_sharded(self.man.spec, a.x_ptrs, a.grad_ptrs, self.x.dtype, self.x.device, pairs, targets,
                                      loss_spec, sp, self.acc)
        table = a.next_table()
        _ops.peer_barrier(table, 0, self.x.device)
        self.opt.step()
        _ops.peer_barrier(table, 1, self.x.device)
        return a.acc_out[0]

    def gather(self):
        """The full (N, ...) point table, rebuilt from every rank's shard (an all-gather; for validation / snapshots)."""
        full = gather_cyclic(self.x, self.pg)
        self._full.data = full
        return full


def window_order(idx_j, n_points, segments):
    """Permutation that puts a pair batch into (window of the target row, original position) order: window w holds the
    pairs whose target j lies in rows [w n / segments, (w + 1) n / segments).  Applied to a source-grouped batch it
    keeps every source's pairs consecutive inside each window.  Launch the reordered lists with `segments=segments`
    (gm_pairs_t.segments): the pair kernel then walks window after window with its whole grid, so the gradient rows it
    scatters into and the point rows it gathers stay inside one L2-sized window at a time (measured on B200: the fused
    SPD 4x4 kernel leaves its 3.3 GB-per-launch random DRAM traffic bound and becomes issue bound).  idx_j: int tensor
    (a packed hop count in the top byte is ignored)."""
    j = idx_j.long() & 0x00ffffff if idx_j.dtype == torch.int32 else idx_j.long()
    window = (j * int(segments)) // int(n_points)
    return torch.sort(window, stable=True).indices


def window_groups(sources, offsets, idx_j, n_points, segments):
    """A source-grouped batch (sources int32 (G,), offsets int64 (G + 1,), targets idx_j (P,)) in window order: returns
    (order, group_rows, group_offsets) with `order` = window_order(idx_j, n_points, segments) and the (window, source)
    groups of the reordered batch -- group w * G + g holds the pairs of source g whose target lies in window w (possibly
    none), group_rows[w * G + g] = sources[g].  Feed `idx_j[order]` etc. with these to step_host_grouped(segments=...)
    or pack_hops2."""
    G = sources.numel()
    counts = offsets[1:] - offsets[:-1]
    group = torch.repeat_interleave(torch.arange(G, dtype=torch.int64), counts)
    order = window_order(idx_j, n_points, segments)
    j = idx_j.long() & 0x00ffffff if idx_j.dtype == torch.int32 else idx_j.long()
    key = ((j[order] * int(segments)) // int(n_points)) * G + group[order]
    group_counts = torch.bincount(key, minlength=int(segments) * G)
    group_offsets = torch.cat([torch.zeros(1, dtype=torch.int64), group_counts.cumsum(0)])
    return order, sources.repeat(int(segments)).contiguous(), group_offsets


class ProductPairTrainer:
    """(I, J, hops) pair batches through a PRODUCT-manifold embedding -- BASELINE config 3 ("product SPD 3x3 x Lorentz 5,
    sampled pairs").  The distance of a pair is sum_f softplus(scale_f) * d_f^2 (modules.py:84-88); one step is

        gm_pairs_product_fused (ONE launch: every factor's d2, the loss, sum l' d2_f per factor, every factor's
        gradient scatter-add)  ->  the optimizer kernels

    for products of at most one SPD factor with up to three of Lorentz / Sphere / Euclidean, and otherwise

        F x gm_pairs_dist2  ->  gm_product_loss (loss term, dL/dm per pair, sum l' d2_f per factor)
        ->  F x gm_pairs_grad (scatter-add of softplus(scale_f) * dL/dm * d(d2_f)/dx)  ->  the optimizer kernels

    with the reference's semantics of `loss.backward(); optimizer.step()`.  `scale_optimizer` (optional: any optimizer
    over embedding.scales, e.g. the second RiemannianAdam group of experiments/run_grid.py:25-28) receives
    d loss / d scale_f = sigmoid(scale_f) * sum_k l'_k d2_f,k and is stepped after the points.  With a process group
    the pair batch is sharded over the ranks and gradients, loss and scale gradients are all-reduced (replicated
    update)."""

    def __init__(self, embedding, optimizer, objective, max_hops_sq, alpha=1.0, scale_optimizer=None,
                 process_group=None, fused=None):
        self.emb, self.opt, self.obj = embedding, optimizer, objective
        self.max_hops_sq, self.alpha, self.pg = float(max_hops_sq), alpha, process_group
        self.scale_opt = scale_optimizer
        self.xs = list(embedding.xs)
        self.mans = list(embedding.manifolds)
        self.scales = list(getattr(embedding, 'scales', ()))
        if any(hasattr(m, 'get_c') for m in self.mans):
            raise ValueError('Universal factors carry a curvature gradient: train them through BatchedObjective')
        self.grads = [torch.zeros_like(x, memory_format=torch.contiguous_format) for x in self.xs]
        for x, g in zip(self.xs, self.grads):
            x.grad = g
        # one launch for all factors where the fused product kernel takes the factor list (fused=False: the F + 1 + F
        # launches above, kept for the other products and as the A/B of the fused kernel)
        can_fuse = _ops.product_fusable([m.spec for m in self.mans], [x.dtype for x in self.xs])
        self.fused = can_fuse if fused is None else (bool(fused) and can_fuse)

    def step(self, idx_i, idx_j, hops, epoch=1):
        """One training step on device tensors (int32/int64 indices, uint8/int16 hop counts); returns the (device,
        float64) loss of the batch."""
        dev = self.xs[0].device
        pairs = _ops.PairSet.from_lists(idx_i, idx_j, dev)
        targets = _ops.TargetSpec.hops(hops, self.max_hops_sq)
        loss_spec = self.obj.loss_spec(epoch=epoch, alpha=self.alpha)
        sps = [_softplus_value(s) for s in self.scales] if self.scales else [1.0] * len(self.xs)
        if self.fused:
            for gx in self.grads:
                gx.zero_()
            acc = _ops.pairs_product_fused([m.spec for m in self.mans], [x.detach() for x in self.xs], pairs, targets,
                                           loss_spec, sps, self.grads)
        else:
            d2s = [_ops.pairs_dist2(m.spec, x.detach(), x.detach(), pairs) for m, x in zip(self.mans, self.xs)]
            acc, g = _ops.product_loss(d2s, sps, targets, loss_spec)
            for m, x, gx, sp in zip(self.mans, self.xs, self.grads, sps):
                gx.zero_()
                _ops.pairs_grad(m.spec, x.detach(), x.detach(), pairs, g, gx, gx, coef=sp)
        if self.pg is not None and torch.distributed.get_world_size(self.pg) > 1:
            for gx in self.grads:
                torch.distributed.all_reduce(gx, group=self.pg)
            torch.distributed.all_reduce(acc, group=self.pg)
        self.opt.step()
        if self.scale_opt is not None:
            for f, s in enumerate(self.scales):
                s.grad = (acc[1 + f] * torch.sigmoid(s.detach().double())).to(s.dtype).reshape(s.shape)
            self.scale_opt.step()
        return acc[0]
