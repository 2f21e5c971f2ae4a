"""Tensor-level wrappers over the C-ABI (include/gm_kernels.h) and the autograd
Functions the manifold classes are built from.

Every function here launches hand-written sm_100a kernels from libgm_b200.so on
the current CUDA stream of the tensors' device.  Nothing falls back to PyTorch.
"""
import ctypes

import torch

from . import _lib as L


class ManifoldSpec:
    """(kind, n, p, flags, wmin, wmax) of one manifold; dtype is taken from the tensors."""

    __slots__ = ('kind', 'n', 'p', 'flags', 'wmin', 'wmax', 'point_shape', 'c_source', '_keep')

    def __init__(self, kind, n, p=0, flags=0, wmin=1e-8, wmax=1e8, point_shape=None, c_source=None):
        self.kind, self.n, self.p, self.flags, self.wmin, self.wmax = kind, n, p, flags, wmin, wmax
        self.point_shape = tuple(point_shape)
        self.c_source = c_source  # Universal: callable returning the current curvature tensor get_c()
        self._keep = None

    def c_struct(self, dtype, device=None, c=None, c_grad=None, wmin=None):
        """gm_manifold_t for tensors of `dtype`.  Universal: `c` (default: c_source()) is passed as a DEVICE scalar so
        that no host sync is needed while a curvature optimizer updates it; `c_grad` is an optional float64 CUDA
        scalar that the backward kernels add d(loss)/dc to."""
        c_dev = None
        if self.kind == L.GM_UNIVERSAL:
            if c is None:
                c = self.c_source()
            c = c.detach().reshape(-1)[:1].to(dtype=dtype)
            if device is not None and c.device != device:
                c = c.to(device)
            L.require_cuda(c)
            self._keep = c = c.contiguous()  # alive until the next launch on this (stream-ordered) allocator
            c_dev = c.data_ptr()
        return L.Manifold(kind=self.kind, dtype=L.dtype_code(dtype), n=self.n, p=self.p, flags=self.flags,
                          reserved=0, wmin=self.wmin if wmin is None else wmin, wmax=self.wmax, c_dev=c_dev,
                          c_grad=None if c_grad is None else c_grad.data_ptr())

    @property
    def numel(self):
        k = 1
        for s in self.point_shape:
            k *= s
        return k


def _no_function_modes(fn):
    """Run a launcher with torch-function modes off.  `torch.set_default_device('cuda')` (what run.py does, like the
    reference's set_default_tensor_type) is a TorchFunctionMode: every tensor attribute a launcher touches (data_ptr,
    is_contiguous, dtype, ...) then costs ~1.5 us instead of ~0.1 us, which dominates the step on small node batches.
    Everything below passes devices explicitly, so the default-device mode has nothing to contribute here."""
    import functools

    @functools.wraps(fn)
    def wrapper(*args, **kwargs):
        with torch._C.DisableTorchFunction():
            return fn(*args, **kwargs)
    return wrapper


def _prep(t):
    L.require_cuda(t)
    return t if t.is_contiguous() else t.contiguous()


def _index_tensor(idx, device):
    """int32/int64 contiguous index tensor on `device` and its idx64 flag."""
    if idx.dtype not in (torch.int32, torch.int64):
        idx = idx.long()
    idx = idx.to(device)
    return (idx if idx.is_contiguous() else idx.contiguous()), int(idx.dtype == torch.int64)


class PairSet:
    """Which pairs a launch covers (mirrors gm_pairs_t); keeps the index tensors alive."""

    def __init__(self, mode, P, idx_i=None, idx_j=None, B=0, nodes=None, idx64=0, k0=0, levels=None, slots=None,
                 n_nodes=0, per_src=0, seed=0, segments=0):
        self.mode, self.P, self.idx_i, self.idx_j, self.B, self.nodes, self.idx64 = mode, P, idx_i, idx_j, B, nodes, idx64
        self.k0 = k0
        self.segments = int(segments)
        self.levels, self.slots, self.n_nodes, self.per_src, self.seed = levels, slots, n_nodes, per_src, seed

    @staticmethod
    def sampled(sources, levels, per_src, seed, slots=None, P=None):
        """Pairs drawn on the device (GM_PAIRS_SAMPLED): for every source g, `per_src` targets j != sources[g] from the
        counter hash of (seed, pair number), hop counts read from row slots[g] (default g) of the resident uint8
        (S, N) matrix `levels`.  sources / slots: int32 device tensors."""
        if sources.dtype != torch.int32 or not sources.is_cuda or levels.dtype != torch.uint8 or levels.ndim != 2:
            raise ValueError('sampled pairs: int32 CUDA sources and a uint8 (S, N) level matrix')
        if slots is not None and (slots.dtype != torch.int32 or slots.numel() != sources.numel()):
            raise ValueError('sampled pairs: slots must be int32, one per source')
        if slots is None and sources.numel() > levels.shape[0]:
            raise ValueError('sampled pairs: without slots, source g reads row g of the level matrix: more sources '
                             'than rows')
        n = levels.shape[1]
        if n >= (1 << 24):
            raise ValueError('sampled pairs need fewer than 2^24 nodes')
        total = sources.numel() * int(per_src)
        return PairSet(L.GM_PAIRS_SAMPLED, total if P is None else P, idx_i=sources.contiguous(),
                       levels=levels.contiguous(), slots=None if slots is None else slots.contiguous(), n_nodes=n,
                       per_src=int(per_src), seed=int(seed) & 0xFFFFFFFFFFFFFFFF)

    @staticmethod
    def elementwise(P):
        return PairSet(L.GM_PAIRS_ELEMENTWISE, P)

    @staticmethod
    def from_lists(idx_i, idx_j, device, segments=0):
        """Explicit pair lists.  `segments` (optional locality hint, gm_pairs_t.segments): the lists are that many
        consecutive parts of ceil(P / segments) pairs which the training kernels walk one after another with the whole
        grid -- for batches ordered by (window of the target row, source), see engine.window_order."""
        if not 0 <= int(segments) <= 64:
            raise ValueError('segments must be in [0, 64]')
        i, f64 = _index_tensor(idx_i, device)
        j, g64 = _index_tensor(idx_j, device)
        if f64 != g64:
            i, j, f64 = i.long(), j.long(), 1
        if i.shape != j.shape or i.ndim != 1:
            raise ValueError('pair index lists must be 1-D tensors of the same length')
        return PairSet(L.GM_PAIRS_LIST, i.numel(), idx_i=i, idx_j=j, idx64=f64, segments=segments)

    @staticmethod
    def triu(B, nodes=None, device=None, k0=0, P=None):
        """All a<b pairs of a batch of B rows in torch.triu_indices(B, B, 1) order; `nodes` maps batch position
        to row of the parameter (None: the batch *is* the tensor).  (k0, P) restricts the launch to pairs
        [k0, k0+P) of the triangle (chunked validation, pair-sharded ranks)."""
        f64 = 0
        if nodes is not None:
            nodes, f64 = _index_tensor(nodes, device)
            if nodes.numel() != B:
                raise ValueError('len(nodes) must equal B')
        total = B * (B - 1) // 2
        if P is None:
            P = total - k0
        if k0 < 0 or P < 0 or k0 + P > total:
            raise ValueError(f'pair range [{k0}, {k0 + P}) outside the triangle of {total} pairs')
        return PairSet(L.GM_PAIRS_TRIU, P, B=B, nodes=nodes, idx64=f64, k0=k0)

    def slice(self, rank, world):
        """The contiguous share of this pair set that `rank` of `world` ranks evaluates (sizes differ by <= 1)."""
        base, extra = divmod(self.P, world)
        lo = rank * base + min(rank, extra)
        n = base + (1 if rank < extra else 0)
        if self.mode == L.GM_PAIRS_TRIU:
            return PairSet(self.mode, n, B=self.B, nodes=self.nodes, idx64=self.idx64, k0=self.k0 + lo)
        if self.mode == L.GM_PAIRS_LIST:
            return PairSet(self.mode, n, idx_i=self.idx_i[lo:lo + n], idx_j=self.idx_j[lo:lo + n], idx64=self.idx64)
        raise ValueError('elementwise pair sets are not sharded')

    def c_struct(self):
        return L.Pairs(mode=self.mode, idx64=self.idx64, P=self.P,
                       idx_i=None if self.idx_i is None else self.idx_i.data_ptr(),
                       idx_j=None if self.idx_j is None else self.idx_j.data_ptr(), B=self.B,
                       nodes=None if self.nodes is None else self.nodes.data_ptr(), k0=self.k0,
                       levels=None if self.levels is None else self.levels.data_ptr(),
                       slots=None if self.slots is None else self.slots.data_ptr(), n_nodes=self.n_nodes,
                       per_src=self.per_src, seed=self.seed, segments=self.segments, reserved=0)


@_no_function_modes
def pairs_dist2(spec, xa, xb, pairs, c=None, wmin=None):
    xa, xb = _prep(xa), _prep(xb)
    if xa.dtype != xb.dtype:
        raise RuntimeError('dtype mismatch between the two endpoint tensors')
    out = torch.empty(pairs.P, dtype=xa.dtype, device=xa.device)
    m, p = spec.c_struct(xa.dtype, xa.device, c=c, wmin=wmin), pairs.c_struct()
    with torch.cuda.device(xa.device):
        rc = L.lib().gm_pairs_dist2(ctypes.byref(m), L.ptr(xa), L.ptr(xb), ctypes.byref(p), L.ptr(out),
                                    L.stream_ptr(xa.device))
    L.check(rc, 'gm_pairs_dist2')
    return out


@_no_function_modes
def pairs_grad(spec, xa, xb, pairs, gout, ga, gb, coef=1.0, c=None, c_grad=None):
    """ga/gb += coef * gout[k] * d(d2_k)/d(rows) (ELEMENTWISE: plain stores).  Universal: c_grad (float64 CUDA
    scalar) += coef * sum_k gout[k] * d(d2_k)/dc."""
    xa, xb, gout = _prep(xa), _prep(xb), _prep(gout)
    if gout.dtype != xa.dtype:
        gout = gout.to(xa.dtype)
    m, p = spec.c_struct(xa.dtype, xa.device, c=c, c_grad=c_grad), pairs.c_struct()
    with torch.cuda.device(xa.device):
        rc = L.lib().gm_pairs_grad(ctypes.byref(m), L.ptr(xa), L.ptr(xb), ctypes.byref(p), L.ptr(gout), float(coef),
                                   L.ptr(ga), L.ptr(gb), L.stream_ptr(xa.device))
    L.check(rc, 'gm_pairs_grad')


class LossSpec:
    def __init__(self, kind, inc_l1=True, inc_l2=True, alpha=1.0, eps=1.0):
        self.kind, self.inc_l1, self.inc_l2, self.alpha, self.eps = kind, inc_l1, inc_l2, alpha, eps

    def c_struct(self):
        return L.Loss(kind=self.kind, inc_l1=int(self.inc_l1), inc_l2=int(self.inc_l2), reserved=0,
                      alpha=float(self.alpha), eps=float(self.eps))


class TargetSpec:
    def __init__(self, mode, data, ld=0, max_sq=1.0):
        self.mode, self.data, self.ld, self.max_sq = mode, data, ld, max_sq

    @staticmethod
    def vector(t):
        return TargetSpec(L.GM_TGT_VECTOR, _prep(t))

    @staticmethod
    def dense(mat):
        mat = _prep(mat)
        return TargetSpec(L.GM_TGT_DENSE, mat, ld=mat.shape[1])

    @staticmethod
    def hops(h, max_sq):
        h = _prep(h)
        if h.dtype == torch.uint8:
            return TargetSpec(L.GM_TGT_HOPS_U8, h, max_sq=max_sq)
        if h.dtype in (torch.uint16, torch.int16):
            return TargetSpec(L.GM_TGT_HOPS_U16, h, max_sq=max_sq)
        raise RuntimeError('hop-count targets must be uint8 or uint16')

    @staticmethod
    def hops_packed(max_sq):
        """Hop count in the top byte of the int32 second-endpoint index (LIST pairs, < 2^24 rows)."""
        return TargetSpec(L.GM_TGT_HOPS_PACKED, None, max_sq=max_sq)

    def c_struct(self):
        return L.Targets(mode=self.mode, reserved=0, data=None if self.data is None else self.data.data_ptr(),
                         ld=self.ld, max_sq=float(self.max_sq))


@_no_function_modes
def pairs_loss_fused(spec, x, pairs, targets, loss, scale_sp, grad, acc=None, want_d2=False, c=None, c_grad=None):
    """One kernel: distances, loss and gradient.  Returns (acc, d2 or None); acc is a 2-element float64 tensor
    [sum loss, sum l'(m) * d2] that is accumulated into (pass a zeroed one or None).  Universal: c_grad (float64
    CUDA scalar) += d(loss)/dc."""
    x = _prep(x)
    if targets.mode in (L.GM_TGT_VECTOR, L.GM_TGT_DENSE) and targets.data.dtype != x.dtype:
        raise RuntimeError('targets must have the dtype of the embedding')
    if acc is None:
        acc = torch.zeros(2, dtype=torch.float64, device=x.device)
    d2 = torch.empty(pairs.P, dtype=x.dtype, device=x.device) if want_d2 else None
    m, p, t, l = (spec.c_struct(x.dtype, x.device, c=c, c_grad=c_grad), pairs.c_struct(), targets.c_struct(),
                  loss.c_struct())
    with torch.cuda.device(x.device):
        rc = L.lib().gm_pairs_loss_fused(ctypes.byref(m), L.ptr(x), ctypes.byref(p), ctypes.byref(t), ctypes.byref(l),
                                         float(scale_sp), L.ptr(d2), L.ptr(acc), L.ptr(grad),
                                         L.stream_ptr(x.device))
    L.check(rc, 'gm_pairs_loss_fused')
    return acc, d2


@_no_function_modes
def pairs_loss_fused_sharded(spec, x_ptrs, grad_ptrs, dtype, device, pairs, targets, loss, scale_sp, acc, want_d2=False):
    """gm_pairs_loss_fused_sharded: the fused training kernel over ROW-SHARDED tables.  x_ptrs / grad_ptrs: device
    addresses (ints) of every rank's point / gradient shard as mapped into this process, in rank order (a power-of-two
    count); global row v is row v // world of shard v % world.  Gradient rows are added into the owning shards; acc
    (2 float64) is accumulated into.  Returns (acc, d2 or None)."""
    W = len(x_ptrs)
    if W != len(grad_ptrs) or W < 1 or W > L.GM_MAX_PEERS or W & (W - 1):
        raise ValueError('row shards: a power-of-two number of ranks, at most %d' % L.GM_MAX_PEERS)
    sh = L.RowShards()
    sh.world = W
    for r in range(W):
        sh.x[r], sh.grad[r] = int(x_ptrs[r]), int(grad_ptrs[r])
    d2 = torch.empty(pairs.P, dtype=dtype, device=device) if want_d2 else None
    m, p, t, l = spec.c_struct(dtype, device), pairs.c_struct(), targets.c_struct(), loss.c_struct()
    with torch.cuda.device(device):
        rc = L.lib().gm_pairs_loss_fused_sharded(ctypes.byref(m), ctypes.byref(sh), ctypes.byref(p), ctypes.byref(t),
                                                 ctypes.byref(l), float(scale_sp), L.ptr(d2), L.ptr(acc),
                                                 L.stream_ptr(device))
    L.check(rc, 'gm_pairs_loss_fused_sharded')
    return acc, d2


def peer_barrier(table, phase, device):
    """gm_peer_barrier over the flag blocks of a peer table (graphembed.parallel.ShardedArena.next_table())."""
    with torch.cuda.device(device):
        rc = L.lib().gm_peer_barrier(ctypes.byref(table), int(phase), L.stream_ptr(device))
    L.check(rc, 'gm_peer_barrier')


@_no_function_modes
def segment_sum(src, chunk_start, chunk_end, out, order=None, dst=None):
    """gm_segment_sum: out[dst[c]] = sum (left to right) of src[order[k]] for chunk_start[c] <= k < chunk_end[c]; rows of
    E = src.shape[1:].numel() elements, int64 index tensors, plain stores (bit-reproducible)."""
    L.require_cuda(src, chunk_start, chunk_end, out, order, dst)
    src = _prep(src)
    if out.dtype != src.dtype or not out.is_contiguous():
        raise RuntimeError('segment_sum: out must be a contiguous tensor of the dtype of src')
    for t in (chunk_start, chunk_end, order, dst):
        if t is not None and (t.dtype != torch.int64 or not t.is_contiguous()):
            raise RuntimeError('segment_sum: index tensors must be contiguous int64')
    E = 1
    for d in src.shape[1:]:
        E *= d
    n = chunk_start.numel()
    if chunk_end.numel() != n or (dst is not None and dst.numel() != n):
        raise ValueError('segment_sum: chunk_start, chunk_end and dst must have one entry per chunk')
    with torch.cuda.device(src.device):
        rc = L.lib().gm_segment_sum(L.dtype_code(src.dtype), E, L.ptr(src), L.ptr(order), L.ptr(chunk_start),
                                    L.ptr(chunk_end), L.ptr(dst), n, L.ptr(out), L.stream_ptr(src.device))
    L.check(rc, 'gm_segment_sum')
    return out


def scatter_add_rows_deterministic(rows, index, out, chunk=128):
    """out[index[k]] += rows[k] for all k, as a FIXED-ORDER sum (out must be zero on entry: rows of `out` that receive
    something are overwritten with their sum, the others left alone).  Entries of a destination row are taken in
    ascending k (stable sort), in chunks of `chunk` entries (level 1), then the chunk sums in order (level 2)."""
    index = index.reshape(-1).long()
    order = torch.sort(index, stable=True).indices.contiguous()
    dest, counts = torch.unique_consecutive(index[order], return_counts=True)
    seg_start = torch.cumsum(counts, 0) - counts
    n_ch = (counts + (chunk - 1)) // chunk
    ch_first = torch.cumsum(n_ch, 0) - n_ch              # first chunk of every segment
    seg_of = torch.repeat_interleave(torch.arange(dest.numel(), device=index.device), n_ch)
    within = torch.arange(seg_of.numel(), device=index.device) - ch_first[seg_of]
    c_start = (seg_start[seg_of] + within * chunk).contiguous()
    c_end = torch.minimum(c_start + chunk, (seg_start + counts)[seg_of]).contiguous()
    partial = torch.empty((seg_of.numel(),) + tuple(rows.shape[1:]), dtype=rows.dtype, device=rows.device)
    segment_sum(rows, c_start, c_end, partial, order=order)
    segment_sum(partial, ch_first.contiguous(), (ch_first + n_ch).contiguous(), out, dst=dest.contiguous())
    return out


FUSABLE_VECTOR_KINDS = (L.GM_LORENTZ, L.GM_SPHERE, L.GM_EUCLIDEAN)
MAX_FUSED_VECTOR_FACTORS = 3


def product_fusable(specs, dtypes):
    """Does gm_pairs_product_fused take this factor list?  (At most one SPD factor, up to three of Lorentz / Sphere /
    Euclidean, 2 <= F <= 4, one dtype -- include/gm_kernels.h.)"""
    kinds = [sp.kind for sp in specs]
    n_spd = sum(k in (L.GM_SPD_AI, L.GM_SPD_STEIN) for k in kinds)
    n_vec = sum(k in FUSABLE_VECTOR_KINDS for k in kinds)
    return (2 <= len(kinds) <= 1 + MAX_FUSED_VECTOR_FACTORS and n_spd + n_vec == len(kinds) and n_spd <= 1
            and n_vec <= MAX_FUSED_VECTOR_FACTORS and len(set(dtypes)) == 1)


@_no_function_modes
def pairs_product_fused(specs, xs, pairs, targets, loss, sp_list, grads, acc=None):
    """One kernel for a product manifold: every factor's d2, the loss of m = sum_f sp_f d2_f and every factor's gradient
    (accumulated into grads[f]).  Returns acc (float64, 1 + F: [sum loss, sum l' d2_f ...], accumulated into)."""
    F = len(specs)
    xs = [_prep(x) for x in xs]
    dtype, device = xs[0].dtype, xs[0].device
    if acc is None:
        acc = torch.zeros(1 + F, dtype=torch.float64, device=device)
    mans = (L.Manifold * F)(*[sp.c_struct(dtype, device) for sp in specs])
    xp = (ctypes.c_void_p * F)(*[x.data_ptr() for x in xs])
    gp = (ctypes.c_void_p * F)(*[g.data_ptr() for g in grads])
    sps = (ctypes.c_double * F)(*[float(s) for s in sp_list])
    p, t, l = pairs.c_struct(), targets.c_struct(), loss.c_struct()
    with torch.cuda.device(device):
        rc = L.lib().gm_pairs_product_fused(F, mans, xp, ctypes.byref(p), ctypes.byref(t), ctypes.byref(l), sps,
                                            L.ptr(acc), gp, L.stream_ptr(device))
    L.check(rc, 'gm_pairs_product_fused')
    return acc


@_no_function_modes
def product_loss(d2_list, sp_list, targets, loss, want_g=True, pairs=None):
    """Loss over the product distance m = sum_f sp_f * d2_f.  Returns (acc[1+F] float64, dL/dm per pair).  DENSE
    targets (the (N, N) matrix of GraphDataset) need `pairs`, whose node ids index the matrix."""
    F = len(d2_list)
    d2_list = [_prep(d) for d in d2_list]
    dtype, device, P = d2_list[0].dtype, d2_list[0].device, d2_list[0].numel()
    acc = torch.zeros(1 + F, dtype=torch.float64, device=device)
    g = torch.empty(P, dtype=dtype, device=device) if want_g else None
    ptrs = (ctypes.c_void_p * F)(*[d.data_ptr() for d in d2_list])
    sps = (ctypes.c_double * F)(*[float(s) for s in sp_list])
    t, l = targets.c_struct(), loss.c_struct()
    pc = None if pairs is None else ctypes.byref(pairs.c_struct())
    with torch.cuda.device(device):
        rc = L.lib().gm_product_loss(L.dtype_code(dtype), F, ptrs, sps, pc, ctypes.byref(t), ctypes.byref(l), P,
                                     L.ptr(acc), L.ptr(g), L.stream_ptr(device))
    L.check(rc, 'gm_product_loss')
    return acc, g


def _factor_args(d2_list, sp_list):
    F = len(d2_list)
    ptrs = (ctypes.c_void_p * F)(*[d.data_ptr() for d in d2_list])
    sps = (ctypes.c_double * F)(*[float(s) for s in sp_list])
    return F, ptrs, sps


@_no_function_modes
def pairs_metrics(d2_list, sp_list, pairs, targets, squared=True, acc=None):
    """Adds the validation-metric moments of the given pairs to `acc` (8 float64 slots):
    [count, sum |m-g|/g, sum m, sum g, sum m^2, sum g^2, sum m g] with m = sqrt(sum_f sp_f d2_f), g = sqrt(target)
    (squared=True) or m = d2_list[0], g = target (squared=False)."""
    d2_list = [_prep(d) for d in d2_list]
    dtype, device = d2_list[0].dtype, d2_list[0].device
    if acc is None:
        acc = torch.zeros(8, dtype=torch.float64, device=device)
    if targets.mode in (L.GM_TGT_VECTOR, L.GM_TGT_DENSE) and targets.data.dtype != dtype:
        raise RuntimeError('targets must have the dtype of the distances')
    F, ptrs, sps = _factor_args(d2_list, sp_list)
    p, t = pairs.c_struct(), targets.c_struct()
    with torch.cuda.device(device):
        rc = L.lib().gm_pairs_metrics(L.dtype_code(dtype), F, ptrs, sps, ctypes.byref(p), ctypes.byref(t),
                                      int(bool(squared)), L.ptr(acc), L.stream_ptr(device))
    L.check(rc, 'gm_pairs_metrics')
    return acc


def sne_kl(d2_list, sp_list, gdists, alpha, inclusive, want_g=True):
    """KL objective with the stochastic-neighbour model over all pairs of a batch (condensed vectors).
    Returns (acc[1+F] float64: [KL, sum_k g_k d2_f[k] ...], dKL/dm per pair)."""
    d2_list = [_prep(d) for d in d2_list]
    dtype, device, P = d2_list[0].dtype, d2_list[0].device, d2_list[0].numel()
    gdists = _prep(gdists.to(dtype))
    if gdists.numel() != P:
        raise ValueError('graph and manifold distance vectors differ in length')
    import math
    B = math.ceil(math.sqrt(2 * P))
    if B * (B - 1) // 2 != P:
        raise ValueError(f'{P} is not the number of pairs of a batch')
    F, ptrs, sps = _factor_args(d2_list, sp_list)
    acc = torch.zeros(1 + F, dtype=torch.float64, device=device)
    stats = torch.empty(3 * B, dtype=dtype, device=device)
    g = torch.empty(P, dtype=dtype, device=device) if want_g else None
    with torch.cuda.device(device):
        st = L.stream_ptr(device)
        rc = L.lib().gm_sne_row_stats(L.dtype_code(dtype), F, ptrs, sps, L.ptr(gdists), B, float(alpha),
                                      int(bool(inclusive)), L.ptr(stats), st)
        L.check(rc, 'gm_sne_row_stats')
        rc = L.lib().gm_sne_pair_terms(L.dtype_code(dtype), F, ptrs, sps, L.ptr(gdists), B, float(alpha),
                                       int(bool(inclusive)), L.ptr(stats), L.ptr(acc), L.ptr(g), st)
        L.check(rc, 'gm_sne_pair_terms')
    return acc, g


@_no_function_modes
def point_op(spec, op, x, u=None, v=None, scalar=False):
    x = _prep(x)
    u = None if u is None else _prep(u.to(x.dtype))
    v = None if v is None else _prep(v.to(x.dtype))
    nd = len(spec.point_shape)
    if tuple(x.shape[x.ndim - nd:]) != spec.point_shape:
        raise RuntimeError(f'expected points of shape (..., {spec.point_shape}), got {tuple(x.shape)}')
    batch = x.shape[:x.ndim - nd]
    N = 1
    for b in batch:
        N *= b
    out = torch.empty(batch if scalar else x.shape, dtype=x.dtype, device=x.device)
    m = spec.c_struct(x.dtype, x.device)
    with torch.cuda.device(x.device):
        rc = L.lib().gm_point_op(ctypes.byref(m), op, L.ptr(x), L.ptr(u), L.ptr(v), L.ptr(out), N,
                                 L.stream_ptr(x.device))
    L.check(rc, 'gm_point_op')
    return out


@_no_function_modes
def optim_step(spec, cfg, x, grad, buf1=None, buf2=None):
    """In-place fused optimizer update of the (N, ...) parameter `x`."""
    L.require_cuda(x, grad, buf1, buf2)
    if not x.is_contiguous():
        raise RuntimeError('parameters must be contiguous')
    grad = _prep(grad.to(x.dtype))
    N = x.numel() // spec.numel
    m = spec.c_struct(x.dtype, x.device)
    with torch.cuda.device(x.device):
        rc = L.lib().gm_optim_step(ctypes.byref(m), ctypes.byref(cfg), L.ptr(x), L.ptr(grad), L.ptr(buf1),
                                   L.ptr(buf2), N, L.stream_ptr(x.device))
    L.check(rc, 'gm_optim_step')


@_no_function_modes
def optim_step_peer(spec, cfg, arena, own_rows, buf1=None, buf2=None):
    """Fused reduce-scatter + optimizer update + all-gather over NVLink peer memory (gm_optim_step_peer): updates the
    rows of arena.x this rank owns from the sum of every rank's arena.grad and publishes them to every rank."""
    L.require_cuda(arena.x, buf1, buf2)
    m = spec.c_struct(arena.x.dtype, arena.x.device)
    table = arena.next_table()
    with torch.cuda.device(arena.x.device):
        rc = L.lib().gm_optim_step_peer(ctypes.byref(m), ctypes.byref(cfg), ctypes.byref(table), L.ptr(buf1),
                                        L.ptr(buf2), own_rows, L.stream_ptr(arena.x.device))
    L.check(rc, 'gm_optim_step_peer')


# ----------------------------------------------------------------------------
# autograd Functions
# ----------------------------------------------------------------------------
class _Dist2Elementwise(torch.autograd.Function):
    """d2[k] = dist^2(x[k], y[k]); backward writes per-row gradients."""

    @staticmethod
    def forward(ctx, x, y, spec, c=None, wmin=None):
        ctx.spec = spec
        x, y = _prep(x), _prep(y)
        ctx.c = None if c is None else c.detach()
        ctx.save_for_backward(x, y)
        nd = len(spec.point_shape)
        ctx.batch_shape = x.shape[:x.ndim - nd]
        d2 = pairs_dist2(spec, x, y, PairSet.elementwise(x.numel() // spec.numel), c=c, wmin=wmin)
        return d2.view(ctx.batch_shape)

    @staticmethod
    def backward(ctx, g):
        x, y = ctx.saved_tensors
        gx, gy = torch.empty_like(x), torch.empty_like(y)
        gc = _curvature_grad_buffer(ctx.c, ctx.needs_input_grad[3])
        pairs_grad(ctx.spec, x, y, PairSet.elementwise(x.numel() // ctx.spec.numel), g.reshape(-1), gx, gy,
                   c=ctx.c, c_grad=gc)
        return gx, gy, None, _curvature_grad(ctx.c, gc), None


def _curvature_grad_buffer(c, wanted):
    """float64 device accumulator for d(loss)/dc when the (Universal) curvature tensor wants a gradient."""
    if c is None or not wanted:
        return None
    return torch.zeros(1, dtype=torch.float64, device=c.device)


def _curvature_grad(c, gc):
    return None if gc is None else gc.to(c.dtype).reshape(c.shape)


class _Dist2Indexed(torch.autograd.Function):
    """d2 over a PairSet (LIST or TRIU) of rows of one parameter tensor; backward accumulates into a dense
    gradient of x's shape (the fused equivalent of x[I], x[J] gathers + index_put_ backward)."""

    @staticmethod
    def forward(ctx, x, spec, pairs, c=None, wmin=None):
        ctx.spec, ctx.pairs, ctx.c = spec, pairs, (None if c is None else c.detach())
        x = _prep(x)
        ctx.save_for_backward(x)
        return pairs_dist2(spec, x, x, pairs, c=c, wmin=wmin)

    @staticmethod
    def backward(ctx, g):
        x, = ctx.saved_tensors
        gx = torch.zeros_like(x)
        gc = _curvature_grad_buffer(ctx.c, ctx.needs_input_grad[3])
        pairs_grad(ctx.spec, x, x, ctx.pairs, g, gx, gx, c=ctx.c, c_grad=gc)
        return gx, None, None, _curvature_grad(ctx.c, gc), None


def dist2_elementwise(spec, x, y, c=None, wmin=None):
    """`c`: the Universal manifold's curvature tensor get_c() (receives a gradient); None otherwise."""
    return _Dist2Elementwise.apply(x, y, spec, c, wmin)


def dist2_indexed(spec, x, pairs, c=None, wmin=None):
    return _Dist2Indexed.apply(x, spec, pairs, c, wmin)


@_no_function_modes
def unpack_pairs2(words, base, offsets, out, group_rows=None, out_i=None):
    """gm_unpack_pairs2: 2-byte delta words (engine.pack_hops2) of a source-grouped batch -> out[k] = j | hops << 24.
    words int16 (P,), base int32 (G,), offsets int64 (G + 1,), out int32 (>= P,), all on one CUDA device.  With
    group_rows int32 (G,) and out_i int32 (>= P,) the first-endpoint vector out_i[k] = group_rows[g] is written in the
    same pass (expand_groups folded in)."""
    L.require_cuda(words, base, offsets, out, group_rows, out_i)
    G = base.numel()
    if (words.dtype != torch.int16 or base.dtype != torch.int32 or offsets.dtype != torch.int64
            or out.dtype != torch.int32 or offsets.numel() != G + 1 or out.numel() < words.numel()):
        raise ValueError('unpack_pairs2: int16 words, int32 base (G,), int64 offsets (G + 1,), int32 output of P words')
    if (group_rows is None) != (out_i is None):
        raise ValueError('unpack_pairs2: group_rows and out_i go together')
    if group_rows is not None and (group_rows.dtype != torch.int32 or out_i.dtype != torch.int32
                                   or group_rows.numel() != G or out_i.numel() < words.numel()):
        raise ValueError('unpack_pairs2: int32 group_rows (G,) and int32 out_i of P words')
    with torch.cuda.device(out.device):
        rc = L.lib().gm_unpack_pairs2(L.ptr(words), L.ptr(base), L.ptr(offsets), G, L.ptr(out), L.ptr(group_rows),
                                      L.ptr(out_i), L.stream_ptr(out.device))
    L.check(rc, 'gm_unpack_pairs2')


def unpack_pairs3(src3, P, out):
    """3-byte pair words (engine.pack_hops3) -> out[k] = (hops << 24) | j, the GM_TGT_HOPS_PACKED form (all CUDA)."""
    L.require_cuda(src3, out)
    if src3.dtype != torch.uint8 or out.dtype != torch.int32 or src3.numel() < 3 * P or out.numel() < P:
        raise ValueError('unpack_pairs3: uint8 source of 3*P bytes, int32 output of P words')
    rc = L.lib().gm_unpack_pairs3(L.ptr(src3), P, L.ptr(out), L.stream_ptr(out.device))
    L.check(rc, 'gm_unpack_pairs3')
    return out


def expand_groups(group_rows, offsets, out):
    """out[k] = group_rows[g] for offsets[g] <= k < offsets[g+1] (int32 rows, int64 offsets, int32 out; all CUDA)."""
    L.require_cuda(group_rows, offsets, out)
    G, P = group_rows.numel(), out.numel()
    if offsets.numel() != G + 1 or group_rows.dtype != torch.int32 or out.dtype != torch.int32 or \
            offsets.dtype != torch.int64:
        raise ValueError('expand_groups: int32 rows (G,), int64 offsets (G+1,), int32 out (P,)')
    rc = L.lib().gm_expand_groups(L.ptr(group_rows), L.ptr(offsets), G, L.ptr(out), P, L.stream_ptr(out.device))
    L.check(rc, 'gm_expand_groups')
    return out
