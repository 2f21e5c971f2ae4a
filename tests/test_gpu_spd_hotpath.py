"""The SPD pair kernels on the training path, at training scale, against a pair-level fp64 reference
(tests/helpers_hotpath.py): spd_pair_stream_kernel with warps that walk many iterations (pipeline rotation, the
cached inverse Cholesky factor of the first endpoint, run-length gradient accumulation and its flushes), window-ordered
segmented walks including the SPEC instantiation bench.py launches, drawn (SAMPLED) pairs, TRIU slices with DENSE
targets, the backward-only kernel with separate input and output tables, and one PairTrainer step.

Every launch is compared per pair and per gradient row, separately for each input class:
  A bench-like (rand ir=0.1)  B moderate (ir=1.0)  C spectra log-uniform in [1e-2, 1e2]  D near-duplicate rows, bitwise
  copies (d2 at its wmin floor) and i == j self-pairs  E spectra in [1e-3, 1e3] (with wmin=1e-4, wmax=1e4 the
  generalised eigenvalues leave [wmin, wmax] and the straight-through clamps act).
"""
import pytest
import torch

import helpers_hotpath as H

pytestmark = pytest.mark.gpu
DEV = torch.device('cuda', 0)
MAX_SQ = 64.0
S = float(torch.nn.functional.softplus(torch.tensor(0.5)))  # fp32 value, as bench.py's scale
# 2^21 pairs, ragged (not a multiple of 32 or of any run length): with at most 16 blocks of 4 warps per SM the grid
# has at most SMs x 64 warps, so a warp walks >= P / (32 x 148 x 64) ~ 7 positions of 32 pairs in a plain launch
P_MAIN = (1 << 21) - 13
N_MAIN = {H.CA: 24576, H.CB: 12288, H.CD: 12288, H.CC: 8192, H.CE: 8192}  # 65536 rows: windows of 8192 rows at W = 8


@pytest.fixture(scope='module', autouse=True)
def _one_host_thread():
    """The reference runs batched 4x4 / 6x6 LAPACK calls and index_add_ over millions of small rows: one thread is as
    fast as many for these, and avoids pathological thread wake-ups on many-core hosts."""
    n = torch.get_num_threads()
    torch.set_num_threads(1)
    yield
    torch.set_num_threads(n)


def _max_warps():
    return torch.cuda.get_device_properties(DEV).multi_processor_count * 64


def _hops(P, seed):
    return torch.randint(1, 9, (P,), generator=torch.Generator().manual_seed(seed), dtype=torch.uint8)


@pytest.fixture(scope='module')
def main4():
    x, cls, partner = H.point_table(4, N_MAIN, seed=11)
    I, J = H.grouped_pairs(cls, partner, P_MAIN, seed=12, weights={H.CA: 4, H.CB: 2, H.CD: 2, H.CC: 1, H.CE: 1})
    ref = H.PairReference(x, I, J, 4)
    pcls = H.pair_classes(cls, I, J)
    return dict(x=x, cls=cls, I=I, J=J, hops=_hops(P_MAIN, 13), ref=ref, pcls=pcls,
                rcls=H.row_classes(cls, (I, J), pcls))


def _fused(man_spec, x, I, J, hops, target, idx64=False, segments=0, dtype=torch.float32, vec=None):
    """One gm_pairs_loss_fused launch (QuotientLoss, epoch 1) -> (d2, grad, acc) on the host."""
    from graphembed import _ops, _lib as L
    from graphembed.engine import pack_hops
    xd = x.to(DEV, dtype).contiguous()
    it = torch.int64 if idx64 else torch.int32
    Id = I.to(it).to(DEV)
    if target == 'packed':
        Jd = pack_hops(J.int(), hops).to(DEV)
        tg = _ops.TargetSpec.hops_packed(MAX_SQ)
    else:
        Jd = J.to(it).to(DEV)
        tg = _ops.TargetSpec.hops(hops.to(DEV), MAX_SQ) if target == 'u8' else _ops.TargetSpec.vector(vec.to(DEV, dtype))
    pairs = _ops.PairSet.from_lists(Id, Jd, DEV, segments=segments)
    grad = torch.zeros_like(xd)
    acc, d2 = _ops.pairs_loss_fused(man_spec, xd, pairs, tg, _ops.LossSpec(L.GM_LOSS_QUOTIENT, True, True, 1.0, 0.5),
                                    S, grad, want_d2=True)
    torch.cuda.synchronize()
    return d2.cpu(), grad.cpu(), acc.cpu()


def _check_fused(what, dtype, out, ref, g, pcls, rcls, I, J):
    d2, grad, acc = out
    chk = H.Checker(dtype, what)
    chk.d2(d2, ref, pcls)
    w = H.loss_weights('quotient', g, d2, S)[2]  # weights on the kernel's own distances (QuotientLoss has kinks)
    chk.grad([(grad, [(I, 'gx'), (J, 'gy')])], ref, w, [rcls])
    chk.acc(acc, 'quotient', g, d2, ref, pcls, S)
    print('\n' + chk.report())
    chk.assert_ok()


# ---------------------------------------------------------------------------------------------------------------------
# grouped LIST, plain and window-ordered
# ---------------------------------------------------------------------------------------------------------------------
LIST_CASES = [  # (index type, target, segments)
    ('i32', 'packed', 0), ('i32', 'u8', 0), ('i32', 'vector', 0), ('i64', 'u8', 0),
    ('i32', 'packed', 2), ('i32', 'packed', 4),  # SPEC instantiation (int32, HOPS_PACKED, segments > 1)
    ('i32', 'u8', 4),  # generic segmented kernel
]


@pytest.mark.parametrize('idx,target,W', LIST_CASES)
def test_list_fused_spd4_f32(main4, idx, target, W):
    from graphembed.engine import window_order
    from graphembed.manifolds import SymmetricPositiveDefinite
    m = main4
    I, J, hops, ref = m['I'], m['J'], m['hops'], m['ref']
    pcls = m['pcls']
    if W:
        # the segmented walk needs P >= W x 32 x warps; warps <= SMs x 64 (16 blocks of 4 warps per SM at most)
        assert P_MAIN >= W * 32 * _max_warps(), 'too few pairs for a segmented walk on this GPU'
        order = window_order(J.int(), m['x'].shape[0], W)
        I, J, hops, ref, pcls = I[order], J[order], hops[order], ref.permuted(order), pcls[order]
    vec = None
    if target == 'vector':
        vec = torch.rand(I.numel(), generator=torch.Generator().manual_seed(14)) * 0.9 + 0.05
        g = vec.double()
    else:
        g = H.targets_from_hops(hops, MAX_SQ, torch.float32)
    out = _fused(SymmetricPositiveDefinite(4).spec, m['x'], I, J, hops, target, idx64=idx == 'i64', segments=W, vec=vec)
    _check_fused(f'SPD4 f32 LIST {idx} {target} W={W}', torch.float32, out, ref, g, pcls, m['rcls'], I, J)


def test_list_fused_spd4_f64(main4):
    """fp64 bars (1e-10) on classes A, B, D.  Classes C and E (condition numbers 1e4 and 1e6, generalised eigenvalues
    spread over up to 12 decades) are not compared: there the fp64 LAPACK reference is itself not accurate to 1e-10
    (kernel and reference differ by 1.7e-10 and 2.6e-8 relative in d2), so such a bar would not say which is wrong."""
    from graphembed.manifolds import SymmetricPositiveDefinite
    m = main4
    g = H.targets_from_hops(m['hops'], MAX_SQ, torch.float64)
    out = _fused(SymmetricPositiveDefinite(4).spec, m['x'], m['I'], m['J'], m['hops'], 'packed', dtype=torch.float64)
    skip = len(H.NAMES)
    pcls = torch.where(m['pcls'] >= H.CC, skip, m['pcls'])
    rcls = torch.where(m['rcls'] >= H.CC, skip, m['rcls'])
    _check_fused('SPD4 f64 LIST i32 packed', torch.float64, out, m['ref'], g, pcls, rcls, m['I'], m['J'])


def test_d2_bitwise_across_paths(main4):
    """Per-pair out_d2 is the same bits through the plain walk, the generic segmented walk, SPEC and K_FWD."""
    from graphembed import _ops
    from graphembed.engine import window_order
    from graphembed.manifolds import SymmetricPositiveDefinite
    m = main4
    spec = SymmetricPositiveDefinite(4).spec
    order = window_order(m['J'].int(), m['x'].shape[0], 4)
    Io, Jo, ho = m['I'][order], m['J'][order], m['hops'][order]
    plain = _fused(spec, m['x'], m['I'], m['J'], m['hops'], 'packed')[0]
    spec_w = _fused(spec, m['x'], Io, Jo, ho, 'packed', segments=4)[0]
    generic_w = _fused(spec, m['x'], Io, Jo, ho, 'u8', segments=4)[0]
    xd = m['x'].to(DEV)
    fwd = _ops.pairs_dist2(spec, xd, xd, _ops.PairSet.from_lists(m['I'].int().to(DEV), m['J'].int().to(DEV), DEV)).cpu()
    assert torch.equal(plain, fwd)
    assert torch.equal(plain[order], spec_w)
    assert torch.equal(plain[order], generic_w)


# ---------------------------------------------------------------------------------------------------------------------
# backward-only kernel: separate input / output tables
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('tables', ['distinct', 'aliased'])
def test_grad_bwd_spd4_f32(main4, tables):
    """gm_pairs_grad with xa != xb and ga != gb: xb is xa with its rows permuted and the second endpoints renumbered
    to match, so every pair sees the same two matrices as in the reference -- a read of the wrong table, or a gradient
    written to the wrong one, changes the answer.  Distinct tables go through a window-ordered segmented walk."""
    from graphembed import _ops
    from graphembed.engine import window_order
    from graphembed.manifolds import SymmetricPositiveDefinite
    m = main4
    x, I, J, ref, pcls, cls = m['x'], m['I'], m['J'], m['ref'], m['pcls'], m['cls']
    N = x.shape[0]
    gen = torch.Generator().manual_seed(15)
    gout = torch.rand(I.numel(), generator=gen) * 2 - 1
    coef = 0.37
    spec = SymmetricPositiveDefinite(4).spec
    if tables == 'distinct':
        perm = torch.randperm(N, generator=gen)
        inv = torch.argsort(perm)
        Jb = inv[J]  # xb[Jb] == x[perm[inv[J]]] == x[J]
        order = window_order(Jb.int(), N, 4)
        I, Jb, gout, ref, pcls = I[order], Jb[order], gout[order], ref.permuted(order), pcls[order]
        xa, xb = x.to(DEV), x[perm].contiguous().to(DEV)
        ga, gb = torch.zeros_like(xa), torch.zeros_like(xb)
        pairs = _ops.PairSet.from_lists(I.int().to(DEV), Jb.int().to(DEV), DEV, segments=4)
        _ops.pairs_grad(spec, xa, xb, pairs, gout.to(DEV), ga, gb, coef=coef)
        w = coef * gout.double()
        out = [(ga.cpu(), [(I, 'gx')]), (gb.cpu(), [(Jb, 'gy')])]
        rcls = [H.row_classes(cls, (I,), pcls), H.row_classes(cls[perm], (Jb,), pcls)]
    else:
        xa = x.to(DEV)
        ga = torch.zeros_like(xa)
        pairs = _ops.PairSet.from_lists(I.int().to(DEV), J.int().to(DEV), DEV)
        _ops.pairs_grad(spec, xa, xa, pairs, gout.to(DEV), ga, ga, coef=coef)
        w = coef * gout.double()
        out = [(ga.cpu(), [(I, 'gx'), (J, 'gy')])]
        rcls = [m['rcls']]
    chk = H.Checker(torch.float32, f'SPD4 f32 K_BWD {tables}')
    chk.grad(out, ref, w, rcls)
    print('\n' + chk.report())
    chk.assert_ok()


# ---------------------------------------------------------------------------------------------------------------------
# clamps: wmin = 1e-4, wmax = 1e4
# ---------------------------------------------------------------------------------------------------------------------
def test_clamped_spectrum_spd4_f32(main4):
    from graphembed.manifolds import SymmetricPositiveDefinite
    m = main4
    P = (1 << 18) - 3
    I, J = H.grouped_pairs(m['cls'], torch.full_like(m['cls'], -1), P, seed=16,
                           weights={H.CA: 1, H.CB: 1, H.CC: 1, H.CE: 4})
    ref = H.PairReference(m['x'], I, J, 4, wmin=1e-4, wmax=1e4)
    pcls = H.pair_classes(m['cls'], I, J)
    hops = _hops(P, 17)
    man = SymmetricPositiveDefinite(4, wmin=1e-4, wmax=1e4)
    out = _fused(man.spec, m['x'], I, J, hops, 'packed')
    _check_fused('SPD4 f32 LIST wmin=1e-4 wmax=1e4', torch.float32, out, ref, H.targets_from_hops(hops, MAX_SQ, torch.float32),
                 pcls, H.row_classes(m['cls'], (I, J), pcls), I, J)


# ---------------------------------------------------------------------------------------------------------------------
# SAMPLED pairs
# ---------------------------------------------------------------------------------------------------------------------
def test_sampled_spd4_f32(main4):
    """Pairs drawn on the device over the bench-like and moderate rows: per_src not a power of two, P not a multiple
    of it, a uint8 level table addressed through a non-identity slot map."""
    import numpy as np
    import sampler_oracle
    from graphembed import _ops, _lib as L
    from graphembed.manifolds import SymmetricPositiveDefinite
    m = main4
    n_sub = N_MAIN[H.CA] + N_MAIN[H.CB]  # class blocks A, B come first
    x, cls = m['x'][:n_sub].contiguous(), m['cls'][:n_sub]
    gen = torch.Generator().manual_seed(18)
    G, per_src = 175, 3000
    P = G * per_src - 77
    sources = torch.randperm(n_sub, generator=gen)[:G].int()
    slots = torch.randperm(G, generator=gen).int()
    levels = torch.randint(1, 9, (G, n_sub), generator=gen, dtype=torch.uint8)
    seed = 0x1234567
    I, J, hops = sampler_oracle.sample_pairs(sources.numpy(), levels.numpy(), per_src, seed, slots=slots.numpy(), P=P)
    I, J, hops = torch.from_numpy(I).long(), torch.from_numpy(J).long(), torch.from_numpy(np.ascontiguousarray(hops))
    ref = H.PairReference(x, I, J, 4)
    pcls = H.pair_classes(cls, I, J)
    xd = x.to(DEV)
    grad = torch.zeros_like(xd)
    pairs = _ops.PairSet.sampled(sources.to(DEV), levels.to(DEV), per_src, seed, slots=slots.to(DEV), P=P)
    acc, d2 = _ops.pairs_loss_fused(SymmetricPositiveDefinite(4).spec, xd, pairs, _ops.TargetSpec.hops_packed(MAX_SQ),
                                    _ops.LossSpec(L.GM_LOSS_QUOTIENT, True, True, 1.0, 0.5), S, grad, want_d2=True)
    _check_fused('SPD4 f32 SAMPLED', torch.float32, (d2.cpu(), grad.cpu(), acc.cpu()), ref,
                 H.targets_from_hops(hops, MAX_SQ, torch.float32), pcls, H.row_classes(cls, (I, J), pcls), I, J)


# ---------------------------------------------------------------------------------------------------------------------
# TRIU slice with DENSE targets
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def triu4():
    x, cls, _ = H.point_table(4, {H.CA: 2048, H.CB: 2048}, seed=21)
    gen = torch.Generator().manual_seed(22)
    B = 1536
    nodes = torch.randperm(x.shape[0], generator=gen)[:B]
    ia, ib = torch.triu_indices(B, B, 1)
    k0 = int(torch.nonzero(ia == 100)[0]) + 37  # starts inside row 100 of the triangle ...
    P = ia.numel() - k0 - 1234                  # ... and ends inside a row too
    I, J = nodes[ia[k0:k0 + P]], nodes[ib[k0:k0 + P]]
    h = torch.randint(1, 9, (x.shape[0], x.shape[0]), generator=gen, dtype=torch.uint8)
    h = torch.triu(h, 1) + torch.triu(h, 1).T
    ref = H.PairReference(x, I, J, 4)
    pcls = H.pair_classes(cls, I, J)
    return dict(x=x, cls=cls, nodes=nodes, B=B, k0=k0, P=P, I=I, J=J, h=h, ref=ref, pcls=pcls,
                rcls=H.row_classes(cls, (I, J), pcls))


@pytest.mark.parametrize('dtype', [torch.float32, torch.float64])
def test_triu_dense_spd4(triu4, dtype):
    from graphembed import _ops, _lib as L
    from graphembed.manifolds import SymmetricPositiveDefinite
    t = triu4
    dense = (t['h'].to(dtype) ** 2) / MAX_SQ
    xd = t['x'].to(DEV, dtype)
    it = torch.int32 if dtype == torch.float32 else torch.int64
    pairs = _ops.PairSet.triu(t['B'], nodes=t['nodes'].to(it).to(DEV), device=DEV, k0=t['k0'], P=t['P'])
    grad = torch.zeros_like(xd)
    acc, d2 = _ops.pairs_loss_fused(SymmetricPositiveDefinite(4).spec, xd, pairs, _ops.TargetSpec.dense(dense.to(DEV)),
                                    _ops.LossSpec(L.GM_LOSS_QUOTIENT, True, True, 1.0, 0.5), S, grad, want_d2=True)
    g = dense[t['I'], t['J']].double()
    _check_fused(f'SPD4 {str(dtype)[6:]} TRIU k0={t["k0"]} DENSE', dtype, (d2.cpu(), grad.cpu(), acc.cpu()), t['ref'], g,
                 t['pcls'], t['rcls'], t['I'], t['J'])


# ---------------------------------------------------------------------------------------------------------------------
# SPD 6x6 (config 4's kernel)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def spd6_check():
    from graphembed.manifolds import SymmetricPositiveDefinite
    x, cls, partner = H.point_table(6, {H.CA: 8192, H.CB: 4096, H.CD: 4096, H.CC: 2048}, seed=31)
    P = (1 << 19) - 7
    I, J = H.grouped_pairs(cls, partner, P, seed=32)
    ref = H.PairReference(x, I, J, 6)
    pcls = H.pair_classes(cls, I, J)
    hops = _hops(P, 33)
    d2, grad, acc = _fused(SymmetricPositiveDefinite(6).spec, x, I, J, hops, 'packed')
    g = H.targets_from_hops(hops, MAX_SQ, torch.float32)
    chk = H.Checker(torch.float32, 'SPD6 f32 LIST i32 packed')
    chk.d2(d2, ref, pcls)
    chk.grad([(grad, [(I, 'gx'), (J, 'gy')])], ref, H.loss_weights('quotient', g, d2, S)[2],
             [H.row_classes(cls, (I, J), pcls)])
    chk.acc(acc, 'quotient', g, d2, ref, pcls, S)
    print('\n' + chk.report())
    return chk


def test_list_fused_spd6_f32(spd6_check):
    """Config 4's kernel with warps that walk several iterations.  On spectra over 4 decades (class C) the loss summed
    over the class is the bar that caught a bias of the 6x6 Jacobi eigenvalues (gm_math.cuh, jacobi_eigh)."""
    spd6_check.assert_ok()


# ---------------------------------------------------------------------------------------------------------------------
# one bench step: PairTrainer.step_host_grouped on window-grouped 2-byte words, RAdam exact with clipping
# ---------------------------------------------------------------------------------------------------------------------
def test_trainer_step_spd4_f32(main4):
    import manifolds_oracle as O
    from graphembed.engine import PairTrainer, pack_hops2, window_groups
    from graphembed.manifolds import SymmetricPositiveDefinite
    from graphembed.modules import ManifoldEmbedding, _softplus_value
    from graphembed.objectives import QuotientLoss
    from graphembed.optim import RiemannianAdam
    m = main4
    x, I, J, hops, ref = m['x'], m['I'], m['J'], m['hops'], m['ref']
    N, W = x.shape[0], 8
    # the source groups of the batch (runs of one first endpoint), then the (window, source) groups of bench.py
    change = torch.ones(I.numel(), dtype=torch.bool)
    change[1:] = I[1:] != I[:-1]
    starts = torch.nonzero(change).flatten()
    sources = I[starts].int()
    offsets = torch.cat([starts, torch.tensor([I.numel()])])
    order, src_groups, goff = window_groups(sources, offsets, J.int(), N, W)
    words, bases, order2 = pack_hops2(goff, J.int()[order].contiguous(), hops[order].contiguous())
    perm = order[order2]  # pair k of the step is pair perm[k] of the batch
    emb = ManifoldEmbedding(N, [SymmetricPositiveDefinite(4)], device=DEV, dtype=torch.float32)
    emb.xs[0].data.copy_(x.to(DEV))
    sp = float(_softplus_value(emb.scales[0]))
    opt = RiemannianAdam(emb.xs, lr=0.01, max_grad_norm=100, exact=True)
    tr = PairTrainer(emb, opt, QuotientLoss(), max_hops_sq=MAX_SQ)
    loss = tr.step_host_grouped(src_groups.pin_memory(), goff.pin_memory(), words.pin_memory(), None, epoch=1,
                                segments=W, bases=bases.pin_memory())
    x_new = emb.xs[0].detach().cpu()
    assert torch.equal(I[perm].int(), src_groups.repeat_interleave(goff[1:] - goff[:-1]))
    # reference: loss on fp64 distances; gradient weights on the kernel's own distances (the same bits in every walk
    # order: test_d2_bitwise_across_paths), fp64 / fp32 sums, then the oracle's RAdam step
    g = H.targets_from_hops(hops, MAX_SQ, torch.float32)
    d2_k = _fused(SymmetricPositiveDefinite(4).spec, x, I, J, hops, 'packed')[0]
    w = H.loss_weights('quotient', g, d2_k, sp)[2]
    G64 = torch.zeros(x.shape, dtype=torch.float64).index_add_(0, I, w.view(-1, 1, 1) * ref.gx_64)
    G64.index_add_(0, J, w.view(-1, 1, 1) * ref.gy_64)
    G32 = torch.zeros(x.shape).index_add_(0, I, w.float().view(-1, 1, 1) * ref.gx_32)
    G32.index_add_(0, J, w.float().view(-1, 1, 1) * ref.gy_32)
    x64 = O.radam_step(O.SpdOracle(4), x.double(), G64, {}, lr=0.01, max_grad_norm=100, exact=True)
    x32 = O.radam_step(O.SpdOracle(4), x.float(), G32, {}, lr=0.01, max_grad_norm=100, exact=True)
    chk = H.Checker(torch.float32, 'SPD4 f32 PairTrainer.step_host_grouped (2-byte words, W=8)')
    chk.scalar('loss contract', loss, H.loss_weights('quotient', g, ref.d2_64, sp)[0],
               H.loss_fp32('quotient', g.float(), ref.d2_32, sp))
    chk.table('points after RAdam', x_new, x64, x32, m['rcls'])
    print('\n' + chk.report())
    chk.assert_ok()
