"""GPU tests of GM_PAIRS_SAMPLED (pairs drawn inside the pair kernels): the device draw equals the host statement
oracle/sampler_oracle.py bit for bit -- indices and hop counts -- for the SPD streaming kernel, the generic SPD
kernel and the vector-manifold kernels, at toy size and at BASELINE config 5's full size (2 M nodes, 2^24 pairs); and
PairTrainer.step_sampled / step_sampled_host is the same step as PairTrainer.step on the host-drawn lists."""
import numpy as np
import pytest
import torch

import sampler_oracle as S
from helpers import rel_err

pytestmark = pytest.mark.gpu
DEV = torch.device('cuda', 0)


def _levels(G, N, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(1, 12, (G, N), generator=g, dtype=torch.uint8)


@pytest.mark.parametrize('per_src', [64, 100])  # a power of two (shift) and a general divisor
def test_device_draw_equals_host_statement(per_src):
    """Euclidean points x[v] = (v, v^2) in fp64: d2 identifies (i, j) exactly; the fused loss identifies the hops."""
    from graphembed import _ops, _lib as L
    from graphembed.manifolds import Euclidean, Lorentz, SymmetricPositiveDefinite
    N, G, seed = 5000, 37, 0xDEADBEEF12345
    levels = _levels(G + 5, N, 1)
    rng = np.random.RandomState(3)
    src = rng.choice(N, G, replace=False).astype(np.int32)
    slots = rng.permutation(G + 5)[:G].astype(np.int32)
    I, J, H = S.sample_pairs(src, levels.numpy(), per_src, seed, slots=slots)
    P = G * per_src
    lv, sd, sl = levels.to(DEV), torch.from_numpy(src).to(DEV), torch.from_numpy(slots).to(DEV)
    sampled = _ops.PairSet.sampled(sd, lv, per_src, seed, slots=sl)
    listed = _ops.PairSet.from_lists(torch.from_numpy(I).to(DEV), torch.from_numpy(J).to(DEV), DEV)
    assert sampled.P == P
    v = torch.arange(N, dtype=torch.float64, device=DEV)
    x = torch.stack([v, v * v], dim=1).contiguous()
    man = Euclidean(2)
    d_s = _ops.pairs_dist2(man.spec, x, x, sampled)
    d_l = _ops.pairs_dist2(man.spec, x, x, listed)
    assert torch.equal(d_s, d_l)
    want = (I.astype(np.float64) - J) ** 2 + (I.astype(np.float64) ** 2 - J.astype(np.float64) ** 2) ** 2
    assert np.array_equal(d_s.cpu().numpy(), want)
    # hop counts: fused loss with packed targets, sampled vs explicit (j | hop << 24) list, every kernel family
    packed = torch.from_numpy((J.astype(np.int64) | (H.astype(np.int64) << 24)).astype(np.int32)).to(DEV)
    listed_p = _ops.PairSet.from_lists(torch.from_numpy(I).to(DEV), packed, DEV)
    tg = _ops.TargetSpec.hops_packed(121.0)
    spec = _ops.LossSpec(L.GM_LOSS_QUOTIENT, True, True, alpha=1.0, eps=0.5)
    torch.manual_seed(0)
    hint32 = torch.empty(0, device=DEV, dtype=torch.float32)
    for man, xs in ((SymmetricPositiveDefinite(4), None), (SymmetricPositiveDefinite(3), None), (Lorentz(6), None)):
        xs = man.rand(N, out=hint32, ir=0.5).contiguous()
        outs = []
        for pairs in (sampled, listed_p):
            grad = torch.zeros_like(xs)
            acc, d2 = _ops.pairs_loss_fused(man.spec, xs, pairs, tg, spec, 0.9, grad, want_d2=True)
            outs.append((acc.clone(), d2, grad))
        assert torch.equal(outs[0][1], outs[1][1]), type(man).__name__
        assert rel_err(outs[0][0], outs[1][0]) < 1e-12
        assert rel_err(outs[0][2], outs[1][2]) < 1e-5  # float atomics: same terms, different arrival order


def test_validation_of_sampled_pairs():
    from graphembed import _ops, _lib as L
    from graphembed.manifolds import SymmetricPositiveDefinite
    lv = _levels(4, 100, 0).to(DEV)
    src = torch.arange(4, dtype=torch.int32, device=DEV)
    pairs = _ops.PairSet.sampled(src, lv, 8, 1)
    man = SymmetricPositiveDefinite(2)
    x = man.rand(100, out=torch.empty(0, device=DEV, dtype=torch.float32)).contiguous()
    spec = _ops.LossSpec(L.GM_LOSS_STRESS)
    with pytest.raises(RuntimeError):  # drawn pairs bring their own hop counts: only packed targets
        _ops.pairs_loss_fused(man.spec, x, pairs, _ops.TargetSpec.vector(torch.ones(32, device=DEV)), spec, 1.0,
                              torch.zeros_like(x))
    with pytest.raises(ValueError):
        _ops.PairSet.sampled(src.long(), lv, 8, 1)
    with pytest.raises(ValueError):  # source 4 would read row 4 of a 4-row level matrix
        _ops.PairSet.sampled(torch.arange(5, dtype=torch.int32, device=DEV), lv, 8, 1)
    _ops.PairSet.sampled(torch.arange(5, dtype=torch.int32, device=DEV), lv, 8, 1,
                         slots=torch.zeros(5, dtype=torch.int32, device=DEV))


def test_step_sampled_is_the_step_on_the_host_drawn_lists():
    from graphembed.engine import PairTrainer, pack_hops
    from graphembed.manifolds import SymmetricPositiveDefinite
    from graphembed.modules import ManifoldEmbedding
    from graphembed.objectives import QuotientLoss
    from graphembed.optim import RiemannianAdam
    N, G, per = 3000, 50, 256
    levels = _levels(G, N, 5)
    lv = levels.to(DEV)
    res = []
    for mode in ('sampled_host', 'lists'):
        torch.manual_seed(1)
        emb = ManifoldEmbedding(N, [SymmetricPositiveDefinite(4)], device=DEV, dtype=torch.float32)
        opt = RiemannianAdam(emb.xs, lr=0.01, max_grad_norm=100, exact=True)
        tr = PairTrainer(emb, opt, QuotientLoss(), max_hops_sq=121.0)
        losses = []
        for step in range(3):
            src = np.random.RandomState(step).choice(N, G, replace=False).astype(np.int32)
            seed = 77 + (step << 32)
            if mode == 'sampled_host':
                losses.append(tr.step_sampled_host(torch.from_numpy(src).pin_memory(), lv, per, seed, epoch=1))
            else:
                I, J, H = S.sample_pairs(src, levels.numpy(), per, seed)
                jp = pack_hops(torch.from_numpy(J), torch.from_numpy(H))
                losses.append(tr.step(torch.from_numpy(I).to(DEV), jp.to(DEV), None, epoch=1).item())
        res.append((losses, emb.xs[0].detach().cpu()))
    assert max(abs(a - b) / abs(b) for a, b in zip(*[r[0] for r in res])) < 1e-6
    assert rel_err(res[0][1], res[1][1]) < 1e-5


def test_full_size_draw_config5():
    """2 M nodes, 1024 sources x 16384 targets = 2^24 pairs: the streaming kernel's draw against the host statement
    (d2 bitwise equal to the LIST launch on the host-drawn pairs), loss equal, finite gradient."""
    from graphembed import _ops, _lib as L
    from graphembed.manifolds import SymmetricPositiveDefinite
    N, G, per, seed = 2_000_000, 1024, 16384, 0x1234ABCD5678
    g = torch.Generator().manual_seed(9)
    levels = torch.randint(1, 20, (64, N), generator=g, dtype=torch.uint8)  # 64 resident rows, shared through slots
    slots = torch.randint(64, (G,), generator=g, dtype=torch.int32)
    src = torch.randperm(N, generator=g)[:G].int()
    I, J, H = S.sample_pairs(src.numpy(), levels.numpy(), per, seed, slots=slots.numpy())
    man = SymmetricPositiveDefinite(4)
    torch.manual_seed(0)
    x = man.rand(N, out=torch.empty(0, device=DEV, dtype=torch.float32)).contiguous()
    lv = levels.to(DEV)
    sampled = _ops.PairSet.sampled(src.to(DEV), lv, per, seed, slots=slots.to(DEV))
    packed = torch.from_numpy((J.astype(np.int64) | (H.astype(np.int64) << 24)).astype(np.int32)).to(DEV)
    listed = _ops.PairSet.from_lists(torch.from_numpy(I).to(DEV), packed, DEV)
    tg = _ops.TargetSpec.hops_packed(361.0)
    spec = _ops.LossSpec(L.GM_LOSS_QUOTIENT, True, True, alpha=1.0, eps=0.5)
    outs = []
    for pairs in (sampled, listed):
        grad = torch.zeros_like(x)
        acc, d2 = _ops.pairs_loss_fused(man.spec, x, pairs, tg, spec, 0.97, grad, want_d2=True)
        outs.append((acc.clone(), d2, grad))
    assert torch.equal(outs[0][1], outs[1][1])
    assert rel_err(outs[0][0], outs[1][0]) < 1e-12
    assert rel_err(outs[0][2], outs[1][2]) < 1e-5 and torch.isfinite(outs[0][2]).all()


def test_registered_custom_ops_match_the_python_api():
    """torch.ops.graphembed_b200.* (the torch custom-op layer over the C-ABI) against the manifold API / _ops."""
    from graphembed import _ops, _torch_ops, _lib as L
    from graphembed.data import bfs_levels, edges_to_csr
    from graphembed.manifolds import SymmetricPositiveDefinite
    ns = torch.ops.graphembed_b200
    man = SymmetricPositiveDefinite(4)
    torch.manual_seed(0)
    x = man.rand(500, out=torch.empty(0, device=DEV, dtype=torch.float32), ir=0.7).contiguous()
    g = torch.Generator().manual_seed(0)
    I = torch.randint(500, (4000,), generator=g, dtype=torch.int32).to(DEV)
    J = ((I.cpu() + 1 + torch.randint(499, (4000,), generator=g, dtype=torch.int32)) % 500).to(DEV)
    H = torch.randint(1, 9, (4000,), generator=g, dtype=torch.uint8).to(DEV)
    margs = _torch_ops.manifold_args(man.spec)
    assert torch.equal(ns.pair_dist2(x, I, J, *margs), man.pair_dist2(x, I, J))
    grad_a, acc_a = torch.zeros_like(x), torch.zeros(2, dtype=torch.float64, device=DEV)
    ns.pairs_loss_fused(x, I, J, H, *margs, L.GM_LOSS_QUOTIENT, True, True, 1.0, 0.5, 64.0, 0.9, grad_a, acc_a)
    grad_b = torch.zeros_like(x)
    acc_b, _ = _ops.pairs_loss_fused(man.spec, x, _ops.PairSet.from_lists(I, J, DEV), _ops.TargetSpec.hops(H, 64.0),
                                     _ops.LossSpec(L.GM_LOSS_QUOTIENT, True, True, alpha=1.0, eps=0.5), 0.9, grad_b)
    assert rel_err(acc_a, acc_b) < 1e-12 and rel_err(grad_a, grad_b) < 1e-5
    rowptr, colidx = edges_to_csr(50, np.stack([np.arange(1, 50), np.arange(49) // 2], 1))
    rp, ci = torch.as_tensor(rowptr, device=DEV), torch.as_tensor(colidx, device=DEV)
    src = torch.arange(7, dtype=torch.int32, device=DEV)
    assert torch.equal(ns.bfs_levels(rp, ci, src), bfs_levels(rp, ci, sources=src, device=DEV))
    with pytest.raises(NotImplementedError):  # no CPU kernel behind the ops
        ns.pair_dist2(x.cpu(), I.cpu(), J.cpu(), *margs)


@pytest.mark.parametrize('fused', [True, False])
@pytest.mark.parametrize('dtype', [torch.float64, torch.float32])
def test_product_pair_trainer_vs_oracle(dtype, fused):
    """BASELINE config 3's "product SPD 3x3 x Lorentz 5, sampled pairs": three steps of ProductPairTrainer (points by
    RiemannianAdam, the two scales by a second RiemannianAdam as run_grid.py:25-28 groups them) against the oracle's
    autograd + optimizer restatement on the same explicit pair lists."""
    import manifolds_oracle as O
    from graphembed.engine import ProductPairTrainer
    from graphembed.manifolds import Lorentz, SymmetricPositiveDefinite
    from graphembed.modules import ManifoldEmbedding
    from graphembed.objectives import QuotientLoss
    from graphembed.optim import RiemannianAdam
    N, P = 400, 6000
    torch.manual_seed(3)
    emb = ManifoldEmbedding(N, [SymmetricPositiveDefinite(3), Lorentz(5)], device=DEV, dtype=dtype)
    with torch.no_grad():  # spread the default init (points within 1e-2 of each other are fp32-cancellation limited)
        emb.xs[0].copy_(emb.manifolds[0].rand(N, out=torch.empty(0, device=DEV, dtype=dtype), ir=0.8))
        emb.xs[1].copy_(emb.manifolds[1].rand(N, out=torch.empty(0, device=DEV, dtype=dtype), ir=0.8))
    x0 = [x.detach().cpu().clone() for x in emb.xs]
    opt = RiemannianAdam(emb.xs, lr=0.01, max_grad_norm=100, exact=True)
    sopt = RiemannianAdam(list(emb.scales), lr=0.01)
    tr = ProductPairTrainer(emb, opt, QuotientLoss(), max_hops_sq=64.0, scale_optimizer=sopt, fused=fused)
    assert tr.fused == fused  # SPD x Lorentz is a product the one-launch kernel takes
    g = torch.Generator().manual_seed(1)
    oracles = [O.SpdOracle(3), O.LorentzOracle(5)]
    xs = [t.clone() for t in x0]
    scales = [torch.tensor(0.5, dtype=dtype) for _ in range(2)]
    states, sstates = [{}, {}], [{}, {}]
    eu = O.EuclideanOracle(1)
    for step in range(3):
        I = torch.randint(N, (P,), generator=g, dtype=torch.int32)
        J = ((I + 1 + torch.randint(N - 1, (P,), generator=g, dtype=torch.int32)) % N).int()
        H = torch.randint(1, 9, (P,), generator=g, dtype=torch.uint8)
        loss = tr.step(I.to(DEV), J.to(DEV), H.to(DEV), epoch=step + 1).item()
        leaves = [x.clone().requires_grad_() for x in xs]
        sl = [s.clone().requires_grad_() for s in scales]
        m = O.product_dist2(oracles, leaves, sl, lambda o, x: o.dist2(x[I.long()], x[J.long()]))
        lo = O.quotient_loss(H.to(dtype).pow(2) / 64.0, m, 1.0, step + 1)
        lo.backward()
        t = 1e-10 if dtype == torch.float64 else 2e-5
        assert abs(loss - lo.item()) <= t * abs(lo.item()), (step, loss, lo.item())
        xs = [O.radam_step(o, x, leaf.grad, st, lr=0.01, max_grad_norm=100, exact=True).detach()
              for o, x, leaf, st in zip(oracles, xs, leaves, states)]
        scales = [O.radam_step(eu, s.reshape(1), sg.grad.reshape(1), st, lr=0.01).reshape(()).detach()
                  for s, sg, st in zip(scales, sl, sstates)]
    t = 1e-10 if dtype == torch.float64 else 2e-5
    for f in range(2):
        assert rel_err(emb.xs[f].detach(), xs[f]) < t
        assert abs(float(emb.scales[f].detach()) - float(scales[f])) <= t * abs(float(scales[f]))
    assert abs(float(emb.scales[0].detach()) - 0.5) > 1e-3  # the scales moved, and the kernels followed them


PRODUCTS = {
    'spd3xlorentz5': [('spd', 3, False), ('lorentz', 5)],
    'lorentz4xspd4stein': [('lorentz', 4), ('spd', 4, True)],
    'lorentz3xlorentz6': [('lorentz', 3), ('lorentz', 6)],
    'sphere4xspd2xeuclidean3xlorentz8': [('sphere', 4), ('spd', 2, False), ('euclidean', 3), ('lorentz', 8)],
    'euclidean5xsphere3xlorentz4': [('euclidean', 5), ('sphere', 3), ('lorentz', 4)],
}


def _make_factor(desc):
    from graphembed import manifolds as M
    if desc[0] == 'spd':
        return M.SymmetricPositiveDefinite(desc[1], use_stein_div=desc[2])
    return {'lorentz': M.Lorentz, 'sphere': M.Sphere, 'euclidean': M.Euclidean}[desc[0]](desc[1])


@pytest.mark.parametrize('mode', ['list_hops', 'triu_dense'])
@pytest.mark.parametrize('dtype', [torch.float64, torch.float32])
@pytest.mark.parametrize('name', sorted(PRODUCTS))
def test_fused_product_kernel_vs_unfused_sequence(name, dtype, mode):
    """gm_pairs_product_fused (one launch) against gm_pairs_dist2 x F -> gm_product_loss -> gm_pairs_grad x F (which the
    oracle tests pin): loss and per-factor scale sums to rounding, every factor's gradient table to the dtype's
    tolerance; factor order (the left-to-right sum of modules.py:84-88) with the SPD factor in any slot."""
    from graphembed import _lib as L, _ops
    mans = [_make_factor(d) for d in PRODUCTS[name]]
    N = 300
    torch.manual_seed(11)
    xs = [m.rand(N, out=torch.empty(0, device=DEV, dtype=dtype), ir=0.7).contiguous() for m in mans]
    sps = [0.6 + 0.25 * f for f in range(len(mans))]
    g = torch.Generator().manual_seed(2)
    if mode == 'list_hops':
        P = 5000 + 77
        I = torch.randint(N, (P,), generator=g, dtype=torch.int32).sort().values
        J = ((I + 1 + torch.randint(N - 1, (P,), generator=g, dtype=torch.int32)) % N).int()
        H = torch.randint(1, 9, (P,), generator=g, dtype=torch.uint8)
        pairs = _ops.PairSet.from_lists(I.to(DEV), J.to(DEV), DEV)
        targets = _ops.TargetSpec.hops(H.to(DEV), 64.0)
    else:
        B = 97
        nodes = torch.randperm(N, generator=g)[:B].to(DEV)
        dense = (torch.rand(N, N, generator=g, dtype=torch.float64) + 0.05).to(dtype).to(DEV)
        dense = (dense + dense.T).contiguous()
        pairs = _ops.PairSet.triu(B, nodes=nodes)
        targets = _ops.TargetSpec.dense(dense)
    for kind in (L.GM_LOSS_QUOTIENT, L.GM_LOSS_STRESS):
        spec = _ops.LossSpec(kind, True, True, alpha=0.7, eps=0.5)
        d2s = [_ops.pairs_dist2(m.spec, x, x, pairs) for m, x in zip(mans, xs)]
        acc_u, gw = _ops.product_loss(d2s, sps, targets, spec, pairs=pairs if mode == 'triu_dense' else None)
        grads_u = [torch.zeros_like(x) for x in xs]
        for m, x, gx, sp in zip(mans, xs, grads_u, sps):
            _ops.pairs_grad(m.spec, x, x, pairs, gw, gx, gx, coef=sp)
        grads_f = [torch.zeros_like(x) for x in xs]
        acc_f = _ops.pairs_product_fused([m.spec for m in mans], xs, pairs, targets, spec, sps, grads_f)
        t, ta = (1e-11, 1e-12) if dtype == torch.float64 else (2e-5, 1e-6)
        assert rel_err(acc_f, acc_u) < ta, (acc_f, acc_u)
        for gf, gu in zip(grads_f, grads_u):
            assert torch.isfinite(gf).all() and rel_err(gf, gu) < t, rel_err(gf, gu)


def test_fused_product_kernel_declines_other_products():
    from graphembed import _lib as L, _ops
    from graphembed import manifolds as M
    for mans in ([M.SymmetricPositiveDefinite(2), M.SymmetricPositiveDefinite(3)], [M.Grassmann(5, 2), M.Lorentz(4)],
                 [M.Lorentz(3)] * 5):
        assert not _ops.product_fusable([m.spec for m in mans], [torch.float32] * len(mans))
        xs = [m.rand(20, out=torch.empty(0, device=DEV, dtype=torch.float32)).contiguous() for m in mans]
        I = torch.arange(10, dtype=torch.int32, device=DEV)
        pairs = _ops.PairSet.from_lists(I, I + 10, DEV)
        targets = _ops.TargetSpec.hops(torch.ones(10, dtype=torch.uint8, device=DEV), 64.0)
        spec = _ops.LossSpec(L.GM_LOSS_QUOTIENT, True, True, alpha=1.0, eps=0.5)
        with pytest.raises(RuntimeError, match='GM_EUNSUPPORTED'):
            _ops.pairs_product_fused([m.spec for m in mans], xs, pairs, targets, spec, [1.0] * len(mans),
                                     [torch.zeros_like(x) for x in xs])
    assert _ops.product_fusable([M.SymmetricPositiveDefinite(3).spec, M.Lorentz(5).spec], [torch.float32] * 2)
    assert not _ops.product_fusable([M.SymmetricPositiveDefinite(3).spec, M.Lorentz(5).spec],
                                    [torch.float32, torch.float64])


def test_three_byte_pair_upload_format():
    """pack_hops3 (j | (hops - 1) << 21 in 3 bytes) expands on the device to exactly pack_hops' 4-byte words, for any
    length (the 4-pair vector path and the ragged tail), and step_host_grouped on it is the same step."""
    from graphembed import _ops
    from graphembed.engine import PairTrainer, pack_hops, pack_hops3
    from graphembed.manifolds import SymmetricPositiveDefinite
    from graphembed.modules import ManifoldEmbedding
    from graphembed.objectives import QuotientLoss
    from graphembed.optim import RiemannianAdam
    g = torch.Generator().manual_seed(0)
    for P in (1, 3, 4, 5, 1023, 40000):
        J = torch.randint(1 << 21, (P,), generator=g, dtype=torch.int32)
        H = torch.randint(1, 9, (P,), generator=g, dtype=torch.uint8)
        b3 = pack_hops3(J, H)
        assert b3.dtype == torch.uint8 and b3.numel() == (3 * P + 3) // 4 * 4
        out = torch.empty(P, dtype=torch.int32, device=DEV)
        _ops.unpack_pairs3(b3.to(DEV), P, out)
        assert torch.equal(out.cpu(), pack_hops(J, H))
    with pytest.raises(ValueError):
        pack_hops3(torch.tensor([1 << 21], dtype=torch.int32), torch.tensor([1], dtype=torch.uint8))
    with pytest.raises(ValueError):
        pack_hops3(torch.tensor([5], dtype=torch.int32), torch.tensor([9], dtype=torch.uint8))
    n, G, per = 300, 37, 129
    res = []
    for three in (False, True):
        torch.manual_seed(3)
        emb = ManifoldEmbedding(n, [SymmetricPositiveDefinite(4)], device=DEV, dtype=torch.float32)
        opt = RiemannianAdam(emb.xs, lr=0.01, max_grad_norm=100, exact=True)
        tr = PairTrainer(emb, opt, QuotientLoss(), max_hops_sq=64.0)
        gg = torch.Generator().manual_seed(5)
        losses = []
        for step in range(3):
            src = torch.randperm(n, generator=gg)[:G].int()
            offsets = torch.arange(G + 1, dtype=torch.int64) * per
            I = src.repeat_interleave(per)
            J = torch.randint(n - 1, (G * per,), generator=gg, dtype=torch.int32)
            J = torch.where(J >= I, J + 1, J).contiguous()
            H = torch.randint(1, 9, (G * per,), generator=gg, dtype=torch.uint8)
            words = (pack_hops3 if three else pack_hops)(J, H)
            losses.append(tr.step_host_grouped(src.pin_memory(), offsets.pin_memory(), words.pin_memory(), None, epoch=1))
        res.append((losses, emb.xs[0].detach().cpu().clone()))
    assert max(abs(a - b) / abs(b) for a, b in zip(res[0][0], res[1][0])) < 1e-6
    assert rel_err(res[0][1], res[1][1]) < 1e-5
