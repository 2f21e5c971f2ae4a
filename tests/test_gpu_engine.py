"""GPU parity of the rows added around the pair kernels (SURVEY 8a A1, 8f-1, 8f-2, 8f-4): the TrainingEngine epoch
loop with streamed validation metrics, the KL/SNE objective, sub-ranges of the pair triangle (pair-sharded ranks),
the packed (j | hops << 24) pair format and the on-disk files -- against golden vectors produced by the real
reference (tests/golden/engine_runs_f64.npz, objectives_*.npz) and against the oracle."""
import os

import numpy as np
import pytest
import torch

import manifolds_oracle as O
from helpers import load_golden, rel_err
from helpers_engine import ENGINE_SEED, N_EPOCHS, RUNS, load_engine_golden

pytestmark = pytest.mark.gpu
DEV = torch.device('cuda', 0)


def _manifold(fam, n):
    from graphembed.manifolds import Lorentz, SymmetricPositiveDefinite
    return SymmetricPositiveDefinite(n) if fam == 'spd' else Lorentz(n)


def _targets_from_bfs(g, n):
    from graphembed.data import bfs_levels, edges_to_csr
    from graphembed.data.graph import levels_to_condensed
    rowptr, colidx = edges_to_csr(n, g['edges'].numpy())
    cond = levels_to_condensed(bfs_levels(rowptr, colidx), torch.float64)
    assert torch.equal(cond.cpu(), g['hops_condensed'])  # BFS targets bit-exact
    return cond


@pytest.mark.parametrize('tag', sorted(RUNS))
def test_training_engine_vs_reference_engine(tag, tmp_path):
    """3 epochs of graphembed.train.TrainingEngine (validation every epoch) against the reference's own engine:
    same randperm batches (CPU generator, same seed), step losses, pearsonr / average_distortion per epoch, final
    points, best-loss bookkeeping and the files written."""
    from graphembed.data import GraphDataset
    from graphembed.modules import ManifoldEmbedding
    from graphembed.objectives import KLDiveregenceLoss, QuotientLoss
    from graphembed.optim import RiemannianAdam, RiemannianSGD
    from graphembed.train import TrainingEngine
    g = load_engine_golden()
    n = 63
    factors, objective, (oname, okw), ekw = RUNS[tag]
    ds = GraphDataset(_targets_from_bfs(g, n))
    emb = ManifoldEmbedding(n, [_manifold(f, k) for f, k in factors], device=DEV, dtype=torch.float64)
    with torch.no_grad():
        for i, x in enumerate(emb.xs):
            x.copy_(g[f'{tag}_x0_{i}'].to(DEV))
    opt = (RiemannianSGD if oname == 'rsgd' else RiemannianAdam)(emb.xs, **okw)
    obj = QuotientLoss() if objective == 'quotient' else KLDiveregenceLoss('sne', inclusive=True)
    eng = TrainingEngine(embedding=emb, optimizer=opt, objective_fn=obj, n_epochs=N_EPOCHS, val_every_epochs=1,
                         save_dir=str(tmp_path), tensorboard=False, **ekw)
    torch.manual_seed(ENGINE_SEED)
    eng(ds)
    hist = eng.writer.history
    got = np.array([v for _, v in hist[str(obj)]])
    assert np.allclose(got, g[f'{tag}_step_loss'].numpy(), rtol=1e-9), (got, g[f'{tag}_step_loss'])
    for m in ('pearsonr', 'average_distortion'):
        got = np.array([v for _, v in hist[m]])
        assert np.allclose(got, g[f'{tag}_{m}'].numpy(), rtol=1e-8), (m, got, g[f'{tag}_{m}'])
    for i, x in enumerate(emb.xs):
        assert rel_err(x.data, g[f'{tag}_xT_{i}']) < 1e-9
    assert sorted(os.listdir(tmp_path)) == list(g[f'{tag}_files'])
    best_epoch, best_loss = int(g[f'{tag}_best'][0]), float(g[f'{tag}_best'][1])
    assert abs(float(open(tmp_path / f'best_loss_{best_epoch}').read()) - best_loss) < 2e-6 * max(1.0, best_loss)
    sd = torch.load(tmp_path / 'best_embedding.pth')
    assert sorted(sd.keys()) == list(g[f'{tag}_state_keys'])
    # resume from the snapshot directory (train.py:349-352)
    emb2 = ManifoldEmbedding(n, [_manifold(f, k) for f, k in factors], device=DEV, dtype=torch.float64)
    TrainingEngine(embedding=emb2, optimizer=opt, objective_fn=obj, snapshot_path=str(tmp_path), save_dir=str(tmp_path))
    assert torch.equal(emb2.xs[0].data, emb.xs[0].data)


@pytest.mark.parametrize('tag', ['f64', 'f32'])
def test_kl_sne_and_vector_metrics_vs_golden(tag):
    from graphembed import metrics
    from graphembed.objectives import KLDiveregenceLoss
    g = load_golden('objectives', tag)
    t = 1e-10 if tag == 'f64' else 1e-5
    for inc in (1, 0):
        m = g['m'].to(DEV).requires_grad_()
        loss = KLDiveregenceLoss('sne', inclusive=bool(inc))(g['g'].to(DEV), m, alpha=float(g['alpha']))
        (2.0 * loss).backward()
        ref = g[f'kl_{inc}_loss'].item()
        assert abs(loss.item() - ref) <= t * abs(ref)
        assert rel_err(m.grad / 2.0, g[f'kl_{inc}_grad']) < t
    assert abs(metrics.pearsonr(g['m'].to(DEV), g['g'].to(DEV)).item() - g['pearsonr'].item()) < t
    assert abs(metrics.average_distortion(g['m'].to(DEV), g['g'].to(DEV)).item() - g['average_distortion'].item()) < t
    with pytest.raises(ValueError):
        KLDiveregenceLoss('nope')


@pytest.mark.parametrize('dtype', [torch.float64, torch.float32])
def test_kl_sne_larger_batch_vs_oracle(dtype):
    """B = 300 nodes (44 850 pairs): strided and contiguous halves of every row, product of two factors via autograd."""
    from graphembed.objectives import KLDiveregenceLoss
    gen = torch.Generator().manual_seed(3)
    B = 300
    P = B * (B - 1) // 2
    g = (torch.rand(P, generator=gen, dtype=torch.float64) * 0.9 + 0.05).to(dtype)
    m0 = (torch.rand(P, generator=gen, dtype=torch.float64) * 3.0 + 0.01).to(dtype)
    for inc in (True, False):
        mo = m0.clone().requires_grad_()
        lo = O.kl_sne_loss(g, mo, 7.0, inclusive=inc)
        lo.backward()
        m = m0.to(DEV).requires_grad_()
        l = KLDiveregenceLoss('sne', inclusive=inc)(g.to(DEV), m, alpha=7.0)
        l.backward()
        t = 1e-10 if dtype == torch.float64 else 2e-5
        assert abs(l.item() - lo.item()) <= t * abs(lo.item())
        assert rel_err(m.grad, mo.grad) < (1e-10 if dtype == torch.float64 else 1e-4)


@pytest.mark.parametrize('name', ['spd4', 'spd6', 'lorentz11', 'grassmann6_2'])
def test_triangle_slices_equal_whole(name):
    """Pairs [k0, k0+P) of the triangle (what one rank of a pair-sharded job evaluates): distances of the slices
    concatenate to the full pdist, fused losses / gradients of the slices add up to the full batch."""
    from graphembed import _ops
    from helpers import make_product
    man = make_product(name)
    torch.manual_seed(5)
    for dtype in (torch.float64, torch.float32):
        n, B = 70, 41
        hint = torch.empty(0, device=DEV, dtype=dtype)
        x = (man.rand(n, out=hint, ir=1.0) if hasattr(man, 'rand') and 'grassmann' not in name
             else man.rand_uniform(n, out=hint)).contiguous()
        nodes = torch.randperm(n)[:B].to(DEV)
        full = _ops.PairSet.triu(B, nodes, DEV)
        d_full = _ops.pairs_dist2(man.spec, x, x, full)
        tg = torch.rand(full.P, device=DEV, dtype=dtype) + 0.2
        spec = _ops.LossSpec(0, True, True, alpha=1.3, eps=0.25)
        g_full = torch.zeros_like(x)
        acc_full, _ = _ops.pairs_loss_fused(man.spec, x, full, _ops.TargetSpec.vector(tg), spec, 0.9, g_full)
        parts, g_sum, acc_sum = [], torch.zeros_like(x), torch.zeros(2, dtype=torch.float64, device=DEV)
        for r in range(3):
            sl = full.slice(r, 3)
            lo = sl.k0
            parts.append(_ops.pairs_dist2(man.spec, x, x, sl))
            _ops.pairs_loss_fused(man.spec, x, sl, _ops.TargetSpec.vector(tg[lo:lo + sl.P].contiguous()), spec, 0.9,
                                  g_sum, acc_sum)
        assert torch.equal(torch.cat(parts), d_full)
        t = 1e-11 if dtype == torch.float64 else 2e-5
        assert rel_err(acc_sum, acc_full) < t
        assert rel_err(g_sum, g_full) < (t if dtype == torch.float64 else 2e-4)


def test_streamed_validation_moments_chunking_and_oracle():
    """validation_moments in chunks of 1000 pairs == one chunk == the oracle's materialised metrics (fp32 and fp64),
    for a product embedding."""
    from graphembed import metrics
    from graphembed.data import GraphDataset
    from graphembed.manifolds import Lorentz, SymmetricPositiveDefinite
    from graphembed.modules import ManifoldEmbedding
    n = 90
    gen = torch.Generator().manual_seed(0)
    hops = torch.randint(1, 12, (n * (n - 1) // 2,), generator=gen).double()
    for dtype in (torch.float64, torch.float32):
        torch.manual_seed(1)
        emb = ManifoldEmbedding(n, [SymmetricPositiveDefinite(4), Lorentz(6)], device=DEV, dtype=dtype)
        ds = GraphDataset(hops.to(device=DEV, dtype=dtype))
        a1 = metrics.validation_moments(emb, ds, chunk_pairs=1000)
        a2 = metrics.validation_moments(emb, ds)
        assert a1[0].item() == n * (n - 1) // 2 and rel_err(a1, a2) < 1e-12
        half = metrics.validation_moments(emb, ds, pair_range=(0, 2000)) + \
            metrics.validation_moments(emb, ds, chunk_pairs=777, pair_range=(2000, n * (n - 1) // 2))
        assert rel_err(half, a2) < 1e-12
        mom = metrics.PairMoments(a1.cpu())
        ref = O.validation_metrics([O.SpdOracle(4), O.LorentzOracle(6)], [x.detach().cpu() for x in emb.xs],
                                   [s.detach().cpu() for s in emb.scales], O.dataset_targets(hops, dtype))
        t = 1e-10 if dtype == torch.float64 else 2e-4
        assert abs(mom.pearsonr - ref['pearsonr']) < t and abs(mom.average_distortion - ref['average_distortion']) < t


def test_packed_hop_format_matches_separate_vectors():
    """(j | hops << 24) pairs give bit-identical loss and gradient to separate int32 j + uint8 hops, through the
    streaming kernel (SPD4 fp32) and the generic one (SPD6, Lorentz), and through the grouped host upload."""
    from graphembed import _ops
    from graphembed.engine import PairTrainer, pack_hops
    from graphembed.manifolds import Lorentz, SymmetricPositiveDefinite
    from graphembed.modules import ManifoldEmbedding
    from graphembed.objectives import QuotientLoss
    from graphembed.optim import RiemannianAdam
    gen = torch.Generator().manual_seed(9)
    n, G, per = 5000, 37, 211
    P = G * per
    src = torch.randperm(n, generator=gen)[:G].int()
    I = src.repeat_interleave(per).contiguous()
    J = torch.randint(n, (P,), generator=gen, dtype=torch.int32)
    hops = torch.randint(1, 30, (P,), generator=gen, dtype=torch.uint8)
    Jp = pack_hops(J, hops)
    assert torch.equal(Jp & 0xFFFFFF, J) and torch.equal((Jp >> 24).to(torch.uint8), hops)
    spec = _ops.LossSpec(0, True, True, alpha=1.0, eps=0.5)
    for man in (SymmetricPositiveDefinite(4), SymmetricPositiveDefinite(6), Lorentz(7)):
        torch.manual_seed(2)
        x = man.rand(n, out=torch.empty(0, device=DEV, dtype=torch.float32), ir=1.0).contiguous()
        ga, gb = torch.zeros_like(x), torch.zeros_like(x)
        acc_a, _ = _ops.pairs_loss_fused(man.spec, x, _ops.PairSet.from_lists(I, J, DEV),
                                         _ops.TargetSpec.hops(hops.to(DEV), 900.0), spec, 0.97, ga)
        acc_b, _ = _ops.pairs_loss_fused(man.spec, x, _ops.PairSet.from_lists(I, Jp, DEV),
                                         _ops.TargetSpec.hops_packed(900.0), spec, 0.97, gb)
        assert rel_err(acc_b, acc_a) < 1e-12
        assert rel_err(gb, ga) < 1e-5  # atomics: summation order differs run to run
    # grouped host upload, packed vs unpacked
    offsets = (torch.arange(G + 1, dtype=torch.int64) * per)
    outs = []
    for packed in (False, True):
        torch.manual_seed(4)
        emb = ManifoldEmbedding(n, [SymmetricPositiveDefinite(4)], device=DEV, dtype=torch.float32)
        tr = PairTrainer(emb, RiemannianAdam(emb.xs, lr=0.01, max_grad_norm=100, exact=True), QuotientLoss(),
                         max_hops_sq=900.0)
        args = (src.pin_memory(), offsets.pin_memory(), (Jp if packed else J).pin_memory(),
                None if packed else hops.pin_memory())
        loss = tr.step_host_grouped(*args, epoch=1)
        outs.append((loss, emb.xs[0].detach().clone()))
    assert abs(outs[0][0] - outs[1][0]) <= 1e-6 * abs(outs[0][0])
    assert rel_err(outs[1][1], outs[0][1]) < 1e-5
    with pytest.raises(ValueError):
        pack_hops(torch.tensor([1 << 24], dtype=torch.int32), torch.tensor([1], dtype=torch.uint8))


def _two_gpu_engine_worker(rank, world, port, q):
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, os.path.join(root, 'matrix-manifolds_b200'))
    sys.path.insert(0, os.path.join(root, 'tests'))
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    import torch.distributed as dist
    dev = torch.device('cuda', rank)
    torch.cuda.set_device(dev)
    dist.init_process_group('nccl', rank=rank, world_size=world, device_id=dev)
    from graphembed.data import GraphDataset
    from graphembed.manifolds import SymmetricPositiveDefinite
    from graphembed.modules import ManifoldEmbedding
    from graphembed.objectives import QuotientLoss
    from graphembed.optim import RiemannianSGD
    from graphembed.train import TrainingEngine
    from helpers_engine import load_engine_golden
    import tempfile
    g = load_engine_golden()
    emb = ManifoldEmbedding(63, [SymmetricPositiveDefinite(3)], device=dev, dtype=torch.float64)
    with torch.no_grad():
        emb.xs[0].copy_(g['spd3_batched_x0_0'].to(dev))
    opt = RiemannianSGD(emb.xs, lr=0.01, max_grad_norm=20, exact=True)
    eng = TrainingEngine(embedding=emb, optimizer=opt, objective_fn=QuotientLoss(), n_epochs=3, val_every_epochs=1,
                         alpha=1.0, batch_size=52, save_dir=tempfile.mkdtemp(), tensorboard=False,
                         process_group=dist.group.WORLD)
    torch.manual_seed(1234)
    eng(GraphDataset(g['hops_condensed'].to(dev)))
    if rank == 0:
        h = eng.writer.history
        q.put(([v for _, v in h['quotient_loss']], [v for _, v in h['average_distortion']],
               emb.xs[0].detach().cpu().numpy()))
    dist.barrier()
    dist.destroy_process_group()


def test_two_gpu_sharded_engine_matches_reference_engine():
    """TrainingEngine with a process group (pairs of every batch split over 2 ranks, all-reduce of gradient and
    loss, validation moments summed over ranks) reproduces the single-process reference run."""
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    import torch.multiprocessing as mp
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 33500 + os.getpid() % 2000
    procs = [ctx.Process(target=_two_gpu_engine_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    losses, dist_metric, xT = q.get(timeout=300)
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    g = load_engine_golden()
    assert np.allclose(losses, g['spd3_batched_step_loss'].numpy(), rtol=1e-9)
    assert np.allclose(dist_metric, g['spd3_batched_average_distortion'].numpy(), rtol=1e-8)
    assert rel_err(torch.from_numpy(xT), g['spd3_batched_xT_0']) < 1e-9


def test_deferred_loss_readback_matches_blocking_steps():
    """defer_loss=True (loss copied to pinned memory asynchronously, returned one step late) gives the same loss
    sequence and the same trajectory as the blocking step_host_grouped."""
    from graphembed.engine import PairTrainer, pack_hops
    from graphembed.manifolds import SymmetricPositiveDefinite
    from graphembed.modules import ManifoldEmbedding
    from graphembed.objectives import QuotientLoss
    from graphembed.optim import RiemannianAdam
    gen = torch.Generator().manual_seed(21)
    n, G, per = 3000, 16, 128
    batches = []
    for _ in range(3):
        src = torch.randperm(n, generator=gen)[:G].int().pin_memory()
        J = torch.randint(n, (G * per,), generator=gen, dtype=torch.int32)
        hops = torch.randint(1, 9, (G * per,), generator=gen, dtype=torch.uint8)
        offs = (torch.arange(G + 1, dtype=torch.int64) * per).pin_memory()
        batches.append((src, offs, pack_hops(J, hops).pin_memory(), None))
    runs = []
    for defer in (False, True):
        torch.manual_seed(8)
        emb = ManifoldEmbedding(n, [SymmetricPositiveDefinite(4)], device=DEV, dtype=torch.float32)
        tr = PairTrainer(emb, RiemannianAdam(emb.xs, lr=0.01, max_grad_norm=100, exact=True), QuotientLoss(),
                         max_hops_sq=64.0)
        losses = []
        for k in range(5):
            losses.append(tr.step_host_grouped(*batches[k % 3], epoch=1, next_batch=batches[(k + 1) % 3],
                                               defer_loss=defer))
        if defer:
            assert losses[0] is None
            losses = losses[1:] + [tr.flush_loss()]
            assert tr.flush_loss() is None
        runs.append((losses, emb.xs[0].detach().clone()))
    assert np.allclose(runs[0][0], runs[1][0], rtol=1e-5)
    assert rel_err(runs[1][1], runs[0][1]) < 1e-4


@pytest.mark.parametrize('dtype', [torch.float64, torch.float32])
def test_lean_step_equals_autograd_step(dtype, tmp_path):
    """TrainingEngine's tape-free step (zero -> gm_pairs_loss_fused -> optimizer kernel) against its own autograd path
    (BatchedObjective + loss.backward()) on node mini-batches, incl. a trained scale (curvature optimizer): same step
    losses, metrics, points and scale up to the summation order of the gradient atomics."""
    from graphembed.data import GraphDataset
    from graphembed.manifolds import SymmetricPositiveDefinite
    from graphembed.modules import ManifoldEmbedding
    from graphembed.objectives import QuotientLoss
    from graphembed.optim import RiemannianAdam
    from graphembed.train import TrainingEngine
    from helpers_engine import load_engine_golden
    g = load_engine_golden()
    outs = []
    for lean in (True, False):
        torch.manual_seed(3)
        emb = ManifoldEmbedding(63, [SymmetricPositiveDefinite(4)], device=DEV, dtype=dtype)
        opt = RiemannianAdam(emb.xs, lr=0.01, max_grad_norm=100, exact=True)
        copt = torch.optim.SGD(list(emb.curvature_params), lr=1e-3)
        eng = TrainingEngine(embedding=emb, optimizer=[opt, copt], objective_fn=QuotientLoss(), n_epochs=4,
                             val_every_epochs=2, alpha=1.0, batch_size=30, drop_last_n=3, save_dir=str(tmp_path),
                             tensorboard=False)
        ds = GraphDataset(g['hops_condensed'].to(device=DEV, dtype=dtype))
        if not lean:
            eng._lean = dict(ok=False, dataset=ds)
        torch.manual_seed(1234)
        eng(ds)
        assert eng._lean['ok'] == lean
        h = eng.writer.history
        outs.append(([v for _, v in h['quotient_loss']], [v for _, v in h['average_distortion']],
                     emb.xs[0].detach().clone(), emb.scales[0].detach().clone()))
    t = 1e-11 if dtype == torch.float64 else 1e-5
    assert len(outs[0][0]) == 12 and np.allclose(outs[0][0], outs[1][0], rtol=t)
    assert np.allclose(outs[0][1], outs[1][1], rtol=t)
    assert rel_err(outs[0][2], outs[1][2]) < t and rel_err(outs[0][3], outs[1][3]) < t
    assert abs(outs[0][3].item() - 0.5) > 1e-6  # the scale really was trained


@pytest.mark.parametrize('kind', ['manifold_product', 'universal_product'])
def test_lean_step_equals_autograd_step_for_products(kind, tmp_path):
    """Same as above for several factors: a ManifoldEmbedding product with trained scales (SGD on the scales) and a
    products.Embedding of Universal factors with trained curvatures -- the lean path runs gm_pairs_dist2 per factor,
    gm_product_loss on the dense targets, gm_pairs_grad per factor (with the curvature gradient)."""
    from graphembed.data import GraphDataset
    from graphembed.manifolds import Lorentz, SymmetricPositiveDefinite
    from graphembed.modules import ManifoldEmbedding
    from graphembed.objectives import QuotientLoss
    from graphembed.optim import RiemannianAdam
    from graphembed.products import Embedding
    from graphembed.train import TrainingEngine
    from helpers_engine import load_engine_golden
    g = load_engine_golden()
    outs = []
    for lean in (True, False):
        torch.manual_seed(3)
        if kind == 'manifold_product':
            emb = ManifoldEmbedding(63, [SymmetricPositiveDefinite(3), Lorentz(5)], device=DEV, dtype=torch.float64)
        else:
            emb = Embedding(63, [3, 2], c_init=0.4, device=DEV, dtype=torch.float64)
            with torch.no_grad():
                emb.manifolds[1].c.fill_(-0.6)
                for x in emb.xs:
                    x.mul_(30.0)
        opt = RiemannianAdam(emb.xs, lr=0.01, max_grad_norm=100, exact=True)
        copt = torch.optim.SGD(list(emb.curvature_params), lr=1e-4)
        eng = TrainingEngine(embedding=emb, optimizer=[opt, copt], objective_fn=QuotientLoss(), n_epochs=3,
                             val_every_epochs=3, alpha=1.0, batch_size=30, drop_last_n=3, save_dir=str(tmp_path),
                             tensorboard=False)
        ds = GraphDataset(g['hops_condensed'].to(device=DEV, dtype=torch.float64))
        if not lean:
            eng._lean = dict(ok=False, dataset=ds)
        torch.manual_seed(1234)
        eng(ds)
        assert eng._lean['ok'] == lean
        h = eng.writer.history
        outs.append(([v for _, v in h['quotient_loss']], [x.detach().clone() for x in emb.xs],
                     [p.detach().clone() for p in emb.curvature_params]))
    assert len(outs[0][0]) == 9 and np.allclose(outs[0][0], outs[1][0], rtol=1e-11)
    for a, b in zip(outs[0][1] + outs[0][2], outs[1][1] + outs[1][2]):
        assert rel_err(a, b) < 1e-10
    start = 0.5 if kind == 'manifold_product' else 0.4
    assert abs(outs[0][2][0].item() - start) > 1e-7  # scale / curvature parameters really were trained


def test_optimizer_zero_grad_after_step_matches_explicit_memset():
    """RiemannianAdam on a parameter marked _gm_zero_grad_after_step (what ShardedPairTrainer sets) lets the optimizer
    kernel clear every gradient row it has read (gm_optim_t.zero_grad), so the gradient buffer is zeroed once before
    the first step only: 4 pair-kernel + optimizer steps against the explicit zero -> pairs -> update sequence."""
    from graphembed import _ops, _lib as L
    from graphembed.manifolds import SymmetricPositiveDefinite
    from graphembed.modules import ManifoldEmbedding
    from graphembed.objectives import QuotientLoss
    from graphembed.optim import RiemannianAdam
    n, P = 3000, 50000
    g = torch.Generator().manual_seed(9)
    batches = []
    for _ in range(4):
        I = torch.randint(n, (P,), generator=g, dtype=torch.int32)
        J = (I + 1 + torch.randint(n - 1, (P,), generator=g, dtype=torch.int32)) % n
        batches.append((I.to(DEV), J.to(DEV), torch.randint(1, 9, (P,), generator=g, dtype=torch.uint8).to(DEV)))
    torch.manual_seed(5)
    emb = ManifoldEmbedding(n, [SymmetricPositiveDefinite(4)], device=DEV, dtype=torch.float64)
    man = emb.manifolds[0]
    x = emb.xs[0]
    x_ref = x.detach().clone()
    sp = float(torch.nn.functional.softplus(torch.tensor(0.5)))
    x.grad = torch.zeros_like(x)
    x._gm_zero_grad_after_step = True
    opt = RiemannianAdam(emb.xs, lr=0.01, max_grad_norm=100, exact=True)
    losses = []
    for k, (I, J, H) in enumerate(batches):
        acc, _ = _ops.pairs_loss_fused(man.spec, x.detach(), _ops.PairSet.from_lists(I, J, DEV),
                                       _ops.TargetSpec.hops(H, 64.0), QuotientLoss().loss_spec(epoch=k + 1, alpha=1.0),
                                       sp, x.grad)
        losses.append(acc[0].item())
        opt.step()
        assert float(x.grad.abs().max().item()) == 0.0  # handed back cleared
    # explicit sequence on a copy
    m, v = torch.zeros_like(x_ref), torch.zeros_like(x_ref)
    ref_losses = []
    for k, (I, J, H) in enumerate(batches):
        grad = torch.zeros_like(x_ref)
        acc, _ = _ops.pairs_loss_fused(man.spec, x_ref, _ops.PairSet.from_lists(I, J, DEV), _ops.TargetSpec.hops(H, 64.0),
                                       QuotientLoss().loss_spec(epoch=k + 1, alpha=1.0), sp, grad)
        cfg = L.Optim(kind=L.GM_OPT_RADAM, exact=1, has_clip=1, step=k + 1, has_momentum=0, first_step=int(k == 0),
                      grassmann_retr_qr=0, zero_grad=0, lr=0.01, beta1=0.9, beta2=0.999, momentum=0.0, dampening=0.0,
                      max_grad_norm=100.0, eps=1e-8)
        _ops.optim_step(man.spec, cfg, x_ref, grad, m, v)
        assert float(grad.abs().max().item()) > 0.0  # zero_grad=0 leaves the gradient alone
        ref_losses.append(acc[0].item())
    assert np.allclose(losses, ref_losses, rtol=1e-9)  # fp64 loss atomics: summation order differs
    assert rel_err(emb.xs[0].detach(), x_ref) < 1e-10


@pytest.mark.parametrize('case', ['spd4_radam_f32', 'lorentz_rsgd_momentum_f64', 'grassmann_qr_radam_f64',
                                  'product_spd3_lorentz5_radam_f64', 'product_stein2_sphere4_rsgd_f32'])
def test_epoch_kernel_equals_step_loop(case, tmp_path, monkeypatch):
    """gm_train_epoch (all slices of an epoch launched from one native call) against the Python step loop (lean step
    per slice, GM_EPOCH_KERNEL=0): same per-step losses, metrics, points and optimizer state, incl. the dropped tail
    slice, RSGD's momentum seeding on the very first step and the Grassmann qr retraction flag."""
    from graphembed.data import GraphDataset
    from graphembed.manifolds import Grassmann, Lorentz, SymmetricPositiveDefinite
    from graphembed.modules import ManifoldEmbedding
    from graphembed.objectives import QuotientLoss, StressLoss
    from graphembed.optim import RiemannianAdam, RiemannianSGD
    from graphembed.train import TrainingEngine
    from helpers_engine import load_engine_golden
    g = load_engine_golden()
    dtype = torch.float32 if case.endswith('f32') else torch.float64
    outs = []
    for native in ('1', '0'):
        monkeypatch.setenv('GM_EPOCH_KERNEL', native)
        torch.manual_seed(3)
        if case.startswith('spd4'):
            emb = ManifoldEmbedding(63, [SymmetricPositiveDefinite(4)], device=DEV, dtype=dtype)
            opt, obj = RiemannianAdam(emb.xs, lr=0.01, max_grad_norm=100, exact=True), QuotientLoss()
        elif case.startswith('lorentz'):
            emb = ManifoldEmbedding(63, [Lorentz(6)], device=DEV, dtype=dtype)
            opt, obj = RiemannianSGD(emb.xs, lr=1e-3, momentum=0.9, dampening=0.1, max_grad_norm=10), StressLoss()
        elif case.startswith('product_spd3'):  # gm_train_epoch_product
            emb = ManifoldEmbedding(63, [SymmetricPositiveDefinite(3), Lorentz(5)], device=DEV, dtype=dtype)
            opt, obj = RiemannianAdam(emb.xs, lr=0.01, max_grad_norm=100, exact=True), QuotientLoss()
        elif case.startswith('product_stein2'):
            from graphembed.manifolds import Sphere
            sph = Sphere(4)
            emb = ManifoldEmbedding(63, [SymmetricPositiveDefinite(2, use_stein_div=True), sph], device=DEV, dtype=dtype)
            opt, obj = RiemannianSGD(emb.xs, lr=1e-3, momentum=0.5, max_grad_norm=10), QuotientLoss(inc_l2=False)
        else:
            man = Grassmann(6, 2, retr='qr')
            emb = ManifoldEmbedding(63, [man], device=DEV, dtype=dtype)
            with torch.no_grad():
                emb.xs[0].copy_(man.rand_uniform(63, out=torch.empty(0, device=DEV, dtype=dtype)))
            opt, obj = RiemannianAdam(emb.xs, lr=0.01), QuotientLoss()
        eng = TrainingEngine(embedding=emb, optimizer=opt, objective_fn=obj, n_epochs=3, val_every_epochs=3, alpha=1.0,
                             batch_size=20, drop_last_n=5, save_dir=str(tmp_path), tensorboard=False)
        ds = GraphDataset(g['hops_condensed'].to(device=DEV, dtype=dtype))
        torch.manual_seed(1234)
        eng(ds)
        assert eng._lean['ok'] and eng._lean['epoch_ok'] == (native == '1')
        h = eng.writer.history
        state = {f'{f}.{k}': (v.clone() if torch.is_tensor(v) else v) for f, x in enumerate(emb.xs)
                 for k, v in opt.state[x].items()}
        outs.append(([v for _, v in h[str(obj)]], [v for _, v in h['average_distortion']],
                     [x.detach().clone() for x in emb.xs], [x.grad.detach().clone() for x in emb.xs], state))
    t = 1e-10 if dtype == torch.float64 else 2e-5
    assert len(outs[0][0]) == 9  # 63 nodes = 3 slices of 20 + a tail of 3 < drop_last_n, 3 epochs
    assert np.allclose(outs[0][0], outs[1][0], rtol=t) and np.allclose(outs[0][1], outs[1][1], rtol=t)
    for a, b in zip(outs[0][2], outs[1][2]):
        assert rel_err(a, b) < t
    for a, b in zip(outs[0][3], outs[1][3]):
        assert rel_err(a, b) < t * 10
    for key, val in outs[1][4].items():
        if torch.is_tensor(val):
            assert rel_err(outs[0][4][key], val) < t * 10
        else:
            assert outs[0][4][key] == val  # RAdam's step counter advanced once per slice
