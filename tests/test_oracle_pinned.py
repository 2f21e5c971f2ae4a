"""Pins the oracle (oracle/manifolds_oracle.py) to the real reference: every function is compared with golden
vectors produced by running dalab/matrix-manifolds itself (tests/golden/make_golden.py).  CPU only."""
import numpy as np
import pytest
import torch

import manifolds_oracle as O
from helpers import CASES, DTYPES, is_spd, load_golden, make_oracle, rel_err, sym

TOL = {'f64': 1e-12, 'f32': 2e-5}


@pytest.mark.parametrize('tag', ['f64', 'f32'])
@pytest.mark.parametrize('name', sorted(CASES))
def test_dist_and_grad(name, tag):
    g = load_golden(name, tag)
    man = make_oracle(name)
    x, y = g['x'].clone().requires_grad_(), g['y'].clone().requires_grad_()
    d2 = man.dist2(x, y)
    (d2 * g['w']).sum().backward()
    fix = sym if is_spd(name) else (lambda t: t)
    assert rel_err(d2.detach(), g['dist2']) < TOL[tag]
    assert rel_err(fix(x.grad), fix(g['gx'])) < TOL[tag] * 10
    assert rel_err(fix(y.grad), fix(g['gy'])) < TOL[tag] * 10


@pytest.mark.parametrize('tag', ['f64', 'f32'])
@pytest.mark.parametrize('name', sorted(CASES))
def test_pdist_losses(name, tag):
    g = load_golden(name, tag)
    man = make_oracle(name)
    fix = sym if is_spd(name) else (lambda t: t)
    for lname, fn in (('quot', lambda t, m: O.quotient_loss(t, m, 1.7, 3)),
                      ('quot_l1', lambda t, m: O.quotient_loss(t, m, 1.7, 3, inc_l2=False)),
                      ('stress', O.stress_loss)):
        x = g['x'].clone().requires_grad_()
        pd2 = man.pdist2(x)
        loss = fn(g['targets'], 0.9 * pd2)
        loss.backward()
        assert rel_err(pd2.detach(), g['pdist2']) < TOL[tag]
        assert abs(loss.item() - g[f'loss_{lname}'].item()) <= TOL[tag] * 10 * abs(g[f'loss_{lname}'].item())
        assert rel_err(fix(x.grad), fix(g[f'grad_{lname}'])) < TOL[tag] * 50


@pytest.mark.parametrize('tag', ['f64', 'f32'])
@pytest.mark.parametrize('name', sorted(CASES))
def test_point_ops(name, tag):
    g = load_golden(name, tag)
    man = make_oracle(name)
    x, y, u, v, eg = g['x'], g['y'], g['u'], g['v'], g['eg']
    t = TOL[tag] * 20
    assert rel_err(man.exp(x, u), g['exp']) < t
    assert rel_err(man.retr(x, u), g['retr']) < t
    assert rel_err(man.log(x, y), g['log']) < t * 50
    assert rel_err(man.proju(x, eg), g['proju']) < t
    assert rel_err(man.egrad2rgrad(x, eg), g['egrad2rgrad']) < t
    assert rel_err(man.transp(x, y, u), g['transp']) < t
    assert rel_err(man.inner(x, u, v), g['inner']) < t
    assert rel_err(man.norm(x, u).pow(2).reshape(-1), g['norm2'].reshape(-1)) < t


OPTS = {
    'radam_clip': ('radam', dict(lr=0.05, max_grad_norm=1.5)),
    'radam_exact': ('radam', dict(lr=0.05, exact=True)),
    'rsgd_exact_clip': ('rsgd', dict(lr=0.05, max_grad_norm=0.5, exact=True)),
    'rsgd_momentum': ('rsgd', dict(lr=0.05, momentum=0.9, dampening=0.1)),
}


@pytest.mark.parametrize('tag', ['f64', 'f32'])
@pytest.mark.parametrize('oname', sorted(OPTS))
@pytest.mark.parametrize('name', sorted(CASES))
def test_optimizer_trajectories(name, oname, tag):
    g = load_golden(name, tag)
    man = make_oracle(name)
    kind, kw = OPTS[oname]
    x, state = g['x'].clone(), {}
    for k in range(3):
        step = O.radam_step if kind == 'radam' else O.rsgd_step
        x = step(man, x, g['opt_grads'][k], state, **kw)
        assert rel_err(x, g[f'{oname}_x'][k]) < TOL[tag] * 50
    for key in ('exp_avg', 'exp_avg_sq', 'momentum_buffer'):
        if f'{oname}_{key}' in g:
            assert rel_err(state[key], g[f'{oname}_{key}']) < TOL[tag] * 50


# ---- objectives / metrics / epoch loop added with the TrainingEngine row (SURVEY 8f-1, 8f-2) ------------------------
@pytest.mark.parametrize('tag', ['f64', 'f32'])
def test_kl_sne_and_metrics_vs_reference(tag):
    g = load_golden('objectives', tag)
    t = 1e-12 if tag == 'f64' else 1e-5
    for inc in (1, 0):
        m = g['m'].clone().requires_grad_()
        loss = O.kl_sne_loss(g['g'], m, float(g['alpha']), inclusive=bool(inc))
        loss.backward()
        assert abs(loss.item() - g[f'kl_{inc}_loss'].item()) <= t * abs(g[f'kl_{inc}_loss'].item())
        assert rel_err(m.grad, g[f'kl_{inc}_grad']) < t
    assert abs(O.pearsonr(g['m'], g['g']).item() - g['pearsonr'].item()) < t
    assert abs(O.average_distortion(g['m'], g['g']).item() - g['average_distortion'].item()) < t


@pytest.mark.parametrize('tag', ['spd3_full', 'spd3_batched', 'spd2_kl', 'prod_radam'])
def test_epoch_loop_vs_reference_training_engine(tag):
    """oracle/engine_oracle.py against the real TrainingEngine's step losses, per-epoch metrics and final points."""
    import engine_oracle as E
    from helpers_engine import RUNS, ENGINE_SEED, N_EPOCHS, load_engine_golden
    g = load_engine_golden()
    factors, objective, (oname, okw), ekw = RUNS[tag]
    oracles = [O.SpdOracle(n) if fam == 'spd' else O.LorentzOracle(n) for fam, n in factors]
    xs = [g[f'{tag}_x0_{i}'].clone() for i in range(len(factors))]
    scales = [torch.tensor(0.5, dtype=torch.float64) for _ in factors]
    if objective == 'quotient':
        loss_fn = lambda t, m, alpha, epoch: O.quotient_loss(t, m, alpha, epoch)
    else:
        loss_fn = lambda t, m, alpha, epoch: O.kl_sne_loss(t, m, alpha, inclusive=True)
    step = O.rsgd_step if oname == 'rsgd' else O.radam_step
    step_fn = lambda f, o, x, grad, st: step(o, x, grad, st, **okw)
    ekw = dict(ekw)
    out = E.run_engine(oracles, xs, scales, g['hops_condensed'], loss_fn, step_fn, N_EPOCHS, ekw.pop('alpha'),
                       seed=ENGINE_SEED, **ekw)
    assert np.allclose(out['step_loss'], g[f'{tag}_step_loss'].numpy(), rtol=1e-10)
    assert np.allclose(out['pearsonr'], g[f'{tag}_pearsonr'].numpy(), rtol=1e-9)
    assert np.allclose(out['average_distortion'], g[f'{tag}_average_distortion'].numpy(), rtol=1e-10)
    for i, x in enumerate(out['xs']):
        assert rel_err(x, g[f'{tag}_xT_{i}']) < 1e-10
    assert out['best'][0] == int(g[f'{tag}_best'][0]) and abs(out['best'][1] - g[f'{tag}_best'][1].item()) < 1e-5
