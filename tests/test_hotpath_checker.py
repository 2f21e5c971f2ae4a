"""The checker of tests/helpers_hotpath.py has teeth: with the reference's own fp32 answer standing in for a kernel it
passes, and it fails when that answer loses one pair's contribution to one row, doubles it, adds one second-endpoint
gradient to the first endpoint's row, or moves one pair's d2 by 1e-4 relative.  CPU only."""
import pytest
import torch

import helpers_hotpath as H

N_ROWS = {H.CA: 1536, H.CB: 768, H.CD: 768, H.CC: 512, H.CE: 512}
P = (1 << 16) - 5
S = 0.93
MAX_SQ = 64.0


@pytest.fixture(scope='module')
def fake_launch():
    x, cls, partner = H.point_table(4, N_ROWS, seed=5)
    I, J = H.grouped_pairs(cls, partner, P, seed=6)
    ref = H.PairReference(x, I, J, 4)
    hops = torch.randint(1, 9, (P,), generator=torch.Generator().manual_seed(7), dtype=torch.uint8)
    g = H.targets_from_hops(hops, MAX_SQ, torch.float32)
    pcls = H.pair_classes(cls, I, J)
    rcls = H.row_classes(cls, (I, J), pcls)
    # the "kernel": the reference's fp32 distances, gradients summed in fp32 with weights on its own d2
    d2 = ref.d2_32.clone()
    _, _, w = H.loss_weights('quotient', g, d2, S)
    grad = torch.zeros(x.shape, dtype=torch.float32)
    grad.index_add_(0, I, w.float().view(-1, 1, 1) * ref.gx_32)
    grad.index_add_(0, J, w.float().view(-1, 1, 1) * ref.gy_32)
    acc = torch.tensor(H.loss_weights('quotient', g, d2, S)[:2], dtype=torch.float64)
    # a class-A pair whose contribution to its first endpoint is above the median of its class
    size = (w.abs().view(-1, 1) * ref.gx_64.reshape(P, -1).abs()).amax(1)
    a = torch.nonzero((pcls == H.CA) & (I != J)).flatten()
    k = int(a[size[a] >= size[a].median()][len(a) // 7])
    return dict(x=x, g=g, I=I, J=J, ref=ref, pcls=pcls, rcls=rcls, d2=d2, w=w, grad=grad, acc=acc, k=k)


def _check(f, d2=None, grad=None):
    chk = H.Checker(torch.float32, 'fp32 oracle as kernel')
    chk.d2(f['d2'] if d2 is None else d2, f['ref'], f['pcls'])
    chk.grad([(f['grad'] if grad is None else grad, [(f['I'], 'gx'), (f['J'], 'gy')])], f['ref'], f['w'], [f['rcls']])
    chk.acc(f['acc'], 'quotient', f['g'], f['d2'] if d2 is None else d2, f['ref'], f['pcls'], S)
    return chk


def test_reference_fp32_passes(fake_launch):
    _check(fake_launch).assert_ok()


def _contribution(f, side):
    k = f['k']
    return (f['w'][k].float() * getattr(f['ref'], side + '_32')[k])


@pytest.mark.parametrize('mutation', ['dropped', 'doubled', 'gy_to_first_endpoint'])
def test_one_wrong_contribution_fails(fake_launch, mutation):
    f = fake_launch
    k, i, j = f['k'], int(f['I'][f['k']]), int(f['J'][f['k']])
    grad = f['grad'].clone()
    if mutation == 'dropped':
        grad[i] -= _contribution(f, 'gx')
    elif mutation == 'doubled':
        grad[i] += _contribution(f, 'gx')
    else:
        grad[j] -= _contribution(f, 'gy')
        grad[i] += _contribution(f, 'gy')
    chk = _check(f, grad=grad)
    assert chk.failures, chk.report()
    assert all('per row' in s or 'contract' in s for s in chk.failures)


def test_one_wrong_distance_fails(fake_launch):
    f = fake_launch
    d2 = f['d2'].clone()
    d2[f['k']] *= 1.0 + 1e-4
    chk = _check(f, d2=d2)
    assert any('d2 class A per pair' in s for s in chk.failures), chk.report()
