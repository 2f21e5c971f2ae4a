"""GPU tests of PairTrainer's steps from pinned host tensors (step_host, step_host_grouped in its 5-, 4-, 3- and 2-byte
formats, step_sampled_host) where the prefetched next batch is not the batch of the next call, where batches grow
while a prefetch is in flight, and where one trainer switches between the formats: every sequence is the same
sequence of device-resident steps (PairTrainer.step on the decoded lists, step_sampled for the sampled pairs)."""
import pytest
import torch

from helpers import rel_err

pytestmark = pytest.mark.gpu
DEV = torch.device('cuda', 0)
N = 3000  # below 8192 rows, so every batch fits the 2-byte words
FORMATS = ['5', '4', '3', '2', 'lists']


class _Batch:
    """One source-grouped pair batch (ragged groups, some empty) in every upload format, and its decoded lists."""

    def __init__(self, seed, G, per):
        from graphembed.engine import pack_hops, pack_hops2, pack_hops3
        g = torch.Generator().manual_seed(seed)
        src = torch.randperm(N, generator=g)[:G].int()
        counts = torch.randint(0, 2 * per + 1, (G,), generator=g)
        offsets = torch.cat([torch.zeros(1, dtype=torch.int64), counts.cumsum(0)])
        I = src.repeat_interleave(counts)
        J = torch.randint(N - 1, (I.numel(),), generator=g, dtype=torch.int32)
        J = torch.where(J >= I, J + 1, J).contiguous()
        H = torch.randint(1, 9, (I.numel(),), generator=g, dtype=torch.uint8)
        words, bases, order = pack_hops2(offsets, J, H)
        Jp = pack_hops(J, H)
        pin = lambda t: t.pin_memory()  # noqa: E731
        s, o = pin(src), pin(offsets)
        self.host = {'5': (s, o, pin(J), pin(H), None), '5w': (s, o, pin(J), pin(H.to(torch.int16)), None),
                     '4': (s, o, pin(Jp), None, None), '3': (s, o, pin(pack_hops3(J, H)), None, None),
                     '2': (s, o, pin(words), None, pin(bases)),
                     'lists': (pin(I), pin(J), pin(H)), 'lists_w': (pin(I), pin(J), pin(H.to(torch.int16)))}
        self.lists = {'5': (I, J, H), '5w': (I, J, H.to(torch.int16)), '4': (I, Jp, None), '3': (I, Jp, None),
                      '2': (I, pack_hops(J[order].contiguous(), H[order].contiguous()), None),
                      'lists': (I, J, H), 'lists_w': (I, J, H.to(torch.int16))}


def _host(b, fmt, nxt=None):
    """The host-input call on batch b in format fmt; nxt = (batch, format) of the prefetched next batch."""
    ahead = None if nxt is None else nxt[0].host[nxt[1]]
    if fmt.startswith('lists'):
        return lambda tr: tr.step_host(*b.host[fmt], epoch=1, next_batch=ahead)
    h = b.host[fmt]
    return lambda tr: tr.step_host_grouped(*h[:4], epoch=1, next_batch=ahead, bases=h[4])


def _listed(b, fmt):
    I, J, H = b.lists[fmt]
    return lambda tr: tr.step(I.to(DEV), J.to(DEV), None if H is None else H.to(DEV), epoch=1).item()


class _Sampled:
    def __init__(self, seed, G=30, per=64):
        g = torch.Generator().manual_seed(seed)
        self.levels = torch.randint(1, 9, (G + 3, N), generator=g, dtype=torch.uint8).to(DEV)
        self.src = torch.randperm(N, generator=g)[:G].int()
        self.slots = torch.randperm(G + 3, generator=g)[:G].int()
        self.per, self.seed = per, 0x5EED + seed

    def host(self):
        src, slots = self.src.pin_memory(), self.slots.pin_memory()
        return lambda tr: tr.step_sampled_host(src, self.levels, self.per, self.seed, slots=slots, epoch=1)

    def device(self):
        return lambda tr: tr.step_sampled(self.src.to(DEV), self.levels, self.per, self.seed, slots=self.slots.to(DEV),
                                          epoch=1).item()


def _check(host_calls, device_calls):
    from graphembed.engine import PairTrainer
    from graphembed.manifolds import SymmetricPositiveDefinite
    from graphembed.modules import ManifoldEmbedding
    from graphembed.objectives import QuotientLoss
    from graphembed.optim import RiemannianAdam
    runs = []
    for calls in (host_calls, device_calls):
        torch.manual_seed(3)
        emb = ManifoldEmbedding(N, [SymmetricPositiveDefinite(4)], device=DEV, dtype=torch.float32)
        tr = PairTrainer(emb, RiemannianAdam(emb.xs, lr=0.01, max_grad_norm=100, exact=True), QuotientLoss(),
                         max_hops_sq=64.0)
        runs.append(([call(tr) for call in calls], emb.xs[0].detach().cpu().clone()))
    (got, x), (want, x_ref) = runs
    assert max(abs(a - b) / abs(b) for a, b in zip(got, want)) < 1e-6, (got, want)
    assert rel_err(x, x_ref) < 2e-5


@pytest.mark.parametrize('fmt', FORMATS)
def test_prefetched_batch_not_taken(fmt):
    """The batch prefetched with next_batch is followed by a call with another batch (B, and later A, are never the
    batch of the call after their prefetch); taken prefetches and blocking calls in between."""
    A, B, C, D = (_Batch(s, 24, 60) for s in range(4))
    _check([_host(A, fmt, (B, fmt)), _host(C, fmt, (D, fmt)), _host(D, fmt), _host(B, fmt, (A, fmt)), _host(C, fmt)],
           [_listed(A, fmt), _listed(C, fmt), _listed(D, fmt), _listed(B, fmt), _listed(C, fmt)])


@pytest.mark.parametrize('fmt', FORMATS)
def test_batches_growing_while_a_prefetch_is_in_flight(fmt):
    """A batch with more sources and pairs than any before arrives while a prefetch is outstanding, and prefetches a
    next batch larger still; the small batch is prefetched after the large ones."""
    S1, S2, L, XL = _Batch(10, 20, 40), _Batch(11, 20, 40), _Batch(12, 40, 120), _Batch(13, 64, 300)
    _check([_host(S1, fmt, (S2, fmt)), _host(L, fmt, (XL, fmt)), _host(XL, fmt, (S2, fmt)), _host(S2, fmt),
            _host(XL, fmt)],
           [_listed(S1, fmt), _listed(L, fmt), _listed(XL, fmt), _listed(S2, fmt), _listed(XL, fmt)])


def test_one_trainer_alternating_every_host_format():
    """Every grouped format (with uint8 and int16 hop counts), step_host and step_sampled_host through one trainer,
    prefetching across formats and discarding a prefetch at a sampled step."""
    A, B, C, D = (_Batch(20 + s, 24 + 8 * s, 40 + 30 * s) for s in range(4))
    S1, S2 = _Sampled(1), _Sampled(2)
    seq = [('5', A, ('4', B)), ('4', B, ('3', C)), ('3', C, ('2', D)), ('2', D, ('5', A)), S1,
           ('lists', A, ('lists_w', B)), ('lists_w', B, None), ('5w', C, ('2', A)), ('2', A, None), S2, ('3', D, None)]
    host, device = [], []
    for item in seq:
        if isinstance(item, _Sampled):
            host.append(item.host())
            device.append(item.device())
        else:
            fmt, b, nxt = item
            host.append(_host(b, fmt, None if nxt is None else (nxt[1], nxt[0])))
            device.append(_listed(b, fmt))
    _check(host, device)
