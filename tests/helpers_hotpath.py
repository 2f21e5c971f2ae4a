"""Pair-level fp64 reference of the SPD pair kernels and a checker that localises errors to one pair or one gradient
row (tests/test_gpu_spd_hotpath.py, tests/test_hotpath_checker.py).

Everything here is plain torch on the CPU, built on the pinned oracle (oracle/manifolds_oracle.py):

* `PairReference` runs `SpdOracle.dist2` under autograd on the gathered rows of every pair, once in fp64 and once in
  fp32 (the reference's own fp32 answer, which sets the fp32 error budget as `helpers.assert_parity` does): per-pair d2
  and per-pair gradients gx_k (first endpoint), gy_k (second endpoint).
* `loss_weights` turns distances into the loss terms and the per-pair weights w_k = l'(g_k, s d2_k) s in fp64.
* `Checker` compares a launch's d2 vector, gradient table(s) and accumulator with the reference, every bar evaluated
  separately per input class so that ill-conditioned rows cannot loosen the bar for well-conditioned ones:

  contract bar      max-norm relative error <= max(1e-5, 2 x the fp32 reference's error)   (fp64: <= 1e-10)
  localisation bar  per pair  e_k = |d2 - d2_64| / max(d2_64, 1e-2),
                    per row   e_r = max|G[r] - G_ref[r]| / A[r],  A[r] = sum over the row's contributions of
                              |w_k| max|contrib_k|;
                    max e of a class <= max(1e-5, 2 x max e of the fp32 reference)          (fp64: <= 1e-10)
                    One missing, doubled or misrouted contribution moves e_r by about 1 / degree(r).
                    Rows that receive no contribution must stay exactly zero.
  accumulator bar   acc[0], acc[1] against the fp64 sums on the kernel's OWN d2: 1e-6 relative (fp64: 1e-12) --
                    the block reductions, separated from distance error.
"""
import torch

import manifolds_oracle as O

# input classes, in order of severity: a pair's class is the worse of its endpoints' classes, a gradient row's class
# the worst of its own and those of the pairs that touch it
NAMES = ('A', 'B', 'D', 'C', 'E')
CA, CB, CD, CC, CE = range(5)
DESCRIPTION = {CA: 'bench-like (rand ir=0.1)', CB: 'moderate (rand ir=1.0)', CD: 'near-duplicates / copies / self-pairs',
               CC: 'spread spectra [1e-2, 1e2]', CE: 'spectra [1e-3, 1e3]'}
F32_FLOOR, F32_FACTOR, F64_BAR = 1e-5, 2.0, 1e-10
ACC_BAR = {torch.float32: 1e-6, torch.float64: 1e-12}
D2_FLOOR = 1e-2


# ---------------------------------------------------------------------------------------------------------------------
# inputs
# ---------------------------------------------------------------------------------------------------------------------
def _spectra(n, count, lo, hi, gen):
    """SPD matrices with eigenvalues log-uniform in [10^lo, 10^hi] and random rotations (fp64)."""
    q, _ = torch.linalg.qr(torch.randn(count, n, n, dtype=torch.float64, generator=gen))
    lam = 10.0 ** (lo + (hi - lo) * torch.rand(count, n, dtype=torch.float64, generator=gen))
    return q @ torch.diag_embed(lam) @ q.mT


def point_table(n, counts, seed):
    """fp32 table of SPD n x n rows in class blocks.  counts: {class: rows}.  Class D rows come in (copy, base) couples:
    half of the block are bench-like base rows, the other half copies of them -- a quarter bitwise equal, the rest
    base * (1 + delta S) with S symmetric noise in [-1, 1] and delta log-uniform in [1e-6, 1e-3].
    Returns (x (N, n, n) float32, cls (N,) int64, partner (N,) int64: the row a D row was copied from / to, or -1)."""
    gen = torch.Generator().manual_seed(seed)
    orc = O.SpdOracle(n)
    blocks, cls, partner = [], [], []
    base_row = 0
    for c in sorted(counts, key=lambda c: c):
        m = counts[c]
        if c == CA:
            x = orc.rand(m, ir=0.1, generator=gen)
        elif c == CB:
            x = orc.rand(m, ir=1.0, generator=gen)
        elif c == CC:
            x = _spectra(n, m, -2.0, 2.0, gen)
        elif c == CE:
            x = _spectra(n, m, -3.0, 3.0, gen)
        else:
            nb = m // 2
            base = orc.rand(nb, ir=0.1, generator=gen)
            src = torch.randint(nb, (m - nb,), generator=gen)
            delta = 10.0 ** (-6.0 + 3.0 * torch.rand(m - nb, 1, 1, dtype=torch.float64, generator=gen))
            s = 2.0 * torch.rand(m - nb, n, n, dtype=torch.float64, generator=gen) - 1.0
            s = 0.5 * (s + s.mT)
            exact = torch.rand(m - nb, 1, 1, generator=gen) < 0.25
            base32 = base.float().double()  # copies of the fp32 rows: exact copies stay bitwise equal
            copies = torch.where(exact, base32[src], base32[src] * (1.0 + delta * s))
            x = torch.cat([base32, copies])
            p = torch.full((m,), -1, dtype=torch.int64)
            p[nb:] = base_row + src
            p[src] = base_row + nb + torch.arange(m - nb)  # (one of) its copies
            partner.append(p)
        if c != CD:
            partner.append(torch.full((m,), -1, dtype=torch.int64))
        blocks.append((0.5 * (x + x.mT)).float())  # exactly symmetric in fp32
        cls.append(torch.full((m,), c, dtype=torch.int64))
        base_row += m
    return torch.cat(blocks).contiguous(), torch.cat(cls), torch.cat(partner)


def grouped_pairs(cls, partner, P, seed, weights=None, long_share=0.75):
    """Source-grouped pair LIST of exactly P pairs with both endpoints in the same class block: runs of one source
    (long: 1000-5000 consecutive pairs, the run-length accumulator's case; short: 1-48, so that warps mix sources),
    groups in random order.  In class D a quarter of the targets are the source's copy / original and 1 % are the
    source itself (i == j).  Returns (I, J) int64."""
    gen = torch.Generator().manual_seed(seed)
    present = [c for c in range(len(NAMES)) if bool((cls == c).any())]
    weights = weights or {c: 1.0 for c in present}
    wv = torch.tensor([weights.get(c, 0.0) for c in present], dtype=torch.float64)
    lens, gcls = [], []
    total = 0
    while total < P:
        long_run = float(torch.rand(1, generator=gen)) < (long_share / (long_share + (1 - long_share) * 120))
        L = int(torch.randint(1000, 5001, (1,), generator=gen)) if long_run else int(torch.randint(1, 49, (1,), generator=gen))
        lens.append(L)
        gcls.append(present[int(torch.multinomial(wv, 1, generator=gen))])
        total += L
    lens, gcls = torch.tensor(lens), torch.tensor(gcls)
    lo = torch.tensor([int(torch.nonzero(cls == c)[0]) if c in present else 0 for c in range(len(NAMES))])
    size = torch.bincount(cls, minlength=len(NAMES))
    src = lo[gcls] + (torch.rand(len(lens), generator=gen) * size[gcls]).long()
    I = src.repeat_interleave(lens)[:P]
    pc = gcls.repeat_interleave(lens)[:P]
    J = torch.randint(1 << 62, (P,), generator=gen) % (size[pc] - 1)
    J = lo[pc] + J
    J = torch.where(J >= I, J + 1, J)
    if CD in present:
        d = pc == CD
        u = torch.rand(P, generator=gen)
        dup = d & (u < 0.25) & (partner[I] >= 0)
        J = torch.where(dup, partner[I], J)
        J = torch.where(d & (u > 0.99), I, J)
    return I.contiguous(), J.contiguous()


def pair_classes(cls, I, J):
    return torch.maximum(cls[I], cls[J])


def row_classes(cls, parts, pcls):
    """Class of every gradient row: the worst of its own and those of the pairs that touch it.
    parts: index vectors of the rows the pairs' contributions go to (e.g. (I, J))."""
    rc = cls.clone()
    for rows in parts:
        rc.scatter_reduce_(0, rows, pcls, reduce='amax')
    return rc


# ---------------------------------------------------------------------------------------------------------------------
# reference
# ---------------------------------------------------------------------------------------------------------------------
class PairReference:
    """Per-pair d2 and gradients of SpdOracle(n, wmin, wmax).dist2 for the pairs (I, J) of table x (fp32 values), in
    fp64 (d2_64, gx_64, gy_64) and in fp32 (d2_32, gx_32, gy_32; skipped with fp32=False).  x[I] and x[J] are separate
    leaf tensors, so self-pairs get both gradients."""

    def __init__(self, x, I, J, n, wmin=1e-8, wmax=1e8, chunk=1 << 17, fp32=True):
        self.I, self.J, self.n = I, J, n
        orc = O.SpdOracle(n, wmin=wmin, wmax=wmax)
        self.d2_64, self.gx_64, self.gy_64 = self._run(orc, x.double(), I, J, chunk)
        self.d2_32 = self.gx_32 = self.gy_32 = None
        if fp32:
            self.d2_32, self.gx_32, self.gy_32 = self._run(orc, x.float(), I, J, chunk)

    @staticmethod
    def _run(orc, x, I, J, chunk):
        P = I.numel()
        d2 = torch.empty(P, dtype=x.dtype)
        gx = torch.empty((P,) + tuple(x.shape[1:]), dtype=x.dtype)
        gy = torch.empty_like(gx)
        for s in range(0, P, chunk):
            a = x[I[s:s + chunk]].requires_grad_()
            b = x[J[s:s + chunk]].requires_grad_()
            d = orc.dist2(a, b)
            ga, gb = torch.autograd.grad(d.sum(), (a, b))
            d2[s:s + chunk], gx[s:s + chunk], gy[s:s + chunk] = d.detach(), ga, gb
        return d2, gx, gy

    def permuted(self, order):
        """The reference of the same pairs in another order (pair k of the result = pair order[k])."""
        r = PairReference.__new__(PairReference)
        r.I, r.J, r.n = self.I[order], self.J[order], self.n
        for k in ('d2_64', 'gx_64', 'gy_64', 'd2_32', 'gx_32', 'gy_32'):
            v = getattr(self, k)
            setattr(r, k, None if v is None else v[order])
        return r


def targets_from_hops(hops, max_sq, dtype):
    """(h^2) / max in the kernel's dtype (dataset.py:11-12), as fp64: the target is an input of the launch."""
    h = hops.to(dtype)
    return ((h * h) / max_sq).double()


def loss_weights(kind, g, d2, s, alpha=1.0, epoch=1):
    """fp64 (sum of loss terms, sum l'(m) d2, per-pair weight w = l'(g, s d2) s) of QuotientLoss / StressLoss at
    m = s d2 (objectives.py through the oracle; abs' = sign with sign(0) = 0, as the kernels)."""
    d2 = d2.double()
    m = (s * d2).requires_grad_()
    if kind == 'quotient':
        loss = O.quotient_loss(g.double(), m, alpha, epoch)
    else:
        loss = O.stress_loss(g.double(), m)
    dm, = torch.autograd.grad(loss, m)
    return loss.item(), (dm * d2).sum().item(), dm * s


def loss_fp32(kind, g, d2, s, alpha=1.0, epoch=1):
    """The reference's own fp32 loss of fp32 distances (the fp32 error budget of acc[0])."""
    m = torch.tensor(s, dtype=torch.float32) * d2.float()
    if kind == 'quotient':
        return O.quotient_loss(g.float(), m, alpha, epoch).item()
    return O.stress_loss(g.float(), m).item()


# ---------------------------------------------------------------------------------------------------------------------
# checker
# ---------------------------------------------------------------------------------------------------------------------
def _class_max(v, cls):
    """Per-class maximum of the non-negative per-item values v (boolean masks are avoided: they are slow on many-core
    hosts for tensors of this size)."""
    return torch.zeros(len(NAMES) + 1, dtype=torch.float64).scatter_reduce_(0, cls, v.double(), 'amax', include_self=True)


def _item_max(t):
    return t.double().abs().reshape(t.shape[0], -1).amax(1)


def _class_errors(got, ref, cls, scale):
    """Per class: (max-norm relative error, max localised error |got - ref| / scale) of items (rows / pairs)."""
    diff = _item_max(got.double() - ref)
    rel = _class_max(diff, cls) / _class_max(_item_max(ref), cls).clamp(min=1e-300)
    return rel, _class_max(diff / scale, cls)


class Checker:
    """Collects the bars of one launch; `failures` lists every bar that was missed, `lines` every value measured."""

    def __init__(self, dtype, what=''):
        self.dtype, self.what = dtype, what
        self.failures, self.lines = [], []

    def _bar(self, name, e_got, e_ref):
        bound = F64_BAR if self.dtype == torch.float64 else max(F32_FLOOR, F32_FACTOR * e_ref)
        ok = e_got <= bound
        ref_txt = '' if self.dtype == torch.float64 else f' (fp32 reference {e_ref:.2e})'
        line = f'{self.what} {name}: {e_got:.2e} <= {bound:.2e}{ref_txt}' + ('' if ok else '  FAILED')
        self.lines.append(line)
        if not ok:
            self.failures.append(line)

    def _classes(self, name, got, t64, t32, cls, scale=None):
        """Contract (and, with `scale`, localisation) bars of items (pairs / rows) per class; class len(NAMES) = skip."""
        present = torch.bincount(cls, minlength=len(NAMES) + 1)[:len(NAMES)] > 0
        sc = torch.ones(cls.shape, dtype=torch.float64) if scale is None else scale
        rel, loc = _class_errors(got, t64, cls, sc)
        rel32, loc32 = _class_errors(t32, t64, cls, sc) if t32 is not None else (rel * 0, loc * 0)
        for c in range(len(NAMES)):
            if present[c]:
                self._bar(f'{name} class {NAMES[c]} contract', rel[c].item(), rel32[c].item())
                if scale is not None:
                    self._bar(f'{name} class {NAMES[c]} per {"pair" if name == "d2" else "row"}', loc[c].item(),
                              loc32[c].item())

    def d2(self, got, ref, pcls):
        """Contract and localisation bars of the per-pair distances, per pair class."""
        self._classes('d2', got.cpu(), ref.d2_64, ref.d2_32, pcls, ref.d2_64.clamp(min=D2_FLOOR))

    def grad(self, tables, ref, w, rcls):
        """Contract and localisation bars of gradient tables, per row class.
        tables: list of (kernel table (N, n, n), [(rows, 'gx' | 'gy'), ...]) -- the contributions each table receives:
        the first endpoint's gradient gx_k goes to row rows[k] of the table it is listed under, likewise gy_k.
        w: fp64 per-pair weights.  rcls: list (one per table) of per-row classes."""
        for ti, (got, parts) in enumerate(tables):
            got = got.cpu()
            N = got.shape[0]
            g64 = torch.zeros(got.shape, dtype=torch.float64)
            g32 = torch.zeros(got.shape, dtype=torch.float32) if ref.gx_32 is not None else None
            A = torch.zeros(N, dtype=torch.float64)
            for rows, side in parts:
                contrib = w.view(-1, 1, 1) * getattr(ref, side + '_64')
                g64.index_add_(0, rows, contrib)
                A.index_add_(0, rows, _item_max(contrib))
                if g32 is not None:
                    g32.index_add_(0, rows, w.float().view(-1, 1, 1) * getattr(ref, side + '_32'))
            idle = A == 0
            stray = idle & (_item_max(got) != 0)
            if bool(stray.any()):
                bad = torch.nonzero(stray).flatten()[:5].tolist()
                self.failures.append(f'{self.what} grad[{ti}]: rows that receive no pair are not zero: {bad}')
            rc = torch.where(idle, len(NAMES), rcls[ti])
            self._classes(f'grad[{ti}]', got, g64, g32, rc, torch.where(idle, 1.0, A))

    def acc(self, acc, kind, g, d2, ref, pcls, s):
        """acc = kernel [sum loss, sum l' d2] of a launch with targets g, kernel distances d2 and scale s.
        Accumulator bar: both entries against the fp64 sums on the kernel's own d2.  Contract bar, per pair class, for
        both sums: the fp64 sum over the class's pairs on the kernel's d2 (which acc is, to the accumulator bar) against
        the same on the reference's fp64 d2, budget from the same sums on the reference's fp32 d2; in the second sum
        l' is taken at the fp64 d2 throughout."""
        d2 = d2.cpu().double()
        own = loss_weights(kind, g, d2, s)[:2]
        bar = ACC_BAR[self.dtype]
        for name, got, want in (('acc[0]', float(acc[0]), own[0]), ('acc[1]', float(acc[1]), own[1])):
            e = abs(got - want) / max(abs(want), 1e-300)
            line = f'{self.what} {name} accumulator (own d2): {e:.2e} <= {bar:.0e}' + ('' if e <= bar else '  FAILED')
            self.lines.append(line)
            if e > bar:
                self.failures.append(line)
        for c in range(len(NAMES)):
            idx = torch.nonzero(pcls == c).flatten()
            if not idx.numel():
                continue
            r64 = loss_weights(kind, g[idx], ref.d2_64[idx], s)
            lk = loss_weights(kind, g[idx], d2[idx], s)[0]
            l32 = None if ref.d2_32 is None else loss_fp32(kind, g[idx], ref.d2_32[idx], s)
            self.scalar(f'loss class {NAMES[c]} contract', lk, r64[0], l32)
            # sum l'(m) d2 with l' taken at the fp64 d2 on every side: l' of QuotientLoss jumps at its kinks, where a
            # last-bit difference in d2 flips a term (the kernel's own l' is checked by the accumulator bar)
            dm = r64[2] / s
            a32 = None if ref.d2_32 is None else (dm * ref.d2_32[idx].double()).sum().item()
            self.scalar(f'sum l\'d2 class {NAMES[c]} contract', (dm * d2[idx]).sum().item(), r64[1], a32)

    def scalar(self, name, got, want64, want32):
        self._bar(name, abs(got - want64) / abs(want64), 0.0 if want32 is None else abs(want32 - want64) / abs(want64))

    def table(self, name, got, want64, want32, rcls):
        """Contract bar of a point table (e.g. after an optimizer step), per row class."""
        self._classes(name, got.cpu(), want64, want32, rcls)

    def report(self):
        return '\n'.join(self.lines)

    def assert_ok(self):
        assert not self.failures, '\n'.join(self.failures) + '\n--- all bars ---\n' + self.report()
