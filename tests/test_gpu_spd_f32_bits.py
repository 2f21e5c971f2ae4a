"""fp32 SPD (affine-invariant) kernels, bit for bit: SHA-256 digests of the output bytes of seeded launches, compared
with tests/golden/spd_f32_bits.json, a table recorded with the library as it was before the window-ordered 4x4 pair
kernel (SPEC) rotated its Jacobi eigenvectors with packed FP32x2 instructions.  The packed form rounds every lane as
the scalar form did, so the bytes must not move.

  test_spec_kernel_bitwise   the kernel that changed: one window-ordered 4x4 launch with packed hop counts, checked
                             (torch.profiler) to run the SPEC instantiation.  Its per-pair d2 and its gradient table
                             are digested; every row is the first endpoint of exactly one pair and the second of
                             exactly one, so each gradient row receives two fp32 atomic adds onto zero, whose result
                             does not depend on their order.
  test_spd_f32_outputs_bitwise   the other users of jacobi_eigh, n = 2, 3, 4, 6: forward-only distances, elementwise
                             gradients (the non-streaming pair kernel) and one exact RiemannianAdam update of fixed
                             (x, g).  Their machine code is the same as before; this guards that it stays so.

Not covered: a PairTrainer(deterministic=True) step -- it runs the same forward-only and elementwise-gradient kernels
and the same optimizer kernel as the second test.  The fused loss is a double atomic and is not digested.

`python tests/test_gpu_spd_f32_bits.py` rewrites the table with the library that graphembed loads (GM_B200_LIB)."""
import hashlib
import json
import os
import re
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
for _p in (os.path.join(os.path.dirname(HERE), 'matrix-manifolds_b200'), os.path.join(os.path.dirname(HERE), 'oracle'), HERE):
    if _p not in sys.path:
        sys.path.insert(0, _p)
import helpers_hotpath as H  # noqa: E402

pytestmark = pytest.mark.gpu
TABLE = os.path.join(HERE, 'golden', 'spd_f32_bits.json')
DEV = torch.device('cuda', 0)
NS = (2, 3, 4, 6)
ROWS = {H.CA: 512, H.CB: 256, H.CC: 256, H.CD: 256, H.CE: 256}
P = 40_000
# SPEC launch: 2^18 pairs over 2^18 rows in W = 2 windows.  The segmented walk needs P >= W x 32 x warps, and the 4x4
# fp32 streaming kernel runs at most 4 blocks of 4 warps per SM (128 registers): 2 x 32 x 148 x 16 = 151,552 on a B200.
SPEC_ROWS = {H.CA: 131072, H.CB: 32768, H.CD: 32768, H.CC: 32768, H.CE: 32768}
SPEC_W = 2
MAX_SQ = 64.0


def _digest(t):
    b = t.detach().contiguous().cpu().numpy().tobytes()
    return {'sha256': hashlib.sha256(b).hexdigest(), 'sample': [float(v) for v in t.detach().reshape(-1)[:4].cpu()]}


def _outputs(n):
    from graphembed import _ops, _lib as L
    x, cls, partner = H.point_table(n, ROWS, seed=100 + n)
    I, J = H.grouped_pairs(cls, partner, P, seed=200 + n, weights={H.CA: 4, H.CB: 2, H.CD: 2, H.CC: 1, H.CE: 1})
    spec = _ops.ManifoldSpec(L.GM_SPD_AI, n, point_shape=(n, n), wmin=1e-4, wmax=1e4)
    xd = x.to(DEV).contiguous()
    out = {}
    out['dist2'] = _ops.pairs_dist2(spec, xd, xd, _ops.PairSet.from_lists(I.int().to(DEV), J.int().to(DEV), DEV))
    gout = torch.linspace(-1.0, 1.0, P, device=DEV)
    ga, gb = torch.zeros((P, n, n), device=DEV), torch.zeros((P, n, n), device=DEV)
    _ops.pairs_grad(spec, xd[I.to(DEV)].contiguous(), xd[J.to(DEV)].contiguous(), _ops.PairSet.elementwise(P), gout,
                    ga, gb, coef=0.5)
    out['grad_a'], out['grad_b'] = ga, gb
    # one exact RiemannianAdam update (first step) of fixed points and gradients
    xo = xd.clone()
    g = torch.randn(xo.shape, generator=torch.Generator().manual_seed(400 + n)).to(DEV)
    g = 1e-2 * (g + g.transpose(-1, -2))
    m1, m2 = torch.zeros_like(xo), torch.zeros_like(xo)
    cfg = L.Optim(kind=L.GM_OPT_RADAM, exact=1, has_clip=0, step=1, has_momentum=0, first_step=1,
                  grassmann_retr_qr=0, zero_grad=0, lr=1e-2, beta1=0.9, beta2=0.999, momentum=0.0, dampening=0.0,
                  max_grad_norm=0.0, eps=1e-8)
    _ops.optim_step(spec, cfg, xo, g, m1, m2)
    out['radam_x'], out['radam_m1'], out['radam_m2'] = xo, m1, m2
    torch.cuda.synchronize()
    return {k: _digest(v) for k, v in out.items()}


def _spec_outputs():
    """One SPEC launch -> (digests, names of the kernels it ran)."""
    from graphembed import _ops, _lib as L
    from graphembed.engine import pack_hops, window_order
    x, _, _ = H.point_table(4, SPEC_ROWS, seed=500)
    R = x.shape[0]
    gen = torch.Generator().manual_seed(501)
    I, J = torch.randperm(R, generator=gen), torch.randperm(R, generator=gen)  # every row once per side
    hops = torch.randint(1, 9, (R,), generator=gen, dtype=torch.uint8)
    order = window_order(J.int(), R, SPEC_W)
    I, J, hops = I[order], J[order], hops[order]
    assert R >= SPEC_W * 32 * torch.cuda.get_device_properties(DEV).multi_processor_count * 16
    spec = _ops.ManifoldSpec(L.GM_SPD_AI, 4, point_shape=(4, 4))  # bench.py's wmin / wmax
    xd = x.to(DEV).contiguous()
    pairs = _ops.PairSet.from_lists(I.int().to(DEV), pack_hops(J.int(), hops).to(DEV), DEV, segments=SPEC_W)
    grad = torch.zeros_like(xd)
    loss = _ops.LossSpec(L.GM_LOSS_QUOTIENT, True, True, 1.0, 0.5)
    scale = float(torch.nn.functional.softplus(torch.tensor(0.5)))
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        _, d2 = _ops.pairs_loss_fused(spec, xd, pairs, _ops.TargetSpec.hops_packed(MAX_SQ), loss, scale, grad,
                                      want_d2=True)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if 'spd_pair' in e.name]
    return {'spec_d2': _digest(d2), 'spec_grad': _digest(grad)}, names


@pytest.fixture(scope='module')
def table():
    with open(TABLE) as f:
        return json.load(f)


def _compare(got, want, what):
    assert sorted(got) == sorted(want)
    bad = {k: (got[k]['sample'], want[k]['sample']) for k in want if got[k]['sha256'] != want[k]['sha256']}
    assert not bad, f'{what}: outputs moved (got, recorded samples): {bad}'


def test_spec_kernel_bitwise(table):
    got, names = _spec_outputs()
    assert names and all(re.search(r'spd_pair_stream_kernel<.*,\s*1>|Li1ELi1EEEvT_', nm) for nm in names), \
        f'the launch did not run the SPEC instantiation: {names}'
    _compare(got, table['spec'], 'SPEC 4x4 launch')


@pytest.mark.parametrize('n', NS)
def test_spd_f32_outputs_bitwise(table, n):
    _compare(_outputs(n), table[str(n)], f'n={n}')


if __name__ == '__main__':
    res = {str(n): _outputs(n) for n in NS}
    res['spec'], names = _spec_outputs()
    print('SPEC launch ran:', names)
    with open(TABLE, 'w') as f:
        json.dump(res, f, indent=1, sort_keys=True)
        f.write('\n')
    print('wrote', TABLE)
