"""CPU-side checks of the drop-in boundary: the shared library loads, exports every symbol include/gm_kernels.h
declares, rejects bad arguments with error codes (no launch), and the Python layer fails loudly without CUDA."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, 'include', 'gm_kernels.h')).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(gm_[a-z0-9_]+)\s*\(', text)))


def test_library_exports_every_declared_symbol():
    from graphembed import _lib
    lib = _lib.lib()
    declared = _declared_symbols()
    assert len(declared) >= 14
    for name in declared:
        assert hasattr(lib, name), f'{name} declared in gm_kernels.h but not exported'
    assert set(declared) == set(_lib.EXPORTED_SYMBOLS)
    assert b'sm_100a' in lib.gm_version()


def test_argument_validation_without_gpu():
    from graphembed import _lib as L
    lib = L.lib()
    man = L.Manifold(kind=L.GM_SPD_AI, dtype=L.GM_F32, n=4, p=0, flags=0, reserved=0, wmin=1e-8, wmax=1e8)
    assert lib.gm_supported(ctypes.byref(man)) == 1
    bad = L.Manifold(kind=L.GM_SPD_AI, dtype=L.GM_F32, n=11, p=0, flags=0, reserved=0, wmin=1e-8, wmax=1e8)
    assert lib.gm_supported(ctypes.byref(bad)) == 0
    bad = L.Manifold(kind=L.GM_SPD_AI, dtype=L.GM_F32, n=4, p=0, flags=L.GM_FAST_CHOL, reserved=0, wmin=0, wmax=1)
    assert lib.gm_supported(ctypes.byref(bad)) == 0
    pairs = L.Pairs(mode=L.GM_PAIRS_TRIU, idx64=0, P=11, idx_i=None, idx_j=None, B=5, nodes=None)  # > 5*4/2
    assert lib.gm_pairs_dist2(ctypes.byref(man), None, None, ctypes.byref(pairs), None, None) == -1
    pairs = L.Pairs(mode=L.GM_PAIRS_TRIU, idx64=0, P=7, idx_i=None, idx_j=None, B=5, nodes=None, k0=4)  # 4+7 > 10
    assert lib.gm_pairs_dist2(ctypes.byref(man), None, None, ctypes.byref(pairs), None, None) == -1
    pairs = L.Pairs(mode=L.GM_PAIRS_TRIU, idx64=0, P=6, idx_i=None, idx_j=None, B=5, nodes=None, k0=4)  # slice ok
    assert lib.gm_pairs_dist2(ctypes.byref(man), None, None, ctypes.byref(pairs), None, None) == -3
    pairs = L.Pairs(mode=L.GM_PAIRS_TRIU, idx64=0, P=10, idx_i=None, idx_j=None, B=5, nodes=None)
    assert lib.gm_pairs_dist2(ctypes.byref(man), None, None, ctypes.byref(pairs), None, None) == -3  # NULL data
    empty = L.Pairs(mode=L.GM_PAIRS_LIST, idx64=0, P=0, idx_i=None, idx_j=None, B=0, nodes=None)
    assert lib.gm_pairs_dist2(ctypes.byref(man), None, None, ctypes.byref(empty), None, None) == 0  # empty input
    assert lib.gm_bfs_workspace_bytes(1000, 64) >= 3 * 1000 * 8
    assert lib.gm_launch_count() == 0 or torch.cuda.is_available()


def test_peer_update_argument_validation_without_gpu():
    """gm_optim_step_peer rejects malformed peer tables before any launch (struct layout check included)."""
    from graphembed import _lib as L
    lib = L.lib()
    man = L.Manifold(kind=L.GM_SPD_AI, dtype=L.GM_F32, n=4, p=0, flags=0, reserved=0, wmin=1e-8, wmax=1e8)
    opt = L.Optim(kind=L.GM_OPT_RSGD, exact=0, has_clip=0, step=0, has_momentum=0, first_step=0, grassmann_retr_qr=0,
                  reserved=0, lr=0.1, beta1=0, beta2=0, momentum=0, dampening=0, max_grad_norm=0, eps=1e-8)
    t = L.Peers()
    t.world, t.rank, t.row_lo, t.epoch, t.n_acc = 2, 0, 0, 1, 0
    call = lambda n=8: lib.gm_optim_step_peer(ctypes.byref(man), ctypes.byref(opt), ctypes.byref(t), None, None, n, None)  # noqa: E731
    assert call() == -3  # NULL tables
    t.world = 9
    assert call() == -1  # more ranks than GM_MAX_PEERS
    t.world, t.rank = 2, 2
    assert call() == -1  # rank out of range
    t.rank, t.epoch = 0, 0
    assert call() == -1  # epochs start at 1
    t.epoch = 1
    assert call(0) == -1  # every rank must own rows
    assert ctypes.sizeof(L.Peers) == 8 + 8 + 8 + 4 * 8 * L.GM_MAX_PEERS + 8 + 8 + 8  # ... + gsum (pipelined exchange)
    assert lib.gm_peer_alloc(0, ctypes.byref(ctypes.c_void_p())) == -1
    assert lib.gm_peer_export(None, None) == -3


def test_no_cpu_fallback():
    from graphembed.manifolds import SymmetricPositiveDefinite, Lorentz
    from graphembed.modules import ManifoldParameter
    from graphembed.optim import RiemannianAdam
    man = SymmetricPositiveDefinite(3)
    x = torch.eye(3).repeat(4, 1, 1)
    with pytest.raises(RuntimeError, match='CUDA'):
        man.pdist(x)
    with pytest.raises(RuntimeError, match='CUDA'):
        man.exp(x, torch.zeros_like(x))
    with pytest.raises(RuntimeError, match='CUDA'):
        Lorentz(4).rand(3)
    p = ManifoldParameter(x.clone(), manifold=man)
    p.grad = torch.zeros_like(x)
    with pytest.raises(RuntimeError, match='CUDA'):
        RiemannianAdam([p]).step()


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, 'matrix-manifolds_b200', 'graphembed')
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith('.py'):
                src = open(os.path.join(dirpath, f)).read()
                assert 'oracle' not in src.replace('no CPU', ''), f'{f} mentions the oracle'
                assert 'manifolds_oracle' not in src and 'ref_import' not in src


def test_reference_api_surface():
    """Same class names / ctor signatures / method names as the reference (SURVEY 8b)."""
    import inspect
    from graphembed import manifolds, optim, modules, objectives
    for cls in ('Manifold', 'Euclidean', 'Grassmann', 'Lorentz', 'SymmetricPositiveDefinite', 'Sphere'):
        assert hasattr(manifolds, cls)
    for meth in ('ndim', 'dim', 'zero', 'zero_vec', 'inner', 'norm', 'proju', 'projx', 'egrad2rgrad', 'exp', 'retr',
                 'log', 'dist', 'pdist', 'transp', 'rand', 'rand_uniform', 'randvec'):
        assert hasattr(manifolds.Manifold, meth), meth
    sig = inspect.signature(manifolds.SymmetricPositiveDefinite.__init__)
    assert list(sig.parameters)[1:] == ['n', 'fast_symeig', 'fast_chol', 'use_stein_div', 'wmin', 'wmax']
    assert list(inspect.signature(optim.RiemannianAdam.__init__).parameters)[1:] == \
        ['params', 'lr', 'betas', 'nc', 'max_grad_norm', 'exact']
    assert list(inspect.signature(optim.RiemannianSGD.__init__).parameters)[1:] == \
        ['params', 'lr', 'momentum', 'dampening', 'max_grad_norm', 'exact']
    assert {'xs', 'scales'} <= set(dir(modules.ManifoldEmbedding)) | {'xs', 'scales'}
    for name in ('QuotientLoss', 'StressLoss', 'Sum', 'ObjectiveFunction'):
        assert hasattr(objectives, name)
    with pytest.raises(ValueError):
        objectives.QuotientLoss(inc_l1=False, inc_l2=False)
    with pytest.raises(ValueError):
        manifolds.Grassmann(5, 2, retr='nope')
    assert manifolds.SymmetricPositiveDefinite(4).dim == 10 and manifolds.Lorentz(11).dim == 10
    assert manifolds.Grassmann(6, 2).dim == 8 and str(manifolds.Lorentz(5)) == 'Lorentzian space of dimension 5'


def test_new_entry_points_validate_arguments():
    """gm_pairs_metrics / gm_sne_* / packed hop targets: bad arguments are rejected before any launch."""
    from graphembed import _lib as L
    lib = L.lib()
    one = (ctypes.c_void_p * 1)(ctypes.c_void_p(16))
    sp = (ctypes.c_double * 1)(1.0)
    pairs = L.Pairs(mode=L.GM_PAIRS_ELEMENTWISE, idx64=0, P=0, idx_i=None, idx_j=None, B=0, nodes=None, k0=0)
    tg = L.Targets(mode=L.GM_TGT_VECTOR, reserved=0, data=None, ld=0, max_sq=1.0)
    acc = ctypes.c_void_p(32)
    assert lib.gm_pairs_metrics(L.GM_F32, 1, one, sp, ctypes.byref(pairs), ctypes.byref(tg), 1, acc, None) == 0  # empty
    assert lib.gm_pairs_metrics(L.GM_F32, 9, one, sp, ctypes.byref(pairs), ctypes.byref(tg), 1, acc, None) == -1
    assert lib.gm_pairs_metrics(5, 1, one, sp, ctypes.byref(pairs), ctypes.byref(tg), 1, acc, None) == -1
    pairs.P = 4
    assert lib.gm_pairs_metrics(L.GM_F32, 1, one, sp, ctypes.byref(pairs), ctypes.byref(tg), 1, acc, None) == -3
    assert lib.gm_sne_row_stats(L.GM_F64, 1, one, sp, None, 1, 1.0, 1, None, None) == 0  # B < 2: nothing to do
    assert lib.gm_sne_row_stats(L.GM_F64, 1, one, sp, None, 5, 1.0, 1, None, None) == -3
    assert lib.gm_sne_pair_terms(L.GM_F64, 0, one, sp, None, 5, 1.0, 1, None, None, None, None) == -1
    # packed hop counts need int32 LIST pairs
    man = L.Manifold(kind=L.GM_SPD_AI, dtype=L.GM_F32, n=4, p=0, flags=0, reserved=0, wmin=1e-8, wmax=1e8)
    loss = L.Loss(kind=L.GM_LOSS_QUOTIENT, inc_l1=1, inc_l2=1, reserved=0, alpha=1.0, eps=0.5)
    tgp = L.Targets(mode=L.GM_TGT_HOPS_PACKED, reserved=0, data=None, ld=0, max_sq=9.0)
    p64 = L.Pairs(mode=L.GM_PAIRS_LIST, idx64=1, P=3, idx_i=16, idx_j=16, B=0, nodes=None, k0=0)
    assert lib.gm_pairs_loss_fused(ctypes.byref(man), None, ctypes.byref(p64), ctypes.byref(tgp), ctypes.byref(loss),
                                   1.0, None, None, None, None) == -1
    ptri = L.Pairs(mode=L.GM_PAIRS_TRIU, idx64=0, P=3, idx_i=None, idx_j=None, B=3, nodes=None, k0=0)
    assert lib.gm_pairs_loss_fused(ctypes.byref(man), None, ctypes.byref(ptri), ctypes.byref(tgp), ctypes.byref(loss),
                                   1.0, None, None, None, None) == -1


def test_pair_set_slices_cover_the_triangle():
    from graphembed import _ops
    ps = _ops.PairSet.triu(9)
    parts = [ps.slice(r, 4) for r in range(4)]
    assert [p.P for p in parts] == [9, 9, 9, 9] and [p.k0 for p in parts] == [0, 9, 18, 27]
    parts = [_ops.PairSet.triu(5).slice(r, 3) for r in range(3)]
    assert [(p.k0, p.P) for p in parts] == [(0, 4), (4, 3), (7, 3)]
    with pytest.raises(ValueError):
        _ops.PairSet.triu(5, k0=8, P=3)


def test_yaml_config_grammar(tmp_path):
    """object / closure nodes of the run.py YAML schema (example_config.yaml) build the drop-in classes."""
    from graphembed.config import parse_config
    from graphembed.manifolds import SymmetricPositiveDefinite
    from graphembed.objectives import KLDiveregenceLoss
    cfg = tmp_path / 'c.yaml'
    cfg.write_text("""
save_dir_root: './runs/run'
input_graph: 'g.edges.gz'
embedding:
  closure:
    name: graphembed.modules.ManifoldEmbedding
    params:
      manifolds:
        - object:
            name: graphembed.manifolds.SymmetricPositiveDefinite
            params:
              n: 2
              use_stein_div: False
objective_fn:
  closure:
    name: graphembed.objectives.KLDiveregenceLoss
    params:
      inference_model: 'sne'
      inclusive: True
training_params:
  alpha: 10.0
  n_epochs: 1500
  batch_size: null
embedding_optimizer:
  closure:
    name: graphembed.optim.RiemannianAdam
    params:
      lr: 0.01
      max_grad_norm: 100
      exact: False
lr:
  object:
    name: math.sqrt
    params: [16.0]
""")
    c = parse_config(str(cfg))
    assert callable(c['embedding']) and callable(c['embedding_optimizer'])
    assert isinstance(c['objective_fn'], KLDiveregenceLoss) and c['objective_fn'].inclusive is True
    assert c['training_params'] == dict(alpha=10.0, n_epochs=1500, batch_size=None)
    assert c['lr'] == 4.0
    p = torch.nn.Parameter(torch.zeros(2, 2, 2))
    p.manifold = SymmetricPositiveDefinite(2)
    opt = c['embedding_optimizer']([p])
    assert type(opt).__name__ == 'RiemannianAdam' and opt.defaults['lr'] == 0.01 and opt.defaults['max_grad_norm'] == 100
    with pytest.raises(RuntimeError, match='CUDA'):  # the closure reaches the (GPU-only) initialiser
        c['embedding'](5)


def test_universal_has_no_cpu_path_and_mirrors_the_reference_surface():
    """SURVEY 8f-3: the Universal manifold / products.Embedding classes exist under the reference's module paths,
    construct without a GPU, and refuse to compute on CPU tensors (no fallback)."""
    from graphembed import _lib as L
    from graphembed.manifolds import Universal
    from graphembed.products import Embedding, TrainingEngine  # noqa: F401
    man = Universal(4, c_init=-0.3, keep_sign_fixed=True)
    assert man.ndim == 1 and man.dim == 4 and str(man) == 'Universal 4-dimensional manifold'
    assert abs(man.get_c().item() + (0.001 + torch.nn.functional.softplus(torch.tensor(-0.3)).item())) < 1e-6
    assert abs(man.get_K().item() + man.get_c().item()) < 1e-12 and man.get_R().item() > 0
    assert [n for n, _ in man.named_parameters()] == ['c']
    x = torch.zeros(3, 4)
    assert man.proju(x, x) is x
    with pytest.raises(RuntimeError):
        man.dist(x, x)
    with pytest.raises(RuntimeError):
        man.exp(x, x)
    with pytest.raises(ValueError):
        TrainingEngine(stabilize_every_epochs=2)
    m = L.Manifold(kind=L.GM_UNIVERSAL, dtype=L.GM_F32, n=4, p=0, flags=0, reserved=0, wmin=1e-8, wmax=1e8)
    assert L.lib().gm_supported(ctypes.byref(m)) == 0  # c_dev missing
    m.c_dev = 16
    assert L.lib().gm_supported(ctypes.byref(m)) == 1


def test_new_entry_points_validate_arguments_without_gpu():
    """gm_rank_metrics / gm_train_epoch / gm_train_epoch_product reject bad arguments with error codes before touching
    the device (nothing is launched on this GPU-less box)."""
    from graphembed import _lib as L
    lib = L.lib()
    # gm_rank_metrics: sizes, layer count, empty root range, NULL buffers
    args = lambda **kw: [kw.get('dtype', L.GM_F32), None, None, kw.get('N', 100), kw.get('lo', 0), kw.get('hi', 100), 1,  # noqa: E731
                         9, kw.get('layers', 5), None, None, None, None, None, None, None, None]
    assert lib.gm_rank_metrics(*args(dtype=7)) == -1
    assert lib.gm_rank_metrics(*args(N=1)) == -1
    assert lib.gm_rank_metrics(*args(hi=101)) == -1
    assert lib.gm_rank_metrics(*args(layers=1)) == -1 and lib.gm_rank_metrics(*args(layers=257)) == -1
    assert lib.gm_rank_metrics(*args(lo=40, hi=40)) == 0  # nothing to do
    assert lib.gm_rank_metrics(*args()) == -3
    # gm_train_epoch
    man = L.Manifold(kind=L.GM_LORENTZ, dtype=L.GM_F32, n=5, p=0, flags=0, reserved=0, wmin=1e-8, wmax=1e8)
    opt = L.Optim(kind=L.GM_OPT_RADAM, exact=1, has_clip=0, step=1, has_momentum=0, first_step=1, grassmann_retr_qr=0,
                  zero_grad=0, lr=0.01, beta1=0.9, beta2=0.999, momentum=0.0, dampening=0.0, max_grad_norm=0.0, eps=1e-8)
    tgt = L.Targets(mode=L.GM_TGT_DENSE, reserved=0, data=64, ld=10, max_sq=1.0)
    loss = L.Loss(kind=L.GM_LOSS_QUOTIENT, inc_l1=1, inc_l2=1, reserved=0, alpha=1.0, eps=0.5)
    n_steps = ctypes.c_int64(-1)
    call = lambda m=man, t=tgt, batch=4, x=None: lib.gm_train_epoch(  # noqa: E731
        ctypes.byref(m), ctypes.byref(opt), x, None, None, None, 10, None, 1, 10, batch, 2, ctypes.byref(t),
        ctypes.byref(loss), 1.0, None, 3, ctypes.byref(n_steps), None)
    assert call() == -3 and n_steps.value == 0  # NULL tables
    assert call(batch=1) == -1
    vec_tgt = L.Targets(mode=L.GM_TGT_VECTOR, reserved=0, data=64, ld=0, max_sq=1.0)
    assert call(t=vec_tgt) == -1  # node batches index the DENSE target matrix
    uni = L.Manifold(kind=L.GM_UNIVERSAL, dtype=L.GM_F32, n=5, p=0, flags=0, reserved=0, wmin=1e-8, wmax=1e8, c_dev=64)
    assert call(m=uni) == -2  # curvature gradients need the autograd-side chain rule
    # gm_train_epoch_product: F range and NULL arrays
    mans = (L.Manifold * 2)(man, man)
    opts = (L.Optim * 2)(opt, opt)
    null2 = (ctypes.c_void_p * 2)(None, None)
    sp = (ctypes.c_double * 2)(1.0, 1.0)
    prod = lambda F: lib.gm_train_epoch_product(F, mans, opts, null2, null2, null2, null2, 10, None, 1, 10, 4, 2,  # noqa: E731
                                                 ctypes.byref(tgt), ctypes.byref(loss), sp, null2, None, None, 3,
                                                 ctypes.byref(n_steps), None)
    assert prod(0) == -1 and prod(9) == -1
    assert prod(2) in (-1, -3)


# ---- request contract: the return code of every entry point over a fixed grid of requests ------------------------
# Every device pointer in every request is NULL (host arrays are real but hold NULL device pointers), so no request
# can reach a launch, an allocation or a memset.  The grid runs in a child process that sees no GPU.
GOLDEN_CODES = os.path.join(ROOT, 'tests', 'golden', 'cabi_request_codes.json')
_CODE_CHARS = {0: '0', 1: '1', -1: 'I', -2: 'U', -3: 'N'}  # gm_supported returns 1 / 0


def _request_grid(L, lib):
    """Yields (entry point, label, thunk returning the code) in a deterministic order."""
    import itertools
    c = ctypes
    vp8 = lambda: (c.c_void_p * 8)()  # noqa: E731  (host array of 8 NULL device pointers)

    def man(kind, dtype=L.GM_F32, n=4, p=0, flags=0):
        return L.Manifold(kind=kind, dtype=dtype, n=n, p=p, flags=flags, reserved=0, wmin=1e-8, wmax=1e8)

    mans = {'none': None, 'spd4': man(L.GM_SPD_AI), 'spd2ec64': man(L.GM_SPD_AI, L.GM_F64, 2, 0, 3),
            'spd3e': man(L.GM_SPD_AI, n=3, flags=L.GM_FAST_EIG), 'spd4c': man(L.GM_SPD_AI, flags=L.GM_FAST_CHOL),
            'spd11': man(L.GM_SPD_AI, n=11), 'stein2c': man(L.GM_SPD_STEIN, n=2, flags=L.GM_FAST_CHOL),
            'stein0': man(L.GM_SPD_STEIN, n=0), 'lor5': man(L.GM_LORENTZ, n=5), 'lor1': man(L.GM_LORENTZ, n=1),
            'sph3': man(L.GM_SPHERE, n=3), 'euc0': man(L.GM_EUCLIDEAN, n=0), 'euc7d': man(L.GM_EUCLIDEAN, L.GM_F64, 7),
            'uni4': man(L.GM_UNIVERSAL), 'gr6_2s': man(L.GM_GRASSMANN, n=6, p=2, flags=L.GM_FAST_SVD),
            'gr6_6': man(L.GM_GRASSMANN, n=6, p=6), 'gr3_4': man(L.GM_GRASSMANN, n=3, p=4),
            'gr6_3s': man(L.GM_GRASSMANN, n=6, p=3, flags=L.GM_FAST_SVD), 'kind7': man(7), 'dtype2': man(0, 2)}
    small = {k: mans[k] for k in ('none', 'spd4', 'lor5', 'spd11')}

    def pr(mode, P, **kw):
        return L.Pairs(mode=mode, P=P, **kw)
    S = L.GM_PAIRS_SAMPLED
    samp = dict(per_src=4, n_nodes=100)
    pairs = {'none': None, 'ew0': pr(0, 0), 'ew5': pr(0, 5), 'ew-1': pr(0, -1),
             'list0': pr(1, 0), 'list8': pr(1, 8), 'list8i64': pr(1, 8, idx64=1), 'list0i64': pr(1, 0, idx64=1),
             'list_seg-1': pr(1, 8, segments=-1), 'list_seg65': pr(1, 8, segments=65), 'list_seg4': pr(1, 8, segments=4),
             'triu10': pr(2, 10, B=5), 'triu_k4p7': pr(2, 7, B=5, k0=4), 'triu_k4p6': pr(2, 6, B=5, k0=4),
             'triu_B-1': pr(2, 0, B=-1), 'triu_k-1': pr(2, 1, B=5, k0=-1), 'triu0': pr(2, 0, B=0),
             'samp8': pr(S, 8, **samp), 'samp0': pr(S, 0, **samp), 'samp_i64': pr(S, 0, idx64=1, **samp),
             'samp_per0': pr(S, 0, per_src=0, n_nodes=100), 'samp_n1': pr(S, 0, per_src=4, n_nodes=1),
             'samp_n2^24': pr(S, 0, per_src=4, n_nodes=1 << 24), 'mode4': pr(4, 0), 'mode-1': pr(-1, 0)}
    tgts = {'none': None}
    for m in (-1, 0, 1, 2, 3, 4, 5):
        tgts[f't{m}'] = L.Targets(mode=m, reserved=0, data=None, ld=5, max_sq=9.0)
    losses = {'none': None}
    for kind, l1, l2 in ((0, 1, 1), (0, 0, 0), (0, 1, 0), (0, 0, 1), (1, 0, 0), (2, 1, 1)):
        losses[f'l{kind}{l1}{l2}'] = L.Loss(kind=kind, inc_l1=l1, inc_l2=l2, reserved=0, alpha=1.0, eps=0.5)
    loss4 = {k: losses[k] for k in ('none', 'l011', 'l000', 'l211')}
    ep_tgts = {k: tgts[k] for k in ('none', 't0', 't1', 't5')}
    opts = {'none': None}
    for name, kind, step, mom in (('sgd', 0, 0, 0), ('sgdm', 0, 0, 1), ('adam0', 1, 0, 0), ('adam1', 1, 1, 0),
                                  ('kind2', 2, 1, 0)):
        opts[name] = L.Optim(kind=kind, exact=1, has_clip=0, step=step, has_momentum=mom, first_step=1,
                             grassmann_retr_qr=0, zero_grad=0, lr=0.01, beta1=0.9, beta2=0.999, momentum=0.9 * mom,
                             dampening=0.0, max_grad_norm=0.0, eps=1e-8)
    ref = lambda s: None if s is None else c.byref(s)  # noqa: E731

    def grid(*named):
        return itertools.product(*[list(d.items()) for d in named])

    def label(*parts):
        return ' '.join(k for k, _ in parts)

    for kind in range(-1, 8):
        for dtype, n, p, flags in itertools.product((0, 1, 2), (0, 1, 2, 3, 4, 5, 10, 11), (0, 1, 2, 3, 5, 6),
                                                    (0, 1, 2, 4, 7)):
            m = man(kind, dtype, n, p, flags)
            yield 'gm_supported', f'{kind} {dtype} {n} {p} {flags}', lambda m=m: lib.gm_supported(c.byref(m))

    for mm, pp in grid(mans, pairs):
        yield 'gm_pairs_dist2', label(mm, pp), \
            lambda m=mm[1], p=pp[1]: lib.gm_pairs_dist2(ref(m), None, None, ref(p), None, None)
        yield 'gm_pairs_grad', label(mm, pp), \
            lambda m=mm[1], p=pp[1]: lib.gm_pairs_grad(ref(m), None, None, ref(p), None, 1.0, None, None, None)

    mid = {k: mans[k] for k in ('none', 'spd4', 'lor5', 'spd11', 'gr6_2s', 'dtype2')}
    for mm, pp, tt, ll in grid(mid, pairs, tgts, losses):
        yield 'gm_pairs_loss_fused', label(mm, pp, tt, ll), \
            lambda m=mm[1], p=pp[1], t=tt[1], lo=ll[1]: lib.gm_pairs_loss_fused(
                ref(m), None, ref(p), ref(t), ref(lo), 1.0, None, None, None, None)

    shards = {'none': None}
    for w in (0, 1, 2, 3, 9):
        shards[f'w{w}'] = L.RowShards(world=w)
    for ss, mm, pp, tt, ll in grid(shards, small, pairs, tgts, loss4):
        yield 'gm_pairs_loss_fused_sharded', label(ss, mm, pp, tt, ll), \
            lambda s=ss[1], m=mm[1], p=pp[1], t=tt[1], lo=ll[1]: lib.gm_pairs_loss_fused_sharded(
                ref(m), ref(s), ref(p), ref(t), ref(lo), 1.0, None, None, None)

    def man_array(*ms):
        arr = (L.Manifold * 8)()
        for i in range(8):
            arr[i] = ms[min(i, len(ms) - 1)]
        return arr
    M = mans
    factor_lists = {'F0': (0, man_array(M['spd4'])), 'F1': (1, man_array(M['spd4'])),
                    'spd+lor': (2, man_array(M['spd4'], M['lor5'])), 'lor+sph': (2, man_array(M['lor5'], M['sph3'])),
                    'spd+spd': (2, man_array(M['spd4'], M['spd4'])),
                    'spd+euc64': (2, man_array(M['spd4'], M['euc7d'])),
                    'spd+gr': (2, man_array(M['spd4'], M['gr6_2s'])), 'spd+lor1': (2, man_array(M['spd4'], M['lor1'])),
                    'spd+lor*3': (4, man_array(M['spd4'], M['lor5'])), 'spd+lor*4': (5, man_array(M['spd4'], M['lor5'])),
                    'F9': (9, man_array(M['spd4']))}
    sp8 = (c.c_double * 8)(*[1.0] * 8)
    for ff, pp, tt, ll in grid(factor_lists, pairs, tgts, losses):
        yield 'gm_pairs_product_fused', label(ff, pp, tt, ll), \
            lambda F=ff[1], p=pp[1], t=tt[1], lo=ll[1]: lib.gm_pairs_product_fused(
                F[0], F[1], vp8(), ref(p), ref(t), ref(lo), sp8, None, vp8(), None)
    fl = factor_lists['spd+lor']
    for which in range(4):
        args = [fl[1], vp8(), sp8, vp8()]
        args[which] = None
        yield 'gm_pairs_product_fused', f'null{which}', lambda a=args: lib.gm_pairs_product_fused(
            2, a[0], a[1], ref(pairs['list8']), ref(tgts['t0']), ref(losses['l011']), a[2], None, a[3], None)

    # acc is a device pointer, so every request below stops at its NULL check
    for (F, dtype, P), pp, tt, ll in itertools.product(((0, 0, 4), (1, 0, 4), (9, 0, 4), (2, 2, 4), (2, 0, -1), (2, 0, 0)),
                                                       pairs.items(), ep_tgts.items(), (('none', None), ('l011', losses['l011']))):
        yield 'gm_product_loss', f'{F} {dtype} {P} ' + label(pp, tt, ll), \
            lambda F=F, dt=dtype, P=P, p=pp[1], t=tt[1], lo=ll[1]: lib.gm_product_loss(
                dt, F, vp8(), sp8, ref(p), ref(t), ref(lo), P, None, None, None)
        yield 'gm_pairs_metrics', f'{F} {dtype} {P} ' + label(pp, tt, ll), \
            lambda F=F, dt=dtype, sq=P & 1, p=pp[1], t=tt[1]: lib.gm_pairs_metrics(
                dt, F, vp8(), sp8, ref(p), ref(t), sq, None, None)

    for mm, oo, N in itertools.product(mans.items(), opts.items(), (-1, 0, 5)):
        yield 'gm_optim_step', label(mm, oo) + f' {N}', lambda m=mm[1], o=oo[1], N=N: lib.gm_optim_step(
            ref(m), ref(o), None, None, None, None, N, None)
        for op in range(-1, 12):
            if oo[0] == 'none':
                yield 'gm_point_op', label(mm) + f' {op} {N}', lambda m=mm[1], op=op, N=N: lib.gm_point_op(
                    ref(m), op, None, None, None, None, N, None)

    peers = {'none': None}
    for w, r, row_lo, epoch, n_acc in itertools.product((0, 1, 2, 9), (-1, 0, 2), (-1, 0), (0, 1), (-1, 0, 65)):
        t = L.Peers()
        t.world, t.rank, t.row_lo, t.epoch, t.n_acc = w, r, row_lo, epoch, n_acc
        peers[f'w{w} r{r} lo{row_lo} e{epoch} a{n_acc}'] = t
    for pe in peers.items():
        for phase in (-1, 0, 1, 2):
            yield 'gm_peer_barrier', label(pe) + f' {phase}', lambda t=pe[1], ph=phase: lib.gm_peer_barrier(
                ref(t), ph, None)
    for mm, oo, pe, N in itertools.product(small.items(), opts.items(), peers.items(), (0, 4)):
        yield 'gm_optim_step_peer', label(mm, oo, pe) + f' {N}', lambda m=mm[1], o=oo[1], t=pe[1], N=N: \
            lib.gm_optim_step_peer(ref(m), ref(o), ref(t), None, None, N, None)

    # (N, n_perm, batch_nodes, max_steps): valid, then one of them out of range
    sizes = ((10, 10, 4, 3), (0, 10, 4, 3), (10, -1, 4, 3), (10, 10, 1, 3), (10, 10, 4, -1))
    ep_mans = {k: mans[k] for k in ('none', 'spd4', 'lor5', 'spd11', 'uni4')}
    n_steps = c.c_int64(0)
    for mm, oo, tt, ll, sz, ns in itertools.product(ep_mans.items(), opts.items(), ep_tgts.items(), loss4.items(),
                                                    sizes, (0, 1)):
        yield 'gm_train_epoch', label(mm, oo, tt, ll) + f' {sz} {ns}', \
            lambda m=mm[1], o=oo[1], t=tt[1], lo=ll[1], sz=sz, ns=ns: lib.gm_train_epoch(
                ref(m), ref(o), None, None, None, None, sz[0], None, 0, sz[1], sz[2], 2, ref(t), ref(lo), 1.0, None,
                sz[3], c.byref(n_steps) if ns else None, None)
    opt_lists = {'sgd': (L.Optim * 8)(*[opts['sgd']] * 8), 'adam0': (L.Optim * 8)(*[opts['adam0']] * 8),
                 'kind2': (L.Optim * 8)(*[opts['kind2']] * 8)}
    for ff, oo, tt, ll, sz in itertools.product(factor_lists.items(), opt_lists.items(),
                                                {k: tgts[k] for k in ('none', 't1', 't0')}.items(),
                                                {k: losses[k] for k in ('none', 'l011')}.items(), sizes):
        yield 'gm_train_epoch_product', label(ff, oo, tt, ll) + f' {sz}', \
            lambda F=ff[1], o=oo[1], t=tt[1], lo=ll[1], sz=sz: lib.gm_train_epoch_product(
                F[0], F[1], o, vp8(), vp8(), vp8(), vp8(), sz[0], None, 0, sz[1], sz[2], 2, ref(t), ref(lo), sp8, vp8(),
                None, None, sz[3], c.byref(n_steps), None)
    for which in range(10):
        args = [factor_lists['spd+lor'][1], opt_lists['sgd'], vp8(), vp8(), vp8(), vp8(), tgts['t1'], losses['l011'],
                sp8, vp8()]
        args[which] = None
        yield 'gm_train_epoch_product', f'null{which}', lambda a=args: lib.gm_train_epoch_product(
            2, a[0], a[1], a[2], a[3], a[4], a[5], 10, None, 0, 10, 4, 2, ref(a[6]), ref(a[7]), a[8], a[9], None, None,
            3, c.byref(n_steps), None)


def _request_codes():
    """{entry point: one character per request of the grid} and the launch count afterwards."""
    from graphembed import _lib as L
    lib = L.lib()
    codes, labels = {}, {}
    for name, lab, call in _request_grid(L, lib):
        codes.setdefault(name, []).append(_CODE_CHARS.get(call(), 'X'))
        labels.setdefault(name, []).append(lab)
    return {k: ''.join(v) for k, v in codes.items()}, labels, int(lib.gm_launch_count())


def test_request_codes_match_the_recorded_table():
    """Each entry point returns, for every request of the grid, the code recorded in tests/golden: check order and
    error codes are part of the C ABI."""
    import json
    import subprocess
    import sys
    env = dict(os.environ, CUDA_VISIBLE_DEVICES='')
    out = subprocess.run([sys.executable, os.path.abspath(__file__), '--dump'], env=env, capture_output=True,
                         text=True, check=True).stdout
    got = json.loads(out.splitlines()[-1])
    assert got['launches'] == 0
    want = json.load(open(GOLDEN_CODES))['codes']
    assert sorted(got['codes']) == sorted(want)
    for name, codes in want.items():
        bad = [(got['labels'][name][i], codes[i], got['codes'][name][i])
               for i in range(len(codes)) if got['codes'][name][i] != codes[i]]
        assert len(got['codes'][name]) == len(codes) and not bad, (name, bad[:10])


if __name__ == '__main__':
    # `python tests/test_cabi.py` rewrites the recorded table; `--dump` prints this build's codes as one JSON line
    import json
    import sys
    for p in (os.path.join(ROOT, 'matrix-manifolds_b200'),):
        sys.path.insert(0, p)
    codes, labels, launches = _request_codes()
    if '--dump' in sys.argv:
        print(json.dumps({'codes': codes, 'labels': labels, 'launches': launches}))
    else:
        assert launches == 0
        with open(GOLDEN_CODES, 'w') as f:
            json.dump({'legend': {v: k for k, v in _CODE_CHARS.items()}, 'codes': codes}, f, indent=0)
            f.write('\n')
