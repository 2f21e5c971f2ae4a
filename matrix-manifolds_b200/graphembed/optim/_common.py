"""Shared plumbing of the two Riemannian optimizers: resolve the manifold of a
parameter and launch the fused in-place update kernel (gm_optim_step)."""
import torch

from .. import _lib as L
from .. import _ops
from .. import _torch_ops


def spec_of(param):
    """ManifoldSpec of a parameter.  Plain tensors are treated like the reference treats them, as
    Euclidean(1): every op is elementwise except the norm, taken over the last axis
    (optim/radam.py:62-65, optim/rsgd.py:56-59)."""
    manifold = getattr(param, 'manifold', None)
    if manifold is not None and hasattr(manifold, 'spec'):
        return manifold.spec, manifold
    last = param.shape[-1] if param.ndim > 0 else 1
    return _ops.ManifoldSpec(L.GM_EUCLIDEAN, last, point_shape=(last,)), None


def fused_step(param, grad, cfg, buf1=None, buf2=None):
    spec, manifold = spec_of(param)
    cfg.grassmann_retr_qr = int(getattr(manifold, 'retr_kind', 'svd') == 'qr')
    # a training loop that owns the gradient buffer (engine.ShardedPairTrainer) lets the update kernel hand it back zeroed
    cfg.zero_grad = int(getattr(param, '_gm_zero_grad_after_step', False) and grad.is_contiguous()
                        and grad.dtype == param.dtype)
    with torch.no_grad():
        arena = getattr(param, '_gm_peer_arena', None)
        if arena is not None:  # multi-GPU owner update over NVLink peer memory (graphembed.parallel.PeerArena):
            # `param` aliases the owned rows of arena.x; the gradient is the sum of every rank's arena.grad rows
            _ops.optim_step_peer(spec, cfg, arena, param.shape[0], buf1, buf2)
        elif spec.kind == L.GM_UNIVERSAL or grad.dtype != param.dtype or not grad.is_contiguous():
            _ops.optim_step(spec, cfg, param.data, grad, buf1, buf2)  # needs the curvature tensor / a gradient copy
        else:  # the registered custom op torch.ops.graphembed_b200.optim_step
            _torch_ops.optim_step(spec, cfg, param.data, grad, buf1, buf2)
    # The kernel wrote through the raw pointer: neither tensor._version nor data_ptr() changed, so anything cached
    # against them (modules._softplus_value: the host copy of softplus(scale)) must be dropped explicitly.
    if getattr(param, '_gm_softplus', None) is not None:
        param._gm_softplus = None
