"""``torch.autograd.Function`` custom ops over the C ABI (``include/dair_pll_b200.h``).

These are the seam between the unchanged Python host API
(:class:`dair_pll_b200.multibody_learnable_system.MultibodyLearnableSystem`) and the
sm_100a kernels.  Tensors must be CUDA, contiguous, fp64 or fp32; there is no CPU path.
"""
from collections import namedtuple
from typing import Optional, Tuple

import torch
from torch import Tensor

from dair_pll_b200 import _lib

_SUFFIX = {torch.float64: 'f64', torch.float32: 'f32'}
_workspaces = {}


def _workspace(device: torch.device, stream: int) -> Tensor:
    """Per-(device, stream) scratch for the gradient reduction (the library never allocates)."""
    key = (device.index, stream)
    ws = _workspaces.get(key)
    if ws is None:
        ws = torch.empty(_lib.load().dpll_workspace_bytes(), dtype=torch.uint8, device=device)
        _workspaces[key] = ws
    return ws


def _call(name: str, device, *args, dtype: Optional[torch.dtype] = None, workspace: bool = False) -> None:
    """Calls the C entry point ``name`` -- ``name_f64`` / ``name_f32`` when ``dtype`` is given -- on ``device``'s current
    stream, which every entry point takes last; tensors are passed as their data pointers, ``None`` as NULL.  With
    ``workspace`` the device's scratch buffer and its size go before the stream.  A non-zero return code raises.
    ``args`` stays referenced until the entry point has been enqueued: callers pass temporaries (casts, contiguous
    copies) inline, and the caching allocator must not hand their memory out before the launch is on the stream."""
    if dtype is not None:
        name = f'{name}_{_SUFFIX[dtype]}'
    ptrs = [a.data_ptr() if isinstance(a, Tensor) else a for a in args]
    with torch.cuda.device(device):
        stream = torch.cuda.current_stream().cuda_stream
        if workspace:
            ws = _workspace(device, stream)
            ptrs += [ws.data_ptr(), ws.numel()]
        _lib.check(getattr(_lib.load(), name)(*ptrs, stream), name)


def set_loss_variant(variant: int) -> None:
    """Selects the cube loss kernel: 0 = warp-level wavefront kernel, static sample ranges (default; bitwise
    reproducible), 1 = one sample per thread (A/B measurements), 2 = wavefront kernel with dynamic sample distribution
    (faster by the load imbalance, gradient sums reproducible only to rounding).  The elbow loss always runs its
    wavefront kernel."""
    # a process-wide setting, not a launch: no device and no stream, so not through _call
    _lib.check(_lib.load().dpll_set_loss_variant(variant), 'dpll_set_loss_variant')


def _check_inputs(*tensors: Optional[Tensor], f64_only: Optional[str] = None) -> torch.dtype:
    """The common dtype of the CUDA tensors given (``None`` entries are skipped); ``f64_only``: the message of the
    TypeError raised when it is not float64."""
    tensors = [t for t in tensors if t is not None]
    dtype = tensors[0].dtype
    if dtype not in _SUFFIX:
        raise TypeError(f'dair_pll_b200 kernels support float64/float32, got {dtype}')
    for t in tensors:
        if not t.is_cuda:
            raise RuntimeError('dair_pll_b200 has no CPU path: tensors must live on a CUDA device')
        if t.dtype != dtype:
            raise TypeError(f'mixed dtypes: {t.dtype} vs {dtype}')
    if f64_only is not None and dtype != torch.float64:
        raise TypeError(f64_only)
    return dtype


def _check_states(n_x: int, x: Tensor, x_plus: Optional[Tensor] = None) -> None:
    if x.dim() != 2 or x.shape[1] != n_x or (x_plus is not None and x_plus.shape != x.shape):
        got = tuple(x.shape) if x_plus is None else f'{tuple(x.shape)} / {tuple(x_plus.shape)}'
        raise ValueError(f'expected (B,{n_x}) states, got {got}')


_Like = namedtuple('_Like', 'shape dtype')      # what _split reads of a tensor


def _split(g: Tensor, *like) -> list:
    """Consecutive pieces of the flat gradient ``g``, one per tensor (or :class:`_Like`) of ``like``, with its shape and
    dtype."""
    out, off = [], 0
    for t in like:
        n = t.shape.numel()
        out.append(g[off:off + n].reshape(t.shape).to(t.dtype))
        off += n
    return out


def _fused_grad(grad: Tensor, grad_loss: Tensor, rerun) -> Tensor:
    """Parameter gradient of sum_b grad_loss[b] loss_b for a loss whose forward launch already returned
    ``grad`` = d(sum_b loss_b)/d params (envelope theorem).  A stride-0 upstream gradient (``loss.sum()``) is provably
    uniform: one scale.  Otherwise (``loss.mean()`` materialises its uniform gradient) uniformity is decided on the
    DEVICE: ``rerun(weight, skip_flag, grad_out)`` launches the weighted pass, which the kernel skips when the int32
    ``skip_flag`` is set, and the scaled fused gradient is selected.  No host read, so the backward can be captured
    into a CUDA graph."""
    if grad_loss.numel() == 0:
        return torch.zeros_like(grad)
    if grad_loss.dim() == 1 and grad_loss.stride(0) == 0:
        return grad * grad_loss[0]
    grad_loss = grad_loss.contiguous()
    lo, hi = torch.aminmax(grad_loss)
    uniform = lo == hi
    gw = torch.zeros_like(grad)
    rerun(grad_loss, uniform.to(torch.int32), gw)
    return torch.where(uniform, grad * lo, gw)


def _f64(t: Optional[Tensor]) -> Optional[Tensor]:
    return None if t is None else t.detach().to(torch.float64).contiguous()


def _summed_backward(name: str, x: Tensor, params, widths, *args, steps: int = 1):
    """Backward through a rollout or step entry point ``name`` that writes PER-SAMPLE gradients: it is called with
    ``args`` (tensors cast to contiguous float64) followed by zeroed float64 (B, w) buffers, one per entry of
    ``widths``, the parameter gradient first; an empty batch or rollout launches nothing.  Returns the parameter
    gradient summed over the batch and split as ``params``, then the other buffers."""
    B = x.shape[0]
    bufs = [torch.zeros((B, w), dtype=torch.float64, device=x.device) for w in widths]
    if B > 0 and steps > 0:
        _call(name, x.device, *(_f64(a) if isinstance(a, Tensor) else a for a in args), *bufs)
    return (*_split(bufs[0].sum(0), *params), *bufs[1:])


def cube_loss_raw(x: Tensor, x_plus: Tensor, inertia: Tensor, mu_pair: Tensor, half: Tensor, dt: float,
                  eps: float, weight: Optional[Tensor] = None, want_grad: bool = True,
                  want_force: bool = False, want_iters: bool = False, want_loss: bool = True,
                  skip_flag: Optional[Tensor] = None, grad_out: Optional[Tensor] = None):
    """Direct call of ``dpll_cube_loss_*``.  x, x_plus (B,13).  Returns
    (loss (B,), grad (14,) | None, loss_sum (1,), force (B,12) | None, iters (B,) | None)."""
    dtype = _check_inputs(x, x_plus, inertia, mu_pair, half)
    x, x_plus = x.contiguous(), x_plus.contiguous()
    inertia, mu_pair, half = inertia.contiguous(), mu_pair.contiguous(), half.contiguous()
    _check_states(13, x, x_plus)
    if inertia.numel() != 10 or mu_pair.numel() != 1 or half.numel() != 3:
        raise ValueError('cube parameters must be inertia (10), mu_pair (1), half (3)')
    B = x.shape[0]
    dev = x.device
    loss = torch.empty(B, dtype=dtype, device=dev) if want_loss else None
    grad = (grad_out if grad_out is not None else torch.empty(14, dtype=dtype, device=dev)) if want_grad else None
    loss_sum = torch.empty(1, dtype=dtype, device=dev)
    force = torch.empty((B, 12), dtype=dtype, device=dev) if want_force else None
    iters = torch.empty(B, dtype=torch.int32, device=dev) if want_iters else None
    if weight is not None:
        weight = weight.to(dtype).contiguous()
    _call('dpll_cube_loss', dev, x, x_plus, weight, inertia, mu_pair, half, dt, eps, B, loss, force, iters, grad, loss_sum,
          skip_flag, dtype=dtype, workspace=True)
    return loss, grad, loss_sum, force, iters


class CubeContactNetsLoss(torch.autograd.Function):
    """loss (B,) = ContactNets loss of the cube; differentiable w.r.t. the callable-level
    parameters (inertia 10-vector, combined friction, box half lengths).  x and x_plus are
    data (no gradient), as in the reference's training loop (drake_experiment.py:202-224).

    The backward is fused into the forward kernel (envelope theorem,
    multibody_learnable_system.py:172-175): the forward launch already returns
    d(sum_b loss_b)/d params.  When the upstream gradient is uniform (``loss.sum()`` /
    ``loss.mean()``) the backward is a 14-element scale; otherwise the kernel is re-run with
    per-sample weights.  Uniformity is decided on the device (skip flag), never by a host sync.
    """

    @staticmethod
    def forward(ctx, x, x_plus, inertia, mu_pair, half, dt, eps):
        need = any(ctx.needs_input_grad[2:5])
        loss, grad, _, _, _ = cube_loss_raw(x, x_plus, inertia, mu_pair, half, dt, eps, want_grad=need)
        ctx.dt, ctx.eps = dt, eps
        if need:
            ctx.save_for_backward(grad, x, x_plus, inertia, mu_pair, half)
        return loss

    @staticmethod
    def backward(ctx, grad_loss):
        grad, x, x_plus, inertia, mu_pair, half = ctx.saved_tensors
        g = _fused_grad(grad, grad_loss, lambda w, skip, out: cube_loss_raw(
            x, x_plus, inertia, mu_pair, half, ctx.dt, ctx.eps, weight=w, want_loss=False, skip_flag=skip, grad_out=out))
        return (None, None, *_split(g, inertia, mu_pair, half), None, None)


LOSS_DYNAMIC = 1     # DPLL_LOSS_DYNAMIC (include/dair_pll_b200.h)
LOSS_RACE = 2        # DPLL_LOSS_RACE: the head of a cost-ordered batch is solved by the racing kernel (small launches)


def _rows(t: Tensor, n_x: int):
    """(B, n_x) tensor -> (tensor, row stride in elements); rows must be contiguous, their spacing is free (so
    the training loop's ``x_past[..., -1, :]`` views, drake_experiment.py:217-218, are read in place)."""
    if t.dim() != 2 or t.shape[1] != n_x:
        raise ValueError(f'expected (B,{n_x}) states, got {tuple(t.shape)}')
    if t.shape[0] > 1 and (t.stride(1) != 1 or t.stride(0) < n_x):
        t = t.contiguous()
    elif t.shape[0] <= 1 and t.stride(1) != 1:
        t = t.contiguous()
    return t, (t.stride(0) if t.shape[0] > 1 else n_x)


def cube_loss_leaf_raw(x: Tensor, x_plus: Tensor, theta: Tensor, friction: Tensor, length: Tensor, dt: float,
                       eps: float, weight: Optional[Tensor] = None, want_grad: bool = True, want_loss: bool = True,
                       skip_flag: Optional[Tensor] = None, grad_out: Optional[Tensor] = None):
    """Direct call of ``dpll_cube_loss_leaf_*``: parameters are the module's learnable leaves
    (theta (1,10), friction_params (2,) [box, ground], length_params (1,3)).  Returns
    (loss (B,) | None, grad_leaf (15,) | None, loss_sum (1,))."""
    dtype = _check_inputs(x, x_plus, theta, friction, length)
    x, x_plus = x.contiguous(), x_plus.contiguous()
    theta, friction, length = theta.contiguous(), friction.contiguous(), length.contiguous()
    _check_states(13, x, x_plus)
    if theta.numel() != 10 or friction.numel() != 2 or length.numel() != 3:
        raise ValueError('cube leaves must be theta (10), friction_params (2), length_params (3)')
    B = x.shape[0]
    dev = x.device
    loss = torch.empty(B, dtype=dtype, device=dev) if want_loss else None
    grad = (grad_out if grad_out is not None else torch.empty(15, dtype=dtype, device=dev)) if want_grad else None
    loss_sum = torch.empty(1, dtype=dtype, device=dev)
    if weight is not None:
        weight = weight.to(dtype).contiguous()
    _call('dpll_cube_loss_leaf', dev, x, x_plus, weight, theta, friction, length, dt, eps, B, loss, None, None, grad,
          loss_sum, skip_flag, dtype=dtype, workspace=True)
    return loss, grad, loss_sum


def cube_loss_leaf_dp_raw(x: Tensor, x_plus: Tensor, theta: Tensor, friction: Tensor, length: Tensor, dt: float,
                          eps: float, flags: int = 0, comm=None, want_loss: bool = True, want_iters: bool = False,
                          u_init: Optional[Tensor] = None, want_u: bool = False):
    """Direct call of ``dpll_cube_loss_leaf_dp_*`` (the training-loop / data-parallel form).  x, x_plus: (B,13)
    with any row stride.  ``comm``: a :class:`dair_pll_b200.parallel.PeerComm` or None.  Returns
    (loss (B,) | None, sums (17,) = [grad_leaf 15 | loss sum | count], means (16,), local (16,), iters | None
    [, u (B,6) if ``want_u``]); with a communicator ``sums`` / ``means`` cover all ranks, ``local`` is this rank's
    share.  ``u_init`` (B,6): warm start of every sample's Newton solve (e.g. last epoch's ``u``)."""
    dtype = _check_inputs(x, x_plus, theta, friction, length)
    x, ldx = _rows(x, 13)
    x_plus, ldxp = _rows(x_plus, 13)
    if x_plus.shape != x.shape:
        raise ValueError(f'x {tuple(x.shape)} and x_plus {tuple(x_plus.shape)} differ')
    theta, friction, length = theta.contiguous(), friction.contiguous(), length.contiguous()
    if theta.numel() != 10 or friction.numel() != 2 or length.numel() != 3:
        raise ValueError('cube leaves must be theta (10), friction_params (2), length_params (3)')
    B, dev = x.shape[0], x.device
    loss = torch.empty(B, dtype=dtype, device=dev) if want_loss else None
    iters = torch.empty(B, dtype=torch.int32, device=dev) if want_iters else None
    out = torch.empty(49, dtype=dtype, device=dev)
    sums, means, local = out[0:17], out[17:33], out[33:49]
    if u_init is not None:
        if tuple(u_init.shape) != (B, 6):
            raise ValueError(f'u_init must be (B,6), got {tuple(u_init.shape)}')
        u_init = u_init.to(dtype).contiguous()
    # with a warm start the optima are written back IN PLACE (every sample reads its row before it writes it): a
    # training loop keeps one (B, 6) buffer per batch and nothing is copied between epochs
    u_out = (u_init if u_init is not None else torch.empty((B, 6), dtype=dtype, device=dev)) if want_u else None
    _call('dpll_cube_loss_leaf_dp', dev, x, ldx, x_plus, ldxp, theta, friction, length, dt, eps, B, flags,
          comm.handle if comm is not None else None, u_init, u_out, loss, iters, sums, means, local, dtype=dtype,
          workspace=True)
    if want_u:
        return loss, sums, means, local, iters, u_out
    return loss, sums, means, local, iters


class CubeContactNetsLossLeaf(torch.autograd.Function):
    """ContactNets loss of the cube as a function of the module's learnable LEAVES: parameter
    preparation and its chain rule run inside the CUDA library (``dpll_cube_loss_leaf_dp_*``), so
    forward + backward is three kernel launches and no PyTorch glue.  Same backward protocol as
    :class:`CubeContactNetsLoss` (fused gradient from the forward launch; device-side skip flag).

    With a communicator (data-parallel step) the gradient this Function returns is the SUM over ranks of every
    rank's vector-Jacobian product -- i.e. the gradient of the sum over ranks of each rank's scalar objective --
    identical bits on every rank.  For ``mean()`` / ``sum()`` of the returned :class:`BatchLoss` the exchange
    happens inside the forward launch's reduction kernel; a general upstream gradient is summed with the
    stand-alone peer all-reduce."""

    @staticmethod
    def forward(ctx, x, x_plus, theta, friction, length, dt, eps, flags, comm, want_iters, u_init=None, want_u=False):
        out = cube_loss_leaf_dp_raw(x, x_plus, theta, friction, length, dt, eps, flags=flags, comm=comm,
                                    want_iters=want_iters, u_init=u_init, want_u=want_u)
        loss, sums, means, local, iters = out[:5]
        # (a warm-start buffer is updated in place and not returned through autograd)
        usol = out[5] if (want_u and u_init is None) else torch.empty(0, dtype=loss.dtype, device=loss.device)
        ctx.dt, ctx.eps, ctx.comm = dt, eps, comm
        if any(ctx.needs_input_grad[2:5]):
            ctx.save_for_backward(local, x, x_plus, theta, friction, length)
        if iters is None:
            iters = torch.empty(0, dtype=torch.int32, device=loss.device)
        # the launch's own (global) sums and means, for BatchLoss.mean() / .sum()
        ctx.mark_non_differentiable(sums, means, iters, usol)
        return loss, sums, means, iters, usol

    @staticmethod
    def backward(ctx, grad_loss, _g_sums, _g_means, _g_iters, _g_u):
        local, x, x_plus, theta, friction, length = ctx.saved_tensors
        g = _fused_grad(local[:15], grad_loss, lambda w, skip, out: cube_loss_leaf_raw(
            x, x_plus, theta, friction, length, ctx.dt, ctx.eps, weight=w, want_loss=False, skip_flag=skip, grad_out=out))
        if ctx.comm is not None:
            g = ctx.comm.all_reduce_sum(g)
        return (None, None, *_split(g, theta, friction, length), None, None, None, None, None, None, None)


class _FusedReduction(torch.autograd.Function):
    """``mean()`` / ``sum()`` of a batch loss taken from the kernel launch that produced it: ``vec`` is the
    launch's [parameter gradient (n) | loss] already summed (or averaged) over the batch -- and over the ranks of
    a data-parallel step --, so the value is a copy of its last element and the backward one scale: no reduction
    over the (B,) loss, no (B,) upstream gradient, no second launch, no collective."""

    @staticmethod
    def forward(ctx, vec, n, *leaves):
        ctx.save_for_backward(vec)
        ctx.n = n
        # only the leaves' shapes and dtypes are kept: the backward does not hold the leaves themselves (nor trip on
        # their version counters if they are updated before it runs)
        ctx.leaves = [_Like(l.shape, l.dtype) for l in leaves]
        return vec[n].clone()

    @staticmethod
    def backward(ctx, g):
        (vec,) = ctx.saved_tensors
        return (None, None, *_split(vec[:ctx.n] * g, *ctx.leaves))


_INPLACE_DUNDERS = {'__iadd__', '__isub__', '__imul__', '__itruediv__', '__ifloordiv__', '__ipow__', '__imod__',
                    '__setitem__'}


class BatchLoss(torch.Tensor):
    """The (*,) loss tensor the module returns: an ordinary tensor whose argument-free ``mean()`` / ``sum()``
    -- what the reference's training loop applies to it (drake_experiment.py:222-223) -- come from the launch
    that produced the losses (:class:`_FusedReduction`).  Every other operation behaves as on a plain tensor
    (and returns plain tensors); in-place modification switches the shortcut off."""

    @classmethod
    def __torch_function__(cls, func, types, args=(), kwargs=None):
        kwargs = kwargs or {}
        name = getattr(func, '__name__', '')
        self = args[0] if args else None
        fused = getattr(self, '_dpll_fused', None) if isinstance(self, BatchLoss) else None
        if fused is not None and name in ('mean', 'sum') and len(args) == 1 and not kwargs:
            sums, means, n, leaves = fused
            return _FusedReduction.apply(means if name == 'mean' else sums, n, *leaves)
        if fused is not None and (name in _INPLACE_DUNDERS or (name.endswith('_') and not name.endswith('__'))):
            self._dpll_fused = None
        with torch._C.DisableTorchFunctionSubclass():
            return func(*args, **kwargs)


def batch_loss(loss: Tensor, sums: Tensor, means: Tensor, n: int, leaves, iters: Optional[Tensor] = None) -> Tensor:
    """Wraps the per-sample loss with the launch's [gradient (n) | loss] sums and means (see :class:`BatchLoss`);
    ``newton_iters`` (B,) int32, when recorded, is the cost hint the data set orders its batches by."""
    out = loss.as_subclass(BatchLoss)
    out._dpll_fused = (sums, means, n, tuple(leaves))
    out.newton_iters = iters
    out.qp_solution = None
    return out


def cube_rollout(x0: Tensor, inertia: Tensor, mu_pair: Tensor, half: Tensor, dt: float, steps: int,
                 eps: float = 1e-4, want_force: bool = False,
                 iters_out: Optional[Tensor] = None) -> Tuple[Tensor, Optional[Tensor]]:
    """(B,13) -> trajectory (B, steps+1, 13) through ``dpll_cube_rollout_*`` (no autograd).  ``iters_out``
    (B,) int32, optional: total Newton iterations of every toss."""
    dtype = _check_inputs(x0, inertia, mu_pair, half)
    x0 = x0.contiguous()
    _check_states(13, x0)
    B = x0.shape[0]
    traj = torch.empty((B, steps + 1, 13), dtype=dtype, device=x0.device)
    force = torch.empty((B, steps, 12), dtype=dtype, device=x0.device) if want_force else None
    _call('dpll_cube_rollout', x0.device, x0, inertia.contiguous(), mu_pair.contiguous(), half.contiguous(), dt, eps, B,
          steps, traj, force, iters_out, dtype=dtype)
    return traj, force


def elbow_loss_raw(x: Tensor, x_plus: Tensor, inertia: Tensor, mu_pair: Tensor, half: Optional[Tensor], kin: Tensor,
                   dt: float, eps: float, weight: Optional[Tensor] = None, want_grad: bool = True,
                   want_force: bool = False, want_iters: bool = False, want_loss: bool = True,
                   skip_flag: Optional[Tensor] = None, grad_out: Optional[Tensor] = None,
                   pts: Optional[Tensor] = None, want_grad_pts: bool = False, flags: int = 0):
    """Direct call of ``dpll_elbow_loss_*`` (``flags``: LOSS_DYNAMIC for cost-ordered batches).  x, x_plus (B,15); inertia (20), mu_pair (2), half (6) or
    witness points pts (B,8,3), kin (12).  Returns (loss (B,) | None, grad (28,) | None, loss_sum (1,),
    force (B,24) | None, iters (B,) | None[, grad_pts (B,8,3)])."""
    dtype = _check_inputs(x, x_plus, inertia, mu_pair, kin, half, pts)
    x, x_plus = x.contiguous(), x_plus.contiguous()
    inertia, mu_pair, kin = inertia.contiguous(), mu_pair.contiguous(), kin.contiguous()
    half = half.contiguous() if half is not None else None
    pts = pts.contiguous() if pts is not None else None
    _check_states(15, x, x_plus)
    if inertia.numel() != 20 or mu_pair.numel() != 2 or kin.numel() != 12 or (half is not None and half.numel() != 6):
        raise ValueError('elbow parameters must be inertia (20), mu_pair (2), half (6), kin (12)')
    if half is None and pts is None:
        raise ValueError('either half lengths (boxes) or witness points (learned geometry) are required')
    if pts is not None and tuple(pts.shape) != (x.shape[0], 8, 3):
        raise ValueError(f'pts must be (B,8,3), got {tuple(pts.shape)}')
    B = x.shape[0]
    dev = x.device
    loss = torch.empty(B, dtype=dtype, device=dev) if want_loss else None
    grad = (grad_out if grad_out is not None else torch.empty(28, dtype=dtype, device=dev)) if want_grad else None
    loss_sum = torch.empty(1, dtype=dtype, device=dev)
    force = torch.empty((B, 24), dtype=dtype, device=dev) if want_force else None
    iters = torch.empty(B, dtype=torch.int32, device=dev) if want_iters else None
    if weight is not None:
        weight = weight.to(dtype).contiguous()
    grad_pts = torch.zeros((B, 8, 3), dtype=dtype, device=dev) if (want_grad_pts and want_grad) else None
    _call('dpll_elbow_loss', dev, x, x_plus, weight, inertia, mu_pair, half, kin, pts, dt, eps, B, flags, loss, force,
          grad_pts, iters, grad, loss_sum, skip_flag, dtype=dtype, workspace=True)
    if want_grad_pts:
        return loss, grad, loss_sum, force, iters, grad_pts
    return loss, grad, loss_sum, force, iters


class ElbowContactNetsLoss(torch.autograd.Function):
    """ContactNets loss of the elbow (floating base + hinge, two boxes); differentiable w.r.t. the
    callable-level parameters (two inertia 10-vectors, two pair frictions, two half-length triples).
    Same fused-backward protocol as :class:`CubeContactNetsLoss`; also returns the launch's
    [gradient (28) | loss] sums and means for :class:`BatchLoss`."""

    @staticmethod
    def forward(ctx, x, x_plus, inertia, mu_pair, half, kin, dt, eps, flags=0, want_iters=False):
        need = any(ctx.needs_input_grad[2:5])
        loss, grad, loss_sum, _, iters = elbow_loss_raw(x, x_plus, inertia, mu_pair, half, kin, dt, eps, want_grad=need,
                                                        want_iters=want_iters, flags=flags)
        ctx.dt, ctx.eps = dt, eps
        if need:
            ctx.save_for_backward(grad, x, x_plus, inertia, mu_pair, half, kin)
        else:
            grad = torch.zeros(28, dtype=loss.dtype, device=loss.device)
        sums = torch.cat((grad, loss_sum))
        means = sums / max(loss.numel(), 1) if loss.numel() > 0 else sums * float('nan')
        if iters is None:
            iters = torch.empty(0, dtype=torch.int32, device=loss.device)
        ctx.mark_non_differentiable(sums, means, iters)
        return loss, sums, means, iters

    @staticmethod
    def backward(ctx, grad_loss, _g_sums, _g_means, _g_iters):
        grad, x, x_plus, inertia, mu_pair, half, kin = ctx.saved_tensors
        g = _fused_grad(grad, grad_loss, lambda w, skip, out: elbow_loss_raw(
            x, x_plus, inertia, mu_pair, half, kin, ctx.dt, ctx.eps, weight=w, want_loss=False, skip_flag=skip, grad_out=out))
        return (None, None, *_split(g, inertia, mu_pair, half), None, None, None, None, None)


class ElbowContactNetsLossPts(torch.autograd.Function):
    """ContactNets loss of the elbow with LEARNED geometry: the 4 + 4 witness points ``pts`` (B,8,3) come
    from the support-function networks (``DeepSupportConvex.get_vertices``).  Differentiable w.r.t.
    inertia (20), mu_pair (2) and ``pts``; the per-sample d loss_b / d pts[b] is produced by the forward
    launch and scaled by the upstream gradient (exact for any upstream weights)."""

    @staticmethod
    def forward(ctx, x, x_plus, inertia, mu_pair, pts, kin, dt, eps):
        need = any(ctx.needs_input_grad[2:5])
        out = elbow_loss_raw(x, x_plus, inertia, mu_pair, None, kin, dt, eps, want_grad=need, pts=pts,
                             want_grad_pts=True)
        loss, grad, gpts = out[0], out[1], out[5]
        ctx.dt, ctx.eps = dt, eps
        if need:
            ctx.save_for_backward(grad, gpts, x, x_plus, inertia, mu_pair, pts, kin)
        return loss

    @staticmethod
    def backward(ctx, grad_loss):
        grad, gpts, x, x_plus, inertia, mu_pair, pts, kin = ctx.saved_tensors
        g = _fused_grad(grad, grad_loss, lambda w, skip, out: elbow_loss_raw(
            x, x_plus, inertia, mu_pair, None, kin, ctx.dt, ctx.eps, weight=w, want_loss=False, skip_flag=skip,
            grad_out=out, pts=pts))
        return (None, None, *_split(g, inertia, mu_pair), gpts * grad_loss.reshape(-1, 1, 1), None, None, None)


def elbow_rollout_saved(x0: Tensor, inertia: Tensor, mu_pair: Tensor, half: Optional[Tensor], kin: Tensor, dt: float,
                        steps: int, eps: float = 1e-4, pts: Optional[Tensor] = None) -> Tuple[Tensor, Tensor]:
    """``dpll_elbow_rollout_saved_f64``: trajectory (B, steps+1, 15) and every step's QP optimum usol (B, steps, 7), which
    the backward (forward-mode tangents) turns into one evaluation per step instead of a dual-number solve.  float64."""
    _check_inputs(x0, inertia, mu_pair, kin)
    B = x0.shape[0]
    traj = torch.empty((B, steps + 1, 15), dtype=torch.float64, device=x0.device)
    usol = torch.empty((B, steps, 7), dtype=torch.float64, device=x0.device)
    _call('dpll_elbow_rollout_saved_f64', x0.device, _f64(x0), _f64(inertia), _f64(mu_pair), _f64(half), _f64(kin), _f64(pts),
          dt, eps, B, steps, traj, usol)
    return traj, usol


def elbow_rollout(x0: Tensor, inertia: Tensor, mu_pair: Tensor, half: Optional[Tensor], kin: Tensor, dt: float,
                  steps: int, eps: float = 1e-4, want_force: bool = False,
                  pts: Optional[Tensor] = None) -> Tuple[Tensor, Optional[Tensor]]:
    """(B,15) -> trajectory (B, steps+1, 15) through ``dpll_elbow_rollout_*`` (no autograd).  With witness
    points ``pts`` (B,8,3) of a learned geometry only a single step is allowed."""
    dtype = _check_inputs(x0, inertia, mu_pair, kin)
    x0 = x0.contiguous()
    _check_states(15, x0)
    B = x0.shape[0]
    traj = torch.empty((B, steps + 1, 15), dtype=dtype, device=x0.device)
    force = torch.empty((B, steps, 24), dtype=dtype, device=x0.device) if want_force else None
    _call('dpll_elbow_rollout', x0.device, x0, inertia.contiguous(), mu_pair.contiguous(),
          half.contiguous() if half is not None else None, kin.contiguous(), pts.contiguous() if pts is not None else None,
          dt, eps, B, steps, traj, force, None, dtype=dtype)
    return traj, force


class CubeRollout(torch.autograd.Function):
    """Differentiable rollout of the learnable cube system: traj (B, steps+1, 13) from x0 (B, 13).
    Forward = ``dpll_cube_rollout_saved_f64`` (keeps every step's QP optimum); backward =
    ``dpll_cube_rollout_backward_f64``, the reverse-mode adjoint: one 6x6 SPD solve per step (implicit
    differentiation of the QP) walking each trajectory backwards -- gradients w.r.t. the callable-level parameters
    and x0, what the reference gets from autograd through ``forward_dynamics`` and sappy's backward
    (multibody_learnable_system.py:293-304) for the prediction loss (experiment.py:230-248).  ``forward_mode=True``
    selects the dual-number backward ``dpll_cube_rollout_grad_f64`` instead (27 tangent rollouts per toss; the
    independent check of the adjoint)."""

    @staticmethod
    def forward(ctx, x0, inertia, mu_pair, half, dt, steps, eps, forward_mode=False):
        B = x0.shape[0]
        a = [_f64(t) for t in (x0, inertia, mu_pair, half)]
        traj = torch.empty((B, steps + 1, 13), dtype=torch.float64, device=x0.device)
        usol = torch.empty((B, steps, 6), dtype=torch.float64, device=x0.device)
        _call('dpll_cube_rollout_saved_f64', x0.device, *a, dt, eps, B, steps, traj, usol)
        ctx.dt, ctx.steps, ctx.eps, ctx.forward_mode = dt, steps, eps, forward_mode
        ctx.save_for_backward(x0, inertia, mu_pair, half, traj, usol)
        return traj.to(x0.dtype)

    @staticmethod
    def backward(ctx, gtraj):
        x0, inertia, mu_pair, half, traj, usol = ctx.saved_tensors
        B, steps, params = x0.shape[0], ctx.steps, (inertia, mu_pair, half)
        if ctx.forward_mode:
            name, start = 'dpll_cube_rollout_grad_f64', (x0,)
        else:
            name, start = 'dpll_cube_rollout_backward_f64', (traj, usol)
        gi, gm, gh, gx0 = _summed_backward(name, x0, params, (14, 13), *start, *params, ctx.dt, ctx.eps, B, steps,
                                           gtraj[:, 1:, :], steps=steps)
        gx = (gx0 + gtraj[:, 0, :].to(torch.float64)).to(x0.dtype)
        return gx, gi, gm, gh, None, None, None, None


class ElbowRollout(torch.autograd.Function):
    """Differentiable rollout of the learnable two-body (elbow) system with box geometries: traj (B, steps+1, 15).
    Backward = ``dpll_elbow_rollout_grad_saved_f64`` (forward-mode tangents, 43 directions per toss; every step's QP
    optimum is kept by the forward, so a dual-number step is one evaluation + one 7x7 solve at it, not a solve)."""

    @staticmethod
    def forward(ctx, x0, inertia, mu_pair, half, kin, dt, steps, eps):
        traj, usol = elbow_rollout_saved(x0, inertia, mu_pair, half, kin, dt, steps, eps)
        ctx.dt, ctx.steps, ctx.eps = dt, steps, eps
        ctx.save_for_backward(x0, inertia, mu_pair, half, kin, usol)
        return traj.to(x0.dtype)

    @staticmethod
    def backward(ctx, gtraj):
        x0, inertia, mu_pair, half, kin, usol = ctx.saved_tensors
        B, steps = x0.shape[0], ctx.steps
        gi, gm, gh, gx0 = _summed_backward('dpll_elbow_rollout_grad_saved_f64', x0, (inertia, mu_pair, half), (28, 15), x0,
                                           inertia, mu_pair, half, kin, usol, ctx.dt, ctx.eps, B, steps, gtraj[:, 1:, :],
                                           steps=steps)
        gx = (gx0 + gtraj[:, 0, :].to(torch.float64)).to(x0.dtype)
        return gx, gi, gm, gh, None, None, None, None


class ElbowStepPts(torch.autograd.Function):
    """ONE differentiable learnable step of the two-body system with learned geometry: x (B,15), witness points pts
    (B,8,3) of the support-function networks -> next state (B,15).  Backward = ``dpll_elbow_step_pts_grad_f64``
    (61 forward-mode directions per sample): cotangents of x, inertia, mu_pair and of the points -- which autograd then
    chains into the network weights through :class:`deep_support_function.ICNNSupport`."""

    @staticmethod
    def forward(ctx, x, inertia, mu_pair, pts, kin, dt, eps):
        traj, usol = elbow_rollout_saved(x, inertia, mu_pair, None, kin, dt, 1, eps, pts=pts)
        ctx.dt, ctx.eps = dt, eps
        ctx.save_for_backward(x, inertia, mu_pair, pts, kin, usol)
        return traj[:, 1].to(x.dtype)

    @staticmethod
    def backward(ctx, gnext):
        x, inertia, mu_pair, pts, kin, usol = ctx.saved_tensors
        gi, gm, gpts, gx = _summed_backward('dpll_elbow_step_pts_grad_f64', x, (inertia, mu_pair), (22, 24, 15), x, inertia,
                                            mu_pair, kin, pts, usol, ctx.dt, ctx.eps, x.shape[0], gnext)
        return gx.to(x.dtype), gi, gm, gpts.reshape(pts.shape).to(pts.dtype), None, None, None


def body_loss_pts_raw(x: Tensor, x_plus: Tensor, inertia: Tensor, mu_pair: Tensor, pts: Tensor, n_contacts: int, dt: float,
                      eps: float, weight: Optional[Tensor] = None, want_grad: bool = True, want_loss: bool = True,
                      want_grad_pts: bool = True, want_iters: bool = False, want_force: bool = False, flags: int = 0,
                      skip_flag: Optional[Tensor] = None, grad_out: Optional[Tensor] = None):
    """Direct call of ``dpll_body_loss_pts_f64`` (``flags``: LOSS_DYNAMIC for cost-ordered batches).  x, x_plus (B,13), inertia
    (10), mu_pair (1), witness points pts (B,4,3) of which the first ``n_contacts`` rows are used.  Returns (loss (B,) | None,
    grad (11,) | None, loss_sum (1,), grad_pts (B,4,3) | None, iters (B,) | None, force (B,12) | None)."""
    _check_inputs(x, x_plus, inertia, mu_pair, pts, f64_only='the witness-point kernels are provided in float64')
    x, x_plus, pts = x.contiguous(), x_plus.contiguous(), pts.contiguous()
    B, dev = x.shape[0], x.device
    _check_states(13, x, x_plus)
    if tuple(pts.shape) != (B, 4, 3):
        raise ValueError(f'pts must be (B,4,3), got {tuple(pts.shape)}')
    loss = torch.empty(B, dtype=x.dtype, device=dev) if want_loss else None
    grad = (grad_out if grad_out is not None else torch.empty(11, dtype=x.dtype, device=dev)) if want_grad else None
    loss_sum = torch.empty(1, dtype=x.dtype, device=dev)
    gpts = torch.empty((B, 4, 3), dtype=x.dtype, device=dev) if want_grad_pts else None
    iters = torch.empty(B, dtype=torch.int32, device=dev) if want_iters else None
    force = torch.empty((B, 12), dtype=x.dtype, device=dev) if want_force else None
    if weight is not None:
        weight = weight.to(x.dtype).contiguous()
    _call('dpll_body_loss_pts_f64', dev, x, x_plus, weight, inertia.contiguous(), mu_pair.contiguous(), pts, n_contacts, dt,
          eps, B, flags, loss, force, gpts, iters, grad, loss_sum, skip_flag, workspace=True)
    return loss, grad, loss_sum, gpts, iters, force


class BodyWitnessPointLoss(torch.autograd.Function):
    """ContactNets loss of a single floating body whose contact set is given by witness points ``pts`` (B,4,3)
    (first ``n_contacts`` rows used) -- Sphere, Polygon, DeepSupportConvex, any plane-convex pair: ``dpll_body_loss_pts_f64``,
    the wavefront kernel.  Differentiable w.r.t. inertia (10), mu_pair (1) and ``pts``; float64.  Returns (loss, iters):
    ``iters`` (B,) int32 Newton directions per sample when ``want_iters``, else empty.  Backward: a uniform upstream
    gradient scales the forward's own sums; other weights take one weighted pass, which the device skips
    (``skip_flag``) when they are uniform after all -- no host read, so the step can be captured into a CUDA graph."""

    @staticmethod
    def forward(ctx, x, x_plus, inertia, mu_pair, pts, n_contacts, dt, eps, flags=0, want_iters=False):
        loss, grad, _, gpts, iters, _ = body_loss_pts_raw(x, x_plus, inertia, mu_pair, pts, n_contacts, dt, eps, flags=flags,
                                                          want_iters=want_iters)
        ctx.args = (n_contacts, dt, eps, flags)
        ctx.save_for_backward(grad, gpts, x, x_plus, inertia, mu_pair, pts)
        if iters is None:
            iters = torch.empty(0, dtype=torch.int32, device=loss.device)
        ctx.mark_non_differentiable(iters)
        return loss, iters

    @staticmethod
    def backward(ctx, grad_loss, _g_iters):
        grad, gpts, x, x_plus, inertia, mu_pair, pts = ctx.saved_tensors
        n_contacts, dt, eps, flags = ctx.args
        g = _fused_grad(grad, grad_loss, lambda w, skip, out: body_loss_pts_raw(
            x, x_plus, inertia, mu_pair, pts, n_contacts, dt, eps, weight=w, want_loss=False, want_grad_pts=False,
            flags=flags, skip_flag=skip, grad_out=out))
        return (None, None, *_split(g, inertia, mu_pair), gpts * grad_loss.reshape(-1, 1, 1), None, None, None, None, None)


def body_step_pts(x: Tensor, inertia: Tensor, mu_pair: Tensor, pts: Tensor, n_contacts: int, dt: float,
                  eps: float = 1e-4) -> Tensor:
    """One learnable time step (B,13) -> (B,13) of a single floating body with witness points (no autograd)."""
    _check_inputs(x, inertia, mu_pair, pts)
    x, pts = x.contiguous(), pts.contiguous()
    out = torch.empty_like(x)
    _call('dpll_body_step_pts_f64', x.device, x, inertia.contiguous(), mu_pair.contiguous(), pts, n_contacts, dt, eps,
          x.shape[0], out, None)
    return out


class BodyStepPts(torch.autograd.Function):
    """ONE differentiable learnable step of a single floating body with witness points (Sphere, Polygon): x (B,13), pts
    (B,4,3) -> next state (B,13).  Backward = ``dpll_body_step_pts_grad_f64`` (36 forward-mode directions per sample); the
    points' cotangent flows on through the caller's autograd graph into the shape parameters and the state."""

    @staticmethod
    def forward(ctx, x, inertia, mu_pair, pts, n_contacts, dt, eps):
        ctx.n_c, ctx.dt, ctx.eps = n_contacts, dt, eps
        ctx.save_for_backward(x, inertia, mu_pair, pts)
        return body_step_pts(x.detach(), inertia.detach(), mu_pair.detach(), pts.detach(), n_contacts, dt, eps)

    @staticmethod
    def backward(ctx, gnext):
        x, inertia, mu_pair, pts = ctx.saved_tensors
        gi, gm, gpts, gx = _summed_backward('dpll_body_step_pts_grad_f64', x, (inertia, mu_pair), (11, 12, 13), x, inertia,
                                            mu_pair, pts, ctx.n_c, ctx.dt, ctx.eps, x.shape[0], gnext)
        return gx.to(x.dtype), gi, gm, gpts.reshape(pts.shape).to(pts.dtype), None, None, None


class ChainContactNetsLoss(torch.autograd.Function):
    """ContactNets loss of a generic floating-base serial chain of ``n`` links (``dpll_chain_loss_f64``,
    csrc/cn_chain.cuh): differentiable w.r.t. inertia (n,10), mu_pair (n), half (n,3); float64."""

    @staticmethod
    def forward(ctx, x, x_plus, inertia, mu_pair, half, kin, n, dt, eps):
        _check_inputs(x, x_plus, inertia, mu_pair, half, kin, f64_only='the generic chain kernels are provided in float64')
        x, x_plus = x.contiguous(), x_plus.contiguous()
        _check_states(13 + 2 * (n - 1), x, x_plus)
        B, dev = x.shape[0], x.device
        loss = torch.empty(B, dtype=x.dtype, device=dev)
        ctx.args = (n, dt, eps)
        ctx.save_for_backward(x, x_plus, inertia, mu_pair, half, kin)
        _call('dpll_chain_loss_f64', dev, n, x, x_plus, None, inertia.contiguous(), mu_pair.contiguous(), half.contiguous(),
              kin.contiguous(), dt, eps, B, loss, None, None, None, None, workspace=True)
        return loss

    @staticmethod
    def backward(ctx, grad_loss):
        x, x_plus, inertia, mu_pair, half, kin = ctx.saved_tensors
        n, dt, eps = ctx.args
        B, dev = x.shape[0], x.device
        g = torch.zeros(14 * n, dtype=x.dtype, device=dev)
        if B > 0:
            _call('dpll_chain_loss_f64', dev, n, x, x_plus, grad_loss.contiguous(), inertia.contiguous(), mu_pair.contiguous(),
                  half.contiguous(), kin.contiguous(), dt, eps, B, None, None, None, g, None, workspace=True)
        return (None, None, *_split(g, inertia, mu_pair, half), None, None, None, None)


def chain_rollout(x0: Tensor, inertia: Tensor, mu_pair: Tensor, half: Tensor, kin: Tensor, n: int, dt: float,
                  steps: int, eps: float = 1e-4) -> Tensor:
    """(B, n_x) -> trajectory (B, steps+1, n_x) of a generic serial chain (``dpll_chain_rollout_f64``, no autograd)."""
    _check_inputs(x0, inertia, mu_pair, half, kin)
    x0 = x0.contiguous()
    B = x0.shape[0]
    traj = torch.empty((B, steps + 1, x0.shape[1]), dtype=x0.dtype, device=x0.device)
    _call('dpll_chain_rollout_f64', x0.device, n, x0, inertia.contiguous(), mu_pair.contiguous(), half.contiguous(),
          kin.contiguous(), dt, eps, B, steps, traj)
    return traj


class ChainRollout(torch.autograd.Function):
    """Differentiable rollout of a generic serial chain of ``n`` links: traj (B, steps+1, n_x).  Backward =
    ``dpll_chain_rollout_grad_f64`` (forward-mode tangents, 14 n + n_x directions per toss).  float64."""

    @staticmethod
    def forward(ctx, x0, inertia, mu_pair, half, kin, n, dt, steps, eps):
        ctx.n, ctx.dt, ctx.steps, ctx.eps = n, dt, steps, eps
        ctx.save_for_backward(x0, inertia, mu_pair, half, kin)
        return chain_rollout(x0.detach(), inertia.detach(), mu_pair.detach(), half.detach(), kin, n, dt, steps, eps)

    @staticmethod
    def backward(ctx, gtraj):
        x0, inertia, mu_pair, half, kin = ctx.saved_tensors
        B, n, steps = x0.shape[0], ctx.n, ctx.steps
        gi, gm, gh, gx0 = _summed_backward('dpll_chain_rollout_grad_f64', x0, (inertia, mu_pair, half), (14 * n, x0.shape[1]),
                                           n, x0, inertia, mu_pair, half, kin, ctx.dt, ctx.eps, B, steps, gtraj[:, 1:, :],
                                           steps=steps)
        gx = (gx0 + gtraj[:, 0, :].to(torch.float64)).to(x0.dtype)
        return gx, gi, gm, gh, None, None, None, None, None


def cube_terms(q: Tensor, v: Tensor, inertia: Tensor, mu_pair: Tensor, half: Tensor):
    """``dpll_cube_terms_f64``: (delassus (B,12,12), M (B,6,6), J (B,12,6), phi (B,4), acc (B,6)) in the order
    ``MultibodyTerms.forward`` returns them (multibody_terms.py:584-609).  fp64 only, no autograd."""
    _check_inputs(q, v, inertia, mu_pair, half, f64_only='cube_terms is provided in float64')
    q, v = q.contiguous(), v.contiguous()
    B, dev = q.shape[0], q.device
    M = torch.empty((B, 6, 6), dtype=q.dtype, device=dev)
    J = torch.empty((B, 12, 6), dtype=q.dtype, device=dev)
    phi = torch.empty((B, 4), dtype=q.dtype, device=dev)
    acc = torch.empty((B, 6), dtype=q.dtype, device=dev)
    D = torch.empty((B, 12, 12), dtype=q.dtype, device=dev)
    _call('dpll_cube_terms_f64', dev, q, v, inertia.contiguous(), mu_pair.contiguous(), half.contiguous(), B, M, J, phi, acc, D)
    return D, M, J, phi, acc


def elbow_terms(q: Tensor, v: Tensor, inertia: Tensor, mu_pair: Tensor, half: Tensor, kin: Tensor):
    """``dpll_elbow_terms_f64``: (delassus (B,24,24), M (B,7,7), J (B,24,7), phi (B,8), acc (B,7)) in the order
    ``MultibodyTerms.forward`` returns them (multibody_terms.py:584-609).  fp64 only, no autograd."""
    _check_inputs(q, v, inertia, mu_pair, half, kin, f64_only='elbow_terms is provided in float64')
    q, v = q.contiguous(), v.contiguous()
    B, dev = q.shape[0], q.device
    M = torch.empty((B, 7, 7), dtype=q.dtype, device=dev)
    J = torch.empty((B, 24, 7), dtype=q.dtype, device=dev)
    phi = torch.empty((B, 8), dtype=q.dtype, device=dev)
    acc = torch.empty((B, 7), dtype=q.dtype, device=dev)
    D = torch.empty((B, 24, 24), dtype=q.dtype, device=dev)
    _call('dpll_elbow_terms_f64', dev, q, v, inertia.contiguous(), mu_pair.contiguous(), half.contiguous(), kin.contiguous(),
          B, M, J, phi, acc, D)
    return D, M, J, phi, acc


class ChainWitnessPointLoss(torch.autograd.Function):
    """ContactNets loss of a generic tree of ``n`` links whose contact sets are given by witness points ``pts``
    (B, n, 4, 3) in link coordinates (``n_pts_packed``: points per slot, 3 bits each) -- spheres, polygons, learned meshes,
    boxes in any frame on any link: ``dpll_chain_loss_pts_f64``.  Differentiable w.r.t. inertia (n,10), mu_pair (n) and
    ``pts``; float64."""

    @staticmethod
    def forward(ctx, x, x_plus, inertia, mu_pair, pts, kin, n, n_pts_packed, dt, eps):
        _check_inputs(x, x_plus, inertia, mu_pair, pts, kin, f64_only='the generic tree kernels are provided in float64')
        n_x = 13 + 2 * (n - 1)
        x, x_plus, pts = x.contiguous(), x_plus.contiguous(), pts.contiguous()
        B, dev = x.shape[0], x.device
        if x.dim() != 2 or x.shape[1] != n_x or x_plus.shape != x.shape or tuple(pts.shape) != (B, n, 4, 3):
            raise ValueError(f'expected (B,{n_x}) states and (B,{n},4,3) points, got {tuple(x.shape)} / {tuple(pts.shape)}')
        loss = torch.empty(B, dtype=x.dtype, device=dev)
        gpts = torch.empty_like(pts)
        _call('dpll_chain_loss_pts_f64', dev, n, x, x_plus, None, inertia.contiguous(), mu_pair.contiguous(), kin.contiguous(),
              pts, n_pts_packed, dt, eps, B, loss, gpts, None, None, workspace=True)
        ctx.args = (n, n_pts_packed, dt, eps)
        ctx.save_for_backward(gpts, x, x_plus, inertia, mu_pair, pts, kin)
        return loss

    @staticmethod
    def backward(ctx, grad_loss):
        gpts, x, x_plus, inertia, mu_pair, pts, kin = ctx.saved_tensors
        n, packed, dt, eps = ctx.args
        B, dev = x.shape[0], x.device
        g = torch.zeros(14 * n, dtype=x.dtype, device=dev)
        if B > 0:
            _call('dpll_chain_loss_pts_f64', dev, n, x, x_plus, grad_loss.contiguous(), inertia.contiguous(),
                  mu_pair.contiguous(), kin.contiguous(), pts, packed, dt, eps, B, None, None, g, None, workspace=True)
        return (None, None, *_split(g, inertia, mu_pair), gpts * grad_loss.reshape(-1, 1, 1, 1), None, None, None, None,
                None)


def chain_terms(q: Tensor, v: Tensor, inertia: Tensor, mu_pair: Tensor, half: Tensor, kin: Tensor, n: int, n_boxes: int):
    """``dpll_chain_terms_f64``: (delassus (B,12g,12g), M (B,nv,nv), J (B,12g,nv), phi (B,4g), acc (B,nv)) of a tree of ``n``
    links with ``g = n_boxes`` boxes, in the order ``MultibodyTerms.forward`` returns them (multibody_terms.py:584-609).
    fp64 only, no autograd."""
    _check_inputs(q, v, inertia, mu_pair, half, kin, f64_only='chain_terms is provided in float64')
    q, v = q.contiguous(), v.contiguous()
    B, dev, nv, k = q.shape[0], q.device, 6 + n - 1, 12 * n_boxes
    M = torch.empty((B, nv, nv), dtype=q.dtype, device=dev)
    J = torch.empty((B, k, nv), dtype=q.dtype, device=dev)
    phi = torch.empty((B, 4 * n_boxes), dtype=q.dtype, device=dev)
    acc = torch.empty((B, nv), dtype=q.dtype, device=dev)
    D = torch.empty((B, k, k), dtype=q.dtype, device=dev)
    _call('dpll_chain_terms_f64', dev, n, n_boxes, q, v, inertia.contiguous(), mu_pair.contiguous(), half.contiguous(),
          kin.contiguous(), B, M, J, phi, acc, D)
    return D, M, J, phi, acc


class LeafPrepare(torch.autograd.Function):
    """Learnable leaves -> callable-level parameters, one launch each way (``dpll_leaf_prepare_f64`` /
    ``dpll_leaf_backward_f64``, csrc/cn_leaf.cu): theta (n_bodies, 10) -> inertia (n_bodies, 10); friction_params
    (n_geoms,) and the collision pairs' geometry indices (int32 (2, n_pairs)) -> pair friction (n_pairs,); length
    parameters (n_len,) -> |.|.  Replaces ~100 elementwise PyTorch launches (and their autograd nodes) per step of the
    systems that have no fused training entry point (two-body tree, generic chains).  float64, CUDA."""

    @staticmethod
    def forward(ctx, theta, friction, pairs, length):
        _check_inputs(theta, friction, length, f64_only='dpll_leaf_prepare is provided in float64')
        theta, friction, length = theta.contiguous(), friction.contiguous(), length.contiguous()
        assert pairs.dtype == torch.int32 and pairs.is_cuda and pairs.is_contiguous() and pairs.shape[0] == 2
        nb, npair, nlen = theta.shape[0], pairs.shape[1], length.numel()
        inertia = torch.empty_like(theta)
        mu = torch.empty(npair, dtype=theta.dtype, device=theta.device)
        half = torch.empty(nlen, dtype=theta.dtype, device=theta.device)
        _call('dpll_leaf_prepare_f64', theta.device, theta, nb, friction, pairs, pairs.data_ptr() + 4 * npair, npair, length,
              nlen, inertia, mu, half)
        ctx.save_for_backward(theta, friction, pairs, length)
        return inertia, mu, half

    @staticmethod
    def backward(ctx, g_inertia, g_mu, g_half):
        theta, friction, pairs, length = ctx.saved_tensors
        nb, npair, nlen = theta.shape[0], pairs.shape[1], length.numel()
        g_theta, g_friction, g_length = torch.empty_like(theta), torch.empty_like(friction), torch.empty_like(length)
        cont = lambda g: None if g is None else g.contiguous()      # noqa: E731
        g_inertia, g_mu, g_half = cont(g_inertia), cont(g_mu), cont(g_half)
        _call('dpll_leaf_backward_f64', theta.device, theta, nb, friction, friction.numel(), pairs, pairs.data_ptr() + 4 * npair,
              npair, length, nlen, g_inertia, g_mu, g_half, g_theta, g_friction, g_length)
        return g_theta, g_friction, None, g_length


_SUPPORT_F64 = 'the support-network kernels are provided in float64'


def elbow_support_directions(q: Tensor, axis: Tensor, pert0: Tensor, pert1: Tensor):
    """``dpll_elbow_support_directions_f64``: q (B, >= 8) rows (any row stride) -> the two links' perturbed, normalised
    support directions (B, n_query, 3) each.  float64, no autograd (directions are data, geometry.py:309-325)."""
    _check_inputs(q, axis, pert0, pert1, f64_only=_SUPPORT_F64)
    if q.dim() != 2 or q.shape[1] < 8 or q.stride(1) != 1:
        raise ValueError(f'expected (B, >= 8) configuration rows with unit column stride, got {tuple(q.shape)}')
    B, nq = q.shape[0], pert0.shape[0]
    d0 = torch.empty((B, nq, 3), dtype=q.dtype, device=q.device)
    d1 = torch.empty((B, nq, 3), dtype=q.dtype, device=q.device)
    _call('dpll_elbow_support_directions_f64', q.device, q, q.stride(0) if B > 1 else q.shape[1], axis.contiguous(),
          pert0.contiguous(), pert1.contiguous(), nq, B, d0, d1)
    return d0, d1


def body_support_directions(q: Tensor, pert: Tensor) -> Tensor:
    """``dpll_body_support_directions_f64``: q (B, >= 4) rows (any row stride, quaternion first) -> the body's perturbed,
    normalised support directions (B, n_query, 3) against the ground.  float64, no autograd (directions are data)."""
    _check_inputs(q, pert, f64_only=_SUPPORT_F64)
    if q.dim() != 2 or q.shape[1] < 4 or q.stride(1) != 1:
        raise ValueError(f'expected (B, >= 4) configuration rows with unit column stride, got {tuple(q.shape)}')
    B, nq = q.shape[0], pert.shape[0]
    d = torch.empty((B, nq, 3), dtype=q.dtype, device=q.device)
    _call('dpll_body_support_directions_f64', q.device, q, q.stride(0) if B > 1 else q.shape[1], pert.contiguous(), nq, B, d)
    return d


def icnn_support_points(d: Tensor, Wd0: Tensor, Wd1: Tensor, Wh: Tensor, wout: Tensor, slope: float) -> Tensor:
    """Support points p (D,3) for unit directions d (D,3), nothing kept for a backward (``ICNNSupport.forward``).
    Width 256: the tensor-core kernel (``icnn_support_points_tc``); other widths: the FP64 layer path."""
    if Wd0.shape[1] == ICNN_TC_WIDTH and not ICNN_FORCE_FP64_PATH:
        return icnn_support_points_tc(d, Wd0, Wd1, Wh, wout, slope)
    return icnn_support_forward(d, Wd0, Wd1, Wh, wout, slope)[0]


def icnn_tc_prepare(Wd0: Tensor, Wd1: Tensor, Wh: Tensor, wout: Tensor, slope: float):
    """``dpll_icnn_tc_prepare_f64``: the four weights -> (digit-plane image, epilogue constants) of the tensor-core kernels."""
    _check_inputs(Wd0, Wd1, Wh, wout, f64_only=_SUPPORT_F64)
    lib = _lib.load()
    Wd0, Wd1, Wh, wout = (t.contiguous() for t in (Wd0, Wd1, Wh, wout))
    dev = Wd0.device
    image = torch.empty(lib.dpll_icnn_tc_image_bytes(), dtype=torch.uint8, device=dev)
    consts = torch.empty(lib.dpll_icnn_tc_const_bytes() // 8, dtype=torch.float64, device=dev)
    _call('dpll_icnn_tc_prepare_f64', dev, Wd0, Wd1, Wh, wout, Wd0.shape[1], slope, image, consts)
    return image, consts


def icnn_support_points_tc(d: Tensor, Wd0: Tensor, Wd1: Tensor, Wh: Tensor, wout: Tensor, slope: float, prepared=None) -> Tensor:
    """``dpll_icnn_tc_support_f64``: support points (D,3) on the tensor cores (``prepared`` = ``icnn_tc_prepare`` output)."""
    _check_inputs(d, Wh, f64_only=_SUPPORT_F64)
    image, consts = prepared if prepared is not None else icnn_tc_prepare(Wd0, Wd1, Wh, wout, slope)
    d, Wh = d.contiguous(), Wh.contiguous()
    D = d.shape[0]
    p = torch.empty((D, 3), dtype=d.dtype, device=d.device)
    _call('dpll_icnn_tc_support_f64', d.device, d, D, image, consts, Wh, Wh.shape[0], slope, p)
    return p


ICNN_TC_BWD_MAX_ROWS = 1 << 20       # rows per backward launch (int32 accumulators of the six row chunks)


def icnn_support_backward_tc(d: Tensor, gp: Tensor, Wh: Tensor, slope: float, prepared):
    """Weight-gradient reductions of the support network on the tensor cores, without a host read: the rows with a non-zero
    cotangent are compacted on the device (``torch.nonzero_static``), their slope masks re-evaluated
    (``dpll_icnn_tc_record_f64``) and contracted (``dpll_icnn_tc_bwd_f64``).  Returns (C (3,W,W), R1 (3,W), S (3)) with
    C_k[j,i] = sum_r gp_k[r] m0[r,j] m1[r,i], R1_k[i] = sum_r gp_k[r] b1[r,i], S_k = sum_r gp_k[r]."""
    _check_inputs(d, gp, Wh)
    lib = _lib.load()
    image, consts = prepared
    W = Wh.shape[0]
    dev = d.device
    C = torch.zeros((3, W, W), dtype=torch.float64, device=dev)
    R1 = torch.zeros((3, W), dtype=torch.float64, device=dev)
    S = torch.zeros(3, dtype=torch.float64, device=dev)
    Wh = Wh.contiguous()
    for lo in range(0, d.shape[0], ICNN_TC_BWD_MAX_ROWS):
        dd, gg = d[lo:lo + ICNN_TC_BWD_MAX_ROWS], gp[lo:lo + ICNN_TC_BWD_MAX_ROWS]
        cap = dd.shape[0]
        ldk = (cap + 127) // 128 * 128
        live = (gg != 0).any(-1)
        idx = torch.nonzero_static(live, size=cap, fill_value=0).reshape(-1)       # first n entries: the live rows, in order
        n = live.sum().reshape(1)
        d_act, g_act = dd.index_select(0, idx), gg.index_select(0, idx)
        amax = gg.abs().amax(0)
        m0t = torch.empty((W, ldk), dtype=torch.uint8, device=dev)
        m1t = torch.empty((W, ldk), dtype=torch.uint8, device=dev)
        planes = torch.empty((lib.dpll_icnn_tc_bwd_planes(), ldk), dtype=torch.int8, device=dev)
        partial = torch.empty(lib.dpll_icnn_tc_bwd_partial_bytes() // 4, dtype=torch.int32, device=dev)
        sums = torch.empty(6 * W + 3, dtype=torch.float64, device=dev)
        Cb = torch.empty((3, W, W), dtype=torch.float64, device=dev)
        _call('dpll_icnn_tc_record_f64', dev, d_act, cap, n, image, consts, Wh, W, slope, m0t, m1t, ldk)
        _call('dpll_icnn_tc_bwd_f64', dev, g_act, n, amax, m0t, m1t, ldk, slope, planes, partial, sums, Cb)
        C += Cb
        R1 += sums[3 * W:6 * W].reshape(3, W)
        S += sums[6 * W:]
    return C, R1, S


ICNN_TC_WIDTH = 256
ICNN_FORCE_FP64_PATH = False        # tests / A-B timing: route width-256 networks through the FP64 layer path too


def icnn_support_forward(d: Tensor, Wd0: Tensor, Wd1: Tensor, Wh: Tensor, wout: Tensor, slope: float):
    """Support points p (D,3) of the depth-2 homogeneous ICNN for unit directions d (D,3), float64, CUDA:
    the ``dpll_icnn_*`` kernels around two FP64 GEMMs.  Returns (p, h0aug, m1, a0) -- the last three are what
    the backward needs."""
    _check_inputs(d, Wd0, Wd1, Wh, wout, f64_only=_SUPPORT_F64)
    d, Wd0 = d.contiguous(), Wd0.contiguous()
    D, W = d.shape[0], Wd0.shape[1]
    dev = d.device
    Wh_a, wo = Wh.abs(), wout.abs()
    h0aug = torch.empty((D, W + 8), dtype=d.dtype, device=dev)
    W_aug = torch.cat((Wh_a, Wd1, torch.zeros((5, W), dtype=d.dtype, device=dev)), 0)
    V1 = (Wd1 * wo).contiguous()
    p = torch.empty((D, 3), dtype=d.dtype, device=dev)
    _call('dpll_icnn_input_f64', dev, d, Wd0, D, W, slope, h0aug)
    m1 = h0aug @ W_aug                                   # z1 = h0 |Wh| + d Wd1
    _call('dpll_icnn_mask_f64', dev, m1, m1.numel(), slope)
    a0 = m1 @ (wo[:, None] * Wh_a.t())                   # T, turned into a0 in place below
    _call('dpll_icnn_output_f64', dev, a0, h0aug, m1, Wd0, V1, D, W, slope, p)
    return p, h0aug, m1, a0


def icnn_support_backward(gp: Tensor, h0aug: Tensor, m1: Tensor, a0: Tensor, Wd0: Tensor, slope: float):
    """Returns (g1 = gp^T m1 (3,W), gWd0 = gp^T a0 (3,W), G = t^T m1 (W,W)) with t = (gp Wd0) o m0."""
    _check_inputs(gp, h0aug, m1, a0, Wd0)
    gp, Wd0 = gp.contiguous(), Wd0.contiguous()
    D, W = m1.shape
    dev = gp.device
    blocks = _lib.load().dpll_icnn_backward_blocks(D)
    t = torch.empty((D, W), dtype=gp.dtype, device=dev)
    part = torch.zeros((max(blocks, 1), 6, W), dtype=gp.dtype, device=dev)   # zeros: D == 0 launches nothing
    _call('dpll_icnn_backward_f64', dev, gp, h0aug, m1, a0, Wd0, D, W, slope, t, part)
    sums = part.sum(0)
    G = t.t() @ m1
    return sums[:3], sums[3:], G


def fma_peak(dtype: torch.dtype, device: torch.device, blocks: int, iters: int, reps: int = 5) -> float:
    """Measured FMA throughput (FLOP/s) of the CUDA cores for ``dtype`` -- roofline denominator.  Best of
    ``reps`` runs (a peak: a run disturbed by clock ramp-up would understate the denominator)."""
    out = torch.empty(blocks * 256, dtype=dtype, device=device)
    stream = torch.cuda.current_stream(out.device)
    best = float('inf')
    _call('dpll_fma_peak', out.device, out, blocks, iters // 4 + 1, dtype=dtype)      # warm-up
    torch.cuda.synchronize(device)
    for _ in range(max(1, reps)):
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record(stream)
        _call('dpll_fma_peak', out.device, out, blocks, iters, dtype=dtype)
        stop.record(stream)
        torch.cuda.synchronize(device)
        best = min(best, start.elapsed_time(stop))
    return blocks * 256 * iters * 16 * 2 / (best * 1e-3)
