"""Autograd bridge for the native UNet: training forward / backward.

Replaces the graph autograd records for ``DDPM_model._train_step`` + ``loss.backward()``
(reference models/diffusion/ddpm.py:111-121,142-144; SURVEY.md Appendix B) with two native calls:
``cm_unet_train_forward`` (forward that keeps activations, GroupNorm statistics and time-MLP
pre-activations resident) and ``cm_unet_backward`` (dgrad / wgrad of every conv on tcgen05,
GroupNorm / SiLU / Dropout3d / attention / time-MLP backward), which fills ONE flat fp32 gradient
buffer.  Data-parallel training is OPT-IN (``enable_data_parallel(module, group)``, called by
``DDPM_model.enable_data_parallel``): the flat buffer is then all-reduced (mean) in a single NCCL call
before the per-parameter views are handed to autograd — the data-parallel exchange step of SURVEY.md
§8(e).  A process group that merely happens to be initialised is never used implicitly.

There is no eager fallback: a missing library or a CPU tensor raises.
"""
from __future__ import annotations

import ctypes as C

import torch


def dropout_layout(plan):
    """[(offset, channels)] per ResnetBlock (plan order) and the row stride of the scale table."""
    if plan._dropout_layout is None:
        plan._dropout_layout = _dropout_layout(plan)
    return plan._dropout_layout


def _dropout_layout(plan):
    n = plan.n
    lib = n.lib()
    ld = C.c_int32()
    nb = lib.cm_unet_dropout_layout(plan.handle, None, None, 0, C.byref(ld))
    offs = (C.c_int32 * nb)()
    chans = (C.c_int32 * nb)()
    lib.cm_unet_dropout_layout(plan.handle, offs, chans, nb, C.byref(ld))
    return [(offs[i], chans[i]) for i in range(nb)], ld.value


def grad_layout(plan):
    if plan._grad_layout is None:
        plan._grad_layout = _grad_layout(plan)
    return plan._grad_layout


def _grad_layout(plan):
    n = plan.n
    lib = n.lib()
    cnt = lib.cm_unet_param_count(plan.handle)
    offs = (C.c_int64 * cnt)()
    total = C.c_int64()
    n.check(lib.cm_unet_grad_layout(plan.handle, offs, cnt, C.byref(total)))
    return [offs[i] for i in range(cnt)], total.value


_DP_UNSET = object()


def enable_data_parallel(module, group=None):
    """Opt in to gradient averaging over ``group`` (None = the default process group).  The caller is
    responsible for starting every rank from the same parameters (DDPM_model.enable_data_parallel
    broadcasts them)."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        raise RuntimeError("enable_data_parallel: torch.distributed is not initialised")
    module._dp_group = group          # None is a valid group handle (the default group)
    module._dp_enabled = True


def disable_data_parallel(module):
    module._dp_enabled = False


def _allreduce_mean(module, flat):
    if not getattr(module, "_dp_enabled", False):
        return
    import torch.distributed as dist
    group = getattr(module, "_dp_group", None)
    world = dist.get_world_size(group)
    if world > 1:
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
        flat.mul_(1.0 / world)


class _UNetFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, module, plan, future, t, past, drop, *params):
        n = plan.n
        B = future.shape[0]
        eps = torch.empty((B, module.output_channels) + tuple(future.shape[2:]), device=future.device,
                          dtype=torch.float32)
        n.check(n.lib().cm_unet_train_forward(plan.handle, n.ptr(future), n.ptr(t), n.ptr(past), n.ptr(eps),
                                              B, n.ptr(drop), n.current_stream()))
        plan.train_token += 1
        ctx.token = plan.train_token
        ctx.plan = plan
        ctx.module = module
        ctx.keep = (future, t, past, drop)        # the native backward reads these buffers again
        ctx.param_meta = [(p.shape, p.requires_grad) for p in params]
        return eps

    @staticmethod
    def backward(ctx, d_eps):
        plan = ctx.plan
        n = plan.n
        if ctx.token != plan.train_token:
            raise RuntimeError(
                "crowdmod-ddpm-4d_b200: the activations of this forward were overwritten by a later "
                "forward or sampling call of the same UNet geometry (one backward per forward, and "
                "nothing else on that geometry in between)")
        offs, total = grad_layout(plan)
        flat = torch.empty(total, device=d_eps.device, dtype=torch.float32)
        d_eps = d_eps.contiguous().float()
        # torch.use_deterministic_algorithms(True) makes the native backward reproducible bit for bit (fixed-order
        # reductions instead of fp32 atomics); the handle keeps the mode, so it is set only when the flag changed
        det = torch.are_deterministic_algorithms_enabled()
        if plan.deterministic != det:
            n.check(n.lib().cm_unet_set_deterministic(plan.handle, int(det)))
            plan.deterministic = det
        n.check(n.lib().cm_unet_backward(plan.handle, n.ptr(d_eps), n.ptr(flat), n.current_stream()))
        _allreduce_mean(ctx.module, flat)
        ctx.module._last_flat_grad = flat
        grads = []
        for (shape, req), off in zip(ctx.param_meta, offs):
            grads.append(flat[off:off + shape.numel()].view(shape) if req else None)
        return (None, None, None, None, None, None) + tuple(grads)


def draw_dropout_scales(module, plan, batch, device):
    """Dropout3d (layers.py:42,70) zeroes whole channels per sample: one scale per (sample, block,
    channel), mask/(1-p).  ``module._injected_dropout`` (list of [B, C_k] masks, plan order) lets a
    parity test supply the masks."""
    p = float(module.dropout_rate)
    injected = getattr(module, "_injected_dropout", None)
    if injected is None and (p <= 0.0 or not module.training):
        return None
    layout, ld = dropout_layout(plan)
    if injected is not None:
        table = torch.ones((batch, ld), device=device, dtype=torch.float32)
        for (off, ch), m in zip(layout, injected):
            table[:, off:off + ch] = m.to(device=device, dtype=torch.float32)
        return table.contiguous()
    if p >= 1.0:
        return torch.zeros((batch, ld), device=device, dtype=torch.float32)
    keep = torch.rand((batch, ld), device=device) >= p
    return (keep.float() / (1.0 - p)).contiguous()


def unet_train_forward(module, future, t, past):
    rows, cols, past_len, future_len = module._geometry(future, past)
    plan = module._plan(rows, cols, past_len, future_len)
    plan.sync(module, need_table=False)
    future = future.detach().contiguous().float()
    past = past.detach().contiguous().float()
    t = t.contiguous().to(torch.int64)
    drop = draw_dropout_scales(module, plan, future.shape[0], future.device)
    return _UNetFunction.apply(module, plan, future, t, past, drop, *plan.tensors(module))
