"""UNet noise-prediction backbone — drop-in for reference models/backbones/unet.py:8-167.

Same constructor, same ``forward(future, t, past) -> eps`` contract, same 169-key (for the ATC
shape) ``state_dict`` and the same default initialisation as the reference, but the forward
pass runs as ONE native plan of hand-written sm_100a kernels (``cm_unet_forward`` in
``include/crowdmod_b200.h``) instead of ~120 eager cuDNN/ATen launches.  The reverse chain
(``sample_chain``) additionally fuses ``DDPM.step`` into the last kernel and replays a CUDA
graph per step (``cm_ddpm_sample``).

There is no CPU or eager-PyTorch path: calling ``forward`` with CPU tensors raises.
"""
from __future__ import annotations

import ctypes as C
import os
import weakref
from typing import Dict, Optional, Tuple

import torch
import torch.nn as nn

from .embeddings import SinusoidalPositionEmbeddings
from .layers import DownSample, ResnetBlock, UpSample


def _native():
    # imported lazily so that building the parameter tree (CPU-only host logic) does not need
    # the shared library; any compute does.
    pkg = __name__.split(".models.")[0] if ".models." in __name__ else None
    if pkg:
        import importlib
        return importlib.import_module(pkg + "._native")
    import _native as n   # package directory itself on sys.path (drop-in mode)
    return n


# native handles live outside the module's __dict__ so that deepcopy / pickling of the
# nn.Module (which the reference's callers may do) never touches ctypes objects
_PLANS: "weakref.WeakKeyDictionary[nn.Module, Dict[Tuple[int, int, int, int], _NativePlan]]" = \
    weakref.WeakKeyDictionary()


def _graph_mode(use_graph) -> int:
    """cm_chain_args.use_graph: False/0 eager, 1 / "step" per-step graph replay, True / 2 / "chain" the whole
    chain as ONE graph (conditional WHILE node)."""
    if use_graph is False or use_graph == 0:
        return 0
    if use_graph is True or use_graph in (2, "chain"):   # before the 1 test: True == 1
        return 2
    if use_graph in (1, "step"):
        return 1
    if use_graph == "eager":
        return 0
    raise ValueError(f"use_graph={use_graph!r}: expected False, True, 'eager', 'step' or 'chain'")


class _NativePlan:
    """One native handle per tensor geometry (rows, cols, past_len, future_len)."""

    def __init__(self, module: "UNet", rows: int, cols: int, past_len: int, future_len: int):
        n = _native()
        self.n = n
        cfg = n.UNetConfig()
        cfg.in_channels = module.input_channels
        cfg.out_channels = module.output_channels
        cfg.num_res_blocks = module.num_res_blocks
        cfg.base_channels = module.base_channels
        mults = list(module.base_channels_multiples)
        cfg.num_levels = len(mults)
        for i, m in enumerate(mults):
            cfg.mult[i] = int(m)
            cfg.attn[i] = int(bool(module.apply_attention[i]))
        cfg.time_multiple = module.time_multiple
        cfg.rows, cfg.cols = rows, cols
        cfg.past_len, cfg.future_len = past_len, future_len
        cfg.table_steps = module.time_embeddings.total_time_steps
        cfg.weight_terms = int(os.environ.get("CROWDMOD_WEIGHT_TERMS", "2"))
        cfg.dgrad_terms = int(os.environ.get("CROWDMOD_DGRAD_TERMS", "2"))
        cfg.train_act_terms = int(os.environ.get("CROWDMOD_TRAIN_ACT_TERMS", "2"))
        self.handle = C.c_void_p()
        n.check(n.lib().cm_unet_create(C.byref(cfg), C.byref(self.handle)))
        self._bound: Optional[Tuple] = None
        self._versions: Optional[Tuple] = None
        self._table_ready = False
        # everything that only depends on the plan is looked up once (169 ctypes calls per name walk)
        self._names = self._query_names()
        self._tensors = None          # parameter / buffer tensors in plan order
        self._ptr_array = None
        self._grad_layout = None
        self._dropout_layout = None
        self.train_token = 0

    def _query_names(self):
        lib = self.n.lib()
        out = []
        buf = C.create_string_buffer(256)
        shape = (C.c_int64 * 5)()
        nd = C.c_int()
        for i in range(lib.cm_unet_param_count(self.handle)):
            self.n.check(lib.cm_unet_param_info(self.handle, i, buf, 256, shape, C.byref(nd)))
            out.append((buf.value.decode(), tuple(shape[j] for j in range(nd.value))))
        return out

    def names(self):
        return self._names

    def tensors(self, module: "UNet"):
        """The module's parameter / buffer tensors in plan (= state_dict) order.  The list is rebuilt when
        the module's tensors were replaced (load_state_dict keeps them, .to() / _apply drops the plan)."""
        if self._tensors is None:
            sd = module.state_dict(keep_vars=True)
            missing = [nm for nm, _ in self._names if nm not in sd]
            if missing:
                raise RuntimeError(f"UNet state_dict lacks {missing[:3]}... expected by the native plan")
            self._tensors = [sd[nm] for nm, _ in self._names]
        return self._tensors

    def invalidate(self):
        """Forget what is bound / packed: the next call re-binds every tensor and re-derives the caches."""
        self._tensors = None
        self._bound = None
        self._versions = None
        self._table_ready = False

    def sync(self, module: "UNet", need_table: bool):
        """(Re)bind fp32 parameter storage (one C call) and re-derive the packed caches (one launch, no
        synchronisation) when a parameter was replaced or modified in place (optimizer.step /
        load_state_dict bump ``_version``; writes through ``p.data`` do NOT: call
        ``UNet.invalidate_native_cache()`` after such surgery)."""
        ts = self.tensors(module)
        ptrs = tuple(t.data_ptr() for t in ts)
        vers = tuple(t._version for t in ts)
        if ptrs == self._bound and vers == self._versions and (self._table_ready or not need_table):
            return
        lib = self.n.lib()
        if ptrs != self._bound:
            for (name, shape), t in zip(self._names, ts):
                if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
                    raise RuntimeError(
                        f"UNet parameter '{name}' must be a contiguous fp32 CUDA tensor "
                        f"(got {t.dtype} on {t.device}); move the module with .to('cuda')")
                if tuple(t.shape) != tuple(shape):
                    raise RuntimeError(f"UNet parameter '{name}': shape {tuple(t.shape)} != plan {tuple(shape)}")
            arr = (C.c_void_p * len(ptrs))(*ptrs)
            self.n.check(lib.cm_unet_bind_params(self.handle, arr, len(ptrs)))
            self._ptr_array = arr
        self.n.check(lib.cm_unet_pack(self.handle, 1 if need_table else 0, self.n.current_stream()))
        self._bound = ptrs
        self._versions = vers
        self._table_ready = bool(need_table)

    def __del__(self):
        try:
            if self.handle:
                self.n.lib().cm_unet_destroy(self.handle)
        except Exception:
            pass


class UNet(nn.Module):
    """UNet architecture to process macroprops sequences (native sm_100a execution)."""

    def __init__(self, input_channels=4, output_channels=4, num_res_blocks=2, base_channels=128,
                 base_channels_multiples=[1, 2, 4, 8],
                 apply_attention=[False, False, True, False, False], dropout_rate=0.1,
                 time_multiple=4, condition="Past"):
        super().__init__()
        self.input_channels = input_channels
        self.output_channels = output_channels
        self.num_res_blocks = num_res_blocks
        self.base_channels = base_channels
        self.base_channels_multiples = list(base_channels_multiples)
        self.apply_attention = list(apply_attention)
        self.dropout_rate = dropout_rate
        self.time_multiple = time_multiple
        self.condition = condition
        emb_dims = base_channels * time_multiple

        # Registration order == reference (unet.py:27-122): identical state_dict and RNG use.
        self.time_embeddings = SinusoidalPositionEmbeddings(time_emb_dims=base_channels,
                                                            time_emb_dims_exp=emb_dims)
        self.first = nn.Conv3d(input_channels, base_channels, kernel_size=3, stride=1, padding="same")
        if condition == "Past":
            self.past_encoding = None

        def block(cin, cout, attn):
            return ResnetBlock(in_channels=cin, out_channels=cout, dropout_rate=dropout_rate,
                               time_emb_dims=emb_dims, apply_attention=attn, condition=condition)

        levels = len(self.base_channels_multiples)
        self.encoder_blocks = nn.ModuleList()
        skip_channels = [base_channels]
        width = base_channels
        for level, mult in enumerate(self.base_channels_multiples):
            cout = base_channels * mult
            for _ in range(num_res_blocks):
                self.encoder_blocks.append(block(width, cout, apply_attention[level]))
                width = cout
                skip_channels.append(width)
            if level != levels - 1:
                self.encoder_blocks.append(DownSample(channels=width))
                skip_channels.append(width)

        self.bottleneck_blocks = nn.ModuleList((block(width, width, True), block(width, width, False)))

        self.decoder_blocks = nn.ModuleList()
        for level in reversed(range(levels)):
            cout = base_channels * self.base_channels_multiples[level]
            for _ in range(num_res_blocks + 1):
                self.decoder_blocks.append(block(skip_channels.pop() + width, cout, apply_attention[level]))
                width = cout
            if level != 0:
                self.decoder_blocks.append(UpSample(width))

        self.final = nn.Sequential(
            nn.GroupNorm(num_groups=8, num_channels=width),
            nn.SiLU(),
            nn.Conv3d(width, output_channels, kernel_size=3, stride=1, padding="same"),
        )

    # ------------------------------------------------------------------ native plumbing
    def _apply(self, fn, *args, **kwargs):
        # .to()/.cuda()/.float() replace parameter storage: drop cached native bindings
        _PLANS.pop(self, None)
        return super()._apply(fn, *args, **kwargs)

    def _plan(self, rows, cols, past_len, future_len) -> _NativePlan:
        key = (rows, cols, past_len, future_len)
        plans = _PLANS.setdefault(self, {})
        plan = plans.get(key)
        if plan is None:
            plan = _NativePlan(self, rows, cols, past_len, future_len)
            plans[key] = plan
        return plan

    @staticmethod
    def _require_cuda(*tensors):
        for t in tensors:
            if t is not None and not t.is_cuda:
                raise RuntimeError(
                    "crowdmod-ddpm-4d_b200 has no CPU path: UNet tensors must live on a CUDA "
                    "(B200, sm_100a) device")

    def _geometry(self, future, past):
        _, _, rows, cols, future_len = future.shape
        past_len = past.shape[4]
        if self.condition != "Past":
            past_len = 0   # unet.py:141-142: x = future only
        return rows, cols, past_len, future_len

    # ------------------------------------------------------------------ reference API
    def forward(self, future, t, past=None):
        """future [B,C,H,W,F] fp32, t [B] int64, past [B,C,H,W,P] fp32 -> eps [B,C,H,W,F]."""
        past_shape = past.shape          # the reference reads past.shape unconditionally (unet.py:133)
        self._require_cuda(future, t, past)
        if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            from .unet_autograd import unet_train_forward   # training fwd/bwd (autograd bridge)
            return unet_train_forward(self, future, t, past)
        n = _native()
        rows, cols, past_len, future_len = self._geometry(future, past)
        plan = self._plan(rows, cols, past_len, future_len)
        plan.sync(self, need_table=False)
        plan.train_token += 1            # the arena is shared: a pending training backward must raise
        future = future.contiguous().float()
        past = past.contiguous().float()
        t = t.contiguous().to(torch.int64)
        B = future.shape[0]
        eps = torch.empty((B, self.output_channels, rows, cols, future_len), device=future.device,
                          dtype=torch.float32)
        if B == 0:                       # the reference's torch ops accept an empty batch and return an empty tensor
            return eps
        n.check(n.lib().cm_unet_forward(plan.handle, n.ptr(future), n.ptr(t), n.ptr(past), n.ptr(eps),
                                        B, n.current_stream()))
        return eps

    # ------------------------------------------------------------------ fused reverse chain
    @torch.no_grad()
    def sample_chain(self, past, x, tsteps, coef, mode=0, noise=None, seed=0, sample_offset=0,
                     history=None, use_graph=True):
        """Runs len(tsteps) reverse steps in place on ``x`` (x_T -> x_0).

        tsteps: int32 CPU tensor [nsteps]; coef: fp32 CPU tensor [nsteps, 8] (see cm_chain_args).
        noise: optional CUDA tensor [nsteps, *x.shape] of injected z; None -> Philox(seed).
        """
        self._require_cuda(past, x, noise, history)
        if x.shape[0] == 0:              # empty sample batch: nothing to denoise (the reference loop is a no-op on it)
            return x
        n = _native()
        rows, cols, past_len, future_len = self._geometry(x, past)
        plan = self._plan(rows, cols, past_len, future_len)
        plan.sync(self, need_table=True)
        plan.train_token += 1
        assert x.is_contiguous() and x.dtype == torch.float32
        assert past.is_contiguous() and past.dtype == torch.float32
        tsteps = tsteps.to(torch.int32).contiguous().cpu()
        coef = coef.to(torch.float32).contiguous().cpu()
        assert coef.shape == (tsteps.numel(), 8)
        if noise is not None:
            assert noise.is_contiguous() and noise.dtype == torch.float32
            assert noise.numel() == tsteps.numel() * x.numel()
        a = n.ChainArgs()
        a.past = past.data_ptr()
        a.x = x.data_ptr()
        a.n = x.shape[0]
        a.nsteps = tsteps.numel()
        a.tsteps = tsteps.data_ptr()
        a.coef = coef.data_ptr()
        a.mode = int(mode)
        a.noise = noise.data_ptr() if noise is not None else None
        a.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        a.sample_offset = int(sample_offset)
        a.history = history.data_ptr() if history is not None else None
        a.use_graph = _graph_mode(use_graph)
        n.check(n.lib().cm_ddpm_sample(plan.handle, C.byref(a), n.current_stream()))
        return x

    def last_chain_launches(self, rows, cols, past_len, future_len) -> int:
        n = _native()
        return int(n.lib().cm_last_chain_launches(self._plan(rows, cols, past_len, future_len).handle))

    def invalidate_native_cache(self):
        """Call after modifying parameters through ``p.data`` (EMA swaps, manual weight surgery): such writes do
        not bump ``_version``, so the packed fp16 weights / time-embedding table would stay stale."""
        for plan in _PLANS.get(self, {}).values():
            plan.invalidate()

    def last_chain_graph_stats(self, rows, cols, past_len, future_len):
        """(cudaGraphLaunch calls of the last chain, whether it had to rebuild its graph)."""
        n = _native()
        h = self._plan(rows, cols, past_len, future_len).handle
        return int(n.lib().cm_last_chain_graph_launches(h)), bool(n.lib().cm_last_chain_graph_rebuilt(h))

    def native_stats(self, rows, cols, past_len, future_len):
        """(kernel launches per forward, algorithmic FLOPs per sample) of the native plan."""
        n = _native()
        plan = self._plan(rows, cols, past_len, future_len)
        return (n.lib().cm_unet_launches_per_forward(plan.handle),
                n.lib().cm_unet_flops_per_sample(plan.handle))
