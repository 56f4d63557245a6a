"""DiT4D_V4 — the reference's second noise-prediction backbone on the native sm_100a plan (SURVEY.md section 8 f2).

Mirror of /root/reference/models/backbones/DiT4D_V4.py: same constructor arguments, the same sub-module tree and
registration order (so the 99-entry ``state_dict`` and the seeded initialisation are identical to the reference's),
the same ``forward(future, t, past) -> [B, C, H, W, F]`` contract.  The sub-modules are parameter containers: the
arithmetic runs in ``csrc/dit.cu`` (``cm_dit_forward`` / ``cm_dit_sample``) — every Linear on the tcgen05 GEMM, the
spatial attention on the attention core, AdaLN / LayerNorm / GELU / temporal cross-attention / (un)patch as bandwidth
kernels, the DDPM / DDIM update fused into the un-patch kernel.

Inference and sampling only: with gradients enabled ``forward`` raises (the training forward / backward of this
backbone is not built; ``DDPM_model.train`` with ``--arch DDPM-DiT`` fails loudly instead of falling back to eager).
"""
from __future__ import annotations

import ctypes as C
import weakref
from typing import Dict, Optional, Tuple

import torch
import torch.nn as nn

from .embeddings import SinusoidalPositionEmbeddings


def _native():
    from ... import _native as n
    n.lib()
    return n


def _no_forward(name):
    def f(self, *a, **k):
        raise RuntimeError(f"{name} is a parameter container: its arithmetic runs inside the fused native DiT plan "
                           "(cm_dit_forward); call DiT4D_V4.forward instead")
    return f


class PatchEmbed4D(nn.Module):
    """Parameters of the patch embedding (reference :6-63): Conv3d with kernel = stride = (t_patch, p, p)."""

    def __init__(self, grid_rows, grid_cols, T_total, patch_size, t_patch_size, in_channels, hidden_size):
        super().__init__()
        assert grid_rows % patch_size == 0, f"grid_rows ({grid_rows}) must be divisible by patch_size ({patch_size})"
        assert grid_cols % patch_size == 0, f"grid_cols ({grid_cols}) must be divisible by patch_size ({patch_size})"
        assert T_total % t_patch_size == 0, f"T_total ({T_total}) must be divisible by t_patch_size ({t_patch_size})"
        self.patch_size, self.t_patch_size = patch_size, t_patch_size
        self.h_patches, self.w_patches, self.t_patches = grid_rows // patch_size, grid_cols // patch_size, T_total // t_patch_size
        self.num_patches = self.h_patches * self.w_patches * self.t_patches
        self.proj = nn.Conv3d(in_channels, hidden_size, kernel_size=(t_patch_size, patch_size, patch_size),
                              stride=(t_patch_size, patch_size, patch_size))

    forward = _no_forward("PatchEmbed4D")


class DiTBlockCA(nn.Module):
    """Parameters of one block (reference :109-141): spatial self-attention, temporal cross-attention, MLP, AdaLN-Zero."""

    def __init__(self, hidden_size, num_heads, N_s, T_p, query_slot_start, mlp_ratio=4.0, dropout_rate=0.0):
        super().__init__()
        self.N_s, self.T_p, self.query_slot_start = N_s, T_p, query_slot_start
        self.norm1 = nn.LayerNorm(hidden_size, elementwise_affine=False, eps=1e-6)
        self.spatial_attn = nn.MultiheadAttention(hidden_size, num_heads, dropout=dropout_rate, batch_first=True)
        self.norm2 = nn.LayerNorm(hidden_size, elementwise_affine=False, eps=1e-6)
        self.temporal_attn = nn.MultiheadAttention(hidden_size, num_heads, dropout=dropout_rate, batch_first=True)
        self.norm3 = nn.LayerNorm(hidden_size, elementwise_affine=False, eps=1e-6)
        mlp_hidden = int(hidden_size * mlp_ratio)
        self.mlp = nn.Sequential(nn.Linear(hidden_size, mlp_hidden), nn.GELU(), nn.Dropout(dropout_rate),
                                 nn.Linear(mlp_hidden, hidden_size), nn.Dropout(dropout_rate))
        self.adaLN_modulation = nn.Sequential(nn.SiLU(), nn.Linear(hidden_size, 9 * hidden_size, bias=True))
        nn.init.zeros_(self.adaLN_modulation[-1].weight)
        nn.init.zeros_(self.adaLN_modulation[-1].bias)

    forward = _no_forward("DiTBlockCA")


class FinalLayer(nn.Module):
    """Parameters of the output projection (reference :213-234)."""

    def __init__(self, hidden_size, patch_size, out_channels, t_patch_size):
        super().__init__()
        self.norm = nn.LayerNorm(hidden_size, elementwise_affine=False, eps=1e-6)
        self.linear = nn.Linear(hidden_size, t_patch_size * out_channels * patch_size * patch_size)
        self.adaLN_modulation = nn.Sequential(nn.SiLU(), nn.Linear(hidden_size, 2 * hidden_size, bias=True))
        nn.init.zeros_(self.adaLN_modulation[-1].weight)
        nn.init.zeros_(self.adaLN_modulation[-1].bias)
        nn.init.zeros_(self.linear.weight)
        nn.init.zeros_(self.linear.bias)

    forward = _no_forward("FinalLayer")


_PLANS: "weakref.WeakKeyDictionary[nn.Module, _DitPlan]" = weakref.WeakKeyDictionary()


class _DitPlan:
    """The native handle of one module (the geometry is part of the constructor arguments)."""

    def __init__(self, m: "DiT4D_V4"):
        n = _native()
        self.n = n
        cfg = n.DitConfig(in_channels=m.input_channels, out_channels=m.output_channels, rows=m.grid_rows, cols=m.grid_cols,
                          past_len=m.past_len, future_len=m.future_len, t_patch=m.t_patch_size, patch=m.patch_size,
                          hidden=m.hidden_size, depth=m.depth, heads=m.num_heads, mlp_hidden=int(m.hidden_size * m.mlp_ratio),
                          time_multiple=m.time_multiple, table_steps=m.dif_time_embeddings.total_time_steps,
                          t_max_slots=m.temporal_pos_embed.shape[1])
        self.handle = C.c_void_p()
        n.check(n.lib().cm_dit_create(C.byref(cfg), C.byref(self.handle)))
        buf = C.create_string_buffer(256)
        shape = (C.c_int64 * 5)()
        nd = C.c_int()
        self.names = []
        for i in range(n.lib().cm_dit_param_count(self.handle)):
            n.check(n.lib().cm_dit_param_info(self.handle, i, buf, 256, shape, C.byref(nd)))
            self.names.append((buf.value.decode(), tuple(shape[j] for j in range(nd.value))))
        self._tensors = None
        self._bound: Optional[Tuple] = None
        self._versions: Optional[Tuple] = None
        self._ptr_array = None

    def invalidate(self):
        self._tensors = self._bound = self._versions = None

    def sync(self, m: "DiT4D_V4"):
        if self._tensors is None:
            sd = m.state_dict(keep_vars=True)
            missing = [nm for nm, _ in self.names if nm not in sd]
            if missing:
                raise RuntimeError(f"DiT4D_V4 state_dict lacks {missing[:3]}... expected by the native plan")
            self._tensors = [sd[nm] for nm, _ in self.names]
        ts = self._tensors
        ptrs = tuple(t.data_ptr() for t in ts)
        vers = tuple(t._version for t in ts)
        if ptrs == self._bound and vers == self._versions:
            return
        lib = self.n.lib()
        if ptrs != self._bound:
            for (name, shape), t in zip(self.names, ts):
                if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
                    raise RuntimeError(f"DiT4D_V4 parameter '{name}' must be a contiguous fp32 CUDA tensor (got {t.dtype} on "
                                       f"{t.device}); move the module with .to('cuda')")
                if tuple(t.shape) != tuple(shape):
                    raise RuntimeError(f"DiT4D_V4 parameter '{name}': shape {tuple(t.shape)} != plan {tuple(shape)}")
            arr = (C.c_void_p * len(ptrs))(*ptrs)
            self.n.check(lib.cm_dit_bind_params(self.handle, arr, len(ptrs)))
            self._ptr_array = arr
        self.n.check(lib.cm_dit_pack(self.handle, self.n.current_stream()))
        self._bound, self._versions = ptrs, vers

    def __del__(self):
        try:
            if self.handle:
                self.n.lib().cm_dit_destroy(self.handle)
        except Exception:
            pass


class DiT4D_V4(nn.Module):
    """DiT backbone with partial temporal tube patching + factorised attention (native sm_100a execution).
    Mirrors UNet's forward signature: forward(future, t, past) -> predicted noise."""

    def __init__(self, input_channels: int = 4, output_channels: int = 4, grid_rows: int = 12, grid_cols: int = 36,
                 past_len: int = 5, future_len: int = 3, t_patch_size: int = 2, patch_size: int = 4, hidden_size: int = 256,
                 depth: int = 6, num_heads: int = 4, mlp_ratio: float = 4.0, dropout_rate: float = 0.1, time_multiple: int = 4,
                 total_time_steps: int = 1000, condition: str = "Past", T_max: int = 32):
        super().__init__()
        assert hidden_size % num_heads == 0
        assert (past_len + future_len) % t_patch_size == 0, \
            f"T_total={past_len + future_len} must be divisible by t_patch={t_patch_size}"
        self.condition = condition
        self.input_channels, self.output_channels = input_channels, output_channels
        self.grid_rows, self.grid_cols = grid_rows, grid_cols
        self.past_len, self.future_len = past_len, future_len
        self.t_patch_size, self.patch_size = t_patch_size, patch_size
        self.hidden_size, self.depth, self.num_heads, self.mlp_ratio = hidden_size, depth, num_heads, mlp_ratio
        self.dropout_rate, self.time_multiple = dropout_rate, time_multiple
        T_total = past_len + future_len
        self.T_p = T_total // t_patch_size
        self.query_slot_start = past_len // t_patch_size
        time_emb_dims_exp = hidden_size * time_multiple
        # registration order == reference (DiT4D_V4.py:263-309): identical state_dict and RNG use
        self.dif_time_embeddings = SinusoidalPositionEmbeddings(total_time_steps=total_time_steps, time_emb_dims=hidden_size,
                                                                time_emb_dims_exp=time_emb_dims_exp)
        self.time_proj = nn.Sequential(nn.Linear(time_emb_dims_exp, hidden_size), nn.SiLU())
        self.patch_embed = PatchEmbed4D(grid_rows, grid_cols, T_total, patch_size, t_patch_size, input_channels, hidden_size)
        self.N_s = self.patch_embed.h_patches * self.patch_embed.w_patches
        self.spatial_pos_embed = nn.Parameter(torch.zeros(1, self.N_s, hidden_size))
        nn.init.trunc_normal_(self.spatial_pos_embed, std=0.02)
        self.temporal_pos_embed = nn.Parameter(torch.zeros(1, T_max // t_patch_size, hidden_size))
        nn.init.trunc_normal_(self.temporal_pos_embed, std=0.02)
        self.blocks = nn.ModuleList([DiTBlockCA(hidden_size=hidden_size, num_heads=num_heads, N_s=self.N_s, T_p=self.T_p,
                                                query_slot_start=self.query_slot_start, mlp_ratio=mlp_ratio,
                                                dropout_rate=dropout_rate) for _ in range(depth)])
        self.final_layer = FinalLayer(hidden_size, patch_size, output_channels, t_patch_size)
        self._init_weights()

    def _init_weights(self):
        for m in self.modules():
            if isinstance(m, nn.Linear):
                nn.init.xavier_uniform_(m.weight)
                if m.bias is not None:
                    nn.init.zeros_(m.bias)
            elif isinstance(m, (nn.Conv2d, nn.Conv3d)):
                nn.init.xavier_uniform_(m.weight.view(m.weight.size(0), -1))
                if m.bias is not None:
                    nn.init.zeros_(m.bias)

    # ------------------------------------------------------------------ native plumbing
    def _apply(self, fn, *args, **kwargs):
        _PLANS.pop(self, None)          # .to()/.cuda()/.float() replace parameter storage
        return super()._apply(fn, *args, **kwargs)

    def _plan(self) -> _DitPlan:
        plan = _PLANS.get(self)
        if plan is None:
            plan = _PLANS[self] = _DitPlan(self)
        return plan

    def invalidate_native_cache(self):
        """Call after modifying parameters through ``p.data`` (such writes do not bump ``_version``)."""
        if self in _PLANS:
            _PLANS[self].invalidate()

    def _check(self, future, past):
        for t in (future, past):
            if t is not None and not t.is_cuda:
                raise RuntimeError("crowdmod-ddpm-4d_b200 has no CPU path: DiT4D_V4 tensors must live on a CUDA (B200, sm_100a) device")
        if self.condition != "Past" or past is None:
            raise NotImplementedError("DiT4D_V4 native plan covers condition='Past' (the only value the reference configs use)")
        want_f = (self.output_channels, self.grid_rows, self.grid_cols, self.future_len)
        want_p = (self.input_channels, self.grid_rows, self.grid_cols, self.past_len)
        if tuple(future.shape[1:]) != want_f or tuple(past.shape[1:]) != want_p:
            raise ValueError(f"DiT4D_V4 was built for future {want_f} / past {want_p}, got {tuple(future.shape[1:])} / {tuple(past.shape[1:])}")

    # ------------------------------------------------------------------ reference API
    def forward(self, future: torch.Tensor, t: torch.Tensor, past: torch.Tensor = None) -> torch.Tensor:
        """future [B,C,H,W,F] fp32, t [B] int64, past [B,C,H,W,P] fp32 -> predicted noise [B,C,H,W,F]."""
        self._check(future, past)
        if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            raise NotImplementedError("training the DiT4D_V4 backbone natively is not built (forward / sampling only); wrap "
                                      "inference in torch.no_grad()")
        n = _native()
        plan = self._plan()
        plan.sync(self)
        future = future.contiguous().float()
        past = past.contiguous().float()
        t = t.contiguous().to(torch.int64)
        B = future.shape[0]
        eps = torch.empty_like(future)
        n.check(n.lib().cm_dit_forward(plan.handle, n.ptr(future), n.ptr(t), n.ptr(past), n.ptr(eps), B, n.current_stream()))
        return eps

    @torch.no_grad()
    def sample_chain(self, past, x, tsteps, coef, mode=0, noise=None, seed=0, sample_offset=0, history=None, use_graph=True):
        """Runs len(tsteps) reverse steps in place on ``x`` (same contract as ``UNet.sample_chain``)."""
        self._check(x, past)
        n = _native()
        plan = self._plan()
        plan.sync(self)
        graph_mode = 0 if use_graph in (False, 0, "eager") else 1     # one captured step, replayed nsteps times
        a, tsteps, coef = n.chain_args(past, x, tsteps, coef, mode, noise, seed, sample_offset, history, graph_mode)
        n.check(n.lib().cm_dit_sample(plan.handle, C.byref(a), n.current_stream()))
        return x

    def native_stats(self, *_):
        """(kernel launches of the last forward / chain, algorithmic FLOPs per sample) of the native plan."""
        n = _native()
        h = self._plan().handle
        return int(n.lib().cm_dit_last_launches(h)), float(n.lib().cm_dit_flops_per_sample(h))
