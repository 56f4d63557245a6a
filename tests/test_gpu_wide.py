"""Wide models: attention heads of 66 ... 128 channels (the streaming tcgen05 forward and the deterministic fp32 backward
of attn_long.cu at every S) and UNet training at base_channels 96 / 128 / 256 (first and final conv weight gradients
through the packed conv weight-gradient kernels), against the CPU oracles with the gates of test_gpu_attn_long.py,
test_gpu_train.py and test_gpu_parity.py."""
import types

import pytest
import torch
import torch.nn.functional as F

from oracle import ddpm_oracle as do
from oracle import dit_oracle as dto
from oracle import unet_oracle as uo
from tests._util import rel_l2

pytestmark = pytest.mark.gpu

EPS_TOL = 1e-3
GRAD_TOL = 1e-3
CHAIN_TOL = 5e-3


@pytest.fixture(scope="module")
def nat():
    import crowdmod_ddpm_4d_b200._native as n
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    n.lib()
    yield n
    assert n.lib().cm_device_error() == 0, "a kernel reported a protocol error"


def _split(x, B, S, C, heads):
    dh = C // heads
    return [t.reshape(B, S, heads, dh).transpose(1, 2) for t in x.split(C, dim=2)]


OP_CASES = [(S, dh) for dh in (66, 96, 128) for S in (1, 54, 64, 128, 129, 168, 432)]


@pytest.mark.parametrize("S,dh", OP_CASES)
def test_attn_core_wide_head_forward_and_backward(nat, S, dh):
    heads = 4
    C_ = heads * dh
    B = 1 + OP_CASES.index((S, dh)) % 3
    g = torch.Generator(device="cuda").manual_seed(13 * S + dh)
    qkv = torch.randn(B, S, 3 * C_, device="cuda", generator=g)
    dctx = torch.randn(B, S, C_, device="cuda", generator=g)
    ctx = torch.zeros(B, S, C_, device="cuda", dtype=torch.half)
    nat.check(nat.lib().cm_op_attn_core(nat.ptr(qkv), nat.ptr(ctx), B, S, C_, heads, nat.current_stream()))
    dqkv = torch.full((B, S, 3 * C_), float("nan"), device="cuda")
    nat.check(nat.lib().cm_op_attn_core_backward(nat.ptr(qkv), nat.ptr(dctx), nat.ptr(dqkv), B, S, C_, heads,
                                                 nat.current_stream()))
    torch.cuda.synchronize()
    x = qkv.double().requires_grad_(True)
    q, k, v = _split(x, B, S, C_, heads)
    p = torch.softmax((q @ k.transpose(-1, -2)) / dh ** 0.5, dim=-1)
    ref = (p @ v).transpose(1, 2).reshape(B, S, C_)
    ref.backward(dctx.double())
    e = rel_l2(ctx.float(), ref.detach())
    print(f"S={S} dh={dh} B={B}: ctx rel-L2 {e:.3e}")
    assert e <= 7e-4
    assert torch.isfinite(dqkv).all()
    for name, sl in (("dQ", slice(0, C_)), ("dK", slice(C_, 2 * C_)), ("dV", slice(2 * C_, 3 * C_))):
        # S = 1: one key, so dQ and dK are zero up to the rounding of P (dP - D cancels); measured against the whole
        # gradient instead
        den = x.grad.norm().item() if S == 1 else x.grad[..., sl].norm().item()
        eg = (dqkv[..., sl].double() - x.grad[..., sl]).norm().item() / den
        print(f"S={S} dh={dh}: {name} rel-L2 {eg:.3e}")
        assert eg <= 1e-5, f"{name} rel-L2 {eg:.3e}"
    if (S, dh) == (168, 128):
        again = torch.empty_like(ctx)
        nat.check(nat.lib().cm_op_attn_core(nat.ptr(qkv), nat.ptr(again), B, S, C_, heads, nat.current_stream()))
        dagain = torch.empty_like(dqkv)
        nat.check(nat.lib().cm_op_attn_core_backward(nat.ptr(qkv), nat.ptr(dctx), nat.ptr(dagain), B, S, C_, heads,
                                                     nat.current_stream()))
        torch.cuda.synchronize()
        assert torch.equal(ctx, again)
        assert torch.equal(dqkv, dagain), "attention backward is not deterministic"


# B: ATC geometry, base 128 (S = 54, dh = 128 at level 2 and in the bottleneck); C: ATC, base 96 (dh = 96);
# D: HERMES 28 x 24 with 8 + 8 frames, base 128 (S = 168, dh = 128: two key tiles);
# E: ATC, base 256, mult [1, 2] (S = 432, dh = 128; the first conv's weight gradient on wgrad_umma with 256 output
#    channels, the final conv's on wgrad_umma with 256 input channels)
MULT3, ATTN3 = [1, 2, 4], [False, False, True, False]
MODELS = {
    "B_atc_base128": dict(rows=12, cols=36, P=5, F=3, base=128, mult=MULT3, attn=ATTN3),
    "C_atc_base96": dict(rows=12, cols=36, P=5, F=3, base=96, mult=MULT3, attn=ATTN3),
    "D_hermes_base128": dict(rows=28, cols=24, P=8, F=8, base=128, mult=MULT3, attn=ATTN3),
    "E_atc_base256_mult12": dict(rows=12, cols=36, P=5, F=3, base=256, mult=[1, 2], attn=[False, True]),
}


def _st(c):
    return dict(num_res_blocks=1, num_levels=len(c["mult"]))


def _unet(c, seed=7, dropout=0.0):
    from crowdmod_ddpm_4d_b200.models.backbones.unet import UNet
    torch.manual_seed(seed)
    net = UNet(input_channels=3, output_channels=3, num_res_blocks=1, base_channels=c["base"],
               base_channels_multiples=c["mult"], apply_attention=c["attn"], dropout_rate=dropout,
               time_multiple=4, condition="Past")
    return net, {k: v.clone() for k, v in net.state_dict().items()}


def _masks(base, B, g):
    """One Dropout3d keep-mask / (1 - p) per ResnetBlock in plan order (num_res_blocks = 1, mult [1, 2, 4]), p = 0.1."""
    blocks = [("encoder_blocks.0", 1), ("encoder_blocks.2", 2), ("encoder_blocks.4", 4), ("bottleneck_blocks.0", 4),
              ("bottleneck_blocks.1", 4), ("decoder_blocks.0", 4), ("decoder_blocks.1", 4), ("decoder_blocks.3", 2),
              ("decoder_blocks.4", 2), ("decoder_blocks.6", 1), ("decoder_blocks.7", 1)]
    return {k: (torch.rand(B, m * base, generator=g) >= 0.1).float() / 0.9 for k, m in blocks}


@pytest.mark.parametrize("name", list(MODELS))
def test_wide_unet_forward_train_step_and_chain_vs_oracle(nat, name):
    from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import DDPM, ddpm_coefficients
    c = MODELS[name]
    ST = _st(c)
    dropout = 0.1 if c["base"] == 96 else 0.0
    net, sd = _unet(c, dropout=dropout)
    B = 2
    past = do.synthetic_macroprops(B, 3, c["rows"], c["cols"], c["P"], 21)
    fut = do.synthetic_macroprops(B, 3, c["rows"], c["cols"], c["F"], 22)
    g = torch.Generator().manual_seed(23)
    x = torch.randn(fut.shape, generator=g)
    t = torch.tensor([3, 871])
    net = net.cuda()
    with torch.no_grad():
        ref = uo.unet_forward(sd, x, t, past, **ST)
        eps = net.eval()(x.cuda(), t.cuda(), past.cuda()).cpu()
    e = rel_l2(eps, ref)
    print(f"{name}: eps rel-L2 vs oracle = {e:.3e}")
    assert e <= EPS_TOL

    # one training step, per-tensor gradients (dropout masks injected into both sides where the model has dropout)
    masks = _masks(c["base"], B, g) if dropout else None
    s = do.schedule(1000, 0.5)
    noise = torch.randn(fut.shape, generator=g)
    sdg = {k: v.detach().clone().requires_grad_(v.dtype.is_floating_point and "time_blocks.0" not in k)
           for k, v in sd.items()}
    loss_ref = do.train_loss(lambda a, b, p: uo.unet_forward(sdg, a, b, p, drop_masks=masks, **ST), s, fut, past, t,
                             noise)
    loss_ref.backward()
    net.train()
    if masks is not None:
        net._injected_dropout = [m.cuda() for m in masks.values()]
    loss = F.mse_loss(net(do.q_sample(s, fut, t, noise).cuda(), t.cuda(), past.cuda()), noise.cuda())
    loss.backward()
    torch.cuda.synchronize()
    assert abs(loss.item() - loss_ref.item()) <= 1e-3 * abs(loss_ref.item())
    num = den = 0.0
    per = {}
    for k, p in net.named_parameters():
        assert (p.grad is None) == (sdg[k].grad is None), k
        if p.grad is None:
            continue
        go = sdg[k].grad.double()
        per[k] = ((p.grad.cpu().double() - go).pow(2).sum().item(), go.pow(2).sum().item())
        num += per[k][0]
        den += per[k][1]
    # tensors whose reference gradient is numerically zero (the k bias under the softmax shift) are compared in
    # absolute terms, as test_gpu_train.py does
    for k, (d, r) in per.items():
        if r ** 0.5 < 1e-9 * den ** 0.5:
            assert dict(net.named_parameters())[k].grad.double().norm().item() < 1e-6 * den ** 0.5, k
    worst, worst_k = max(((d / r) ** 0.5, k) for k, (d, r) in per.items() if r ** 0.5 >= 1e-9 * den ** 0.5)
    eg = (num / den) ** 0.5
    print(f"{name}: loss {loss.item():.6f} vs {loss_ref.item():.6f}, global grad rel-L2 {eg:.3e}, "
          f"worst tensor {worst_k} {worst:.3e}")
    assert eg <= GRAD_TOL
    assert worst <= GRAD_TOL, f"{worst_k}: gradient rel-L2 {worst:.3e}"
    for w in ("first.weight", "final.2.weight"):
        assert rel_l2(dict(net.named_parameters())[w].grad.cpu(), sdg[w].grad) <= GRAD_TOL, w

    # 16-step DDPM chain with injected noise
    T = 16
    sch = do.schedule(T, 0.5)
    x_T = torch.randn(fut.shape, generator=g)
    zs = [torch.randn(fut.shape, generator=g) for _ in range(T)]
    with torch.no_grad():
        x0_ref, _ = do.generate_ddpm(lambda a, b, p: uo.unet_forward(sd, a, b, p, **ST), sch, past, x_T, zs)
    ts, coef = ddpm_coefficients(DDPM(timesteps=T, scale=0.5))
    net.eval()
    xg = x_T.cuda().contiguous()
    net.sample_chain(past.cuda().contiguous(), xg, ts, coef, mode=0, noise=torch.stack(zs).cuda().contiguous())
    torch.cuda.synchronize()
    ec = rel_l2(xg.cpu(), x0_ref)
    print(f"{name}: 16-step chain x0 rel-L2 vs oracle = {ec:.3e}")
    assert ec <= CHAIN_TOL


@pytest.mark.parametrize("base", [96, 128])
def test_wide_train_step_through_driver_loss_decreases(nat, base):
    """DDPM_model._train_step + Adam on a fixed batch (same t and noise every step): the loss goes down."""
    from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import DDPM, DDPM_model
    c = dict(MODELS["B_atc_base128"], base=base)
    net, _ = _unet(c, seed=5, dropout=0.0)
    net = net.cuda().train()
    model = types.SimpleNamespace(denoiser=net)
    fs = DDPM(timesteps=1000, scale=0.5).cuda()
    opt = torch.optim.Adam(net.parameters(), lr=1e-4)
    B = 4
    past = do.synthetic_macroprops(B, 3, 12, 36, 5, 41).cuda()
    fut = do.synthetic_macroprops(B, 3, 12, 36, 3, 42).cuda()
    losses = []
    for _ in range(4):
        torch.manual_seed(17)
        loss = DDPM_model._train_step(model, fut, past, fs)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        losses.append(loss.item())
    print(f"base {base}: losses {losses}")
    assert all(torch.isfinite(torch.tensor(losses)))
    assert losses[-1] < losses[0], losses


def test_dit_hidden512_heads4_vs_oracle_and_chain(nat):
    """DDPM-DiT with hidden 512 and 4 heads (dh = 128) on the ATC geometry: 27 spatial patches per slot."""
    from crowdmod_ddpm_4d_b200.models.backbones.DiT4D_V4 import DiT4D_V4
    from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import DDPM, ddpm_coefficients
    kw = dict(input_channels=3, output_channels=3, grid_rows=12, grid_cols=36, past_len=5, future_len=3,
              t_patch_size=4, patch_size=4, hidden_size=512, depth=2, num_heads=4, mlp_ratio=4.0, dropout_rate=0.0,
              time_multiple=4)
    torch.manual_seed(3)
    net = DiT4D_V4(**kw)
    sd = dto.randomize_zero_init({k: v.detach().clone() for k, v in net.state_dict().items()}, 3)
    net.load_state_dict(sd)
    net = net.cuda().eval()
    B = 2
    g = torch.Generator().manual_seed(8)
    fut = torch.randn(B, 3, 12, 36, 3, generator=g)
    past = do.synthetic_macroprops(B, 3, 12, 36, 5, 12)
    t = torch.tensor([17, 640])
    den = lambda a, b, p: dto.dit_forward(sd, a, b, p, patch=4, t_patch=4, heads=4, depth=2)
    with torch.no_grad():
        ref = den(fut, t, past)
        eps = net(fut.cuda(), t.cuda(), past.cuda()).cpu()
    e = rel_l2(eps, ref)
    print(f"DiT hidden 512: eps rel-L2 vs oracle = {e:.3e}")
    assert e <= EPS_TOL
    T = 8
    sch = do.schedule(T, 0.5)
    x_T = torch.randn(fut.shape, generator=g)
    zs = [torch.randn(fut.shape, generator=g) for _ in range(T)]
    with torch.no_grad():
        x0_ref, _ = do.generate_ddpm(den, sch, past, x_T, zs)
    ts, coef = ddpm_coefficients(DDPM(timesteps=T, scale=0.5))
    xg = x_T.cuda().contiguous()
    net.sample_chain(past.cuda().contiguous(), xg, ts, coef, mode=0, noise=torch.stack(zs).cuda().contiguous())
    torch.cuda.synchronize()
    ec = rel_l2(xg.cpu(), x0_ref)
    print(f"DiT hidden 512: {T}-step chain x0 rel-L2 vs oracle = {ec:.3e}")
    assert ec <= CHAIN_TOL


def test_head_dim_above_128_still_raises(nat):
    """Head dim 256 (e.g. the default UNet()'s bottleneck: 1024 channels, 4 heads) comes back as an error through
    cm_last_error, not as a fallback."""
    B, S, heads, C_ = 1, 8, 4, 1024
    qkv = torch.zeros(B, S, 3 * C_, device="cuda")
    ctx = torch.zeros(B, S, C_, device="cuda", dtype=torch.half)
    rc = nat.lib().cm_op_attn_core(nat.ptr(qkv), nat.ptr(ctx), B, S, C_, heads, nat.current_stream())
    assert rc != 0
    assert b"head dim 256" in nat.lib().cm_last_error()
