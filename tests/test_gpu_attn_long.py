"""Attention over more than 128 tokens per (sample, head): the streaming tcgen05 forward (attn_long_kernel) and the
deterministic two-kernel backward, through the op entry points, the UNet plan (attention at finer levels of the
reference configs), the fused reverse chain and the DiT spatial attention (patch_size = 2 on HERMES)."""
import pytest
import torch

from oracle import ddpm_oracle as do
from oracle import dit_oracle as dto
from oracle import unet_oracle as uo
from tests._util import rel_l2

pytestmark = pytest.mark.gpu

EPS_TOL = 1e-3
GRAD_TOL = 1e-3


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


FWD_CASES = [(S, C) for S in (129, 168, 432, 777, 3456) for C in (32, 64, 128, 256)]


@pytest.mark.parametrize("S,C_", FWD_CASES)
def test_attn_core_long_forward(nat, S, C_):
    """dh = 8 ... 64, one to 27 query tiles, ragged last key tile; fp16 P / V / output as in the S <= 128 kernel."""
    B = 1 + FWD_CASES.index((S, C_)) % 3
    heads = 4
    g = torch.Generator(device="cuda").manual_seed(S + C_)
    qkv = torch.randn(B, S, 3 * C_, device="cuda", generator=g)
    ctx = torch.zeros(B, S, C_, device="cuda", dtype=torch.half)
    nat.check(nat.lib().cm_op_attn_core(nat.ptr(qkv), nat.ptr(ctx), B, S, C_, heads, nat.current_stream()))
    torch.cuda.synchronize()
    q, k, v = _split(qkv, B, S, C_, heads)
    p = torch.softmax((q @ k.transpose(-1, -2)) / (C_ // heads) ** 0.5, dim=-1)
    ref = (p @ v).transpose(1, 2).reshape(B, S, C_)
    e = rel_l2(ctx.float(), ref)
    print(f"S={S} C={C_} B={B}: ctx rel-L2 {e:.3e}")
    assert e <= 7e-4
    again = torch.empty_like(ctx)
    nat.check(nat.lib().cm_op_attn_core(nat.ptr(qkv), nat.ptr(again), B, S, C_, heads, nat.current_stream()))
    torch.cuda.synchronize()
    assert torch.equal(ctx, again)


@pytest.mark.parametrize("S,C_", [(S, C) for S in (129, 168, 432, 777) for C in (32, 64, 128, 256)])
def test_attn_core_long_backward_vs_float64_autograd(nat, S, C_):
    B = 2
    heads = 4
    g = torch.Generator(device="cuda").manual_seed(7 * S + C_)
    qkv = torch.randn(B, S, 3 * C_, device="cuda", generator=g)
    dctx = torch.randn(B, S, C_, device="cuda", generator=g)
    dqkv = torch.full((B, S, 3 * C_), float("nan"), device="cuda")
    nat.check(nat.lib().cm_op_attn_core_backward(nat.ptr(qkv), nat.ptr(dctx), nat.ptr(dqkv), B, S, C_, heads,
                                                 nat.current_stream()))
    torch.cuda.synchronize()
    x = qkv.double().requires_grad_(True)
    q, k, v = _split(x, B, S, C_, heads)
    p = torch.softmax((q @ k.transpose(-1, -2)) / (C_ // heads) ** 0.5, dim=-1)
    (p @ v).transpose(1, 2).reshape(B, S, C_).backward(dctx.double())
    assert torch.isfinite(dqkv).all()
    for name, sl in (("dQ", slice(0, C_)), ("dK", slice(C_, 2 * C_)), ("dV", slice(2 * C_, 3 * C_))):
        e = rel_l2(dqkv[..., sl].double(), x.grad[..., sl])
        print(f"S={S} C={C_}: {name} rel-L2 {e:.3e}")
        assert e <= 1e-5, f"{name} rel-L2 {e:.3e}"
    again = torch.empty_like(dqkv)
    nat.check(nat.lib().cm_op_attn_core_backward(nat.ptr(qkv), nat.ptr(dctx), nat.ptr(again), B, S, C_, heads,
                                                 nat.current_stream()))
    torch.cuda.synchronize()
    assert torch.equal(dqkv, again), "attention backward is not deterministic"


# attention tokens per level = rows * cols * frames / 8^level; base 32 puts dh = 8 / 16 / 32 at levels 0 / 1 / 2
LONG_SHAPES = {
    "HERMES_P8F8_attn_FFT": dict(rows=28, cols=24, P=8, F=8, attn=[False, False, True]),     # S = 168, dh = 32
    "ATC_P5F3_attn_FTT": dict(rows=12, cols=36, P=5, F=3, attn=[False, True, True]),        # S = 432 (dh 16) and 54
    "ETHUCY_P5F3_attn_TFT": dict(rows=8, cols=12, P=5, F=3, attn=[True, False, True]),      # S = 768, dh = 8
}
ST = dict(num_res_blocks=1, num_levels=3)


def _unet(c, seed=7):
    from crowdmod_ddpm_4d_b200.models.backbones.unet import UNet
    kw = dict(input_channels=3, output_channels=3, num_res_blocks=1, base_channels=32,
              base_channels_multiples=[1, 2, 4], apply_attention=c["attn"], dropout_rate=0.0,
              time_multiple=4, condition="Past")
    torch.manual_seed(seed)
    net = UNet(**kw)
    return net, {k: v.clone() for k, v in net.state_dict().items()}


@pytest.mark.parametrize("name", list(LONG_SHAPES))
def test_unet_long_attention_forward_and_train_step_vs_oracle(nat, name):
    import torch.nn.functional as F
    c = LONG_SHAPES[name]
    net, sd = _unet(c)
    B = 2
    past = do.synthetic_macroprops(B, 3, c["rows"], c["cols"], c["P"], 21)
    fut = do.synthetic_macroprops(B, 3, c["rows"], c["cols"], c["F"], 22)
    g = torch.Generator().manual_seed(23)
    x = torch.randn(fut.shape, generator=g)
    t = torch.tensor([3, 871])
    with torch.no_grad():
        ref = uo.unet_forward(sd, x, t, past, **ST)
        eps = net.cuda().eval()(x.cuda(), t.cuda(), past.cuda()).cpu()
    e = rel_l2(eps, ref)
    print(f"{name}: eps rel-L2 vs oracle = {e:.3e}")
    assert e <= EPS_TOL
    s = do.schedule(1000, 0.5)
    noise = torch.randn(fut.shape, generator=g)
    sdg = {k: v.detach().clone().requires_grad_(v.dtype.is_floating_point and "time_blocks.0" not in k)
           for k, v in sd.items()}
    loss_ref = do.train_loss(lambda a, b, p: uo.unet_forward(sdg, a, b, p, **ST), s, fut, past, t, noise)
    loss_ref.backward()
    net.train()
    loss = F.mse_loss(net(do.q_sample(s, fut, t, noise).cuda(), t.cuda(), past.cuda()), noise.cuda())
    loss.backward()
    torch.cuda.synchronize()
    assert abs(loss.item() - loss_ref.item()) <= 1e-3 * abs(loss_ref.item())
    num = den = 0.0
    worst, worst_k = 0.0, None
    for k, p in net.named_parameters():
        if p.grad is None:
            continue
        d = (p.grad.cpu().double() - sdg[k].grad.double()).pow(2).sum().item()
        r = sdg[k].grad.double().pow(2).sum().item()
        num += d
        den += r
        ek = (d / max(r, 1e-300)) ** 0.5
        if ek > worst:
            worst, worst_k = ek, k
    eg = (num / den) ** 0.5
    print(f"{name}: loss {loss.item():.6f} vs {loss_ref.item():.6f}, global grad rel-L2 {eg:.3e}, "
          f"worst tensor {worst_k} {worst:.3e}")
    assert eg <= GRAD_TOL
    assert worst <= GRAD_TOL, f"{worst_k}: gradient rel-L2 {worst:.3e}"


def test_long_attention_chain_vs_oracle_graph_and_permutation(nat):
    """T = 16 DDPM chain with injected noise on the ATC shape with attention at level 1 (S = 432): against the oracle's
    reverse loop, whole-chain graph == eager launches bit for bit, and a batch permutation permutes x_0 bit for bit."""
    from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import DDPM, ddpm_coefficients
    c = LONG_SHAPES["ATC_P5F3_attn_FTT"]
    net, sd = _unet(c, seed=11)
    net = net.cuda().eval()
    T, n = 16, 3
    s = do.schedule(T, 0.5)
    g = torch.Generator().manual_seed(5)
    shape = (n, 3, c["rows"], c["cols"], c["F"])
    past = do.synthetic_macroprops(n, 3, c["rows"], c["cols"], c["P"], 31)
    x_T = torch.randn(shape, generator=g)
    zs = [torch.randn(shape, generator=g) for _ in range(T)]
    with torch.no_grad():
        ref, _ = do.generate_ddpm(lambda a, b, p: uo.unet_forward(sd, a, b, p, **ST), s, past, x_T, zs)
    ts, coef = ddpm_coefficients(DDPM(timesteps=T, scale=0.5))
    noise = torch.stack(zs).cuda().contiguous()
    pg = past.cuda().contiguous()

    def run(p, x0, z, use_graph):
        x = x0.cuda().contiguous()
        net.sample_chain(p, x, ts, coef, mode=0, noise=z, use_graph=use_graph)
        torch.cuda.synchronize()
        return x.cpu()

    xg = run(pg, x_T, noise, "chain")
    e = rel_l2(xg, ref)
    print(f"long-attention chain: x0 rel-L2 vs oracle = {e:.3e}")
    assert e <= 5e-3
    assert torch.equal(run(pg, x_T, noise, False), xg)
    perm = torch.tensor([2, 0, 1])
    xp = run(pg[perm.cuda()].contiguous(), x_T[perm], noise[:, perm.cuda()].contiguous(), "chain")
    assert torch.equal(xp, xg[perm])


def test_dit_168_patches_vs_oracle_and_philox_chain(nat):
    """DDPM-DiT on HERMES 28 x 24 with patch_size 2: 14 * 12 = 168 spatial patches per temporal slot.  Four channels:
    the final layer's width t_patch * C * p^2 must be a multiple of 32 (64 here; 48 with three channels)."""
    from crowdmod_ddpm_4d_b200.models.backbones.DiT4D_V4 import DiT4D_V4
    from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import DDPM, ddpm_coefficients
    kw = dict(input_channels=4, output_channels=4, grid_rows=28, grid_cols=24, past_len=5, future_len=3,
              t_patch_size=4, patch_size=2, hidden_size=128, depth=2, num_heads=4, mlp_ratio=4.0, dropout_rate=0.0,
              time_multiple=4)
    torch.manual_seed(3)
    net = DiT4D_V4(**kw)
    sd = dto.randomize_zero_init({k: v.detach().clone() for k, v in net.state_dict().items()}, 3)
    net.load_state_dict(sd)
    net = net.cuda().eval()
    B = 2
    g = torch.Generator().manual_seed(8)
    fut = torch.randn(B, 4, 28, 24, 3, generator=g)
    past = do.synthetic_macroprops(B, 4, 28, 24, 5, 12)
    t = torch.tensor([17, 640])
    with torch.no_grad():
        ref = dto.dit_forward(sd, fut, t, past, patch=2, t_patch=4, heads=4, depth=2)
        eps = net(fut.cuda(), t.cuda(), past.cuda()).cpu()
    e = rel_l2(eps, ref)
    print(f"DiT Ns=168: eps rel-L2 vs oracle = {e:.3e}")
    assert e <= 1e-3
    ts, coef = ddpm_coefficients(DDPM(timesteps=6, scale=0.5))
    x_T = torch.randn(B, 4, 28, 24, 3, generator=g).cuda()
    run = lambda: net.sample_chain(past.cuda().contiguous(), x_T.clone().contiguous(), ts, coef, mode=0, seed=5)
    a, b = run(), run()
    assert torch.isfinite(a).all()
    assert torch.equal(a, b)
