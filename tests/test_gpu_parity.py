"""GPU parity proper: the CUDA path, called through the reference-facing Python API (which goes
through the C ABI), against (a) the golden vectors generated from the unmodified reference and
(b) the CPU oracle on the same seeded inputs.

Tolerances (BASELINE.json north_star): per-step eps rel-L2 <= 1e-3 (fp16 operands, fp32
accumulate); full chain with identical injected noise: elementwise rel-L2 <= 5e-3 and
per-channel mean/std within 1e-2 * std_ref (SURVEY.md §8d).
"""
import numpy as np
import pytest
import torch

from oracle import ddpm_oracle as do
from oracle import unet_oracle as uo
from tests._util import build_unet, chain_noise, load_golden, rel_l2, structure

pytestmark = pytest.mark.gpu

EPS_TOL = 1e-3


@pytest.fixture(scope="module", autouse=True)
def _no_device_errors():
    import crowdmod_ddpm_4d_b200._native as n
    yield
    assert n.lib().cm_device_error() == 0, "a kernel reported a protocol error"


@pytest.mark.parametrize("name", ["unet_atc_b2", "unet_small_b3", "unet_hermes_b1"])
def test_unet_forward_vs_reference_golden(name):
    meta, a = load_golden(name)
    net = build_unet(meta).cuda().eval()
    with torch.no_grad():
        eps = net(a["future"].cuda(), a["t"].cuda(), a["past"].cuda())
    e = rel_l2(eps.cpu(), a["eps"])
    print(f"{name}: eps rel-L2 vs reference golden = {e:.3e}")
    assert e <= EPS_TOL


def test_unet_forward_vs_oracle_fresh_inputs_b5():
    """Seeded inputs the goldens do not cover: odd batch (ragged last M-tiles), extreme t."""
    meta, _ = load_golden("unet_atc_b2")
    net = build_unet(meta)
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    g = torch.Generator().manual_seed(77)
    B = 5
    future = torch.randn(B, 3, 12, 36, 3, generator=g) * 3.0
    past = do.synthetic_macroprops(B, 3, 12, 36, 5, 99)
    t = torch.tensor([0, 1, 499, 998, 999])
    with torch.no_grad():
        ref = uo.unet_forward(sd, future, t, past, **structure(meta))
        net = net.cuda().eval()
        eps = net(future.cuda(), t.cuda(), past.cuda())
    assert rel_l2(eps.cpu(), ref) <= EPS_TOL
    for b in range(B):                                  # per-sample, not only in aggregate
        assert rel_l2(eps[b].cpu(), ref[b]) <= 2 * EPS_TOL


def test_empty_and_single_sample_batches():
    """Edge cases of the drop-in surface: an empty batch returns an empty tensor (as the reference's torch ops do) from the
    forward and from the fused chain; a single sample equals the same sample inside a batch of 3 bit for bit."""
    meta, a = load_golden("unet_atc_b2")
    net = build_unet(meta).cuda().eval()
    fut, past, t = a["future"].cuda(), a["past"].cuda(), a["t"].cuda()
    with torch.no_grad():
        e0 = net(fut[:0], t[:0], past[:0])
        assert e0.shape == (0,) + tuple(fut.shape[1:]) and e0.dtype == torch.float32
        from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import DDPM, ddpm_coefficients
        ts, coef = ddpm_coefficients(DDPM(timesteps=4, scale=0.5))
        x0 = fut[:0].clone().contiguous()
        assert net.sample_chain(past[:0].contiguous(), x0, ts, coef, mode=0, seed=1).shape[0] == 0
        one = net(fut[:1], t[:1], past[:1])
        three = net(fut[:1].repeat(3, 1, 1, 1, 1), t[:1].repeat(3), past[:1].repeat(3, 1, 1, 1, 1))
    assert torch.equal(one[0], three[0]) and torch.equal(one[0], three[2])
    assert rel_l2(one.cpu(), a["eps"][:1]) <= EPS_TOL


def test_unet_forward_vs_oracle_at_baseline_batch_64():
    """eps against the CPU oracle at the BASELINE batch (config/ATC.yml, B = 64): full SM fill, every persistent
    CTA walks several units, ragged last wave -- the regime bench.py times.  Gate per sample as well."""
    meta, _ = load_golden("unet_atc_b2")
    net = build_unet(meta)
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    g = torch.Generator().manual_seed(64)
    B = 64
    future = torch.randn(B, 3, 12, 36, 3, generator=g)
    past = do.synthetic_macroprops(B, 3, 12, 36, 5, 640)
    t = torch.randint(0, 1000, (B,), generator=g)
    with torch.no_grad():
        ref = uo.unet_forward(sd, future, t, past, **structure(meta))
        eps = net.cuda().eval()(future.cuda(), t.cuda(), past.cuda()).cpu()
    e = rel_l2(eps, ref)
    worst = max(rel_l2(eps[b], ref[b]) for b in range(B))
    print(f"B=64: eps rel-L2 vs oracle = {e:.3e}, worst sample {worst:.3e}")
    assert e <= EPS_TOL
    assert worst <= 1.5 * EPS_TOL


def test_production_batch_1280_forward_and_chain():
    """generate_metrics' default chain batch (config/ATC.yml MODEL.NSAMPLES = 1280, reference
    generate_metrics.py:53-58): ~20 GB workspace, 20x the units per launch.  The batch holds 20 copies of 64
    distinct samples.  Copies inside ONE launch are bit-identical (a sample's result does not depend on where
    it sits in the batch); against the B=64 launch they agree only to the eps tolerance class: a different
    batch size changes tile / slice shapes, hence fp32 summation orders, and a 1e-7 difference flips fp16
    operand roundings downstream (measured, tools/batch_divergence.py: 5e-7 after the first conv grows to
    ~6e-4 at the output -- the same size as the fp16-operand error against the oracle itself).  Two samples
    are checked against the oracle, and a short whole-chain graph must stay finite and shard-consistent."""
    from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import DDPM, ddpm_coefficients
    meta, _ = load_golden("unet_atc_b2")
    net = build_unet(meta)
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    net = net.cuda().eval()
    g = torch.Generator().manual_seed(1280)
    x64 = torch.randn(64, 3, 12, 36, 3, generator=g)
    p64 = do.synthetic_macroprops(64, 3, 12, 36, 5, 1281)
    t64 = torch.randint(0, 1000, (64,), generator=g)
    with torch.no_grad():
        e64 = net(x64.cuda(), t64.cuda(), p64.cuda())
        big = net(x64.repeat(20, 1, 1, 1, 1).cuda(), t64.repeat(20).cuda(), p64.repeat(20, 1, 1, 1, 1).cuda())
        ref = uo.unet_forward(sd, x64[:2], t64[:2], p64[:2], **structure(meta))
    assert big.shape == (1280, 3, 12, 36, 3) and torch.isfinite(big).all()
    for r in range(1, 20):
        assert torch.equal(big[64 * r:64 * (r + 1)], big[:64]), r
    d = rel_l2(big[:64], e64)
    print(f"n=1280 vs B=64 launch on the same samples: rel-L2 {d:.3e}; vs oracle {rel_l2(big[:2].cpu(), ref):.3e}")
    assert d <= 1.5 * EPS_TOL
    assert rel_l2(big[:2].cpu(), ref) <= EPS_TOL
    # short chain at n = 1280 (whole-chain graph), Philox noise, against the same chain on the first 64 samples
    T = 6
    ts, coef = ddpm_coefficients(DDPM(timesteps=T, scale=0.5))
    gx = torch.Generator(device="cuda").manual_seed(3)
    xT = torch.randn(1280, 3, 12, 36, 3, device="cuda", generator=gx)
    past = p64.repeat(20, 1, 1, 1, 1).cuda().contiguous()
    xa = xT.clone()
    net.sample_chain(past, xa, ts, coef, mode=0, seed=77, sample_offset=0)
    xb = xT[:64].clone()
    net.sample_chain(past[:64].contiguous(), xb, ts, coef, mode=0, seed=77, sample_offset=0)
    torch.cuda.synchronize()
    assert torch.isfinite(xa).all()
    assert rel_l2(xa[:64], xb) <= 2e-4


def test_forward_is_batch_permutation_equivariant_full_size():
    """Size-independent property at the BASELINE batch (64): every sample is independent
    (GroupNorm / attention are per-sample), so permuting the batch permutes the output exactly,
    and duplicated samples give bit-identical rows."""
    meta, _ = load_golden("unet_atc_b2")
    net = build_unet(meta).cuda().eval()
    g = torch.Generator(device="cuda").manual_seed(5)
    B = 64
    x = torch.randn(B, 3, 12, 36, 3, device="cuda", generator=g)
    past = torch.randn(B, 3, 12, 36, 5, device="cuda", generator=g)
    x[1], past[1] = x[0], past[0]
    t = torch.full((B,), 123, device="cuda", dtype=torch.long)
    perm = torch.randperm(B, device="cuda", generator=g)
    with torch.no_grad():
        a = net(x, t, past).clone()
        b = net(x[perm].contiguous(), t, past[perm].contiguous())
    assert torch.equal(a[0], a[1])
    assert torch.equal(a[perm], b)
    assert torch.isfinite(a).all()


def _run_chain(meta, a, use_graph=True, history=False):
    from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import DDPM, ddim_coefficients, ddpm_coefficients
    net = build_unet(meta).cuda().eval()
    x_T, zs = chain_noise(meta)
    sampler = DDPM(timesteps=meta["T"], scale=meta["scale"])
    lam = meta["lambda"] if meta["guidance"] == "Sparsity" else 0.0
    if meta["sampler"] == "DDPM":
        ts, coef = ddpm_coefficients(sampler, meta["guidance"], lam)
        zs = zs + [torch.zeros_like(x_T)]               # slot for t = 0 (never read: coef 0)
        mode = 0
    else:
        taus = np.arange(0, meta["T"] - 1, meta["divider"])
        ts, coef = ddim_coefficients(sampler, taus, meta["sigma"], meta["guidance"], lam)
        mode = 1
    noise = torch.stack(zs).cuda().contiguous()
    x = x_T.cuda().contiguous()
    hist = torch.zeros((len(ts) + 1,) + tuple(x.shape), device="cuda") if history else None
    net.sample_chain(a["past"].cuda().contiguous(), x, ts, coef, mode=mode, noise=noise, history=hist,
                     use_graph=use_graph)
    torch.cuda.synchronize()
    return x.cpu(), hist


@pytest.mark.parametrize("name", ["chain_small_ddpm", "chain_small_sparsity", "chain_small_ddim", "chain_atc_T16"])
def test_chain_vs_reference_golden(name):
    meta, a = load_golden(name)
    x0, _ = _run_chain(meta, a)
    ref = a["x0"]
    e = rel_l2(x0, ref)
    print(f"{name}: x0 rel-L2 vs reference golden = {e:.3e}")
    assert e <= 5e-3
    for c in range(3):
        sd = ref[:, c].std().item()
        assert abs(x0[:, c].mean().item() - ref[:, c].mean().item()) <= 1e-2 * sd
        assert abs(x0[:, c].std().item() - sd) <= 1e-2 * sd


def test_full_1000_step_chain_statistics_vs_reference_golden():
    """north_star gate 3: the FULL T = 1000 chain of config/ATC.yml (n = 2) with the reference's own injected
    noise (x_T, then one z per step, SURVEY.md §3.3; reference loop models/diffusion/ddpm.py:206-236): per-channel
    mean / std of x_0 within 1e-2 * std_ref, elementwise rel-L2 <= 5e-3 (random-init chains end at std ~ 20)."""
    meta, a = load_golden("chain_atc_T1000")
    assert meta["T"] == 1000 and meta["n"] == 2
    x0, _ = _run_chain(meta, a)
    ref = a["x0"]
    e = rel_l2(x0, ref)
    print(f"chain_atc_T1000: x0 rel-L2 vs reference golden = {e:.3e}")
    for c in range(3):
        sd = ref[:, c].std().item()
        dm = abs(x0[:, c].mean().item() - ref[:, c].mean().item()) / sd
        ds = abs(x0[:, c].std().item() - sd) / sd
        print(f"  channel {c}: |d mean| = {dm:.2e} std_ref, |d std| = {ds:.2e} std_ref (std_ref {sd:.3f})")
        assert dm <= 1e-2 and ds <= 1e-2
    assert e <= 5e-3


def test_chain_graph_replay_equals_eager_launches_and_history():
    meta, a = load_golden("chain_small_ddpm")
    xg, hg = _run_chain(meta, a, use_graph="chain", history=True)
    xs, hs = _run_chain(meta, a, use_graph="step", history=True)
    xe, he = _run_chain(meta, a, use_graph=False, history=True)
    assert torch.equal(xg, xe) and torch.equal(xs, xe)
    assert torch.equal(hg[1:], he[1:]) and torch.equal(hs[1:], he[1:])
    assert torch.equal(hg[-1].cpu(), xg)


def test_whole_chain_is_one_graph_launch_and_survives_new_seeds_and_buffers():
    """The T-step loop is ONE cudaGraphLaunch (conditional WHILE node); the seed, the shard offset and the
    x / past buffers travel through device memory the handle owns, so a new seed or freshly allocated
    tensors re-use the instantiated graph (no re-capture), and equal seeds give equal chains."""
    from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import DDPM, ddpm_coefficients
    meta, _ = load_golden("unet_small_b3")
    net = build_unet(meta).cuda().eval()
    geo = (4, 4, 2, 2)
    ts, coef = ddpm_coefficients(DDPM(timesteps=9, scale=0.5))
    n = 5
    past = torch.randn(n, 3, 4, 4, 2, device="cuda")
    xT = torch.randn(n, 3, 4, 4, 2, device="cuda")
    outs = []
    for i, seed in enumerate([11, 12, 11]):
        x = xT.clone()                                   # a fresh buffer every call
        p = past.clone()
        net.sample_chain(p, x, ts, coef, mode=0, seed=seed, use_graph="chain")
        launches, rebuilt = net.last_chain_graph_stats(*geo)
        assert launches == 1
        assert rebuilt == (i == 0), (i, rebuilt)
        outs.append(x.clone())
    torch.cuda.synchronize()
    assert torch.equal(outs[0], outs[2]) and not torch.equal(outs[0], outs[1])
    x = xT.clone()
    net.sample_chain(past, x, ts, coef, mode=0, seed=11, use_graph="step")
    assert net.last_chain_graph_stats(*geo) == (9, True)
    assert torch.equal(x, outs[0])


def test_same_length_schedules_back_to_back_equal_a_fresh_handle():
    """One handle runs two different schedules of the same length back to back: the schedule tables are uploaded only
    when they change, so the second chain must see the new tsteps / coef and equal the same chain on a fresh handle."""
    from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import DDPM, ddpm_coefficients
    meta, _ = load_golden("unet_small_b3")
    ts_a, coef_a = ddpm_coefficients(DDPM(timesteps=6, scale=0.5))
    ts_b, coef_b = (v[:6] for v in ddpm_coefficients(DDPM(timesteps=8, scale=0.5)))
    g = torch.Generator(device="cuda").manual_seed(8)
    past = torch.randn(3, 3, 4, 4, 2, device="cuda", generator=g)
    xT = torch.randn(3, 3, 4, 4, 2, device="cuda", generator=g)

    def run(net, ts, coef):
        x = xT.clone()
        net.sample_chain(past, x, ts, coef, mode=0, seed=5)
        return x

    net = build_unet(meta).cuda().eval()
    first = run(net, ts_a, coef_a)
    second = run(net, ts_b, coef_b)
    assert torch.equal(second, run(build_unet(meta).cuda().eval(), ts_b, coef_b))
    assert not torch.equal(first, second)


def test_philox_noise_is_standard_normal_and_shard_invariant():
    """One chain step with coefficients {A=0, C=1} returns exactly the injected z: checks the
    in-kernel Philox/Box-Muller stream and that it depends on the GLOBAL sample index only."""
    meta, _ = load_golden("unet_small_b3")
    net = build_unet(meta).cuda().eval()
    n = 64
    past = torch.zeros(n, 3, 4, 4, 2, device="cuda")
    ts = torch.tensor([5], dtype=torch.int32)
    coef = torch.zeros(1, 8)
    coef[0, 2] = 1.0
    x = torch.zeros(n, 3, 4, 4, 2, device="cuda")
    net.sample_chain(past, x, ts, coef, mode=0, seed=1234, sample_offset=0)
    z = x.clone()
    assert abs(z.mean().item()) < 0.05 and abs(z.std().item() - 1.0) < 0.05
    assert abs((z ** 4).mean().item() - 3.0) < 0.5
    x2 = torch.zeros(n // 2, 3, 4, 4, 2, device="cuda")
    net.sample_chain(past[: n // 2].contiguous(), x2, ts, coef, mode=0, seed=1234, sample_offset=n // 2)
    assert torch.equal(x2, z[n // 2:])
    x3 = torch.zeros(n, 3, 4, 4, 2, device="cuda")
    net.sample_chain(past, x3, ts, coef, mode=0, seed=1235, sample_offset=0)
    assert not torch.equal(x3, z)


def test_ddpm_model_generate_api():
    """The reference-facing driver: DDPM_model._generate_ddpm / _generate_ddim signatures."""
    import os
    from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import DDPM, DDPM_model
    from crowdmod_ddpm_4d_b200.utils.myparser import getYamlConfig
    cfg = getYamlConfig(os.path.join(os.path.dirname(__file__), "configs", "atc_nested.yml"))
    cfg.MODEL.DDPM.TIMESTEPS = 6
    torch.manual_seed(42)
    m = DDPM_model(cfg, "DDPM-UNet", 3)
    assert m.device.type == "cuda"
    sampler = DDPM(timesteps=6, scale=0.5).to(m.device)
    past = do.synthetic_macroprops(4, 3, 12, 36, 5, 1).cuda()
    x, hist = m._generate_ddpm(past, sampler, 4)
    assert x.shape == (4, 3, 12, 36, 3) and len(hist) == 2 and torch.isfinite(x).all()
    x, hist = m._generate_ddpm(past, sampler, 4, history=True)
    assert len(hist) == 7 and torch.equal(hist[-1], x)
    cfg.MODEL.DDPM.GUIDANCE = "Sparsity"
    x, _ = m._generate_ddim(past, np.arange(0, 5, 2), sampler, 4)
    assert torch.isfinite(x).all()
    cfg.MODEL.DDPM.GUIDANCE = "mass_preservation"
    with pytest.raises(NotImplementedError):
        m._generate_ddpm(past, sampler, 4)


# ---------------------------------------------------------------------------------------------
# every BASELINE.json config shape (SURVEY.md §8d): forward + one training step against the CPU
# oracle at a small batch.  ATC and HERMES-CR-120 forwards are also pinned by reference goldens
# above; ATC_medium (base 64, 16 frames, attention S=108, dh=64) and ETH-UCY (8x12 grid, attention
# S=12) have no golden of their own, so the oracle (itself pinned against the reference) is the
# checker.
# ---------------------------------------------------------------------------------------------
BASELINE_SHAPES = {
    "ATC_medium": dict(base=64, rows=12, cols=36, P=8, F=8, attn=[False, False, True]),
    "ETHUCY_ddpm": dict(base=32, rows=8, cols=12, P=5, F=3, attn=[False, False, True, False]),
    "HERMES-CR-120": dict(base=32, rows=28, cols=24, P=5, F=3, attn=[False, False, True, False]),
}


@pytest.mark.parametrize("name", list(BASELINE_SHAPES))
def test_baseline_config_shape_forward_and_train_step_vs_oracle(name):
    import torch.nn.functional as F
    from crowdmod_ddpm_4d_b200.models.backbones.unet import UNet
    c = BASELINE_SHAPES[name]
    kw = dict(input_channels=3, output_channels=3, num_res_blocks=1, base_channels=c["base"],
              base_channels_multiples=[1, 2, 4], apply_attention=c["attn"], dropout_rate=0.0,
              time_multiple=4, condition="Past")
    torch.manual_seed(7)
    net = UNet(**kw)
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    B = 2
    past = do.synthetic_macroprops(B, 3, c["rows"], c["cols"], c["P"], 21)
    fut = do.synthetic_macroprops(B, 3, c["rows"], c["cols"], c["F"], 22)
    g = torch.Generator().manual_seed(23)
    x = torch.randn(fut.shape, generator=g)
    t = torch.tensor([3, 871])
    st = dict(num_res_blocks=1, num_levels=3)
    with torch.no_grad():
        ref = uo.unet_forward(sd, x, t, past, **st)
        eps = net.cuda().eval()(x.cuda(), t.cuda(), past.cuda()).cpu()
    e = rel_l2(eps, ref)
    print(f"{name}: eps rel-L2 vs oracle = {e:.3e}")
    assert e <= EPS_TOL
    # one training step: loss + global gradient vector
    s = do.schedule(1000, 0.5)
    noise = torch.randn(fut.shape, generator=g)
    sdg = {k: v.detach().clone().requires_grad_(v.dtype.is_floating_point and "time_blocks.0" not in k)
           for k, v in sd.items()}
    loss_ref = do.train_loss(lambda a, b, p: uo.unet_forward(sdg, a, b, p, **st), s, fut, past, t, noise)
    loss_ref.backward()
    net.train()
    loss = F.mse_loss(net(do.q_sample(s, fut, t, noise).cuda(), t.cuda(), past.cuda()), noise.cuda())
    loss.backward()
    torch.cuda.synchronize()
    num = den = 0.0
    for k, p in net.named_parameters():
        if p.grad is None:
            continue
        num += (p.grad.cpu().double() - sdg[k].grad.double()).pow(2).sum().item()
        den += sdg[k].grad.double().pow(2).sum().item()
    eg = (num / den) ** 0.5
    print(f"{name}: loss {loss.item():.6f} vs {loss_ref.item():.6f}, global grad rel-L2 = {eg:.3e}")
    assert abs(loss.item() - loss_ref.item()) <= 1e-3 * abs(loss_ref.item())
    # north_star: "training loss and gradients within 1e-3" -- the same GRAD_TOL as tests/test_gpu_train.py.
    # (Round 1 measured 1.11e-3 on the smallest grid with single-fp16 dOut operands in dgrad; the data-gradient
    # convs now take a K-concatenated hi|lo fp16 pair, cm_unet_config.dgrad_terms = 2.)
    assert eg <= 1e-3
