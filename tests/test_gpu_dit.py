"""GPU parity of the second backbone, DiT4D_V4 (SURVEY.md section 8 f2), through the C ABI (cm_dit_forward /
cm_dit_sample) against the golden vectors generated from the unmodified reference and against oracle/dit_oracle.py
(pinned to the live reference).  Gates as for the UNet: per-step eps rel-L2 <= 1e-3 (fp16 operands, hi + lo weights,
fp32 accumulation), chains with the same injected noise rel-L2 <= 5e-3."""
import numpy as np
import pytest
import torch

from oracle import ddpm_oracle as do
from oracle import dit_oracle as dto
from tests._util import build_dit, load_golden, rel_l2

pytestmark = pytest.mark.gpu


def _den(sd, kw):
    return lambda x, t, p: dto.dit_forward(sd, x, t, p, patch=kw["patch_size"], t_patch=kw["t_patch_size"],
                                           heads=kw["num_heads"], depth=kw["depth"])


@pytest.mark.parametrize("name", ["dit_atc_b2", "dit_small_b3"])
def test_dit_eps_vs_reference_golden(name):
    import crowdmod_ddpm_4d_b200._native as nat
    meta, a = load_golden(name)
    net, _ = build_dit(meta)
    net = net.cuda().eval()
    with torch.no_grad():
        eps = net(a["future"].cuda(), torch.tensor(meta["t"]).cuda(), a["past"].cuda()).cpu()
    assert nat.lib().cm_device_error() == 0
    e = rel_l2(eps, a["eps"])
    print(f"{name}: eps rel-L2 vs reference golden = {e:.3e}")
    assert e <= 1e-3
    assert eps.shape == a["eps"].shape


def test_dit_eps_vs_oracle_at_bench_batch_and_batch_invariance():
    """B = 64 (the BASELINE sampling batch) against the oracle; every sample equals its own B = 1 evaluation bit for
    bit up to the GEMM tile position (checked to 1e-5), and a batch permutation permutes the output."""
    meta, _ = load_golden("dit_atc_b2")
    net, sd = build_dit(meta)
    net = net.cuda().eval()
    kw = meta["kw"]
    B = 64
    g = torch.Generator().manual_seed(5)
    fut = torch.randn(B, 3, kw["grid_rows"], kw["grid_cols"], kw["future_len"], generator=g)
    past = do.synthetic_macroprops(B, 3, kw["grid_rows"], kw["grid_cols"], kw["past_len"], 9)
    t = torch.randint(0, 1000, (B,), generator=g)
    with torch.no_grad():
        ref = _den(sd, kw)(fut, t, past)
        eps = net(fut.cuda(), t.cuda(), past.cuda()).cpu()
        perm = torch.randperm(B, generator=g)
        eps_p = net(fut[perm].cuda(), t[perm].cuda(), past[perm].cuda()).cpu()
    e = rel_l2(eps, ref)
    worst = max(rel_l2(eps[i], ref[i]) for i in range(B))
    print(f"DiT B=64: eps rel-L2 vs oracle = {e:.3e}, worst sample {worst:.3e}")
    assert e <= 1e-3 and worst <= 1.5e-3
    assert rel_l2(eps_p, eps[perm]) <= 1e-5


@pytest.mark.parametrize("mode", ["DDPM", "DDIM", "Sparsity"])
def test_dit_chain_vs_oracle(mode):
    """12-step reverse chains with injected noise (reference loops models/diffusion/ddpm.py:206-282) and the update
    fused into the un-patch kernel."""
    from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import DDPM, ddim_coefficients, ddpm_coefficients
    meta, _ = load_golden("dit_small_b3")
    net, sd = build_dit(meta)
    net = net.cuda().eval()
    kw = meta["kw"]
    T, n = 12, 3
    s = do.schedule(T, 0.5)
    g = torch.Generator().manual_seed(3)
    shape = (n, 3, kw["grid_rows"], kw["grid_cols"], kw["future_len"])
    past = do.synthetic_macroprops(n, 3, kw["grid_rows"], kw["grid_cols"], kw["past_len"], 21)
    x_T = torch.randn(shape, generator=g)
    den = _den(sd, kw)
    sampler = DDPM(timesteps=T, scale=0.5)
    guidance, lam = ("Sparsity", 0.1) if mode == "Sparsity" else ("None", 0.0)
    with torch.no_grad():
        if mode == "DDIM":
            taus = np.arange(0, T - 1, 3)
            zs = [torch.randn(shape, generator=g) for _ in range(len(taus))]
            ref = do.generate_ddim(den, s, past, x_T, zs, taus, 0.001)
            ref = ref[0] if isinstance(ref, tuple) else ref
            ts, coef = ddim_coefficients(sampler, taus, 0.001)
            m = 1
        else:
            zs = [torch.randn(shape, generator=g) for _ in range(T)]
            ref, _ = do.generate_ddpm(den, s, past, x_T, zs, guidance=guidance, lam=lam)
            ts, coef = ddpm_coefficients(sampler, guidance, lam)
            m = 0
    x = x_T.cuda().contiguous()
    noise = torch.stack(zs[:ts.numel()]).cuda().contiguous()
    net.sample_chain(past.cuda().contiguous(), x, ts, coef, mode=m, noise=noise)
    torch.cuda.synchronize()
    e = rel_l2(x.cpu(), ref)
    print(f"DiT chain {mode}: x0 rel-L2 vs oracle = {e:.3e}")
    assert e <= 5e-3


def test_dit_philox_chain_is_deterministic_and_shard_invariant():
    from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import DDPM, ddpm_coefficients
    meta, _ = load_golden("dit_small_b3")
    net, _ = build_dit(meta)
    net = net.cuda().eval()
    kw = meta["kw"]
    ts, coef = ddpm_coefficients(DDPM(timesteps=8, scale=0.5))
    past = do.synthetic_macroprops(4, 3, kw["grid_rows"], kw["grid_cols"], kw["past_len"], 1).cuda()
    x_T = torch.randn(4, 3, kw["grid_rows"], kw["grid_cols"], kw["future_len"], generator=torch.Generator().manual_seed(0)).cuda()
    run = lambda p, x, off: net.sample_chain(p.contiguous(), x.clone().contiguous(), ts, coef, mode=0, seed=77, sample_offset=off)
    a, b = run(past, x_T, 0), run(past, x_T, 0)
    assert torch.equal(a, b)
    lo, hi = run(past[:2], x_T[:2], 0), run(past[2:], x_T[2:], 2)     # two shards with global Philox offsets
    assert torch.equal(torch.cat([lo, hi]), a)
    assert not torch.equal(run(past, x_T, 1), a)


def _dit_chain_inputs(meta, n=3):
    kw = meta["kw"]
    shape = (n, 3, kw["grid_rows"], kw["grid_cols"], kw["future_len"])
    past = do.synthetic_macroprops(n, 3, kw["grid_rows"], kw["grid_cols"], kw["past_len"], 4).cuda().contiguous()
    return past, torch.randn(shape, generator=torch.Generator().manual_seed(2)).cuda()


def test_dit_eager_equals_step_graph_with_history():
    """The eager chain and the captured step replayed nsteps times enqueue the same kernels: bitwise-equal x_0 and
    history (Philox noise, Sparsity guidance), and the same launch count."""
    from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import DDPM, ddpm_coefficients
    meta, _ = load_golden("dit_small_b3")
    net, _ = build_dit(meta)
    net = net.cuda().eval()
    ts, coef = ddpm_coefficients(DDPM(timesteps=8, scale=0.5), "Sparsity", 0.1)
    past, x_T = _dit_chain_inputs(meta)
    runs = []
    for use_graph in ("eager", True):
        x = x_T.clone()
        hist = torch.zeros((ts.numel() + 1,) + tuple(x.shape), device="cuda")
        net.sample_chain(past, x, ts, coef, mode=0, seed=9, history=hist, use_graph=use_graph)
        runs.append((x, hist, net.native_stats()[0]))
    (xe, he, le), (xg, hg, lg) = runs
    assert torch.equal(xe, xg) and torch.equal(he[1:], hg[1:]) and torch.equal(hg[-1], xg)
    assert le == lg > 0


def test_dit_same_length_schedules_back_to_back_equal_a_fresh_handle():
    """As for the UNet: a second schedule of the same length on the same handle (new tsteps / coef, same graph shape)
    equals the same chain on a fresh handle."""
    from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import DDPM, ddpm_coefficients
    meta, _ = load_golden("dit_small_b3")
    ts_a, coef_a = ddpm_coefficients(DDPM(timesteps=6, scale=0.5))
    ts_b, coef_b = (v[:6] for v in ddpm_coefficients(DDPM(timesteps=8, scale=0.5)))
    past, x_T = _dit_chain_inputs(meta)

    def run(net, ts, coef):
        x = x_T.clone()
        net.sample_chain(past, x, ts, coef, mode=0, seed=5)
        return x

    net = build_dit(meta)[0].cuda().eval()
    first = run(net, ts_a, coef_a)
    second = run(net, ts_b, coef_b)
    assert torch.equal(second, run(build_dit(meta)[0].cuda().eval(), ts_b, coef_b))
    assert not torch.equal(first, second)


def test_dit_driver_and_training_guard():
    """DDPM_model(arch='DDPM-DiT') builds the backbone from the reference's config keys (ddpm.py:88-104) and samples;
    a training forward raises instead of silently running something else."""
    import types
    from crowdmod_ddpm_4d_b200.models.backbones.DiT4D_V4 import DiT4D_V4
    from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import DDPM, DDPM_model
    ns = types.SimpleNamespace
    dit = ns(CONDITION="Past", PATCH_SIZE=4, T_PATCH_SIZE=4, HIDDEN_SIZE=128, DEPTH=2, NUM_HEADS=4, MLP_RATIO=4.0,
             DROPOUT_RATE=0.1, TIME_EMB_MULT=4,
             TRAIN=ns(EPOCHS=1, SOLVER=ns(LR=1e-4, WEIGHT_DECAY=3e-3, BETAS=[0.5, 0.999],
                                          SCHEDULER=ns(FACTOR=0.5, PATIENCE=10, MIN_LR=1e-6))))
    cfg = ns(MACROPROPS=ns(ROWS=12, COLS=36, EPS=1e-6), DATASET=ns(PAST_LEN=5, FUTURE_LEN=3, BATCH_SIZE=4),
             MODEL=ns(NSAMPLES=4, DDPM=ns(TIMESTEPS=6, SCALE=0.5, SIGMA=0.001, DDIM_DIVIDER=2, GUIDANCE="None", SAMPLER="DDPM",
                                          CHECKPOINTS_TO_KEEP=1, DIT=dit)),
             DATA_FS=ns(SAVE_DIR="/tmp/", OUTPUT_DIR="/tmp/"))
    torch.manual_seed(0)
    model = DDPM_model(cfg, "DDPM-DiT", 3)
    assert isinstance(model.denoiser, DiT4D_V4)
    past = do.synthetic_macroprops(4, 3, 12, 36, 5, 2).cuda()
    x, _ = model._generate_ddpm(past, DDPM(timesteps=6, scale=0.5).to("cuda"), 4)
    assert x.shape == (4, 3, 12, 36, 3) and torch.isfinite(x).all()
    model.denoiser.train()
    with pytest.raises(NotImplementedError):
        model.denoiser(torch.randn(4, 3, 12, 36, 3, device="cuda"), torch.zeros(4, dtype=torch.long, device="cuda"), past)
