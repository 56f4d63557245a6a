"""TEST INFRASTRUCTURE — generates tests/golden/*.npz by running the UNMODIFIED reference
(imported from a checkout of the original project through oracle/ref_shim.py) on CPU fp32.

Run where such a checkout exists:  python -m oracle.make_golden
The reference ships no golden vectors of its own (SURVEY.md §4, §8c); these files pin the
oracle restatement (tests/test_oracle_golden.py) and the CUDA path (tests/test_gpu_parity.py)
without it.

Weights are never stored: every case records the torch seed under which the reference's
``UNet(...)`` was constructed plus a SHA-256 of the resulting state_dict; the product ``UNet``
reproduces the same initialisation (same nn constructors, same order) and the tests check
the hash before using it.
"""
import hashlib
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import ref_shim  # noqa: E402
from oracle.ddpm_oracle import synthetic_macroprops  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def sd_hash(sd):
    h = hashlib.sha256()
    for k in sd:
        h.update(k.encode())
        h.update(sd[k].detach().cpu().contiguous().numpy().tobytes())
    return h.hexdigest()


ATC = dict(input_channels=3, output_channels=3, num_res_blocks=1, base_channels=32,
           base_channels_multiples=[1, 2, 4], apply_attention=[False, False, True, False],
           dropout_rate=0.1, time_multiple=4, condition="Past")
SMALL = dict(input_channels=3, output_channels=3, num_res_blocks=2, base_channels=32,
             base_channels_multiples=[1, 2], apply_attention=[True, True],
             dropout_rate=0.0, time_multiple=4, condition="Past")


def make_cfg(ns, unet_kw, rows, cols, P, F, T, scale, guidance="None", sampler="DDPM", sigma=0.001,
             divider=2, lam=0.004):
    E = ns.EasyDict
    return E({
        "MACROPROPS": {"ROWS": rows, "COLS": cols},
        "DATASET": {"PAST_LEN": P, "FUTURE_LEN": F, "BATCH_SIZE": 4},
        "DATA_FS": {"SAVE_DIR": "/tmp/", "OUTPUT_DIR": "/tmp/"},
        "MODEL": {"NAME": "{}_G_TE{}_PL{}_FL{}_CE{}_{}.pth", "NSAMPLES": 4, "NSAMPLES4PLOTS": 2,
                  "DDPM": {"SAMPLER": sampler, "TIMESTEPS": T, "SCALE": scale, "SIGMA": sigma,
                           "DDIM_DIVIDER": divider, "GUIDANCE": guidance, "LAMBDA_GUIDANCE": lam,
                           "CHECKPOINTS_TO_KEEP": 1,
                           "UNET": {"CONDITION": unet_kw["condition"], "NUM_RES_BLOCKS": unet_kw["num_res_blocks"],
                                    "BASE_CH": unet_kw["base_channels"],
                                    "BASE_CH_MULT": unet_kw["base_channels_multiples"],
                                    "APPLY_ATTENTION": unet_kw["apply_attention"],
                                    "DROPOUT_RATE": unet_kw["dropout_rate"],
                                    "TIME_EMB_MULT": unet_kw["time_multiple"],
                                    "TRAIN": {"EPOCHS": 1, "SOLVER": {
                                        "LR": 5e-5, "WEIGHT_DECAY": 3e-3, "BETAS": [0.5, 0.999],
                                        "SCHEDULER": {"FACTOR": 0.5, "PATIENCE": 10, "MIN_LR": 1e-6}}}}}},
    })


def save(name, meta, **arrays):
    os.makedirs(OUT, exist_ok=True)
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, meta=np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8),
                        **{k: np.asarray(v) for k, v in arrays.items()})
    print("wrote", path, os.path.getsize(path), "bytes")


def unet_case(ns, name, kw, seed, B, rows, cols, P, F, tvals):
    torch.manual_seed(seed)
    net = ns.UNet(**kw).eval()
    past = synthetic_macroprops(B, 3, rows, cols, P, 1234)
    g = torch.Generator().manual_seed(5)
    future = torch.randn(B, 3, rows, cols, F, generator=g)
    t = torch.tensor(tvals, dtype=torch.long)
    with torch.no_grad():
        eps = net(future, t, past)
    save(name, {"kind": "unet_forward", "unet": kw, "seed": seed, "sd_sha256": sd_hash(net.state_dict()),
                "rows": rows, "cols": cols, "P": P, "F": F, "past_seed": 1234, "future_seed": 5},
         future=future.numpy(), past=past.numpy(), t=t.numpy(), eps=eps.numpy())


def chain_case(ns, name, kw, seed, n, rows, cols, P, F, T, scale, guidance, sampler, divider=2, sigma=0.001):
    cfg = make_cfg(ns, kw, rows, cols, P, F, T, scale, guidance, sampler, sigma, divider)
    torch.manual_seed(seed)
    model = ns.DDPM_model(cfg, "DDPM-UNet", 3)
    model.device = torch.device("cpu")
    model.denoiser.to("cpu")
    sampler_mod = ns.DDPM(timesteps=T, scale=scale)
    past = synthetic_macroprops(n, 3, rows, cols, P, 1234)
    torch.manual_seed(seed + 1000)            # noise stream: x_T first, then one z per step
    if sampler == "DDPM":
        x0, _ = model._generate_ddpm(past, sampler_mod, n)
    else:
        taus = np.arange(0, T - 1, divider)
        x0, _ = model._generate_ddim(past, taus, sampler_mod, n)
    save(name, {"kind": "chain", "unet": kw, "seed": seed, "noise_seed": seed + 1000,
                "sd_sha256": sd_hash(model.denoiser.state_dict()), "rows": rows, "cols": cols, "P": P,
                "F": F, "T": T, "scale": scale, "guidance": guidance, "sampler": sampler,
                "divider": divider, "sigma": sigma, "lambda": 0.004, "n": n, "past_seed": 1234},
         past=past.numpy(), x0=x0.numpy())


def train_case(ns, name, kw, seed, B, rows, cols, P, F, T, scale):
    cfg = make_cfg(ns, kw, rows, cols, P, F, T, scale)
    torch.manual_seed(seed)
    model = ns.DDPM_model(cfg, "DDPM-UNet", 3)
    model.device = torch.device("cpu")
    model.denoiser.to("cpu").train()
    fs = ns.DDPM(timesteps=T, scale=scale)
    past = synthetic_macroprops(B, 3, rows, cols, P, 1234)
    future = synthetic_macroprops(B, 3, rows, cols, F, 4321)
    torch.manual_seed(seed + 2000)            # t = randint first, then eps = randn_like(future)
    loss = model._train_step(future, past, fs)
    model.optimizer.zero_grad(set_to_none=True)
    loss.backward()
    names, norms, proj = [], [], []
    g = torch.Generator().manual_seed(99)
    for k, p in model.denoiser.named_parameters():
        if p.grad is None:
            continue
        names.append(k)
        norms.append(p.grad.double().norm().item())
        r = torch.randn(p.shape, generator=g)
        proj.append((p.grad.double() * r.double()).sum().item())
    save(name, {"kind": "train_step", "unet": kw, "seed": seed, "rng_seed": seed + 2000,
                "sd_sha256": sd_hash(model.denoiser.state_dict()), "rows": rows, "cols": cols, "P": P,
                "F": F, "T": T, "scale": scale, "B": B, "names": names, "proj_seed": 99},
         past=past.numpy(), future=future.numpy(), loss=np.float64(loss.item()),
         grad_norms=np.array(norms), grad_proj=np.array(proj))


def schedule_case(ns):
    s = ns.ForwardSampler(timesteps=1000, scale=0.5)
    idx = np.array([0, 1, 10, 100, 500, 998, 999])
    save("schedule_T1000_s0p5", {"kind": "schedule", "T": 1000, "scale": 0.5},
         idx=idx, **{k: getattr(s, k).numpy()[idx] for k in
                     ("beta", "alpha", "alpha_bar", "sqrt_alpha_bar", "one_by_sqrt_alpha",
                      "sqrt_one_minus_alpha_bar")})


def metrics_case(ns, name, n, rows, cols, F, seed, chunk, eps):
    """Reduction metrics of the reference's MetricsGenerator (utils/metrics/metricsGenerator.py:120-186,293-339) on a
    seeded (pred, gt) pair; the pair itself is regenerated from the seed by oracle.metrics_oracle.synthetic_pair."""
    from oracle import metrics_oracle as mo
    pred, gt = mo.synthetic_pair(n, rows, cols, F, seed)
    params = ns.EasyDict({"MPROPS_COUNT": 3})
    gen = ns.MetricsGenerator([torch.from_numpy(p) for p in pred], [torch.from_numpy(g) for g in gt], params, None)
    with np.errstate(all="ignore"):
        gen.compute_psnr_metric(chunk, eps)
        gen.compute_psnr_metric(chunk, eps, masked_flag=True)
        gen.compute_re_density_metric(chunk, eps)
        gen.compute_tv_metric()
    keys = ["PSNR", "MAX_PSNR", "PSNR_OVER_TIME", "MAX_PSNR_OVER_TIME", "MASK_PSNR", "MAX_MASK_PSNR",
            "MASK_PSNR_OVER_TIME", "MAX_MASK_PSNR_OVER_TIME", "RE_DENSITY", "MIN_RE_DENSITY", "TV_OVER_TIME"]
    save(name, {"n": n, "rows": rows, "cols": cols, "F": F, "seed": seed, "chunk": chunk, "eps": eps,
                "ranges": [gen.rho_range, gen.vx_range, gen.vy_range]},
         **{k: gen.data_dict[k] for k in keys})


DIT_ATC = dict(input_channels=3, output_channels=3, grid_rows=12, grid_cols=36, past_len=5, future_len=3, t_patch_size=4,
               patch_size=4, hidden_size=256, depth=6, num_heads=4, mlp_ratio=4.0, dropout_rate=0.1, time_multiple=4)
DIT_SMALL = dict(input_channels=3, output_channels=3, grid_rows=8, grid_cols=12, past_len=4, future_len=4, t_patch_size=2,
                 patch_size=4, hidden_size=128, depth=2, num_heads=4, mlp_ratio=4.0, dropout_rate=0.1, time_multiple=4)


def dit_case(ns, name, kw, seed, B, tvals):
    """DiT4D_V4.forward of the unmodified reference (models/backbones/DiT4D_V4.py:348-375), eval mode, seeded init with
    the zero-initialised AdaLN / final projections filled by oracle.dit_oracle.randomize_zero_init (same seed)."""
    from oracle import dit_oracle as dto
    torch.manual_seed(seed)
    m = ns.DiT4D_V4(**kw).eval()
    init_hash = sd_hash(m.state_dict())
    sd = dto.randomize_zero_init({k: v.detach().clone() for k, v in m.state_dict().items()}, seed)
    m.load_state_dict(sd)
    g = torch.Generator().manual_seed(seed + 1)
    fut = torch.randn(B, kw["input_channels"], kw["grid_rows"], kw["grid_cols"], kw["future_len"], generator=g)
    from oracle import ddpm_oracle as _dpo
    past = _dpo.synthetic_macroprops(B, kw["input_channels"], kw["grid_rows"], kw["grid_cols"], kw["past_len"], seed + 2)
    t = torch.tensor(tvals)
    with torch.no_grad():
        eps = m(fut, t, past)
    save(name, {"kw": kw, "seed": seed, "B": B, "t": tvals, "init_sha256": init_hash, "n_keys": len(sd)},
         future=fut.numpy(), past=past.numpy(), eps=eps.numpy())


def main():
    """python -m oracle.make_golden [case ...]: regenerate every golden, or only the named ones."""
    ns = ref_shim.load()
    torch.set_num_threads(os.cpu_count())
    only = set(sys.argv[1:])
    if only:
        # the full 1000-step chain of BASELINE config #2 at n = 2 (north_star gate 3: output statistics of the
        # whole chain; reference loop models/diffusion/ddpm.py:206-236)
        if "chain_atc_T1000" in only:
            chain_case(ns, "chain_atc_T1000", ATC, 42, 2, 12, 36, 5, 3, 1000, 0.5, "None", "DDPM")
        if "metrics_small" in only:
            metrics_case(ns, "metrics_small", 8, 12, 36, 3, 7, 4, 1e-6)
        if "dit" in only:
            dit_case(ns, "dit_atc_b2", DIT_ATC, 42, 2, [7, 640])
            dit_case(ns, "dit_small_b3", DIT_SMALL, 11, 3, [0, 999, 31])
        return
    schedule_case(ns)
    unet_case(ns, "unet_atc_b2", ATC, 42, 2, 12, 36, 5, 3, [7, 640])
    unet_case(ns, "unet_small_b3", SMALL, 11, 3, 4, 4, 2, 2, [0, 999, 31])
    unet_case(ns, "unet_hermes_b1", ATC, 42, 1, 28, 24, 5, 3, [250])
    chain_case(ns, "chain_small_ddpm", SMALL, 11, 3, 4, 4, 2, 2, 12, 0.5, "None", "DDPM")
    chain_case(ns, "chain_small_sparsity", SMALL, 11, 3, 4, 4, 2, 2, 12, 0.5, "Sparsity", "DDPM")
    chain_case(ns, "chain_small_ddim", SMALL, 11, 3, 4, 4, 2, 2, 12, 0.5, "None", "DDIM", divider=3)
    chain_case(ns, "chain_atc_T16", ATC, 42, 2, 12, 36, 5, 3, 16, 0.5, "None", "DDPM")
    train_case(ns, "train_small", SMALL, 11, 3, 4, 4, 2, 2, 1000, 0.5)
    kw = dict(ATC, dropout_rate=0.0)
    train_case(ns, "train_atc_b2", kw, 42, 2, 12, 36, 5, 3, 1000, 0.5)
    chain_case(ns, "chain_atc_T1000", ATC, 42, 2, 12, 36, 5, 3, 1000, 0.5, "None", "DDPM")
    metrics_case(ns, "metrics_small", 8, 12, 36, 3, 7, 4, 1e-6)
    dit_case(ns, "dit_atc_b2", DIT_ATC, 42, 2, [7, 640])
    dit_case(ns, "dit_small_b3", DIT_SMALL, 11, 3, [0, 999, 31])


if __name__ == "__main__":
    main()
