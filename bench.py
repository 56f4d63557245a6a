#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native DDPM sampling hot path.

Metric (BASELINE.json): sampled sequences/sec for the FULL T-step reverse chain.
Workload at N=1: config/ATC.yml — 1000-step DDPM sampling, batch 64 per GPU, grid 12x36,
past 5 + future 3 frames, UNet base 32 / mult [1,2,4] / attention at the coarsest level,
pretrained-shape random-init weights (torch.manual_seed(42)), synthetic macroprops.

A "step" is ONE full reverse chain (T denoiser evaluations + T fused updates) over one batch.

  python bench.py --gpus N --steps K --warmup W            (native arm; torchrun for N>1)
  python bench.py --impl reference ...                     (CPU oracle port of the reference path)
  python bench.py ... --dump-outputs DIR                   (also writes x_0 of the last timed chain to DIR/x0.npy)

Prints ONE JSON line on rank 0.  Besides the contract keys it carries
  roofline      the tcgen05 conv class of one denoiser step: achieved = EXECUTED FLOPs / summed CUDA-event
                time (the UpSample convs count their 8-tap phase convs), algorithmic_equiv = the dense
                27-tap formulation of SURVEY.md §8(d) over the same time, reported separately
  train         BASELINE config #4 (HERMES-CR-120.yml training step) through DDPM_model
  extra         the other BASELINE configs / batches: n = 1280 (generate_metrics' production batch; under
                torchrun the 1280 samples are split over the ranks = strong scaling), ATC_medium (#3),
                ETH-UCY (#5); one timed chain each
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import torch

# the benchmark may run from a read-only tree: no bytecode caches next to the project's modules
sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

T_STEPS, SCALE = 1000, 0.5
UNIT = "sequences/s"
METRIC = "sampled sequences/sec (full T-step DDPM chain)"


def unet_kwargs(base=32, attn=(False, False, True, False)):
    return dict(input_channels=3, output_channels=3, num_res_blocks=1, base_channels=base,
                base_channels_multiples=[1, 2, 4], apply_attention=list(attn), dropout_rate=0.1,
                time_multiple=4, condition="Past")


# the five BASELINE.json configs by tensor shape (SURVEY.md §8d "Config -> shapes")
WORKLOADS = {
    "atc": dict(cfg="config/ATC.yml", rows=12, cols=36, past=5, fut=3, unet=unet_kwargs()),
    "atc_medium": dict(cfg="config/ATC_medium.yml", rows=12, cols=36, past=8, fut=8,
                       unet=unet_kwargs(64, (False, False, True))),
    "ethucy": dict(cfg="config/ETHUCY_ddpm.yml", rows=8, cols=12, past=5, fut=3, unet=unet_kwargs()),
    "hermes": dict(cfg="config/HERMES-CR-120.yml", rows=28, cols=24, past=5, fut=3, unet=unet_kwargs()),
}
ATC = WORKLOADS["atc"]["unet"]
ROWS, COLS, PAST, FUT = 12, 36, 5, 3


def synthetic_macroprops(n, channels, rows, cols, frames, seed, device="cpu"):
    """SURVEY.md §8(d): occupancy Bernoulli(0.2); rho = mask*(1+Poisson(0.5)); v = mask*N(0,0.5^2)."""
    g = torch.Generator().manual_seed(seed)
    mask = (torch.rand(n, 1, rows, cols, frames, generator=g) < 0.2).float()
    rho = mask * (1 + torch.poisson(torch.full_like(mask, 0.5), generator=g))
    v = mask * torch.randn(n, channels - 1, rows, cols, frames, generator=g) * 0.5
    return torch.cat([rho, v], dim=1).contiguous().to(device)


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"tflops_sustained": p.get("bf16_tflops_sustained", 1426.2),
                "tflops_burst": p.get("bf16_tflops", 1688.0), "hbm_gbs": p.get("hbm_gbs", 6455.6),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"tflops_sustained": 1400.0, "tflops_burst": 1590.0, "hbm_gbs": 6650.0,
            "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi sampling DURING the timed region (B200_PROFILING.md clocks line)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(gpu_index)], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
                for k, v in zip(names, r[5:9]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(k)
            except Exception:
                continue
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_oracle_sample(n, steps, threads):
    """Times `steps` denoiser+update iterations of the reference path's CPU restatement
    (oracle/) at batch n; returns seconds per iteration."""
    from oracle import ddpm_oracle as do
    from oracle import unet_oracle as uo
    from crowdmod_ddpm_4d_b200.models.backbones.unet import UNet
    torch.set_num_threads(threads)
    torch.manual_seed(42)
    sd = UNet(**ATC).state_dict()
    s = do.schedule(T_STEPS, SCALE)
    past = do.synthetic_macroprops(n, 3, ROWS, COLS, PAST, 1234)
    g = torch.Generator().manual_seed(42)
    x = torch.randn(n, 3, ROWS, COLS, FUT, generator=g)

    def one(x, t):
        tt = torch.full((n,), t, dtype=torch.long)
        eps = uo.unet_forward(sd, x, tt, past, num_res_blocks=1, num_levels=3)
        return do.ddpm_step(s, eps, x, t, torch.randn(x.shape, generator=g))

    with torch.no_grad():
        x = one(x, T_STEPS - 1)                       # warm-up
        t0 = time.perf_counter()
        for i in range(steps):
            x = one(x, T_STEPS - 2 - i)
        dt = (time.perf_counter() - t0) / steps
    return dt


def run_reference(args, rank, world):
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    n = args.batch
    it = args.ref_iters
    times = []
    for k in range(args.warmup + args.steps):
        dt = cpu_oracle_sample(n, it, threads)
        if k >= args.warmup:
            times.append(dt)
    s_per_iter = sum(times) / len(times)
    chain_s = s_per_iter * T_STEPS
    value = n / chain_s
    sample = (f"{it} denoiser+DDPM.step iterations at batch {n} per step (of the {T_STEPS}-step chain), "
              f"extrapolated x{T_STEPS}/{it}")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": chain_s * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic macroprops, random-init weights (seed 42)",
        "config": workload_config(n, args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(n, gpus):
    """Identical in both arms (the driver compares the two `config` objects)."""
    return {"workload": "config/ATC.yml: full 1000-step DDPM sampling, batch 64 per GPU, UNet base 32 "
                        "mult [1,2,4], grid 12x36, past 5 + future 3",
            "samples_per_gpu": n, "global_samples": n * gpus, "timesteps": T_STEPS,
            "parallelism": f"sample-sharded x{gpus}, no collective",
            "l2_flush": "256 MiB buffer written between timed chains; per-step working set (~1 GB) > L2",
            "noise": "in-kernel Philox (device-resident), x_T ~ N(0,I)"}


def make_cfg(name):
    """The nested MODEL.DDPM.UNET config (reference config/ATC.yml / HERMES-CR-120.yml schema) of a workload."""
    from crowdmod_ddpm_4d_b200.utils.myparser import YamlParser
    w = WORKLOADS[name]
    u = w["unet"]
    return YamlParser({
        "DATA_FS": {"OUTPUT_DIR": "/tmp/crowdmod_bench_out", "SAVE_DIR": "/tmp/crowdmod_bench_models/"},
        "MACROPROPS": {"ROWS": w["rows"], "COLS": w["cols"]},
        "DATASET": {"NAME": name, "PAST_LEN": w["past"], "FUTURE_LEN": w["fut"], "BATCH_SIZE": 64},
        "MODEL": {"NAME": "{}_B_TE{}_PL{}_FL{}_CE{}_{}.pth", "NSAMPLES": 1280, "NSAMPLES4PLOTS": 20,
                  "DDPM": {"SAMPLER": "DDPM", "TIMESTEPS": T_STEPS, "SCALE": SCALE, "SIGMA": 0.001,
                           "DDIM_DIVIDER": 2, "GUIDANCE": "None", "LAMBDA_GUIDANCE": 0.004,
                           "CHECKPOINTS_TO_KEEP": 7,
                           "UNET": {"CONDITION": "Past", "NUM_RES_BLOCKS": u["num_res_blocks"],
                                    "BASE_CH": u["base_channels"], "BASE_CH_MULT": u["base_channels_multiples"],
                                    "APPLY_ATTENTION": u["apply_attention"], "DROPOUT_RATE": u["dropout_rate"],
                                    "TIME_EMB_MULT": u["time_multiple"],
                                    "TRAIN": {"EPOCHS": 200, "SOLVER": {
                                        "LR": 5e-5, "WEIGHT_DECAY": 3e-3, "BETAS": [0.5, 0.999],
                                        "SCHEDULER": {"FACTOR": 0.5, "PATIENCE": 10, "MIN_LR": 1e-6}}}}}},
    })


def run_native(args, rank, world, local_rank):
    import torch.distributed as dist
    from crowdmod_ddpm_4d_b200 import _native as nat
    from crowdmod_ddpm_4d_b200.models.backbones.unet import UNet
    from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import DDPM, ddpm_coefficients

    if not torch.cuda.is_available():
        raise SystemExit("bench.py (native arm) needs a CUDA device: there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    n = args.batch
    torch.manual_seed(42)
    net = UNet(**ATC).to(dev).eval()
    sampler = DDPM(timesteps=args.timesteps, scale=SCALE)
    tsteps, coef = ddpm_coefficients(sampler)
    past_host = synthetic_macroprops(n, 3, ROWS, COLS, PAST, 1234 + rank).pin_memory()
    past = past_host.to(dev)
    gen = torch.Generator(device=dev).manual_seed(42 + rank)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    terms = int(os.environ.get("CROWDMOD_WEIGHT_TERMS", "2"))

    def chain_device(seed):
        x = torch.randn(n, 3, ROWS, COLS, FUT, device=dev, generator=gen)
        net.sample_chain(past, x, tsteps, coef, mode=0, seed=seed, sample_offset=rank * n, use_graph=True)
        return x

    x0_host = torch.empty(n, 3, ROWS, COLS, FUT).pin_memory()

    def chain_e2e(seed):
        """The call a user makes: host past in, host x_0 out (H2D + D2H inside the timed region)."""
        p = past_host.to(dev, non_blocking=True)
        x = torch.randn(n, 3, ROWS, COLS, FUT, device=dev, generator=gen)
        net.sample_chain(p, x, tsteps, coef, mode=0, seed=seed, sample_offset=rank * n, use_graph=True)
        x0_host.copy_(x, non_blocking=True)
        return x

    # ---- warm-up (graph capture, descriptor build, clocks) ----
    for w in range(max(args.warmup, 3)):
        chain_device(1000 + w)
    barrier()

    # ---- timed: device-resident inputs ----
    clocks = ClockSampler(local_rank) if rank == 0 else None
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    launches = 0
    graph_launches = 0
    rebuilt = 0
    x_last = None
    try:
        barrier()
        for k in range(args.steps):
            flush.fill_(k)
            ev[k][0].record()
            x_last = chain_device(k)
            ev[k][1].record()
            launches += net.last_chain_launches(ROWS, COLS, PAST, FUT)
            gl, rb = net.last_chain_graph_stats(ROWS, COLS, PAST, FUT)
            graph_launches += gl
            rebuilt += int(rb)
        barrier()
    finally:                                      # never leave the nvidia-smi sampler running
        clk = clocks.stop() if clocks else None
    ms = sum(a.elapsed_time(b) for a, b in ev)
    # ---- timed: end to end through the public call with host buffers ----
    chain_e2e(999)
    barrier()
    ev2 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for k in range(args.steps):
        flush.fill_(k)
        ev2[k][0].record()
        chain_e2e(k)
        ev2[k][1].record()
    barrier()
    ms_e2e = sum(a.elapsed_time(b) for a, b in ev2)

    t = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = t.tolist()

    roof = None
    if rank == 0:
        roof = roofline(net, nat, past, n, dev, ms / args.steps / args.timesteps)
    del net, flush
    torch.cuda.empty_cache()

    train = None
    if not args.no_train:
        train = train_bench(rank, world, dev, cpu_baseline=not args.no_cpu_baseline)
    extra = None
    if not args.no_extras:
        extra = extras_bench(rank, world, dev)

    if rank == 0:
        total = n * world * args.steps
        value = total / (ms / 1e3)
        e2e = total / (ms_e2e / 1e3)
        cfg = workload_config(n, world)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f16 operands, f32 accumulate",
            "data": "synthetic macroprops, random-init weights (seed 42)",
            "config": cfg,
            "weight_terms": terms,
            "denoiser_step_ms": ms / args.steps / args.timesteps,
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": past_host.numel() * 4,
                    "d2h_bytes_per_step": x0_host.numel() * 4},
            "gpu_launches": launches,
            "graph": {"cuda_graph_launches_in_timed_region": graph_launches, "chains": args.steps,
                      "graphs_rebuilt_in_timed_region": rebuilt,
                      "kind": "whole T-step chain = one graph (conditional WHILE node)"
                      if graph_launches == args.steps else "one graph per denoiser step, replayed T times"},
            "clocks": clk,
            "roofline": roof,
        }
        if train is not None:
            line["train"] = train
        if extra is not None:
            line["extra"] = extra
        if world == 1 and not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            s_it = cpu_oracle_sample(n, args.ref_iters, threads)
            line["cpu_baseline"] = {
                "value": n / (s_it * T_STEPS), "unit": UNIT, "cores": threads, "kind": "port",
                "sample": f"{args.ref_iters} denoiser+DDPM.step iterations at batch {n} on the host cores "
                          f"(oracle/ restatement of the reference CPU path), extrapolated to {T_STEPS} steps"}
        print(json.dumps(line), flush=True)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"x0": x_last})
    if world > 1:
        dist.destroy_process_group()


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Writes each output of the last timed step as out_dir/<name>.npy (float32), so that two builds run with the
    same arguments can be compared output for output.  The files stay within DUMP_MAX_BYTES in all: an array over
    its share keeps a fixed, seeded subset of its samples (leading dimension)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_MAX_BYTES // len(arrays)
    for name, t in arrays.items():
        a = t.detach().float().cpu().numpy()
        if a.nbytes > share:
            keep = share // (a.nbytes // a.shape[0])
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ---- other BASELINE configs / batches: one timed full chain each ------------------------------------------------
def extras_bench(rank, world, dev):
    import torch.distributed as dist
    from crowdmod_ddpm_4d_b200.models.backbones.unet import UNet
    from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import DDPM, ddpm_coefficients, shard_samples

    tsteps, coef = ddpm_coefficients(DDPM(timesteps=T_STEPS, scale=SCALE))
    ts_short, coef_short = ddpm_coefficients(DDPM(timesteps=8, scale=SCALE))

    def one(name, n_rank, offset, chains=1):
        w = WORKLOADS[name]
        torch.manual_seed(42)
        net = UNet(**w["unet"]).to(dev).eval()
        past = synthetic_macroprops(n_rank, 3, w["rows"], w["cols"], w["past"], 77 + rank, dev)
        gen = torch.Generator(device=dev).manual_seed(7 + rank)
        shape = (n_rank, 3, w["rows"], w["cols"], w["fut"])
        x = torch.randn(shape, device=dev, generator=gen)
        net.sample_chain(past, x, ts_short, coef_short, mode=0, seed=1, sample_offset=offset)     # warm-up
        x = torch.randn(shape, device=dev, generator=gen)
        net.sample_chain(past, x, tsteps, coef, mode=0, seed=2, sample_offset=offset)             # builds the T=1000 graph
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for c in range(chains):
            x = torch.randn(shape, device=dev, generator=gen)
            net.sample_chain(past, x, tsteps, coef, mode=0, seed=3 + c, sample_offset=offset)
        b.record()
        torch.cuda.synchronize()
        ms = torch.tensor([a.elapsed_time(b) / chains], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        fl = net.native_stats(w["rows"], w["cols"], w["past"], w["fut"])[1]
        finite = bool(torch.isfinite(x).all().item())
        del net, past, x
        torch.cuda.empty_cache()
        return ms.item(), fl, finite

    out = {}
    # (1) the production batch of generate_metrics (config/ATC.yml MODEL.NSAMPLES = 1280): strong scaling --
    #     the 1280 samples are split over the ranks, global Philox offsets
    lo, hi = shard_samples(1280, rank, world)
    ms, fl, ok = one("atc", hi - lo, lo)
    out["atc_n1280"] = {"workload": "config/ATC.yml generate_metrics batch: ONE 1000-step chain of 1280 samples "
                                    f"split over {world} GPU(s)", "scaling": "strong", "samples": 1280,
                        "chain_ms": ms, "sequences_per_s": 1280 / (ms * 1e-3),
                        "denoiser_step_ms": ms / T_STEPS, "algorithmic_tflops": fl * 1280 * T_STEPS / (ms * 1e-3) / 1e12,
                        "finite": ok}
    # (2) BASELINE config #3: ATC_medium (base 64, 8+8 frames, attention S=108), 64 samples per GPU, no collective
    ms, fl, ok = one("atc_medium", 64, rank * 64)
    out["atc_medium"] = {"workload": "config/ATC_medium.yml: 1000-step chain, 64 samples per GPU, base 64, past 8 + future 8",
                         "scaling": "weak", "samples": 64 * world, "chain_ms": ms,
                         "sequences_per_s": 64 * world / (ms * 1e-3), "denoiser_step_ms": ms / T_STEPS,
                         "algorithmic_tflops": fl * 64 * world * T_STEPS / (ms * 1e-3) / 1e12, "finite": ok}
    # (3) BASELINE config #5: ETH-UCY (8x12 grid, attention S=12), 64 samples per GPU
    ms, fl, ok = one("ethucy", 64, rank * 64, chains=2)
    out["ethucy"] = {"workload": "config/ETHUCY_ddpm.yml: 1000-step chain, 64 samples per GPU, grid 8x12, past 5 + future 3",
                     "scaling": "weak", "samples": 64 * world, "chain_ms": ms,
                     "sequences_per_s": 64 * world / (ms * 1e-3), "denoiser_step_ms": ms / T_STEPS,
                     "algorithmic_tflops": fl * 64 * world * T_STEPS / (ms * 1e-3) / 1e12, "finite": ok}
    # (4) the second backbone (--arch DDPM-DiT, config/ATC.yml MODEL.DDPM.DIT): 1000-step chain, 64 samples per GPU
    out["dit_atc"] = dit_bench(rank, world, dev, tsteps, coef)
    if rank == 0:
        out.update(feed_and_metrics_bench(dev))
    return out


def dit_bench(rank, world, dev, tsteps, coef):
    """DiT4D_V4 (reference models/backbones/DiT4D_V4.py, config/ATC.yml: patch 4, t_patch 4, hidden 256, depth 6, 4 heads)
    through cm_dit_sample: weak scaling, no collective.  The CPU baseline is the oracle port of the same forward."""
    import torch.distributed as dist
    from crowdmod_ddpm_4d_b200.models.backbones.DiT4D_V4 import DiT4D_V4
    w = WORKLOADS["atc"]
    kw = dict(input_channels=3, output_channels=3, grid_rows=w["rows"], grid_cols=w["cols"], past_len=w["past"],
              future_len=w["fut"], t_patch_size=4, patch_size=4, hidden_size=256, depth=6, num_heads=4, mlp_ratio=4.0,
              dropout_rate=0.1, time_multiple=4)
    torch.manual_seed(42)
    net = DiT4D_V4(**kw).to(dev).eval()
    n = 64
    past = synthetic_macroprops(n, 3, w["rows"], w["cols"], w["past"], 77 + rank, dev)
    gen = torch.Generator(device=dev).manual_seed(7 + rank)
    shape = (n, 3, w["rows"], w["cols"], w["fut"])
    x = torch.randn(shape, device=dev, generator=gen)
    net.sample_chain(past, x, tsteps[:8], coef[:8], mode=0, seed=1, sample_offset=rank * n)      # warm-up
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    x = torch.randn(shape, device=dev, generator=gen)
    t0 = time.perf_counter()
    a.record()
    net.sample_chain(past, x, tsteps, coef, mode=0, seed=3, sample_offset=rank * n)
    b.record()
    t_issue = time.perf_counter() - t0
    torch.cuda.synchronize()
    ms = torch.tensor([a.elapsed_time(b)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    launches, fl = net.native_stats()
    # one forward alone (device events) for the denoiser-step figure without the host loop
    t = torch.full((n,), 500, device=dev, dtype=torch.long)
    with torch.no_grad():
        net(x, t, past)
        torch.cuda.synchronize()
        a.record()
        for _ in range(20):
            net(x, t, past)
        b.record()
        torch.cuda.synchronize()
    fwd_ms = a.elapsed_time(b) / 20
    res = {"workload": "config/ATC.yml MODEL.DDPM.DIT (DiT4D_V4: patch 4, t_patch 4, hidden 256, depth 6, 4 heads): 1000-step "
                       "chain, 64 samples per GPU", "scaling": "weak", "samples": n * world, "chain_ms": ms.item(),
           "sequences_per_s": n * world / (ms.item() * 1e-3), "denoiser_step_ms": ms.item() / T_STEPS,
           "forward_ms_device": fwd_ms, "host_issue_ms_per_step": t_issue * 1e3 / T_STEPS,
           "launches_per_step": launches // T_STEPS, "algorithmic_gflop_per_sample_step": fl / 1e9,
           "algorithmic_tflops": fl * n * world * T_STEPS / (ms.item() * 1e-3) / 1e12, "finite": bool(torch.isfinite(x).all().item())}
    if rank == 0:
        from oracle import dit_oracle as dto
        sd = {k: v.detach().cpu() for k, v in net.state_dict().items()}
        xc, pc, tc = x[:8].cpu(), past[:8].cpu(), t[:8].cpu()
        torch.set_num_threads(os.cpu_count())
        with torch.no_grad():
            dto.dit_forward(sd, xc, tc, pc, patch=4, t_patch=4, heads=4, depth=6)
            t1 = time.perf_counter()
            for _ in range(4):
                dto.dit_forward(sd, xc, tc, pc, patch=4, t_patch=4, heads=4, depth=6)
            cpu_step = (time.perf_counter() - t1) / 4
        res["cpu_baseline"] = {"value": 8 / (cpu_step * T_STEPS), "unit": "sequences/s", "cores": os.cpu_count(), "kind": "port",
                               "sample": "4 denoiser evaluations at batch 8 (of 64) on the host cores (oracle/ restatement of "
                                         "DiT4D_V4.forward), extrapolated to 1000 steps"}
    del net
    torch.cuda.empty_cache()
    return res


def feed_and_metrics_bench(dev):
    """The callers either side of the hot path (SURVEY.md section 8 f3 / f4), rank 0 only, each against the HBM roofline
    (MEASURED_PEAKS.json) with the oracle port of the reference's CPU code timed beside it on a bounded sample:
      * data feed: one epoch of BATCH_SIZE-64 (past, future) windows gathered on the device from HBM-resident raw
        sequences (reference: MacropropsDataset + DataLoader + per-step .to(device), utils/dataset.py:22-53, ddpm.py:136-137);
      * metrics tail: PSNR / MASK_PSNR / RE_DENSITY / TV of generate_metrics' 1280-sample batch
        (reference: utils/metrics/metricsGenerator.py:120-186,293-339)."""
    import types
    import numpy as np
    from crowdmod_ddpm_4d_b200.utils.dataset_gpu import GpuMacropropsDataset, GpuWindowLoader
    from crowdmod_ddpm_4d_b200.utils.metrics_gpu import GpuMetricsGenerator, compute_metrics_gpu
    from oracle import dataset_oracle as dso
    from oracle import metrics_oracle as mo
    hbm = peaks()["hbm_gbs"]
    out = {}
    # ---- data feed: 64 raw ATC sequences of 200 frames, stride 8 -> 1600 windows = 25 batches of 64
    w = WORKLOADS["atc"]
    rng = np.random.default_rng(3)
    seq = rng.normal(size=(64, 3, w["rows"], w["cols"], 200)).astype(np.float32)
    cfg = types.SimpleNamespace(DATASET=types.SimpleNamespace(PAST_LEN=w["past"], FUTURE_LEN=w["fut"]),
                                MACROPROPS=types.SimpleNamespace(EPS=1e-6))
    ds = GpuMacropropsDataset(seq, cfg, 3, stride=8, device=dev)
    loader = GpuWindowLoader(ds, 64, shuffle=True, drop_last=True)
    for _ in loader:      # warm-up epoch
        pass
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    a.record()
    nb = 0
    for _ in range(4):
        for past, fut in loader:
            nb += 1
    b.record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    dev_ms = a.elapsed_time(b) / nb
    per_batch_bytes = 64 * 3 * w["rows"] * w["cols"] * (w["past"] + w["fut"]) * 4 * 2
    # kernel alone (CUDA events around back-to-back gathers of one fixed batch)
    import crowdmod_ddpm_4d_b200._native as nat
    ids = torch.randperm(len(ds), device=dev)[:64].contiguous()
    pbuf, fbuf = ds.gather(ids)
    torch.cuda.synchronize()
    a.record()
    for _ in range(200):
        nat.check(nat.lib().cm_window_gather(nat.ptr(ds.seq_all), 64, 3, w["rows"], w["cols"], 200, nat.ptr(ds._seq_idx),
                                             nat.ptr(ds._t0), nat.ptr(ids), 64, w["past"], w["fut"], nat.ptr(pbuf), nat.ptr(fbuf),
                                             nat.current_stream()))
    b.record()
    torch.cuda.synchronize()
    k_us = a.elapsed_time(b) * 1e3 / 200
    t1 = time.perf_counter()
    torch.manual_seed(0)
    ncpu = 0
    for past, fut in dso.batches(seq, w["past"], w["fut"], 8, 64, shuffle=True, drop_last=True):
        past.to(dev, non_blocking=False), fut.to(dev, non_blocking=False)
        ncpu += 1
    torch.cuda.synchronize()
    cpu_s = time.perf_counter() - t1
    out["data_feed"] = {"workload": "config/ATC.yml windows (past 5 + future 3, stride 8) of 64 HBM-resident raw sequences x 200 "
                                    "frames, shuffled batches of 64", "batches_per_s": nb / wall, "ms_per_batch_device": dev_ms,
                        "gather_kernel_us": k_us,
                        "roofline": {"bound": "hbm", "achieved": per_batch_bytes / (k_us * 1e-6) / 1e9, "peak": hbm, "unit": "GB/s",
                                     "frac": per_batch_bytes / (k_us * 1e-6) / 1e9 / hbm,
                                     "algorithmic_bytes_per_batch": per_batch_bytes},
                        "cpu_baseline": {"value": ncpu / cpu_s, "unit": "batches/s", "cores": 1, "kind": "port",
                                         "sample": f"one epoch ({ncpu} batches): host window slicing + collate + .to(device), "
                                                   "oracle/ restatement of the reference's single-process loader"}}
    # ---- metrics tail at n = 1280
    pred, gt = mo.synthetic_pair(1280, w["rows"], w["cols"], w["fut"], 11)
    pd_, gd = torch.from_numpy(pred).to(dev), torch.from_numpy(gt).to(dev)
    params = types.SimpleNamespace(MPROPS_COUNT=3)
    for _ in range(2):
        gen = GpuMetricsGenerator(pd_, gd, params)
        compute_metrics_gpu(cfg, gen, "ALL", 20)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(5):
        gen = GpuMetricsGenerator(pd_, gd, params)
        compute_metrics_gpu(cfg, gen, "ALL", 20)
    torch.cuda.synchronize()
    gpu_s = (time.perf_counter() - t0) / 5
    outbuf = torch.empty(1280, w["fut"], 21, dtype=torch.float64, device=dev)
    a.record()
    for _ in range(50):
        nat.check(nat.lib().cm_metrics_reduce(nat.ptr(pd_), nat.ptr(gd), 1280, 3, w["rows"], w["cols"], w["fut"], nat.ptr(outbuf),
                                              nat.current_stream()))
    b.record()
    torch.cuda.synchronize()
    k_us = a.elapsed_time(b) * 1e3 / 50
    mbytes = 2 * pred.size * 4
    t1 = time.perf_counter()
    ncpu = 64
    with np.errstate(all="ignore"):
        mo.compute_psnr_metric(pred[:ncpu], gt[:ncpu], 4, 1e-6)
        mo.compute_psnr_metric(pred[:ncpu], gt[:ncpu], 4, 1e-6, masked=True)
        mo.compute_re_density(pred[:ncpu], gt[:ncpu], 4, 1e-6)
        mo.compute_tv_metric(pred[:ncpu], gt[:ncpu])
    cpu_s = (time.perf_counter() - t1) * (1280 / ncpu)
    out["metrics_tail"] = {"workload": "PSNR + MASK_PSNR + RE_DENSITY + TV of 1280 predicted ATC sequences (generate_metrics batch), "
                                       "device tensors in, numpy tables out (one D2H read of 1280 x 3 x 21 doubles)",
                           "samples_per_s": 1280 / gpu_s, "ms_total": gpu_s * 1e3, "reduce_kernel_us": k_us,
                           "roofline": {"bound": "hbm", "achieved": mbytes / (k_us * 1e-6) / 1e9, "peak": hbm, "unit": "GB/s",
                                        "frac": mbytes / (k_us * 1e-6) / 1e9 / hbm, "algorithmic_bytes": mbytes},
                           "cpu_baseline": {"value": 1280 / cpu_s, "unit": "samples/s", "cores": 1, "kind": "port",
                                            "sample": f"{ncpu} of 1280 samples through the oracle/ restatement of the reference's "
                                                      "per-sample numpy loops, extrapolated"}}
    return out


# ---- training leg (BASELINE config #4: HERMES-CR-120.yml, 28x24 grid, batch 64 per GPU) ----------
def train_bench(rank, world, dev, steps=20, warmup=5, cpu_baseline=True):
    """DDPM_model._train_one_epoch's loop body (reference ddpm.py:111-121,132-146) through the reference-facing
    driver object: t ~ U, q-sample, native training forward (tcgen05 fprop), MSE, native backward (dgrad with
    hi|lo dOut pairs / wgrad), ONE flat-gradient all-reduce when world > 1, the driver's own torch.optim.Adam.
    Returns a dict added to the bench line under "train"."""
    import torch.distributed as dist
    from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import DDPM, DDPM_model
    w = WORKLOADS["hermes"]
    n = 64
    torch.manual_seed(42)
    model = DDPM_model(make_cfg("hermes"), "DDPM-UNet", 3)
    if world > 1:
        model.enable_data_parallel()
    net = model.denoiser.train()
    opt = model.optimizer
    fs = DDPM(timesteps=T_STEPS, scale=SCALE).to(dev)
    past = synthetic_macroprops(n, 3, w["rows"], w["cols"], w["past"], 1234 + rank, dev)
    fut = synthetic_macroprops(n, 3, w["rows"], w["cols"], w["fut"], 4321 + rank, dev)

    def step():
        loss = model._train_step(fut, past, fs)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        return loss

    for _ in range(warmup):
        step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    a.record()
    for _ in range(steps):
        loss = step()
    b.record()
    t_issue = time.perf_counter() - t0            # host time to ISSUE the steps (no sync inside)
    torch.cuda.synchronize()
    ms = torch.tensor([a.elapsed_time(b) / steps], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    step_ms = ms.item()
    # forward / backward / optimizer split on rank 0 (events around the native calls)
    e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    torch.cuda.synchronize()
    e[0].record()
    loss = model._train_step(fut, past, fs)
    e[1].record()
    opt.zero_grad(set_to_none=True)
    loss.backward()
    e[2].record()
    opt.step()
    e[3].record()
    torch.cuda.synchronize()
    plan = net._plan(w["rows"], w["cols"], w["past"], w["fut"])
    fl = net.native_stats(w["rows"], w["cols"], w["past"], w["fut"])[1]
    out = {"workload": "config/HERMES-CR-120.yml: DDPM-UNet training step (t~U, q-sample, fwd, MSE, bwd, Adam), "
                       "grid 28x24, past 5 + future 3, batch 64 per GPU, dropout 0.1",
           "steps": steps, "warmup": warmup,
           "step_ms": step_ms, "samples_per_s": n * world / (step_ms * 1e-3),
           "host_issue_ms_per_step": t_issue * 1e3 / steps,
           "fwd_ms": e[0].elapsed_time(e[1]), "bwd_ms": e[1].elapsed_time(e[2]), "adam_ms": e[2].elapsed_time(e[3]),
           "loss": float(loss.item()), "grad_allreduce": "one NCCL all-reduce of the flat fp32 gradient buffer"
           if world > 1 else "none (1 GPU)",
           "dgrad_terms": int(os.environ.get("CROWDMOD_DGRAD_TERMS", "2")),
           "algorithmic_tflops": 3.0 * fl * n / (step_ms * 1e-3) / 1e12,
           "bwd_launches": int(plan.n.lib().cm_last_backward_launches(plan.handle))}
    if cpu_baseline and rank == 0 and world == 1:
        out["cpu_baseline"] = train_cpu_baseline()
    del model, net, opt
    torch.cuda.empty_cache()
    return out


def train_cpu_baseline(n=8):
    """One fwd+bwd of the reference path's CPU restatement on the host cores (bounded sample)."""
    from oracle import ddpm_oracle as do
    from oracle import unet_oracle as uo
    from crowdmod_ddpm_4d_b200.models.backbones.unet import UNet
    w = WORKLOADS["hermes"]
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    torch.manual_seed(42)
    sd = {k: v.detach().clone().requires_grad_(v.dtype.is_floating_point and "time_blocks.0" not in k)
          for k, v in UNet(**ATC).state_dict().items()}
    s = do.schedule(T_STEPS, SCALE)
    past = do.synthetic_macroprops(n, 3, w["rows"], w["cols"], w["past"], 1234)
    fut = do.synthetic_macroprops(n, 3, w["rows"], w["cols"], w["fut"], 4321)
    den = lambda x, tt, p: uo.unet_forward(sd, x, tt, p, num_res_blocks=1, num_levels=3)
    t = torch.randint(0, T_STEPS, (n,))
    eps = torch.randn_like(fut)
    t0 = time.perf_counter()
    do.train_loss(den, s, fut, past, t, eps).backward()
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": "samples/s", "cores": threads, "kind": "port",
            "sample": f"one fwd+bwd at batch {n} (of 64) on the host cores, oracle/ restatement"}


def roofline(net, nat, past, n, dev, step_ms):
    """Dominant kernel class = the tcgen05 implicit-GEMM convs (conv_plane_kernel + conv_umma_kernel).
    achieved = EXECUTED FLOPs of all its launches in one denoiser step / their summed device time, timed live
    with CUDA events around every launch (cm_unet_profile_forward).  The UpSample convs execute 8 phase convs of
    2x2x2 folded taps (8/27 of the dense formulation): the dense-equivalent rate is reported separately."""
    pk = peaks()
    plan = net._plan(ROWS, COLS, PAST, FUT)
    lib = nat.lib()
    nops = lib.cm_unet_op_count(plan.handle)
    x = torch.randn(n, 3, ROWS, COLS, FUT, device=dev)
    t = torch.full((n,), 500, device=dev, dtype=torch.long)
    eps = torch.empty_like(x)
    ms = (C.c_float * nops)()
    best = None
    for _ in range(5):
        nat.check(lib.cm_unet_profile_forward(plan.handle, nat.ptr(x), nat.ptr(t), nat.ptr(past), nat.ptr(eps),
                                              n, nat.current_stream(), ms, nops))
        cur = list(ms)
        if best is None or sum(cur) < sum(best):
            best = cur
    kinds = {0: "first_conv", 1: "gn_silu", 2: "conv_umma", 3: "attn_core", 4: "final_conv"}
    agg = {}
    tag = C.create_string_buffer(128)
    ty = C.c_int()
    fl = C.c_double()
    for i in range(nops):
        lib.cm_unet_op_info(plan.handle, i, tag, 128, C.byref(ty), C.byref(fl))
        kind = kinds[ty.value]
        name = tag.value.decode()
        # the sampling path runs each AttentionBlock (GroupNorm, in_proj, core, out_proj + residual) as ONE
        # fused launch: its four plan ops are one class, not conv / GN work
        if ".attention." in name:
            kind = "attn_block"
        a = agg.setdefault(kind, {"ms": 0.0, "flops": 0.0, "exec_flops": 0.0, "launches": 0})
        a["ms"] += best[i]
        a["flops"] += fl.value * n
        a["exec_flops"] += lib.cm_unet_op_exec_flops(plan.handle, i) * n
        a["launches"] += 1 if best[i] > 0 else 0
    conv = agg["conv_umma"]
    achieved = conv["exec_flops"] / (conv["ms"] * 1e-3) / 1e12
    dense = conv["flops"] / (conv["ms"] * 1e-3) / 1e12
    traffic = None
    tp = os.path.join(ROOT, "profiles", "conv_umma_traffic.json")
    if os.path.exists(tp):
        traffic = json.load(open(tp)).get("dram_bytes_per_launch")
    total_ms = sum(best)
    return {"bound": "tensor", "kernel": "tcgen05 implicit-GEMM conv3d: conv_plane_kernel (levels 0/1) + conv_umma_kernel",
            "achieved": achieved, "peak": pk["tflops_sustained"], "unit": "TFLOP/s",
            "frac": achieved / pk["tflops_sustained"], "traffic": traffic,
            "flops_counted": "executed (UpSample convs as 8 phase convs of 2x2x2 folded taps)",
            "algorithmic_equiv": {"achieved": dense, "frac": dense / pk["tflops_sustained"],
                                  "note": "dense 27-tap formulation of SURVEY.md §8(d) over the same device time"},
            "peak_source": pk["source"] + ", sustained bf16/fp16 dense",
            "launches_per_step": conv["launches"], "avg_launch_us": conv["ms"] * 1e3 / max(conv["launches"], 1),
            "executed_gflop_per_step": conv["exec_flops"] / 1e9,
            "algorithmic_gflop_per_step": conv["flops"] / 1e9,
            "share_of_step": conv["ms"] / total_ms,
            "per_kernel_ms_per_step": {k: round(v["ms"], 4) for k, v in agg.items()},
            "eager_step_ms": total_ms, "graph_step_ms": step_ms,
            "whole_step_tflops_executed": (sum(v["exec_flops"] for v in agg.values()) / 1e12) / (step_ms * 1e-3),
            "whole_step_tflops": (sum(v["flops"] for v in agg.values()) / 1e12) / (step_ms * 1e-3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--batch", type=int, default=64, help="samples per GPU (ATC.yml BATCH_SIZE)")
    ap.add_argument("--timesteps", type=int, default=T_STEPS)
    ap.add_argument("--ref-iters", type=int, default=8, help="CPU denoiser iterations per reference sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the training-step leg (extra key 'train')")
    ap.add_argument("--no-extras", action="store_true", help="skip the n=1280 / ATC_medium / ETH-UCY chains")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write x_0 of the last timed chain (rank 0's samples) as DIR/x0.npy, float32")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs applies to the native arm")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_native(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
