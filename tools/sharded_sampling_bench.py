"""Sharded sampling through the public driver against hand-sharded chains, at one world size per run.

  torchrun --nproc-per-node=N tools/sharded_sampling_bench.py [--reps 3] [--out profiles/sharded_sampling_nN.json]

Two legs on the config/ATC.yml model of bench.py (UNet base 32, mult [1, 2, 4], grid 12 x 36, past 5 + future 3,
random-init weights under seed 42, synthetic macroprops), each a full 1000-step DDPM chain:
  n1280   generate_metrics' production batch: 1 280 samples split over the N ranks (strong scaling, bench.py's
          extra "atc_n1280" leg)
  n64     64 samples per GPU (weak scaling, bench.py's headline leg)
Per leg and repetition, alternating, after one warm-up chain of each kind at the same size:
  driver  DDPM_model._generate_ddpm after enable_data_parallel(): x_T, past and the seed broadcast from rank 0, this
          rank's shard_samples slice, x_0 all-gathered back to every rank
  hand    UNet.sample_chain on this rank's slice with its global sample offset and no collective, as bench.py does
Both are host-clock times from a barrier to the end of a device synchronise, maximum over the ranks.  Rank 0 prints
the JSON document and writes it to --out, with the name and power limit of every GPU read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (the workloads, config and synthetic inputs bench.py times)


def gpu_info(world):
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    lines = [l.strip() for l in q.stdout.splitlines() if l.strip()]
    return lines[:world] or [torch.cuda.get_device_name(0)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="default: profiles/sharded_sampling_n<world>.json")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("sharded_sampling_bench.py needs a CUDA device")
    from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import DDPM, DDPM_model, ddpm_coefficients, shard_samples
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    torch.manual_seed(42)
    model = DDPM_model(bench.make_cfg("atc"), "DDPM-UNet", 3).enable_data_parallel()
    net = model.denoiser.eval()
    sampler = DDPM(timesteps=bench.T_STEPS, scale=bench.SCALE).to(dev)
    tsteps, coef = ddpm_coefficients(sampler)
    w = bench.WORKLOADS["atc"]

    def timed(fn):
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        t = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    legs = {}
    for name, n in (("n1280", 1280), ("n64", 64 * world)):
        past = bench.synthetic_macroprops(n, 3, w["rows"], w["cols"], w["past"], 1234, dev)
        lo, hi = shard_samples(n, model.rank, model.world)
        past_mine = past[lo:hi].contiguous()
        gen = torch.Generator(device=dev).manual_seed(7 + rank)

        def driver():
            model._generate_ddpm(past, sampler, n)

        def hand(seed=1):
            x = torch.randn((hi - lo, 3, w["rows"], w["cols"], w["fut"]), device=dev, generator=gen)
            net.sample_chain(past_mine, x, tsteps, coef, mode=0, seed=seed, sample_offset=lo)

        timed(driver)
        timed(hand)
        t_driver, t_hand = [], []
        for k in range(a.reps):
            t_driver.append(timed(driver))
            t_hand.append(timed(lambda: hand(2 + k)))
        med_d, med_h = statistics.median(t_driver), statistics.median(t_hand)
        legs[name] = {
            "samples": n, "samples_per_gpu": [b - l for l, b in (shard_samples(n, r, world) for r in range(world))],
            "driver_s": t_driver, "hand_s": t_hand,
            "driver_seq_per_s": n / med_d, "hand_seq_per_s": n / med_h,
            "driver_seq_per_s_range": [n / max(t_driver), n / min(t_driver)],
            "hand_seq_per_s_range": [n / max(t_hand), n / min(t_hand)],
            "driver_over_hand_time": med_d / med_h,
        }
    from crowdmod_ddpm_4d_b200 import _native
    _native.check_device_error("sharded_sampling_bench")
    if rank == 0:
        doc = {"gpus": gpu_info(world), "world": world, "timesteps": bench.T_STEPS, "reps": a.reps,
               "workload": "config/ATC.yml DDPM chain (UNet base 32, mult [1, 2, 4], grid 12 x 36, past 5 + future 3), "
                           "random-init weights (seed 42), synthetic macroprops",
               "timing": "host clock from a barrier to the end of a device synchronise, max over ranks; seq/s of the "
                         "median repetition, range over repetitions",
               "legs": legs}
        text = json.dumps(doc, indent=1)
        print(text, flush=True)
        out = a.out or os.path.join(ROOT, "profiles", f"sharded_sampling_n{world}.json")
        with open(out, "w") as f:
            f.write(text + "\n")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
