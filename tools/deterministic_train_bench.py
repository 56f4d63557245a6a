"""Cost of reproducible training: bench.py's training step (DDPM_model._train_step + backward + Adam, batch 64) with
torch.use_deterministic_algorithms off and on, alternating within one process after warm-up, at the HERMES-CR-120 and
ATC geometries.  Also reports the backward's launch count in both modes and the device memory the deterministic
partial-sum scratch takes (cudaMemGetInfo around the first deterministic backward).  Prints one JSON object and writes
it to --out when given.

    python tools/deterministic_train_bench.py --steps 20 --rounds 4 --out profiles/deterministic_train_b200.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")

import torch  # noqa: E402

import bench  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def measure(name, steps, rounds, warmup):
    from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import DDPM, DDPM_model
    w = bench.WORKLOADS[name]
    n = 64
    torch.manual_seed(42)
    model = DDPM_model(bench.make_cfg(name), "DDPM-UNet", 3)
    net = model.denoiser.train()
    opt = model.optimizer
    fs = DDPM(timesteps=bench.T_STEPS, scale=bench.SCALE).cuda()
    past = bench.synthetic_macroprops(n, 3, w["rows"], w["cols"], w["past"], 1234, "cuda")
    fut = bench.synthetic_macroprops(n, 3, w["rows"], w["cols"], w["fut"], 4321, "cuda")
    plan = net._plan(w["rows"], w["cols"], w["past"], w["fut"])
    lib = plan.n.lib()

    def step():
        loss = model._train_step(fut, past, fs)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()

    out = {"workload": f"{w['cfg']}: training step, grid {w['rows']}x{w['cols']}, past {w['past']} + future "
                       f"{w['fut']}, batch {n}, dropout 0.1", "ms_per_step": {"off": [], "on": []}}
    for det in (False, True):
        torch.use_deterministic_algorithms(det)
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info()[0]
        for _ in range(warmup):
            step()
        torch.cuda.synchronize()
        key = "on" if det else "off"
        out.setdefault("bwd_launches", {})[key] = int(lib.cm_last_backward_launches(plan.handle))
        if det:
            out["scratch_bytes_device_delta"] = int(free0 - torch.cuda.mem_get_info()[0])
    for _ in range(rounds):
        for det in (False, True):
            torch.use_deterministic_algorithms(det)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            for _ in range(steps):
                step()
            b.record()
            torch.cuda.synchronize()
            out["ms_per_step"]["on" if det else "off"].append(a.elapsed_time(b) / steps)
    torch.use_deterministic_algorithms(False)
    for k in ("off", "on"):
        v = sorted(out["ms_per_step"][k])
        out[f"median_ms_{k}"] = v[len(v) // 2]
    out["added_ms"] = out["median_ms_on"] - out["median_ms_off"]
    out["added_launches"] = out["bwd_launches"]["on"] - out["bwd_launches"]["off"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="timed steps per window")
    ap.add_argument("--rounds", type=int, default=4, help="alternating (off, on) windows per workload")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("deterministic_train_bench.py needs a CUDA device")
    res = {"card": card(), "steps": args.steps, "rounds": args.rounds,
           "workloads": {name: measure(name, args.steps, args.rounds, args.warmup) for name in ("hermes", "atc")},
           "card_after": card()}
    s = json.dumps(res, indent=1)
    print(s)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
