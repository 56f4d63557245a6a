"""Long-sequence attention (S > 128 tokens per (sample, head)) on the GPU: core forward / backward device time at the
attention shapes of the reference configs, their exponential and tensor rates against the hardware bounds, and the
end-to-end sampling chain and training step of two configs with such attention.

    python tools/attn_long_bench.py --out DIR

Writes DIR/attn_long_bench.json (card name and power limit read in the same run).  Needs a CUDA device.

Core shapes: B = 64 samples, 4 heads.  A forward computes B * heads * S^2 exponentials and 4 * B * S^2 * C algorithmic
FLOP (Q K^T and P V); the tcgen05 kernel issues 3 fp16 products for the scores (hi / lo splits, K = 3 * dhp, dh padded
to dhp = 16 / 32 / 64) and one for P V, which is the executed tensor FLOP count reported beside it.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import torch  # noqa: E402

# (label, S, C): attention tokens of the level and its channel count (base 32; heads 4)
CORE_SHAPES = [
    ("HERMES 28x24 P8+F8, level 2 / DiT patch 2 (168 patches)", 168, 128),
    ("ATC 12x36 P5+F3, level 1", 432, 64),
    ("HERMES 28x24 P5+F3, level 1", 672, 64),
    ("ETH-UCY 8x12 P5+F3, level 0", 768, 32),
    ("ATC 12x36 P5+F3, level 0", 3456, 32),
]
E2E = {
    "HERMES 8+8 [F,F,T]": dict(rows=28, cols=24, P=8, F=8, attn=[False, False, True]),
    "ATC attention [F,T,T]": dict(rows=12, cols=36, P=5, F=3, attn=[False, True, True]),
}
TENSOR_PEAK = 2250e12           # dense FP16 FLOP/s of one B200 (HGX B200 data sheet, 1,000 W)
SFU_EX2_PER_CLK_SM = 16         # MUFU.EX2 results per clock per SM (compute capability 10.0 throughput table)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, plim, mhz = [s.strip() for s in q.split(",")]
    return {"name": name, "power_limit_w": float(plim), "sm_max_mhz": float(mhz),
            "sms": torch.cuda.get_device_properties(0).multi_processor_count}


def timed(fn, iters, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def kernel_ms(fn, match, iters=3):
    """Mean device time per call of the kernels whose name contains `match` (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            fn()
        torch.cuda.synchronize()
    us = sum(e.device_time_total for e in prof.key_averages() if match in e.key)
    return us / 1e3 / iters


def core(nat, info):
    lib, stream = nat.lib(), nat.current_stream()
    B, heads = 64, 4
    ex2_rate = info["sms"] * SFU_EX2_PER_CLK_SM * info["sm_max_mhz"] * 1e6
    rows = []
    for label, S, C in CORE_SHAPES:
        dh = C // heads
        dhp = 16 if dh <= 16 else 32 if dh <= 32 else 64
        g = torch.Generator(device="cuda").manual_seed(S)
        qkv = torch.randn(B, S, 3 * C, device="cuda", generator=g)
        dctx = torch.randn(B, S, C, device="cuda", generator=g)
        ctx = torch.empty(B, S, C, device="cuda", dtype=torch.half)
        dqkv = torch.empty_like(qkv)
        iters = max(5, int(2e9 / (B * heads * S * S)))
        f_ms = timed(lambda: nat.check(lib.cm_op_attn_core(nat.ptr(qkv), nat.ptr(ctx), B, S, C, heads, stream)), iters)
        # the op entry of the backward also reruns the forward into temporaries: time only the two backward kernels
        b_ms = kernel_ms(lambda: nat.check(lib.cm_op_attn_core_backward(nat.ptr(qkv), nat.ptr(dctx), nat.ptr(dqkv), B,
                                                                        S, C, heads, stream)), "attn_long_d")
        exps = B * heads * S * S
        alg = 4.0 * B * S * S * C
        executed = 2.0 * B * heads * S * S * (3 * dhp + dhp)
        bwd_alg = 2.5 * alg                      # S recompute, dP, dV, dK, dQ: five S x S x dh products
        t_exp, t_mma = exps / ex2_rate, executed / TENSOR_PEAK
        rows.append({
            "shape": label, "B": B, "heads": heads, "S": S, "C": C, "dh": dh,
            "fwd_ms": f_ms, "bwd_ms": b_ms,
            "exponentials": exps, "exp_per_s": exps / (f_ms * 1e-3), "exp_rate_share_of_sfu": t_exp / (f_ms * 1e-3),
            "algorithmic_flop": alg, "executed_tensor_flop": executed,
            "tensor_flop_per_s": executed / (f_ms * 1e-3), "tensor_share_of_peak": t_mma / (f_ms * 1e-3),
            "fwd_bound": "exp (SFU)" if t_exp > t_mma else "tensor",
            "bwd_fp32_flop_per_s": bwd_alg / (b_ms * 1e-3),
        })
        print(json.dumps(rows[-1]), flush=True)
    return {"sfu_ex2_per_s": ex2_rate, "tensor_peak_flop_per_s": TENSOR_PEAK, "shapes": rows}


def e2e():
    import torch.nn.functional as F
    from crowdmod_ddpm_4d_b200.models.backbones.unet import UNet
    from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import DDPM, ddpm_coefficients
    from oracle import ddpm_oracle as do
    out = {}
    for name, c in E2E.items():
        torch.manual_seed(0)
        net = UNet(input_channels=3, output_channels=3, num_res_blocks=1, base_channels=32,
                   base_channels_multiples=[1, 2, 4], apply_attention=c["attn"], dropout_rate=0.0, time_multiple=4,
                   condition="Past").cuda()
        n = 64
        past = do.synthetic_macroprops(n, 3, c["rows"], c["cols"], c["P"], 1).cuda().contiguous()
        fut = do.synthetic_macroprops(n, 3, c["rows"], c["cols"], c["F"], 2).cuda().contiguous()
        x = torch.randn(n, 3, c["rows"], c["cols"], c["F"], device="cuda")
        net.eval()
        ts, coef = ddpm_coefficients(DDPM(timesteps=1000, scale=0.5))
        net.sample_chain(past, x.clone(), ts[:8], coef[:8], mode=0, seed=1)
        net.sample_chain(past, x.clone(), ts, coef, mode=0, seed=2)          # builds the whole-chain graph
        torch.cuda.synchronize()
        xs = x.clone()
        t0 = time.perf_counter()
        net.sample_chain(past, xs, ts, coef, mode=0, seed=3)
        torch.cuda.synchronize()
        chain_s = time.perf_counter() - t0
        net.train()
        t = torch.randint(0, 1000, (n,), device="cuda")
        noise = torch.randn_like(fut)

        def step():
            loss = F.mse_loss(net(fut + 0.1 * noise, t, past), noise)
            net.zero_grad(set_to_none=True)
            loss.backward()

        step_ms = timed(step, 20)
        out[name] = {"rows": c["rows"], "cols": c["cols"], "past": c["P"], "future": c["F"], "attention": c["attn"],
                     "base_channels": 32, "samples": n, "chain_steps": 1000, "chain_s": chain_s,
                     "chain_sequences_per_s": n / chain_s, "train_step_ms_fwd_bwd_batch64": step_ms,
                     "finite": bool(torch.isfinite(xs).all().item())}
        print(name, json.dumps(out[name]), flush=True)
        del net
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True, help="output directory")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("attn_long_bench.py needs a CUDA device")
    import crowdmod_ddpm_4d_b200._native as nat
    torch.backends.cuda.matmul.allow_tf32 = False
    info = card()
    res = {"card": info, "core": core(nat, info), "end_to_end": e2e(),
           "device_error": int(nat.lib().cm_device_error())}
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "attn_long_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", os.path.join(args.out, "attn_long_bench.json"))


if __name__ == "__main__":
    main()
