"""Wide-model measurements (attention heads of 128 channels, base_channels 128) on one GPU; prints one JSON document.

  models  B: ATC 12 x 36, 5 + 3 frames, base 128, mult [1, 2, 4], attention at level 2 (S = 54, dh = 128)
          D: HERMES 28 x 24, 8 + 8 frames, the same UNet (S = 168, dh = 128: two key tiles)
          per model: a --chain-steps DDPM chain (whole-chain graph, Philox noise) at --batch samples, and the training
          step (forward + backward, no optimizer) at --batch, both timed with CUDA events after a warm-up
  attention core  forward and backward at dh = 128 against dh = 64 at equal FLOPs (twice the (sample, head) pairs at
          dh = 64), S in {54, 168, 432}; device time of the attention kernels only (torch.profiler); algorithmic FLOPs
          4 * S^2 * dh per (sample, head) forward (QK^T and PV) and 2.5 times that backward (the recomputed scores,
          dP, dV, dK and dQ), as tools/attn_long_bench.py counts them

usage: python tools/wide_bench.py [--batch 64] [--chain-steps 1000] [--out profiles/wide_bench_b200.json]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

MODELS = {
    "B_atc_base128": dict(rows=12, cols=36, P=5, F=3),
    "D_hermes_base128": dict(rows=28, cols=24, P=8, F=8),
}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def timed(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def bench_model(name, c, batch, chain_steps):
    import torch.nn.functional as F
    from crowdmod_ddpm_4d_b200.models.backbones.unet import UNet
    from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import DDPM, ddpm_coefficients
    torch.manual_seed(0)
    net = UNet(input_channels=3, output_channels=3, num_res_blocks=1, base_channels=128,
               base_channels_multiples=[1, 2, 4], apply_attention=[False, False, True, False], dropout_rate=0.0,
               time_multiple=4).cuda()
    past = torch.randn(batch, 3, c["rows"], c["cols"], c["P"], device="cuda")
    fut = torch.randn(batch, 3, c["rows"], c["cols"], c["F"], device="cuda")
    ts, coef = ddpm_coefficients(DDPM(timesteps=chain_steps, scale=0.5))
    net.eval()
    chain = lambda: net.sample_chain(past, fut.clone(), ts, coef, mode=0, seed=1)
    chain()
    torch.cuda.synchronize()
    chain_ms = timed(chain, 2)
    net.train()
    t = torch.randint(0, 1000, (batch,), device="cuda")
    noise = torch.randn_like(fut)

    def step():
        loss = F.mse_loss(net(fut, t, past), noise)
        net.zero_grad(set_to_none=True)
        loss.backward()

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    train_ms = timed(step, 10)
    return dict(batch=batch, chain_steps=chain_steps, chain_ms=round(chain_ms, 2),
                chain_samples_per_s=round(batch / (chain_ms / 1e3), 2),
                chain_step_ms=round(chain_ms / chain_steps, 4), train_step_ms=round(train_ms, 3))


def kernel_ms(fn, match, iters=5):
    """Mean device time per call of the kernels whose name contains `match` (torch.profiler, CUDA activities): the
    op entry of the streaming backward also allocates, reruns the forward for its lse and synchronises, none of which
    belongs to the backward kernels' time."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            fn()
        torch.cuda.synchronize()
    us = sum(e.device_time_total for e in prof.key_averages() if match in e.key)
    assert us > 0, f"no kernel matching {match!r} ran"
    return us / 1e3 / iters


def bench_attention(n):
    rows = []
    lib = n.lib()
    for S in (54, 168, 432):
        for dh, pairs in ((128, 256), (64, 512)):
            heads = 4
            B, C_ = pairs // heads, heads * dh
            streaming = S > 128 or dh > 64                   # attn_uses_long in kernels.cuh
            qkv = torch.randn(B, S, 3 * C_, device="cuda")
            ctx = torch.empty(B, S, C_, device="cuda", dtype=torch.half)
            dctx = torch.randn(B, S, C_, device="cuda")
            dqkv = torch.empty_like(qkv)
            st = n.current_stream()
            fwd = lambda: n.check(lib.cm_op_attn_core(n.ptr(qkv), n.ptr(ctx), B, S, C_, heads, st))
            bwd = lambda: n.check(lib.cm_op_attn_core_backward(n.ptr(qkv), n.ptr(dctx), n.ptr(dqkv), B, S, C_, heads, st))
            f_ms = kernel_ms(fwd, "attn_long_kernel" if streaming else "attn_mma_kernel", iters=20)
            b_ms = kernel_ms(bwd, "attn_long_d" if streaming else "attn_core_backward_kernel")
            ff = 4.0 * S * S * dh * pairs
            rows.append(dict(S=S, dh=dh, pairs=pairs, kernels="streaming" if streaming else "register-resident",
                             fwd_ms=round(f_ms, 4), fwd_tflops=round(ff / f_ms / 1e9, 2),
                             bwd_ms=round(b_ms, 4), bwd_tflops=round(2.5 * ff / b_ms / 1e9, 2)))
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--chain-steps", type=int, default=1000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("wide_bench.py needs a CUDA device")
    import crowdmod_ddpm_4d_b200._native as n
    torch.backends.cuda.matmul.allow_tf32 = False
    res = dict(gpu=gpu_info(), models={k: bench_model(k, c, a.batch, a.chain_steps) for k, c in MODELS.items()},
               attention=bench_attention(n))
    assert n.lib().cm_device_error() == 0
    doc = json.dumps(res, indent=1)
    print(doc)
    if a.out:
        with open(a.out, "w") as f:
            f.write(doc + "\n")


if __name__ == "__main__":
    main()
