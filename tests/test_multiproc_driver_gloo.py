"""Sharded sampling through DDPM_model on CPU (gloo, world sizes 2 and 3): after enable_data_parallel() every rank gets
the chain the group's rank 0 would have run alone, whatever its own RNG state and inputs.  The native backbone is
replaced by a stand-in with the same sample_chain contract, so this covers the driver's broadcasts, shard offsets,
empty shards and the padded gather; tests/test_gpu_multirank_driver.py runs the native chains."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

CFG = os.path.join(os.path.dirname(os.path.abspath(__file__)), "configs", "atc_nested.yml")


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


class _StandInChain:
    """Each sample of x_0 depends only on its own x_T, past, the seed or injected noise and its GLOBAL index
    (sample_offset + i), as in UNet.sample_chain; an empty batch is refused, as cm_dit_sample does."""

    def eval(self):
        return self

    def sample_chain(self, past, x, tsteps, coef, mode=0, noise=None, seed=0, sample_offset=0, history=None,
                     use_graph=True):
        assert x.shape[0] > 0 and past.shape[0] == x.shape[0]
        idx = torch.arange(sample_offset, sample_offset + x.shape[0], dtype=torch.float32).view(-1, 1, 1, 1, 1)
        cond = past.mean(-1, keepdim=True) * 0.1
        for k in range(tsteps.numel()):
            z = noise[k] if noise is not None else torch.sin(idx * 0.37 + float(seed % 9973) + k)
            x.mul_(float(coef[k, 0])).add_(cond + float(coef[k, 5]) * x.sign() + z)
            if history is not None:
                history[k + 1].copy_(x)
        return x


def _models():
    from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import DDPM_model
    from crowdmod_ddpm_4d_b200.utils.myparser import getYamlConfig
    cfg = getYamlConfig(CFG)
    cfg.MODEL.DDPM.TIMESTEPS = 6
    single, sharded = DDPM_model(cfg, "DDPM-UNet", 3), DDPM_model(cfg, "DDPM-UNet", 3)
    sharded.enable_data_parallel()
    single.denoiser = _StandInChain()
    sharded.denoiser = _StandInChain()
    return cfg, single, sharded


def _past(n, seed):
    return torch.randn((n, 3, 12, 36, 5), generator=torch.Generator().manual_seed(seed))


def _worker(rank, world, port, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import DDPM
        cfg, single, sharded = _models()
        sampler = DDPM(timesteps=6, scale=0.5)
        failures = []

        def check(name, fn):
            """fn(model) runs one call; the single-process model gets rank 0's seed and inputs, the sharded one
            this rank's own (different on every rank but 0)."""
            torch.manual_seed(1)
            want = fn(single, _past(5, 10))
            torch.manual_seed(1 + 1000 * rank)
            past = _past(5, 10 + rank)
            past_in = past.clone()
            got = fn(sharded, past)
            if not torch.equal(past, past_in):
                failures.append(f"{name}: the caller's past was overwritten")
            for a, b in zip(got, want):
                if a.shape != b.shape or not torch.equal(a, b):
                    failures.append(f"{name}: {tuple(a.shape)} vs single-process {tuple(b.shape)}")
                    break

        def ddpm(n, history=False):
            def fn(m, past):
                x, over_time = m._generate_ddpm(past[:n].contiguous(), sampler, n, history=history)
                return [x] + list(over_time)
            return fn

        check("ddpm n=5", ddpm(5))
        check("ddpm n=5 history", ddpm(5, True))
        check("ddpm n=1", ddpm(1))              # world - 1 ranks hold an empty shard
        check("ddpm n=2 history", ddpm(2, True))

        cfg.MODEL.DDPM.GUIDANCE = "Sparsity"
        cfg.MODEL.DDPM.LAMBDA_GUIDANCE = 0.004

        def ddim(m, past):
            x, over_time = m._generate_ddim(past, np.arange(0, 5, 2), sampler, 5, history=True)
            return [x, torch.stack(over_time)]
        check("ddim sparsity history", ddim)
        cfg.MODEL.DDPM.GUIDANCE = "None"

        for m in (single, sharded):
            m.noise_source = lambda nsteps, shape, device: torch.randn((nsteps,) + shape, device=device)
        check("noise_source", ddpm(5))
        check("noise_source n=1", ddpm(1))
        out[rank] = failures
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_driver_chain_equals_rank0_single_process(world):
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    assert sorted(out.keys()) == list(range(world))
    assert all(out[r] == [] for r in range(world)), dict(out)


def test_chain_without_data_parallel_calls_the_backbone_once_on_the_whole_batch():
    """Without enable_data_parallel an initialised process group is ignored: one sample_chain call over all samples
    with the model's own sample_offset, and the torch generator advances exactly as before (x_T, then the seed)."""
    from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import DDPM, DDPM_model
    from crowdmod_ddpm_4d_b200.utils.myparser import getYamlConfig
    cfg = getYamlConfig(CFG)
    m = DDPM_model(cfg, "DDPM-UNet", 3)
    calls = []

    class Spy(_StandInChain):
        def sample_chain(self, past, x, tsteps, coef, **kw):
            calls.append((x.shape[0], kw["sample_offset"], kw["seed"]))
            return super().sample_chain(past, x, tsteps, coef, **kw)

    m.denoiser = Spy()
    m.sample_offset = 7
    torch.manual_seed(3)
    m._generate_ddpm(_past(4, 0), DDPM(timesteps=5, scale=0.5), 4)
    torch.manual_seed(3)
    torch.randn(4, 3, 12, 36, 3)
    seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    assert calls == [(4, 7, seed)]
