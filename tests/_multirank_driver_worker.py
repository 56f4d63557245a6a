"""Worker of tests/test_gpu_multirank_driver.py (launched under torchrun, one rank per GPU, NCCL).

DDPM_model with enable_data_parallel() shards every reverse chain over the ranks.  Each rank builds the same models
(same seed) and computes the single-GPU answer itself, with the model run without enable_data_parallel on rank 0's
seed and inputs; the sharded call gets this rank's own seed and inputs, which differ on every rank but 0.
Exits non-zero on any mismatch; rank 0 prints the measured differences.
"""
import os
import sys
import tempfile
import types

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ddpm_oracle as do  # noqa: E402
from tests._util import rel_l2  # noqa: E402

T = 10


def atc_cfg():
    from crowdmod_ddpm_4d_b200.utils.myparser import getYamlConfig
    cfg = getYamlConfig(os.path.join(ROOT, "tests", "configs", "atc_nested.yml"))
    cfg.MODEL.DDPM.TIMESTEPS = T
    cfg.MACROPROPS.EPS = 1e-6
    cfg.METRICS = types.SimpleNamespace(MPROPS_COUNT=3)
    return cfg


def dit_cfg():
    ns = types.SimpleNamespace
    dit = ns(CONDITION="Past", PATCH_SIZE=4, T_PATCH_SIZE=4, HIDDEN_SIZE=128, DEPTH=2, NUM_HEADS=4, MLP_RATIO=4.0,
             DROPOUT_RATE=0.1, TIME_EMB_MULT=4,
             TRAIN=ns(EPOCHS=1, SOLVER=ns(LR=1e-4, WEIGHT_DECAY=3e-3, BETAS=[0.5, 0.999],
                                          SCHEDULER=ns(FACTOR=0.5, PATIENCE=10, MIN_LR=1e-6))))
    return ns(MACROPROPS=ns(ROWS=12, COLS=36, EPS=1e-6), DATASET=ns(PAST_LEN=5, FUTURE_LEN=3, BATCH_SIZE=4),
              MODEL=ns(NSAMPLES=4, DDPM=ns(TIMESTEPS=T, SCALE=0.5, SIGMA=0.001, DDIM_DIVIDER=2, GUIDANCE="None",
                                           SAMPLER="DDPM", CHECKPOINTS_TO_KEEP=1, DIT=dit)),
              DATA_FS=ns(SAVE_DIR="/tmp/", OUTPUT_DIR="/tmp/"))


def pair(cfg, arch):
    """The same weights twice: one model run on its own, one sharded over the group."""
    from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import DDPM_model
    torch.manual_seed(0)
    single = DDPM_model(cfg, arch, 3)
    torch.manual_seed(0)
    sharded = DDPM_model(cfg, arch, 3).enable_data_parallel()
    return single, sharded


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    from crowdmod_ddpm_4d_b200 import _native as nat
    from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import DDPM
    from crowdmod_ddpm_4d_b200.utils.checkpoint import save_checkpoint
    from crowdmod_ddpm_4d_b200.utils.metrics_gpu import GpuMetricsGenerator, compute_metrics_gpu

    def past_of(n, r):
        return do.synthetic_macroprops(n, 3, 12, 36, 5, 600 + r).to(dev)

    def same_on_all_ranks(t):
        t0 = t.clone()
        dist.broadcast(t0, src=0)
        return torch.equal(t0, t)

    errs, fails = {}, []

    def compare(name, fn, gate=1e-4):
        """fn(model, past) -> list of tensors.  Single-GPU: rank 0's seed and past.  Sharded: this rank's own."""
        torch.manual_seed(21)
        want = fn(single, past_of(5, 0))
        torch.manual_seed(21 + 1000 * rank)
        got = fn(sharded, past_of(5, rank))
        e = max(rel_l2(a, b) if a.shape == b.shape else float("inf") for a, b in zip(got, want))
        errs[name] = e
        if e > gate:
            fails.append(f"{name}: rel-L2 {e:.3e} > {gate:.0e}")
        if not all(same_on_all_ranks(a) for a in got):
            fails.append(f"{name}: ranks hold different results")
        return got

    sampler = DDPM(timesteps=T, scale=0.5).to(dev)
    cfg = atc_cfg()
    single, sharded = pair(cfg, "DDPM-UNet")

    def ddpm(n, history=False):
        def fn(m, past):
            x, over_time = m._generate_ddpm(past[:n].contiguous(), sampler, n, history=history)
            return [x.clone()] + [h.clone() for h in over_time]
        return fn

    # n = 5 over the ranks: an uneven split; a rerun with the same seeds gives the same bits
    a = compare("ddpm n=5", ddpm(5))
    b = compare("ddpm n=5 rerun", ddpm(5))
    if not torch.equal(a[0], b[0]):
        fails.append("ddpm n=5: rerun differs")
    compare("ddpm n=1", ddpm(1))                        # every rank but 0 holds an empty shard

    cfg.MODEL.DDPM.GUIDANCE = "Sparsity"
    taus = np.arange(0, T - 1, 2)

    def ddim(m, past):
        x, over_time = m._generate_ddim(past, taus, sampler, 5, history=True)
        return [x.clone(), torch.stack(over_time)]
    h = compare("ddim sparsity history", ddim)[1]
    if tuple(h.shape) != (len(taus) + 1, 5, 3, 12, 36, 3):
        fails.append(f"ddim history shape {tuple(h.shape)}")
    cfg.MODEL.DDPM.GUIDANCE = "None"

    for m in (single, sharded):
        m.noise_source = lambda nsteps, shape, device: torch.randn((nsteps,) + shape, device=device)
    compare("ddpm noise_source", ddpm(5))
    single.noise_source = sharded.noise_source = None

    # generate_metrics on a tiny synthetic loader: rank 0 alone writes files, the tables equal the single-GPU run
    tmp = tempfile.mkdtemp(prefix=f"crowdmod_driver_r{rank}_")
    cfg.DATA_FS.SAVE_DIR = tmp + "/"
    ckpt = save_checkpoint(single.optimizer, single.denoiser, "000", cfg, "DDPM-UNet")

    def loader(r):
        return [(do.synthetic_macroprops(6, 3, 12, 36, 5, 700 + 10 * r + b),
                 do.synthetic_macroprops(6, 3, 12, 36, 3, 800 + 10 * r + b)) for b in range(2)]

    def metrics(m, r, out):
        m.output_dir = out
        torch.manual_seed(31 + 1000 * r)
        preds, gts = m.generate_metrics(loader(r), 2, "ALL", 2, 6, ckpt, out)
        return torch.stack(preds), torch.stack(gts)

    want_pred, want_gt = metrics(single, 0, os.path.join(tmp, "single"))
    got_pred, got_gt = metrics(sharded, rank, os.path.join(tmp, "sharded"))
    errs["generate_metrics x_0"] = rel_l2(got_pred, want_pred)
    if errs["generate_metrics x_0"] > 1e-4 or not torch.equal(got_gt, want_gt):
        fails.append("generate_metrics: predictions or ground truth differ from the single-GPU run")
    wrote = os.path.exists(os.path.join(tmp, "sharded", "metrics_files.json"))
    if wrote != (rank == 0) or (rank != 0 and os.path.exists(os.path.join(tmp, "sharded"))):
        fails.append(f"generate_metrics: rank {rank} {'wrote' if wrote else 'did not write'} its files")
    if rank == 0:
        # rank 0 scores the gathered batch: its tables are the metrics of the returned pairs.  Against the single-GPU
        # run they agree only as far as x_0 does: a shard is a smaller batch, and the conv kernels pick their split-K
        # from the batch, so x_0 differs in the fp32 summation order (rel-L2 ~3e-5 here)
        gen = GpuMetricsGenerator(got_pred, got_gt, cfg.METRICS)
        compute_metrics_gpu(cfg, gen, "ALL", 2)
        for k in ("PSNR", "MASK_PSNR", "PSNR_OVER_TIME", "TV_OVER_TIME", "RE_DENSITY"):
            own = float(np.nanmax(np.abs(sharded.last_metrics[k] - gen.data_dict[k])))
            d = float(np.nanmax(np.abs(sharded.last_metrics[k] - single.last_metrics[k])))
            if "PSNR" not in k:                       # sums over the grid: relative to the table's largest entry
                d /= float(np.nanmax(np.abs(single.last_metrics[k])))
            errs[f"metrics {k} vs returned pairs"] = own
            errs[f"metrics {k} vs single-GPU {'dB' if 'PSNR' in k else 'rel'}"] = d
            if not (own <= 1e-6 and d <= (1e-3 if "PSNR" in k else 1e-4)):
                fails.append(f"generate_metrics: {k} differs by {own:.3e} from its own pairs, {d:.3e} from one GPU")

    # the DiT backbone has the same sample_chain contract (cm_dit_sample, per-step graph by default)
    single, sharded = pair(dit_cfg(), "DDPM-DiT")
    from oracle import dit_oracle as dto             # the zero-initialised projections get seeded noise: eps != 0
    sd = dto.randomize_zero_init({k: v.detach().clone() for k, v in single.denoiser.state_dict().items()}, 5)
    single.denoiser.load_state_dict(sd)
    sharded.denoiser.load_state_dict(sd)
    compare("dit ddpm n=5", ddpm(5))
    compare("dit ddpm n=1", ddpm(1))

    dev_err = nat.lib().cm_device_error()
    if dev_err != 0:
        fails.append(f"device error flag {dev_err}")
    if rank == 0:
        print(f"MULTIRANK_DRIVER world={world}: " + ", ".join(f"{k} {v:.3e}" for k, v in errs.items()), flush=True)
    if fails:
        print(f"rank {rank}: " + "; ".join(fails), flush=True)
    flag = torch.tensor([1 if fails else 0], device=dev)
    dist.all_reduce(flag)
    dist.destroy_process_group()
    sys.exit(1 if flag.item() else 0)


if __name__ == "__main__":
    main()
