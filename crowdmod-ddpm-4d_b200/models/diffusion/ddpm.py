"""DDPM driver — drop-in for reference models/diffusion/ddpm.py:23-392 (DDPM-UNet arch).

Same classes / methods / arguments / attributes:

* ``DDPM(ForwardSampler).step(predicted_noise, xnoise, timestep)`` (ddpm.py:23-38)
* ``DDPM_model(cfg, arch, mprops_count, output_dir=None, from_fixed_past=False)`` with
  ``.denoiser .optimizer .scheduler .device .cfg .arch``, ``.train``, ``.sampling``,
  ``.generate_metrics``, ``._train_step``, ``._train_one_epoch``, ``._generate_ddpm``,
  ``._generate_ddim`` (ddpm.py:40-392)

What changes underneath: ``_generate_ddpm`` / ``_generate_ddim`` hand the whole T-step loop to
the native library (``UNet.sample_chain`` -> ``cm_ddpm_sample``): the per-step update
(``DDPM.step`` / DDIM eq. 12 / Sparsity guidance) is the epilogue of the backbone's last
kernel and each step is a CUDA-graph replay.  The Python side only builds the per-step
coefficient table from the sampler's buffers (bit-identical fp32 values to the reference's).

Plotting (utils/plot/*) and CPU metrics (utils/metrics/*) are outside the hot path: they are
imported from the reference when present on sys.path and skipped (with a log line) otherwise.
"""
import gc
import os
import logging
import re

import numpy as np
import torch
import torch.nn.functional as F

from .forward import ForwardSampler, get_from_idx
from ..backbones.unet import UNet
from ..guidance import sparsityGradient  # noqa: F401  (API parity with the reference module)

try:  # package-relative in alias mode, top-level in drop-in mode
    from ...utils.checkpoint import save_checkpoint, create_directory
except (ImportError, ValueError):  # pragma: no cover
    from utils.checkpoint import save_checkpoint, create_directory

try:
    import wandb as _wandb
except Exception:  # wandb is optional; the reference logs train_loss to it
    _wandb = None


def _wandb_log(d):
    if _wandb is not None and getattr(_wandb, "run", None) is not None:
        _wandb.log(d)


class DDPM(ForwardSampler):
    """One step back in the reverse process (API-compatible stand-alone form; the sampling
    loop itself uses the fused native epilogue, not this method)."""

    def step(self, predicted_noise: torch.Tensor, xnoise: torch.Tensor, timestep: int):
        z = torch.randn_like(xnoise) if timestep > 0 else torch.zeros_like(xnoise)
        beta_t = self.beta[timestep].reshape(-1, 1, 1, 1, 1)
        one_by_sqrt_alpha_t = self.one_by_sqrt_alpha[timestep].reshape(-1, 1, 1, 1, 1)
        sqrt_one_minus_alpha_bar_t = self.sqrt_one_minus_alpha_bar[timestep].reshape(-1, 1, 1, 1, 1)
        xdenoised = (one_by_sqrt_alpha_t * (xnoise - (beta_t / sqrt_one_minus_alpha_bar_t) * predicted_noise)
                     + torch.sqrt(beta_t) * z)
        return xdenoised, torch.sqrt(beta_t), 1 - beta_t


def ddpm_coefficients(sampler: ForwardSampler, guidance="None", lam=0.0):
    """Per-step table for cm_chain_args.coef, mode 0 (ddpm.py:25-38,214-229).

    Row i is the step at t = T-1-i: {1/sqrt(alpha_t), beta_t/sqrt(1-abar_t), sqrt(beta_t) (0 at
    t=0: no noise is added on the last step), 0, 0, lambda*sqrt(beta_t) | 0, 0, 0}; computed in
    fp32 with the reference's own op order."""
    beta = sampler.beta.detach().float().cpu()
    a = sampler.one_by_sqrt_alpha.detach().float().cpu()
    b = sampler.sqrt_one_minus_alpha_bar.detach().float().cpu()
    T = beta.numel()
    ts = torch.arange(T - 1, -1, -1)
    coef = torch.zeros(T, 8, dtype=torch.float32)
    coef[:, 0] = a[ts]
    coef[:, 1] = (beta / b)[ts]
    sig = torch.sqrt(beta)[ts]
    coef[:, 2] = torch.where(ts > 0, sig, torch.zeros_like(sig))
    if guidance == "Sparsity":
        coef[:, 5] = float(lam) * sig
    return ts.to(torch.int32), coef


def ddim_coefficients(sampler: ForwardSampler, taus, sigma_t, guidance="None", lam=0.0):
    """Per-step table for cm_chain_args.coef, mode 1 (ddpm.py:238-282, DDIM eq. 12)."""
    beta = sampler.beta.detach().float().cpu()
    sab = sampler.sqrt_alpha_bar.detach().float().cpu()
    somab = sampler.sqrt_one_minus_alpha_bar.detach().float().cpu()
    T = beta.numel()
    order = [int(t) for t in reversed(list(taus))]
    coef = torch.zeros(len(order), 8, dtype=torch.float32)
    cur = T - 1
    for i, t in enumerate(order):
        coef[i, 0] = somab[cur]
        coef[i, 1] = sab[cur]
        coef[i, 2] = sab[t]
        coef[i, 3] = torch.sqrt(1 - sab[t] ** 2 - sigma_t ** 2)
        coef[i, 4] = float(sigma_t)
        if guidance == "Sparsity":
            coef[i, 5] = float(lam) * torch.sqrt(beta[cur])
        cur = t
    return torch.tensor(order, dtype=torch.int32), coef


def shard_samples(nsamples, rank, world):
    """Contiguous slice [lo, hi) of the sample batch owned by `rank` (SURVEY.md §8e: sampling
    shards the independent sample batch across GPUs with no communication).  `lo` is also the
    shard's `sample_offset`, so the in-kernel Philox noise depends on the GLOBAL sample index and
    the union of the shards equals the single-GPU result."""
    base, rem = divmod(int(nsamples), int(world))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


class _RunningMean:
    """Epoch mean of the step losses (torchmetrics.MeanMetric in the reference, ddpm.py:125,146,150).  The sum
    is kept ON THE DEVICE in fp64 and read once per epoch: the reference's per-step ``loss.item()``
    (ddpm.py:145) would stall the host on every step and leave the GPU idle while Python prepares the next."""

    def __init__(self):
        self.total, self.count = None, 0

    def update(self, v):
        v = v.detach().double() if torch.is_tensor(v) else torch.tensor(float(v), dtype=torch.float64)
        self.total = v.clone() if self.total is None else self.total + v
        self.count += 1

    def compute(self):
        return float(self.total.item()) / max(self.count, 1) if self.total is not None else 0.0


class DDPM_model:
    def __init__(self, cfg, arch, mprops_count, output_dir=None, from_fixed_past=False):
        self.cfg = cfg
        self.arch = arch
        self.mprops_count = mprops_count
        self.output_dir = output_dir
        self.from_fixed_past = from_fixed_past

        self.device = torch.device("cuda" if torch.cuda.is_available() else "cpu")
        self.denoiser_cfg = self._get_denoiser_cfg()
        self.denoiser = self._get_denoiser()
        self.denoiser.to(self.device)

        solver = self.denoiser_cfg.TRAIN.SOLVER
        # same optimizer object / state_dict layout as the reference (ddpm.py:53-56); fused=True runs the
        # coupled-L2 Adam update of all 169 tensors as one multi-tensor kernel instead of ~10 foreach passes
        self.optimizer = torch.optim.Adam(self.denoiser.parameters(), lr=solver.LR,
                                          betas=tuple(solver.BETAS), weight_decay=solver.WEIGHT_DECAY,
                                          fused=self.device.type == "cuda")
        self.scheduler = torch.optim.lr_scheduler.ReduceLROnPlateau(
            self.optimizer, mode='min', factor=solver.SCHEDULER.FACTOR,
            patience=solver.SCHEDULER.PATIENCE, min_lr=solver.SCHEDULER.MIN_LR)
        # Optional hooks for tests / multi-GPU sharding (not part of the reference API):
        self.noise_source = None      # callable(nsteps, shape, device) -> [nsteps,*shape] injected z
        self.sample_offset = 0        # global index of this shard's first sample (Philox counter)
        self.use_cuda_graph = True
        # data-parallel training is opt-in (enable_data_parallel); a process group that merely exists is ignored
        self.data_parallel = False
        self.dp_group = None
        self.rank, self.world = 0, 1

    # ------------------------------------------------------------------ data parallel (SURVEY.md §8e)
    def enable_data_parallel(self, group=None):
        """One process per GPU, global batch split over the ranks: broadcasts rank 0's parameters so every
        replica starts from the same model, then averages the flat gradient buffer with ONE all-reduce per
        step.  The epoch loss is averaged over ranks before ReduceLROnPlateau / best-checkpoint decisions, the
        random extra-checkpoint epochs are drawn on rank 0, and only rank 0 writes checkpoints.

        Sampling is sharded too: every reverse chain (``_generate_ddpm`` / ``_generate_ddim``, hence ``sampling``
        and ``generate_metrics``) takes x_T, ``past``, the noise seed (or the ``noise_source`` noise) from rank 0,
        runs this rank's contiguous slice of the samples (``shard_samples``) and all-gathers x_0 (and the history)
        back to every rank.  The Philox noise is keyed by the global sample index, so x_0 is the single-GPU chain
        that rank 0's inputs give, up to the fp32 summation order of a smaller batch, whatever the other ranks'
        RNG state or data order.  Only rank 0 plots, computes metrics and writes files."""
        import torch.distributed as dist
        from ..backbones.unet_autograd import enable_data_parallel
        if not (dist.is_available() and dist.is_initialized()):
            raise RuntimeError("enable_data_parallel: call torch.distributed.init_process_group first")
        self.dp_group = group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        src = dist.get_global_rank(group, 0) if group is not None else 0
        with torch.no_grad():
            for t in self.denoiser.state_dict().values():
                dist.broadcast(t, src=src, group=group)
        enable_data_parallel(self.denoiser, group)
        self.data_parallel = True
        return self

    def _get_denoiser_cfg(self):
        gen_model_key, backbone_key = self.arch.upper().split('-')
        gen_cfg = getattr(self.cfg.MODEL, gen_model_key)
        return getattr(gen_cfg, backbone_key)

    def _get_denoiser(self):
        if self.arch == "DDPM-UNet":
            c = self.denoiser_cfg
            return UNet(input_channels=self.mprops_count, output_channels=self.mprops_count,
                        num_res_blocks=c.NUM_RES_BLOCKS, base_channels=c.BASE_CH,
                        base_channels_multiples=c.BASE_CH_MULT, apply_attention=c.APPLY_ATTENTION,
                        dropout_rate=c.DROPOUT_RATE, time_multiple=c.TIME_EMB_MULT,
                        condition=c.CONDITION)
        if self.arch == "DDPM-DiT":
            # reference ddpm.py:88-104 (sampling / inference natively; training this backbone raises in forward)
            from ..backbones.DiT4D_V4 import DiT4D_V4
            c = self.denoiser_cfg
            return DiT4D_V4(input_channels=self.mprops_count, output_channels=self.mprops_count,
                            grid_rows=self.cfg.MACROPROPS.ROWS, grid_cols=self.cfg.MACROPROPS.COLS,
                            past_len=self.cfg.DATASET.PAST_LEN, future_len=self.cfg.DATASET.FUTURE_LEN,
                            t_patch_size=c.T_PATCH_SIZE, patch_size=c.PATCH_SIZE, hidden_size=c.HIDDEN_SIZE,
                            depth=c.DEPTH, num_heads=c.NUM_HEADS, mlp_ratio=c.MLP_RATIO, dropout_rate=c.DROPOUT_RATE,
                            time_multiple=c.TIME_EMB_MULT, condition=c.CONDITION)
        raise ValueError(f"Unknown Architecture {self.arch}")

    # ------------------------------------------------------------------ training
    def _train_step(self, future: torch.Tensor, past: torch.Tensor, forward_sampler: DDPM):
        t = torch.randint(low=0, high=forward_sampler.timesteps, size=(future.shape[0],),
                          device=future.device)
        future_macroprops_noisy, eps_true = forward_sampler(future, t)
        eps_predicted = self.denoiser(future_macroprops_noisy, t, past)
        return F.mse_loss(eps_predicted, eps_true)

    def _train_one_epoch(self, forward_sampler: DDPM, loader, epoch):
        loss_record = _RunningMean()
        self.denoiser.train()
        for batched_train_data in loader:
            past_train, future_train = batched_train_data
            past_train = past_train.float().to(device=self.device)
            future_train = future_train.float().to(device=self.device)
            loss = self._train_step(future_train, past_train, forward_sampler)
            self.optimizer.zero_grad(set_to_none=True)
            loss.backward()
            self.optimizer.step()
            loss_record.update(loss.detach())
        epoch_loss = loss_record.compute()
        if self.device.type == "cuda":
            from ..backbones.unet import _native
            _native().check_device_error(f"training epoch {epoch}")   # e.g. a saturated fp16 gradient operand
        if self.data_parallel and self.world > 1:
            import torch.distributed as dist
            t = torch.tensor([epoch_loss], device=self.device, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.dp_group)
            epoch_loss = float(t.item()) / self.world
        return epoch_loss

    def train(self, batched_train_data, baseline_ckpt=None):
        forward_sampler = DDPM(timesteps=self.cfg.MODEL.DDPM.TIMESTEPS, scale=self.cfg.MODEL.DDPM.SCALE)
        forward_sampler.to(self.device)
        if baseline_ckpt is not None:
            self.denoiser.load_state_dict(
                torch.load(baseline_ckpt, map_location=self.device, weights_only=True)['model'])
            self.denoiser.to(self.device)
            logging.info("Baseline checkpoint loaded successfully.")
        best_loss = 1e6
        consecutive_nan_count = 0
        epochs = self.denoiser_cfg.TRAIN.EPOCHS
        epochs_cktp_to_save = np.random.randint(int(epochs * 0.75), epochs + 1,
                                                size=self.cfg.MODEL.DDPM.CHECKPOINTS_TO_KEEP)
        if self.data_parallel and self.world > 1:      # every rank keeps rank 0's draw
            import torch.distributed as dist
            t = torch.as_tensor(epochs_cktp_to_save, dtype=torch.int64, device=self.device)
            src = dist.get_global_rank(self.dp_group, 0) if self.dp_group is not None else 0
            dist.broadcast(t, src=src, group=self.dp_group)
            epochs_cktp_to_save = t.cpu().numpy()
        writer = (not self.data_parallel) or self.rank == 0
        for epoch in range(1, epochs + 1):
            torch.cuda.empty_cache()
            gc.collect()
            epoch_loss = self._train_one_epoch(forward_sampler, batched_train_data, epoch)
            _wandb_log({"train_loss": epoch_loss})
            self.scheduler.step(epoch_loss)
            if np.isnan(epoch_loss):
                consecutive_nan_count += 1
                logging.warning(f"Epoch {epoch}: loss is NaN ({consecutive_nan_count} consecutive)")
                if consecutive_nan_count >= 3:
                    logging.error("Loss has been NaN for 3 consecutive epochs; terminating training early.")
                    if _wandb is not None and getattr(_wandb, "run", None) is not None:
                        _wandb.finish()
                    break
            else:
                consecutive_nan_count = 0
            if epoch_loss < best_loss:
                best_loss = epoch_loss
                if writer:
                    save_checkpoint(self.optimizer, self.denoiser, "000", self.cfg, self.arch)
            if epoch in epochs_cktp_to_save and writer:
                logging.info(f"Epoch {epoch}: in checkpoints_to_keep set, saving model.")
                save_checkpoint(self.optimizer, self.denoiser, epoch, self.cfg, self.arch)
        logging.info(f"Trained model {self.arch} saved in {self.cfg.DATA_FS.SAVE_DIR}")

    # ------------------------------------------------------------------ sampling
    def _chain(self, past, x, tsteps, coef, mode, history):
        past = past.to(self.device).float().contiguous()
        nsteps = tsteps.numel()
        noise = None
        seed = 0
        if self.noise_source is not None:
            noise = self.noise_source(nsteps, tuple(x.shape), x.device).contiguous()
        else:
            seed = int(torch.randint(0, 2 ** 62, (1,)).item())   # consumes torch's generator once
        if self._sharded():
            hist = self._sharded_chain(past, x, tsteps, coef, mode, history, noise, seed)
        else:
            hist = None
            if history:
                hist = torch.empty((nsteps + 1,) + tuple(x.shape), device=x.device, dtype=torch.float32)
                hist[0].copy_(x)
            self.denoiser.sample_chain(past, x, tsteps, coef, mode=mode, noise=noise, seed=seed,
                                       sample_offset=self.sample_offset, history=hist,
                                       use_graph=self.use_cuda_graph)
        if self.device.type == "cuda":
            from ..backbones.unet import _native
            _native().check_device_error("the reverse chain")     # synchronises: x_0 is about to be read anyway
        return hist

    # ------------------------------------------------------------------ sharded sampling (enable_data_parallel)
    def _sharded(self):
        return self.data_parallel and self.world > 1

    def _from_rank0(self, t):
        """The group's rank 0's value of ``t`` on every rank: a contiguous copy on the receiving ranks, so that the
        caller's tensor is never overwritten."""
        import torch.distributed as dist
        buf = t.contiguous() if self.rank == 0 else torch.empty(t.shape, dtype=t.dtype, device=t.device)
        src = dist.get_global_rank(self.dp_group, 0) if self.dp_group is not None else 0
        dist.broadcast(buf, src=src, group=self.dp_group)
        return buf

    def _gather_samples(self, part, n, dim):
        """Every rank's ``shard_samples`` slice of a sample axis (``dim``) concatenated in rank order, on every rank.
        The shards can differ by one sample: each is padded to the largest so that ONE all_gather_into_tensor
        moves them all, and the padding is trimmed afterwards."""
        import torch.distributed as dist
        sizes = [hi - lo for lo, hi in (shard_samples(n, r, self.world) for r in range(self.world))]
        shape = list(part.shape)
        shape[dim] = sizes[0]
        buf = part
        if part.shape[dim] != sizes[0]:
            buf = part.new_zeros(shape)
            buf.narrow(dim, 0, part.shape[dim]).copy_(part)
        out = part.new_empty([self.world * shape[0]] + shape[1:])     # gloo accepts only the concatenated form
        dist.all_gather_into_tensor(out, buf, group=self.dp_group)
        out = out.view([self.world] + shape)
        return torch.cat([out[r].narrow(dim, 0, s) for r, s in enumerate(sizes)], dim)

    def _sharded_chain(self, past, x, tsteps, coef, mode, history, noise, seed):
        """``_chain`` over the data-parallel group.  ``x`` (x_T) already holds rank 0's draw; ``past``, the seed and
        the injected noise are taken from rank 0 too, so the result does not depend on the other ranks' RNG state
        or data order.  This rank runs its slice [lo, hi) of the samples with Philox offset ``sample_offset + lo``,
        then x_0 (in place in ``x``) and the history are gathered back to the full batch."""
        past = self._from_rank0(past)
        seed = int(self._from_rank0(torch.tensor([seed], dtype=torch.int64, device=x.device)).item())
        if noise is not None:
            noise = self._from_rank0(noise)
        n = x.shape[0]
        lo, hi = shard_samples(n, self.rank, self.world)
        mine = x[lo:hi]                  # a contiguous view: the chain runs in place on the caller's x
        hist = None
        if history:
            hist = torch.empty((tsteps.numel() + 1,) + tuple(mine.shape), device=x.device, dtype=torch.float32)
            hist[0].copy_(mine)
        if hi > lo:                      # with n < world some ranks hold no sample (cm_dit_sample rejects n = 0)
            self.denoiser.sample_chain(past[lo:hi], mine, tsteps, coef, mode=mode,
                                       noise=noise[:, lo:hi].contiguous() if noise is not None else None, seed=seed,
                                       sample_offset=self.sample_offset + lo, history=hist,
                                       use_graph=self.use_cuda_graph)
        x.copy_(self._gather_samples(mine, n, 0))
        return self._gather_samples(hist, n, 1) if history else None

    def _guidance(self):
        g = self.cfg.MODEL.DDPM.GUIDANCE
        if g == "mass_preservation":
            raise NotImplementedError("mass_preservation guidance is outside the B200 hot path "
                                      "(SURVEY.md §2 #6)")
        return g, (self.cfg.MODEL.DDPM.LAMBDA_GUIDANCE if g == "Sparsity" else 0.0)

    def _x_T(self, nsamples):
        x = torch.randn((nsamples, self.mprops_count, self.cfg.MACROPROPS.ROWS,
                         self.cfg.MACROPROPS.COLS, self.cfg.DATASET.FUTURE_LEN), device=self.device)
        return self._from_rank0(x) if self._sharded() else x

    @torch.inference_mode()
    def _generate_ddpm(self, past: torch.Tensor, backward_sampler: DDPM, nsamples, history=False):
        self.denoiser.eval()
        xnoisy = self._x_T(nsamples)
        x_T = xnoisy.clone()
        guidance, lam = self._guidance()
        tsteps, coef = ddpm_coefficients(backward_sampler, guidance, lam)
        hist = self._chain(past, xnoisy, tsteps, coef, 0, history)
        over_time = [hist[i] for i in range(hist.shape[0])] if history else [x_T, xnoisy]
        return xnoisy, over_time

    @torch.inference_mode()
    def _generate_ddim(self, past: torch.Tensor, taus, backward_sampler: DDPM, nsamples, history=False):
        self.denoiser.eval()
        sigma_t = self.cfg.MODEL.DDPM.SIGMA
        xnoisy = self._x_T(nsamples)
        x_T = xnoisy.clone()
        guidance, lam = self._guidance()
        tsteps, coef = ddim_coefficients(backward_sampler, taus, sigma_t, guidance, lam)
        hist = self._chain(past, xnoisy, tsteps, coef, 1, history)
        over_time = [hist[i] for i in range(hist.shape[0])] if history else [x_T, xnoisy]
        return xnoisy, over_time

    def _load(self, model_fullname):
        self.denoiser.load_state_dict(
            torch.load(model_fullname, map_location=torch.device('cpu'), weights_only=True)['model'])
        self.denoiser.to(self.device)

    def _predict(self, past, backward_sampler, nsamples):
        timesteps = self.cfg.MODEL.DDPM.TIMESTEPS
        if self.cfg.MODEL.DDPM.SAMPLER == "DDPM":
            x, _ = self._generate_ddpm(past, backward_sampler, nsamples)
            l1 = torch.mean(torch.abs(x[:, 0])).item()
            logging.info(f'L1 norm {l1:.2f} using {self.cfg.MODEL.DDPM.GUIDANCE} guidance')
            return x
        if self.cfg.MODEL.DDPM.SAMPLER == "DDIM":
            taus = np.arange(0, timesteps - 1, self.cfg.MODEL.DDPM.DDIM_DIVIDER)
            logging.info(f'Shape of subset taus:{taus.shape}')
            x, _ = self._generate_ddim(past, taus, backward_sampler, nsamples)
            return x
        logging.info(f"{self.cfg.MODEL.DDPM.SAMPLER} sampler not supported")
        return None

    def sampling(self, batched_test_data, plotType, model_fullname, plotMprop, plotPast, samePastSeq,
                 macropropPlotter):
        logging.info(f'model full name:{model_fullname}')
        writer = (not self.data_parallel) or self.rank == 0
        if writer:
            create_directory(self.output_dir)
        self._load(model_fullname)
        backward_sampler = DDPM(timesteps=self.cfg.MODEL.DDPM.TIMESTEPS, scale=self.cfg.MODEL.DDPM.SCALE)
        backward_sampler.to(self.device)
        if self.from_fixed_past:
            nsamples = batched_test_data.batch_size
            macropropPlotter.samples4plot = nsamples
        else:
            nsamples = self.cfg.MODEL.NSAMPLES4PLOTS
        logging.info(f"Total samples to predict:{nsamples}")
        for batch in batched_test_data:
            past_test, future_test = batch
            past_test = past_test.float().to(device=self.device)
            future_test = future_test.float().to(device=self.device)
            if self.from_fixed_past:
                random_past_idx = torch.arange(nsamples)
            else:
                random_past_idx = torch.randperm(past_test.shape[0])[:nsamples]
                if samePastSeq:
                    random_past_idx.fill_(random_past_idx[0])
            random_past_samples = past_test[random_past_idx]
            random_future_samples = future_test[random_past_idx]
            predictions = self._predict(random_past_samples, backward_sampler, nsamples)
            if not writer:
                return predictions
            try:
                from utils.plot.plot_sampled_mprops import setup_predictions_plot
                setup_predictions_plot(predictions, random_past_idx, random_past_samples,
                                       random_future_samples, model_fullname, plotType, plotMprop,
                                       plotPast, macropropPlotter)
                logging.info(f"All sampling macroprops seqs saved in {self.output_dir}")
            except ImportError:
                logging.info("utils.plot not importable (reference not on sys.path): plots skipped")
            return predictions

    def generate_metrics(self, batched_test_data, chunkRepdPastSeq, metric, batches_to_use,
                         samples_per_batch, model_fullname, output_dir):
        logging.info(f'model full name:{model_fullname}')
        writer = (not self.data_parallel) or self.rank == 0
        if writer:
            create_directory(self.output_dir)
        self._load(model_fullname)
        match = re.search(r'TE\d+_PL\d+_FL\d+_CE\d+_NA', model_fullname)
        backward_sampler = DDPM(timesteps=self.cfg.MODEL.DDPM.TIMESTEPS, scale=self.cfg.MODEL.DDPM.SCALE)
        backward_sampler.to(self.device)
        count_batch = 0
        pred_seq_list, gt_seq_list = [], []
        for batch in batched_test_data:
            logging.info("===" * 20)
            logging.info(f'Computing sampling on batch:{count_batch + 1}')
            past_test, future_test = batch
            past_test = past_test.float().to(device=self.device)
            future_test = future_test.float().to(device=self.device)
            if past_test.shape[0] < samples_per_batch:
                random_past_idx = torch.randperm(past_test.shape[0])
            else:
                random_past_idx = torch.randperm(past_test.shape[0])[:samples_per_batch]
            random_past_idx = torch.repeat_interleave(random_past_idx, chunkRepdPastSeq)[:samples_per_batch]
            random_past_samples = past_test[random_past_idx]
            random_future_samples = future_test[random_past_idx]
            if self._sharded():          # every rank returns the (prediction, ground truth) pairs rank 0 scores
                random_future_samples = self._from_rank0(random_future_samples)
            x = self._predict(random_past_samples, backward_sampler, samples_per_batch)
            for i in range(len(random_past_idx)):
                pred_seq_list.append(x[i])
                gt_seq_list.append(random_future_samples[i])
            count_batch += 1
            if count_batch == batches_to_use:
                break
        if not writer:
            return pred_seq_list, gt_seq_list
        logging.info("===" * 20)
        logging.info(f'Computing metrics on predicted mprops sequences with {self.arch} model.')
        # reduction metrics (PSNR / MASK_PSNR / RE_DENSITY / TV) on the device in one launch; SSIM, the motion-feature
        # histograms and the energy metric stay with the reference's CPU class when it is importable
        from ...utils.metrics_gpu import GpuMetricsGenerator, compute_metrics_gpu
        title = (f"{self.cfg.DATASET.BATCH_SIZE * chunkRepdPastSeq * batches_to_use} samples in total "
                 f"(BS:{self.cfg.DATASET.BATCH_SIZE}, Rep:{chunkRepdPastSeq}, TB:{batches_to_use})-({self.arch})")
        covered = []
        if metric in ("ALL",) + GpuMetricsGenerator.GPU_METRICS:
            gpu_gen = GpuMetricsGenerator(pred_seq_list, gt_seq_list, self.cfg.METRICS, output_dir)
            covered = compute_metrics_gpu(self.cfg, gpu_gen, metric, chunkRepdPastSeq)
            gpu_files = gpu_gen.save_data_metrics(match, title, samples_per_batch)
            self.last_metrics = gpu_gen.data_dict
        rest = metric if metric not in covered else None
        if metric == "ALL" or rest is not None:
            try:
                from utils.metrics.metricsGenerator import MetricsGenerator
            except ImportError:
                logging.info("utils.metrics not importable (reference not on sys.path): SSIM / motion-feature / energy "
                             "metrics skipped")
                return pred_seq_list, gt_seq_list
            ref_gen = MetricsGenerator(pred_seq_list, gt_seq_list, self.cfg.METRICS, output_dir)
            if metric in ('SSIM', 'ALL'):
                ref_gen.compute_ssim_metric(chunkRepdPastSeq)
            if metric in ('MF_MSE', 'MF_BHATT', 'ALL'):
                ref_gen.compute_motion_feature_metrics(metric in ('MF_MSE', 'ALL'), metric in ('MF_BHATT', 'ALL'))
            if metric in ('ENERGY', 'ALLA'):
                ref_gen.compute_energy_metric(chunkRepdPastSeq)
            ref_gen.save_data_metrics(match, title, samples_per_batch)
            if covered:          # the reference rewrote metrics_files.json with its own files only: merge ours back in
                import json
                jp = os.path.join(output_dir, "metrics_files.json")
                files = json.load(open(jp))
                files.update({k: v for k, v in gpu_files.items() if k != "title"})
                json.dump(files, open(jp, "w"), indent=2)
        return pred_seq_list, gt_seq_list
