"""One short training epoch through DDPM_model._train_one_epoch on synthetic ATC-shaped data, for the reproducibility
tests of test_gpu_deterministic.py.  Run as a script it prints the SHA-256 of the final state_dict and the epoch loss
(the cross-process check); imported, ``run`` returns them."""
import hashlib
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")

import numpy as np  # noqa: E402
import torch  # noqa: E402

ROWS, COLS, PAST, FUT = 12, 36, 5, 3


def make_cfg(out_dir):
    from crowdmod_ddpm_4d_b200.utils.myparser import YamlParser
    return YamlParser({
        "DATA_FS": {"OUTPUT_DIR": out_dir, "SAVE_DIR": out_dir + "/"},
        "MACROPROPS": {"ROWS": ROWS, "COLS": COLS},
        "DATASET": {"NAME": "atc", "PAST_LEN": PAST, "FUTURE_LEN": FUT, "BATCH_SIZE": 8},
        "MODEL": {"NAME": "{}_B_TE{}_PL{}_FL{}_CE{}_{}.pth", "NSAMPLES": 8, "NSAMPLES4PLOTS": 2,
                  "DDPM": {"SAMPLER": "DDPM", "TIMESTEPS": 1000, "SCALE": 0.5, "SIGMA": 0.001,
                           "DDIM_DIVIDER": 2, "GUIDANCE": "None", "LAMBDA_GUIDANCE": 0.004,
                           "CHECKPOINTS_TO_KEEP": 7,
                           "UNET": {"CONDITION": "Past", "NUM_RES_BLOCKS": 1, "BASE_CH": 32, "BASE_CH_MULT": [1, 2, 4],
                                    "APPLY_ATTENTION": [False, False, True, False], "DROPOUT_RATE": 0.1,
                                    "TIME_EMB_MULT": 4,
                                    "TRAIN": {"EPOCHS": 1, "SOLVER": {
                                        "LR": 1e-3, "WEIGHT_DECAY": 3e-3, "BETAS": [0.5, 0.999],
                                        "SCHEDULER": {"FACTOR": 0.5, "PATIENCE": 10, "MIN_LR": 1e-6}}}}}},
    })


def state_sha(sd):
    h = hashlib.sha256()
    for k in sorted(sd):
        h.update(k.encode())
        h.update(sd[k].detach().cpu().contiguous().numpy().tobytes())
    return h.hexdigest()


def run(deterministic, seed=11, epochs=1):
    """Fresh DDPM_model under torch.manual_seed(seed); `epochs` passes of _train_one_epoch over 4 batches of 8 windows
    (dropout 0.1, Adam).  Returns (model, [epoch losses], SHA-256 of the final state_dict)."""
    from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import DDPM, DDPM_model
    from crowdmod_ddpm_4d_b200.utils.dataset_gpu import GpuMacropropsDataset, GpuWindowLoader
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(deterministic)
    try:
        torch.manual_seed(seed)
        with tempfile.TemporaryDirectory() as d:
            cfg = make_cfg(d)
            model = DDPM_model(cfg, "DDPM-UNet", 3)
            seq = np.random.default_rng(seed).normal(size=(4, 3, ROWS, COLS, 24)).astype(np.float32)
            seq[:, 0] = np.abs(seq[:, 0])
            ds = GpuMacropropsDataset(seq, cfg, 3, stride=2)
            loader = GpuWindowLoader(ds, 8, shuffle=True, drop_last=True)
            fs = DDPM(timesteps=1000, scale=0.5).cuda()
            losses = [float(model._train_one_epoch(fs, _first(loader, 4), e)) for e in range(epochs)]
            torch.cuda.synchronize()
            return model, losses, state_sha(model.denoiser.state_dict())
    finally:
        torch.use_deterministic_algorithms(prev)


def _first(loader, n):
    out = []
    for i, b in enumerate(loader):
        if i == n:
            break
        out.append(b)
    return out


if __name__ == "__main__":
    _, losses, sha = run(True)
    print(f"SHA {sha} LOSS {losses[0].hex()}")
