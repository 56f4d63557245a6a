"""CPU: host-side logic of the drop-in boundary — config schema + adapter, module tree /
state_dict contract, coefficient tables, checkpoint naming, error behaviour without a GPU."""
import glob
import os

import numpy as np
import pytest
import torch

from crowdmod_ddpm_4d_b200.models.backbones.unet import UNet
from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import (DDPM, DDPM_model, ddim_coefficients,
                                                         ddpm_coefficients)
from crowdmod_ddpm_4d_b200.models.diffusion.forward import ForwardSampler
from crowdmod_ddpm_4d_b200.utils.checkpoint import get_model_fullname, save_checkpoint
from crowdmod_ddpm_4d_b200.utils.myparser import getYamlConfig
from oracle import ddpm_oracle as do
from oracle import ref_shim
from tests._util import build_unet, load_golden

CFG = os.path.join(os.path.dirname(__file__), "configs")
REF_CFG = os.path.join(ref_shim.REF_ROOT, "config")


def test_state_dict_contract_atc():
    meta, _ = load_golden("unet_atc_b2")
    net = build_unet(meta)                       # asserts SHA-256 of the seeded state_dict
    sd = net.state_dict()
    assert len(sd) == 169
    assert sum(p.numel() for p in net.parameters() if p.requires_grad) == 7200099
    assert tuple(sd["time_embeddings.time_blocks.0.weight"].shape) == (1000, 32)
    assert not net.time_embeddings.time_blocks[0].weight.requires_grad
    assert tuple(sd["decoder_blocks.0.attention.mhsa.in_proj_weight"].shape) == (384, 128)
    assert tuple(sd["decoder_blocks.5.upsample.1.weight"].shape) == (64, 64, 3, 3, 3)
    assert tuple(sd["final.2.weight"].shape) == (3, 32, 3, 3, 3)


def test_native_plan_mirrors_state_dict():
    meta, _ = load_golden("unet_small_b3")
    net = build_unet(meta)
    plan = net._plan(4, 4, 2, 2)
    names = plan.names()
    sd = net.state_dict()
    assert [n for n, _ in names] == list(sd.keys())
    assert all(tuple(sd[n].shape) == s for n, s in names)
    launches, flops = net.native_stats(4, 4, 2, 2)
    assert launches > 0 and flops > 0


def test_flops_census_matches_survey():
    meta, _ = load_golden("unet_atc_b2")
    net = build_unet(meta)
    _, flops = net.native_stats(12, 36, 5, 3)
    assert abs(flops / 1e9 - 4.323) < 0.01          # SURVEY.md §6: 4.323 GFLOP/sample/step
    _, flops = net.native_stats(28, 24, 5, 3)
    assert abs(flops / 1e9 - 6.729) < 0.01          # HERMES-CR-120


def test_no_cpu_path():
    meta, a = load_golden("unet_small_b3")
    net = build_unet(meta).eval()
    with torch.no_grad(), pytest.raises(RuntimeError, match="no CPU path"):
        net(a["future"], a["t"], a["past"])


def test_geometry_constraint_is_reported():
    net = UNet(3, 3, 1, 32, [1, 2, 4], [False, False, True], 0.1, 4, "Past")
    from crowdmod_ddpm_4d_b200._native import NativeError
    with pytest.raises(NativeError, match="divisible"):
        net._plan(12, 36, 5, 2)                      # 7 frames: not divisible by 4


def test_forward_sampler_buffers_match_oracle():
    fs = ForwardSampler(timesteps=1000, scale=0.5)
    s = do.schedule(1000, 0.5)
    for k, v in s.items():
        assert torch.equal(getattr(fs, k), v), k
    assert fs.timesteps == 1000
    assert list(dict(fs.named_buffers()).keys()) == ["beta", "alpha", "alpha_bar", "sqrt_alpha_bar",
                                                      "one_by_sqrt_alpha", "sqrt_one_minus_alpha_bar"]


def test_ddpm_step_api_matches_oracle():
    d = DDPM(timesteps=50, scale=0.5)
    s = do.schedule(50, 0.5)
    x = torch.randn(2, 3, 4, 4, 2)
    e = torch.randn_like(x)
    torch.manual_seed(3)
    out, sigma, one_minus_beta = d.step(e, x, 17)
    torch.manual_seed(3)
    z = torch.randn_like(x)
    assert torch.equal(out, do.ddpm_step(s, e, x, 17, z))
    assert torch.equal(sigma.flatten(), torch.sqrt(s["beta"][17]).flatten())
    out0, _, _ = d.step(e, x, 0)
    assert torch.equal(out0, do.ddpm_step(s, e, x, 0, None))


def test_coefficient_tables():
    fs = DDPM(timesteps=1000, scale=0.5)
    ts, coef = ddpm_coefficients(fs, "Sparsity", 0.004)
    assert ts[0].item() == 999 and ts[-1].item() == 0 and coef.shape == (1000, 8)
    assert coef[-1, 2].item() == 0.0                           # no noise at t = 0
    assert torch.equal(coef[:, 0], fs.one_by_sqrt_alpha.flip(0))
    assert torch.equal(coef[:, 1], (fs.beta / fs.sqrt_one_minus_alpha_bar).flip(0))
    assert torch.allclose(coef[:, 5], 0.004 * torch.sqrt(fs.beta).flip(0), rtol=1e-7, atol=0)
    taus = np.arange(0, 999, 90)
    ts, coef = ddim_coefficients(fs, taus, 0.001)
    assert ts.tolist() == list(reversed(taus.tolist()))
    assert coef[0, 0].item() == fs.sqrt_one_minus_alpha_bar[999].item()     # starts from T-1
    assert coef[1, 1].item() == fs.sqrt_alpha_bar[int(taus[-1])].item()     # then previous tau


def test_config_nested_and_legacy_adapter():
    cfg = getYamlConfig(os.path.join(CFG, "atc_nested.yml"))
    assert cfg.MODEL.DDPM.UNET.BASE_CH == 32 and cfg.MODEL.DDPM.LAMBDA_GUIDANCE == 0.004
    m = DDPM_model(cfg, "DDPM-UNet", 3)
    assert isinstance(m.denoiser, UNet) and len(m.denoiser.state_dict()) == 169
    assert m.optimizer.defaults["lr"] == 5e-5 and m.optimizer.defaults["betas"] == (0.5, 0.999)
    assert m.optimizer.defaults["weight_decay"] == 0.003
    with pytest.raises(ValueError, match="Unknown Architecture"):
        DDPM_model(cfg, "ddpm-unet", 3)              # cfg node resolves (upper()), arch string does not
    with pytest.raises(AttributeError):
        DDPM_model(cfg, "DDPM-Foo", 3)               # reference: getattr(cfg.MODEL.DDPM, "FOO")
    with pytest.raises(AttributeError):
        DDPM_model(cfg, "FM-UNet", 3)                            # no MODEL.FM node: same as reference

    leg = getYamlConfig(os.path.join(CFG, "atc_legacy_flat.yml"))
    u = leg.MODEL.DDPM.UNET
    assert u.BASE_CH == 64 and u.TRAIN.EPOCHS == 250 and u.TRAIN.SOLVER.LR == 5e-5
    assert leg.MODEL.DDPM.TIMESTEPS == 1000 and leg.MODEL.DDPM.GUIDANCE == "Sparsity"
    assert leg.MODEL.DDPM.CHECKPOINTS_TO_KEEP == 7 and leg.MODEL.NSAMPLES == 1280
    assert leg.DATA_FS.SAVE_DIR == "saved_models/"
    m = DDPM_model(leg, "DDPM-UNet", 3)
    assert sum(p.numel() for p in m.denoiser.parameters() if p.requires_grad) == 28766915


@pytest.mark.skipif(not os.path.isdir(REF_CFG), reason=ref_shim.MISSING)
@pytest.mark.parametrize("name", ["ATC.yml", "ATC_synthetic.yml", "ATC_medium.yml", "HERMES-CR-120.yml",
                                  "ETHUCY_ddpm.yml"])
def test_all_baseline_configs_load(name):
    cfg = getYamlConfig(os.path.join(REF_CFG, name))
    m = DDPM_model(cfg, "DDPM-UNet", 3)
    assert cfg.MODEL.DDPM.CHECKPOINTS_TO_KEEP >= 1
    rows, cols = cfg.MACROPROPS.ROWS, cfg.MACROPROPS.COLS
    launches, flops = m.denoiser.native_stats(rows, cols, cfg.DATASET.PAST_LEN, cfg.DATASET.FUTURE_LEN)
    assert flops > 0


@pytest.mark.parametrize("name,params,gflop", [
    ("atc_nested.yml", 7200099, 4.323),                    # config/ATC.yml
    ("atc_synthetic_legacy_flat.yml", 7200099, 4.323),     # config/ATC_synthetic.yml
    ("atc_legacy_flat.yml", 28766915, 34.44),              # config/ATC_medium.yml
    ("hermes_nested_model_samples.yml", 7200099, 6.729),   # config/HERMES-CR-120.yml
    ("ethucy_legacy_flat.yml", 7200099, 0.960),            # config/ETHUCY_ddpm.yml
])
def test_baseline_config_schemas_load(name, params, gflop):
    """The five BASELINE configs' schemas and shapes (stored fixtures): they load, build the denoiser and its
    native plan, and give the parameter and FLOP counts of BASELINE.md section 2."""
    cfg = getYamlConfig(os.path.join(CFG, name))
    m = DDPM_model(cfg, "DDPM-UNet", 3)
    assert cfg.MODEL.DDPM.CHECKPOINTS_TO_KEEP >= 1
    assert sum(p.numel() for p in m.denoiser.parameters() if p.requires_grad) == params
    rows, cols = cfg.MACROPROPS.ROWS, cfg.MACROPROPS.COLS
    launches, flops = m.denoiser.native_stats(rows, cols, cfg.DATASET.PAST_LEN, cfg.DATASET.FUTURE_LEN)
    assert launches > 0 and abs(flops / 1e9 - gflop) < 0.01


def test_checkpoint_layout(tmp_path):
    cfg = getYamlConfig(os.path.join(CFG, "atc_nested.yml"))
    cfg.DATA_FS.SAVE_DIR = str(tmp_path) + "/"
    assert get_model_fullname(cfg, "DDPM-UNet", "000").endswith("DDPM-UNet_ATC_TE200_PL5_FL3_CE000_NA.pth")
    m = DDPM_model(cfg, "DDPM-UNet", 3)
    path = save_checkpoint(m.optimizer, m.denoiser, "000", cfg, "DDPM-UNet")
    ck = torch.load(path, weights_only=True)
    assert set(ck.keys()) == {"opt", "model"} and len(ck["model"]) == 169
    m2 = DDPM_model(cfg, "DDPM-UNet", 3)
    m2.denoiser.load_state_dict(ck["model"])
    assert all(torch.equal(a, b) for a, b in zip(m.denoiser.state_dict().values(), m2.denoiser.state_dict().values()))


def test_feed_and_metrics_modules_have_no_cpu_path():
    """The callers either side of the path (SURVEY.md section 8 f3 / f4) refuse CPU tensors instead of falling back."""
    import types
    import numpy as np
    import pytest
    import torch
    from crowdmod_ddpm_4d_b200 import _native
    from crowdmod_ddpm_4d_b200.utils.dataset_gpu import GpuMacropropsDataset
    from crowdmod_ddpm_4d_b200.utils.metrics_gpu import GpuMetricsGenerator
    cfg = types.SimpleNamespace(DATASET=types.SimpleNamespace(PAST_LEN=5, FUTURE_LEN=3))
    seq = np.zeros((2, 3, 4, 4, 12), dtype=np.float32)
    with pytest.raises(_native.NativeError):
        GpuMacropropsDataset(seq, cfg, 3, stride=2, device="cpu")
    with pytest.raises(ValueError):
        GpuMacropropsDataset(seq[0], cfg, 3, stride=2, device="cpu")
    x = torch.zeros(2, 3, 4, 4, 3)
    with pytest.raises(_native.NativeError):
        GpuMetricsGenerator(x, x, types.SimpleNamespace(MPROPS_COUNT=3))
    with pytest.raises(ValueError):
        GpuMetricsGenerator(x, x[:1], types.SimpleNamespace(MPROPS_COUNT=3))
    # headers / file naming follow the reference's MetricsGenerator (metricsGenerator.py:13-35)
    assert GpuMetricsGenerator.HEADERS["RE_DENSITY"] == "re_f6,re_f7,re_f8"
    assert GpuMetricsGenerator.HEADERS["PSNR"] == "rho,vx,vy"


def test_dit_plan_entry_points_work_without_gpu():
    """cm_dit_create validates the reference's constructor constraints (DiT4D_V4.py:26-31, :252-254) and lists the
    99 state_dict entries of the ATC configuration."""
    import ctypes
    import crowdmod_ddpm_4d_b200._native as n
    cfg = n.DitConfig(in_channels=3, out_channels=3, rows=12, cols=36, past_len=5, future_len=3, t_patch=4, patch=4,
                      hidden=256, depth=6, heads=4, mlp_hidden=1024, time_multiple=4, table_steps=1000, t_max_slots=8)
    h = ctypes.c_void_p()
    n.check(n.lib().cm_dit_create(ctypes.byref(cfg), ctypes.byref(h)))
    assert n.lib().cm_dit_param_count(h) == 99
    assert abs(n.lib().cm_dit_flops_per_sample(h) / 1e9 - 0.667) < 0.01
    n.check(n.lib().cm_dit_destroy(h))
    bad = n.DitConfig(in_channels=3, out_channels=3, rows=12, cols=36, past_len=5, future_len=3, t_patch=3, patch=4,
                      hidden=256, depth=6, heads=4, mlp_hidden=1024, time_multiple=4, table_steps=1000, t_max_slots=8)
    assert n.lib().cm_dit_create(ctypes.byref(bad), ctypes.byref(h)) != 0
    assert b"divisible by t_patch" in n.lib().cm_last_error()
