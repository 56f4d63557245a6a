"""CPU: the oracle restatement against the LIVE reference imported from a checkout of the original project
(oracle/ref_shim.py: oracle/_ref/ or $CROWDMOD_REFERENCE; skipped where there is none).  The stored vectors of
tests/golden/ (tests/test_oracle_golden.py) check the oracle against the reference's outputs on other inputs only:
UNet forward at the ATC / HERMES / small geometries, seeded init at base 32, the schedule, whole chains (rel-L2,
not one bit-exact DDPM.step), metrics, DiT at patch 4.  The dataset windows and batch order, the geometries below,
the base-64 init and the DiT patch-2 case are checked here only."""
import pytest
import torch

from oracle import ddpm_oracle as do
from oracle import ref_shim
from oracle import unet_oracle as uo

pytestmark = pytest.mark.skipif(not ref_shim.available(), reason=ref_shim.MISSING)


@pytest.fixture(scope="module")
def ns():
    return ref_shim.load()


@pytest.mark.parametrize("kw,geom", [
    (dict(input_channels=3, output_channels=3, num_res_blocks=1, base_channels=32,
          base_channels_multiples=[1, 2, 4], apply_attention=[False, False, True, False],
          dropout_rate=0.1, time_multiple=4, condition="Past"), (8, 12, 5, 3)),          # ETH-UCY shape
    (dict(input_channels=3, output_channels=3, num_res_blocks=2, base_channels=32,
          base_channels_multiples=[1, 2], apply_attention=[True, False],
          dropout_rate=0.1, time_multiple=2, condition="Past"), (4, 6, 3, 1)),
])
def test_unet_forward_vs_live_reference(ns, kw, geom):
    rows, cols, P, F_ = geom
    torch.manual_seed(3)
    ref = ns.UNet(**kw).eval()
    x = torch.randn(2, 3, rows, cols, F_)
    past = do.synthetic_macroprops(2, 3, rows, cols, P, 77)
    t = torch.tensor([5, 900])
    with torch.no_grad():
        a = ref(x, t, past)
        b = uo.unet_forward(ref.state_dict(), x, t, past, num_res_blocks=kw["num_res_blocks"],
                            num_levels=len(kw["base_channels_multiples"]))
    assert uo.rel_l2(b, a) <= 5e-6


def test_product_module_reproduces_reference_init(ns):
    from crowdmod_ddpm_4d_b200.models.backbones.unet import UNet
    kw = dict(input_channels=3, output_channels=3, num_res_blocks=1, base_channels=64,
              base_channels_multiples=[1, 2, 4], apply_attention=[False, False, True, False],
              dropout_rate=0.1, time_multiple=4, condition="Past")
    torch.manual_seed(42)
    a = ns.UNet(**kw).state_dict()
    torch.manual_seed(42)
    b = UNet(**kw).state_dict()
    assert list(a.keys()) == list(b.keys())
    assert all(torch.equal(a[k], b[k]) for k in a)


def test_schedule_and_step_vs_live_reference(ns):
    ref = ns.DDPM(timesteps=1000, scale=0.5)
    s = do.schedule(1000, 0.5)
    for k, v in s.items():
        assert torch.equal(getattr(ref, k), v), k
    x = torch.randn(2, 3, 4, 4, 2)
    e = torch.randn_like(x)
    torch.manual_seed(9)
    out, _, _ = ref.step(e, x, 321)
    torch.manual_seed(9)
    z = torch.randn_like(x)
    assert torch.equal(out, do.ddpm_step(s, e, x, 321, z))


def test_metrics_oracle_pinned_to_live_reference():
    """SURVEY.md section 8 f3: the numpy restatement equals the unmodified MetricsGenerator on a fresh seeded pair."""
    import numpy as np
    from oracle import metrics_oracle as mo
    ns = ref_shim.load()
    if ns.MetricsGenerator is None:
        pytest.skip("reference metrics module not importable: " + getattr(ns, "metrics_error", ""))
    pred, gt = mo.synthetic_pair(6, 8, 12, 3, 99)
    gen = ns.MetricsGenerator([torch.from_numpy(p) for p in pred], [torch.from_numpy(g) for g in gt],
                              ns.EasyDict({"MPROPS_COUNT": 3}), None)
    with np.errstate(all="ignore"):
        gen.compute_psnr_metric(3, 1e-6)
        gen.compute_psnr_metric(3, 1e-6, masked_flag=True)
        gen.compute_re_density_metric(3, 1e-6)
        gen.compute_tv_metric()
        a = mo.compute_psnr_metric(pred, gt, 3, 1e-6)
        b = mo.compute_psnr_metric(pred, gt, 3, 1e-6, masked=True)
    for k, v in zip(["PSNR", "MAX_PSNR", "PSNR_OVER_TIME", "MAX_PSNR_OVER_TIME"], a):
        np.testing.assert_allclose(v, gen.data_dict[k], rtol=0, atol=1e-12)
    for k, v in zip(["MASK_PSNR", "MAX_MASK_PSNR", "MASK_PSNR_OVER_TIME", "MAX_MASK_PSNR_OVER_TIME"], b):
        np.testing.assert_allclose(v, gen.data_dict[k], rtol=0, atol=1e-12, equal_nan=True)
    re, mre = mo.compute_re_density(pred, gt, 3, 1e-6)
    np.testing.assert_array_equal(re, gen.data_dict["RE_DENSITY"])
    np.testing.assert_array_equal(mre, gen.data_dict["MIN_RE_DENSITY"])
    np.testing.assert_array_equal(mo.compute_tv_metric(pred, gt), gen.data_dict["TV_OVER_TIME"])


def test_dataset_oracle_pinned_to_live_reference():
    """SURVEY.md section 8 f4: window index table, windows and DataLoader batch order equal the unmodified
    MacropropsDataset + torch DataLoader (utils/dataset.py:22-53,169-190), shuffled and not."""
    import numpy as np
    from torch.utils.data import DataLoader
    from oracle import dataset_oracle as dso
    ns = ref_shim.load()
    if ns.MacropropsDataset is None:
        pytest.skip("reference dataset module not importable: " + getattr(ns, "dataset_error", ""))
    rng = np.random.default_rng(5)
    seq = rng.normal(size=(3, 3, 4, 5, 23)).astype(np.float32)
    cfg = ns.EasyDict({"DATASET": {"PAST_LEN": 5, "FUTURE_LEN": 3}})
    ds = ns.MacropropsDataset(seq, cfg, 3, stride=4)
    assert [tuple(i) for i in ds.indices] == dso.window_indices(3, 23, 5, 3, 4)
    for shuffle, drop_last in ((False, False), (True, True), (True, False)):
        torch.manual_seed(1234)
        ref_batches = list(DataLoader(ds, batch_size=4, shuffle=shuffle, drop_last=drop_last))
        torch.manual_seed(1234)
        ours = list(dso.batches(seq, 5, 3, 4, 4, shuffle=shuffle, drop_last=drop_last))
        assert len(ours) == len(ref_batches)
        for (p0, f0), (p1, f1) in zip(ref_batches, ours):
            assert torch.equal(p0, p1) and torch.equal(f0, f1)


@pytest.mark.parametrize("kw,geom", [
    (dict(input_channels=3, output_channels=3, grid_rows=12, grid_cols=36, past_len=5, future_len=3, t_patch_size=4,
          patch_size=4, hidden_size=256, depth=6, num_heads=4, mlp_ratio=4.0, dropout_rate=0.1, time_multiple=4), 2),
    (dict(input_channels=3, output_channels=3, grid_rows=8, grid_cols=12, past_len=5, future_len=3, t_patch_size=2,
          patch_size=2, hidden_size=128, depth=2, num_heads=4, mlp_ratio=4.0, dropout_rate=0.1, time_multiple=4), 3),
])
def test_dit_oracle_and_mirror_pinned_to_live_reference(kw, geom):
    """SURVEY.md section 8 f2: oracle/dit_oracle.py == the unmodified DiT4D_V4.forward (eval), and the product's mirror
    module reproduces the reference's state_dict (keys, shapes, seeded values) bit for bit."""
    from oracle import dit_oracle as dto
    from crowdmod_ddpm_4d_b200.models.backbones.DiT4D_V4 import DiT4D_V4
    ns = ref_shim.load()
    if ns.DiT4D_V4 is None:
        pytest.skip("reference DiT4D_V4 not importable: " + getattr(ns, "dit_error", ""))
    torch.manual_seed(5)
    ref = ns.DiT4D_V4(**kw).eval()
    torch.manual_seed(5)
    mine = DiT4D_V4(**kw)
    rs, ms = ref.state_dict(), mine.state_dict()
    assert list(rs) == list(ms)
    for k in rs:
        assert torch.equal(rs[k], ms[k]), k
    sd = dto.randomize_zero_init({k: v.detach().clone() for k, v in rs.items()}, 1)
    ref.load_state_dict(sd)
    B = geom
    g = torch.Generator().manual_seed(0)
    fut = torch.randn(B, 3, kw["grid_rows"], kw["grid_cols"], kw["future_len"], generator=g)
    past = torch.randn(B, 3, kw["grid_rows"], kw["grid_cols"], kw["past_len"], generator=g)
    t = torch.randint(0, 1000, (B,), generator=g)
    with torch.no_grad():
        want = ref(fut, t, past)
        got = dto.dit_forward(sd, fut, t, past, patch=kw["patch_size"], t_patch=kw["t_patch_size"], heads=kw["num_heads"],
                              depth=kw["depth"])
    assert ((want - got).norm() / want.norm()).item() <= 2e-6
