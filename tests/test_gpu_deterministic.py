"""Reproducible training under torch.use_deterministic_algorithms(True): the fixed-order reductions of cm_unet_backward.

Op level: every reduction the deterministic mode rewrites (wgrad_umma split-K, wgrad_plane's persistent CTAs,
cast_colsum's channel sums, the first / final conv weight and bias gradients) runs twice through its `_det` entry point
at shapes that reach each route; the two results are bitwise equal and each meets the float64 bound the op tests of
test_gpu_ops.py / test_gpu_backward_ops.py set for the same kernel.  Model level: two training steps on identical inputs
(injected Dropout3d masks) give bitwise equal flat gradient buffers, within the oracle gates of test_gpu_train.py.
Driver level: two fresh DDPM_models (and a second process) training one epoch with the flag on end in the same bits.
"""
import os
import subprocess
import sys

import pytest
import torch
import torch.nn.functional as F

from oracle import ddpm_oracle as do
from oracle import unet_oracle as uo
from tests._util import rel_l2

pytestmark = pytest.mark.gpu

NAN = float("nan")
GRAD_TOL = 1e-3
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def nat():
    import crowdmod_ddpm_4d_b200._native as n
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    n.lib()
    assert n.lib().cm_device_error() == 0
    yield n
    assert n.lib().cm_device_error() == 0, "a kernel left the device error flag set"


def gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def twice(fn):
    """fn() -> tuple of output tensors; runs it twice and checks the two runs agree bit for bit."""
    a = [t.clone() for t in fn()]
    b = fn()
    torch.cuda.synchronize()
    for x, y in zip(a, b):
        assert torch.equal(x, y), "deterministic reduction differs between two identical calls"
    return a


# =====================================================================================================================
# weight gradients: wgrad_umma (split-K over gridDim.y) and wgrad_plane (persistent CTAs)
# =====================================================================================================================
def _out_grid(mode, D, H, W):
    if mode == 1:
        return (D - 1) // 2 + 1, (H - 1) // 2 + 1, (W - 1) // 2 + 1
    if mode == 2:
        return 2 * D, 2 * H, 2 * W
    return D, H, W


def _wgrad_ref(mode, act, extra, dout, cout):
    x = act.double().permute(0, 4, 1, 2, 3)
    k = 1 if mode == 3 else 3
    w = torch.zeros(cout, act.shape[-1], k, k, k, dtype=torch.float64, device="cuda", requires_grad=True)
    if mode == 2:
        x = F.interpolate(x, scale_factor=2, mode="nearest")
    y = F.conv3d(x, w, None, stride=2 if mode == 1 else 1, padding=0 if mode == 3 else 1)
    wx = None
    if extra is not None:
        wx = torch.zeros(cout, extra.shape[-1], dtype=torch.float64, device="cuda", requires_grad=True)
        y = y + F.conv3d(extra.double().permute(0, 4, 1, 2, 3), wx[:, :, None, None, None])
    y.backward(dout.double().permute(0, 4, 1, 2, 3))
    return w.grad, (wx.grad if wx is not None else None)


# (mode, B, D, H, W, cin, cout, cin_extra, impl): impl 0 = wgrad_umma, 2 = the plane scheme
WGRAD_CASES = [
    (0, 2, 12, 36, 8, 32, 32, 0, 0),      # wgrad_umma, 7 M tiles x 42 pixel splits
    (0, 2, 6, 18, 4, 64, 64, 32, 0),      # wgrad_umma with the fused match_input rows, 7 splits
    (0, 2, 3, 9, 2, 256, 128, 0, 0),      # BN = 128, BKC = 64
    (2, 1, 6, 18, 4, 64, 64, 0, 0),       # UpSample: 8 phases x 4 splits
    (2, 2, 3, 9, 2, 128, 128, 0, 0),
    (1, 2, 12, 36, 8, 32, 32, 0, 0),      # DownSample
    (3, 3, 3, 9, 2, 128, 384, 0, 0),      # 1x1x1 (attention projections)
    (0, 2, 8, 12, 36, 32, 32, 0, 2),      # plane, ATC 12 x 36 grid
    (0, 1, 8, 28, 24, 32, 32, 0, 2),      # plane, HERMES 28 x 24 grid
    (0, 2, 8, 12, 36, 96, 32, 0, 2),      # three plane chunks
    (0, 2, 8, 12, 36, 32, 32, 96, 2),     # plane + the 1x1x1 source through wgrad_umma
    (0, 40, 8, 12, 36, 64, 32, 0, 2),     # more units than the 148 deterministic CTAs
]


@pytest.mark.parametrize("case", WGRAD_CASES, ids=lambda c: "m%d_B%d_%dx%dx%d_ci%d_co%d_x%d_impl%d" % c)
def test_wgrad_deterministic(nat, case):
    mode, B, D, H, W, cin, cout, cx, impl = case
    g = gen(3)
    act = torch.randn(B, D, H, W, cin, device="cuda", generator=g).half()
    od, oh, ow = _out_grid(mode, D, H, W)
    extra = torch.randn(B, od, oh, ow, cx, device="cuda", generator=g).half() if cx else None
    dout = torch.randn(B, od, oh, ow, cout, device="cuda", generator=g).half()
    k = 1 if mode == 3 else 3

    def run():
        dw = torch.full((cout, cin, k, k, k), NAN, device="cuda")
        dwx = torch.full((cout, cx), NAN, device="cuda") if cx else None
        nat.check(nat.lib().cm_op_conv3d_wgrad_det(mode, nat.ptr(act), B, D, H, W, cin, nat.ptr(extra), cx,
                                                   nat.ptr(dout), cout, nat.ptr(dw), nat.ptr(dwx), impl,
                                                   nat.current_stream()))
        return (dw, dwx) if cx else (dw,)

    out = twice(run)
    rw, rwx = _wgrad_ref(mode, act, extra, dout, cout)
    e = rel_l2(out[0], rw)
    print(f"wgrad det rel-L2 {e:.2e}")
    assert e <= 3e-5, f"wgrad rel-L2 {e:.3e}"
    if cx:
        assert rel_l2(out[1], rwx) <= 3e-5


# =====================================================================================================================
# per-sample channel sums (bias and time-embedding gradients)
# =====================================================================================================================
@pytest.mark.parametrize("case", [(2, 3456, 32, 2), (64, 54, 128, 2), (600, 54, 96, 2), (1, 3456, 256, 2),
                                  (5, 777, 64, 1)], ids=lambda c: "B%d_p%d_C%d_dup%d" % c)
def test_cast_colsum_deterministic(nat, case):
    B, pixels, C_, dup = case
    g = gen(3)
    src = torch.randn(B, pixels, C_, device="cuda", generator=g) * 40.0
    ld = C_ + 8
    colsum0 = torch.randn(B, ld, device="cuda", generator=g)

    def run():
        dst = torch.full((B, pixels, dup * C_), NAN, device="cuda").half()
        acc = torch.full_like(src, NAN)
        colsum = colsum0.clone()
        nat.check(nat.lib().cm_op_cast_colsum_det(nat.ptr(src), nat.ptr(dst), dup, nat.ptr(acc), 1, nat.ptr(colsum),
                                                  ld, B, pixels, C_, nat.current_stream()))
        return dst, acc, colsum

    dst, acc, colsum = twice(run)
    assert torch.equal(dst[..., :C_], src.half()) and torch.equal(acc, src)
    ref = colsum0.double()[:, :C_] + src.double().sum(dim=1)
    scale = colsum0.double()[:, :C_].abs() + src.double().abs().sum(dim=1)
    assert ((colsum[:, :C_].double() - ref).abs() / scale).max().item() <= 1e-6
    assert torch.equal(colsum[:, C_:], colsum0[:, C_:]), "colsum wrote past C"


# =====================================================================================================================
# first / final conv weight and bias gradients
# =====================================================================================================================
@pytest.mark.parametrize("case", [(2, 12, 36, 5, 3, 3, 32), (2, 12, 36, 5, 3, 3, 64), (1, 28, 24, 8, 8, 4, 64),
                                  (3, 2, 3, 6, 5, 3, 32)], ids=lambda c: "B%d_%dx%d_P%d_F%d_ci%d_co%d" % c)
def test_first_conv_wgrad_deterministic(nat, case):
    """The SIMT first-conv kernel (the model's route at base 64; bases 32 and 128 take the packed operand through the
    wgrad kernels above, and their bias through cast_colsum)."""
    B, H, W, P, F_, cin, cout = case
    g = gen(8)
    L = P + F_
    x = torch.randn(B, cin, H, W, F_, device="cuda", generator=g)
    past = torch.randn(B, cin, H, W, P, device="cuda", generator=g)
    dout = torch.randn(B, L, H, W, cout, device="cuda", generator=g)

    def run():
        dw = torch.full((cout, cin, 3, 3, 3), NAN, device="cuda")
        db = torch.full((cout,), NAN, device="cuda")
        nat.check(nat.lib().cm_op_first_conv_wgrad_det(nat.ptr(x), nat.ptr(past), nat.ptr(dout), nat.ptr(dw),
                                                       nat.ptr(db), B, H, W, P, F_, cin, cout, nat.current_stream()))
        return dw, db

    dw, db = twice(run)
    inp = torch.cat([past, x], dim=-1).double()
    w64 = torch.zeros(cout, cin, 3, 3, 3, dtype=torch.float64, device="cuda", requires_grad=True)
    b64 = torch.zeros(cout, dtype=torch.float64, device="cuda", requires_grad=True)
    F.conv3d(inp, w64, b64, padding=1).backward(dout.double().permute(0, 4, 2, 3, 1))
    assert rel_l2(dw, w64.grad) <= 1e-5 and rel_l2(db, b64.grad) <= 1e-5


# (B, H, W, P, F, cin, cout, packed): SIMT weight gradient at cin 32 / 64 (the model's route at base 64), the packed
# operand through the plane chunks at cin 32, 96 and 128 (the model's route at those bases)
FINAL_CASES = [
    (2, 12, 36, 5, 3, 32, 3, 0), (1, 28, 24, 8, 8, 64, 4, 0), (2, 12, 36, 5, 3, 64, 3, 0),
    (2, 12, 36, 5, 3, 32, 3, 1), (1, 28, 24, 8, 8, 128, 4, 1), (2, 12, 36, 5, 3, 96, 3, 1),
]


@pytest.mark.parametrize("case", FINAL_CASES, ids=lambda c: "B%d_%dx%d_P%d_F%d_ci%d_co%d_packed%d" % c)
def test_final_conv_backward_deterministic(nat, case):
    B, H, W, P, F_, cin, cout, packed = case
    scale = 2.0 ** 11
    g = gen(7)
    L = P + F_
    a32 = torch.randn(B, L, H, W, cin, device="cuda", generator=g)
    hi = a32.half()
    lo = (a32 - hi.float()).half()
    act16 = torch.cat([hi, lo], dim=-1).contiguous()
    w = torch.randn(cout, cin, 3, 3, 3, device="cuda", generator=g) / (27 * cin) ** 0.5
    deps = torch.randn(B, cout, H, W, F_, device="cuda", generator=g) * 1e-3

    def run():
        dact = torch.full((B, L, H, W, cin), NAN, device="cuda")
        dw = torch.full_like(w, NAN)
        db = torch.full((cout,), NAN, device="cuda")
        d16 = torch.full((B, L, H, W, 32), NAN, device="cuda").half() if packed else None
        nat.check(nat.lib().cm_op_final_conv_backward_det(
            nat.ptr(deps), scale, nat.ptr(act16), 2 * cin, cin, nat.ptr(w), nat.ptr(dact), nat.ptr(dw), nat.ptr(db),
            B, H, W, L, P, cin, cout, nat.ptr(d16), nat.current_stream()))
        return dact, dw, db

    dact, dw, db = twice(run)
    x = (hi.double() + lo.double()).permute(0, 4, 2, 3, 1).contiguous().requires_grad_(True)
    w64 = w.double().requires_grad_(True)
    b64 = torch.zeros(cout, dtype=torch.float64, device="cuda", requires_grad=True)
    F.conv3d(x, w64, b64, padding=1)[..., P:].backward(deps.double())
    e_act = rel_l2(dact.permute(0, 4, 2, 3, 1) / scale, x.grad)
    e_w, e_b = rel_l2(dw / scale, w64.grad), rel_l2(db / scale, b64.grad)
    print(f"final det dact {e_act:.2e} dw {e_w:.2e} db {e_b:.2e}")
    assert e_act <= 1e-5 and e_b <= 1e-5
    assert e_w <= (6e-4 if packed else 1e-5)      # test_gpu_backward_ops.PACKED_DW_BOUND for the packed route


# =====================================================================================================================
# model level: two training steps on identical inputs, flag on
# =====================================================================================================================
MULT3 = [1, 2, 4]
MODELS = {
    # ATC base 32: plane weight gradients at level 0 (first conv included), res32 forward convs
    "atc_base32": dict(rows=12, cols=36, P=5, F=3, base=32, attn=[False, False, True, False]),
    "hermes_cr120_base32": dict(rows=28, cols=24, P=5, F=3, base=32, attn=[False, False, True, False]),
    # ATC_medium-style base 64: the SIMT first / final conv weight gradients
    "atc_medium_base64": dict(rows=12, cols=36, P=8, F=8, base=64, attn=[False, False, True]),
    # the first conv's weight gradient through wgrad_umma (cout = base), the final conv's through plane chunks
    "atc_base96": dict(rows=12, cols=36, P=5, F=3, base=96, attn=[False, False, True, False]),
    "atc_base128": dict(rows=12, cols=36, P=5, F=3, base=128, attn=[False, False, True, False]),
    # 8 + 8 frames: attention at S = 168 (streaming attention backward)
    "hermes_8p8_base32": dict(rows=28, cols=24, P=8, F=8, base=32, attn=[False, False, True, False]),
}
BLOCKS = [("encoder_blocks.0", 1), ("encoder_blocks.2", 2), ("encoder_blocks.4", 4), ("bottleneck_blocks.0", 4),
          ("bottleneck_blocks.1", 4), ("decoder_blocks.0", 4), ("decoder_blocks.1", 4), ("decoder_blocks.3", 2),
          ("decoder_blocks.4", 2), ("decoder_blocks.6", 1), ("decoder_blocks.7", 1)]


@pytest.mark.parametrize("name", list(MODELS))
def test_train_step_gradients_bitwise_repeatable(nat, name):
    from crowdmod_ddpm_4d_b200.models.backbones.unet import UNet
    c = MODELS[name]
    ST = dict(num_res_blocks=1, num_levels=3)
    torch.manual_seed(7)
    net = UNet(input_channels=3, output_channels=3, num_res_blocks=1, base_channels=c["base"],
               base_channels_multiples=MULT3, apply_attention=c["attn"], dropout_rate=0.1, time_multiple=4,
               condition="Past")
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    B = 2
    g = torch.Generator().manual_seed(23)
    past = do.synthetic_macroprops(B, 3, c["rows"], c["cols"], c["P"], 21)
    fut = do.synthetic_macroprops(B, 3, c["rows"], c["cols"], c["F"], 22)
    t = torch.tensor([3, 871])
    noise = torch.randn(fut.shape, generator=g)
    masks = {k: (torch.rand(B, m * c["base"], generator=g) >= 0.1).float() / 0.9 for k, m in BLOCKS}
    s = do.schedule(1000, 0.5)

    net = net.cuda().train()
    net._injected_dropout = [m.cuda() for m in masks.values()]
    x_t = do.q_sample(s, fut, t, noise).cuda()
    flats = []
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        for _ in range(2):
            net.zero_grad(set_to_none=True)
            loss = F.mse_loss(net(x_t, t.cuda(), past.cuda()), noise.cuda())
            loss.backward()
            torch.cuda.synchronize()
            flats.append(net._last_flat_grad.clone())
    finally:
        torch.use_deterministic_algorithms(prev)
    assert torch.equal(flats[0], flats[1]), f"{name}: flat gradients differ between two identical steps"

    sdg = {k: v.detach().clone().requires_grad_(v.dtype.is_floating_point and "time_blocks.0" not in k)
           for k, v in sd.items()}
    loss_ref = do.train_loss(lambda a, b, p: uo.unet_forward(sdg, a, b, p, drop_masks=masks, **ST), s, fut, past, t,
                             noise)
    loss_ref.backward()
    assert abs(loss.item() - loss_ref.item()) <= 1e-3 * abs(loss_ref.item())
    num = den = 0.0
    per = {}
    for k, p in net.named_parameters():
        if p.grad is None:
            continue
        go = sdg[k].grad.double()
        per[k] = ((p.grad.cpu().double() - go).pow(2).sum().item(), go.pow(2).sum().item())
        num += per[k][0]
        den += per[k][1]
    for k, (d, r) in per.items():
        if r ** 0.5 < 1e-9 * den ** 0.5:        # numerically zero reference gradient: absolute bound
            assert dict(net.named_parameters())[k].grad.double().norm().item() < 1e-6 * den ** 0.5, k
    worst, worst_k = max(((d / r) ** 0.5, k) for k, (d, r) in per.items() if r ** 0.5 >= 1e-9 * den ** 0.5)
    eg = (num / den) ** 0.5
    print(f"{name}: global grad rel-L2 {eg:.3e}, worst tensor {worst_k} {worst:.3e}")
    assert eg <= GRAD_TOL
    assert worst <= GRAD_TOL, f"{worst_k}: gradient rel-L2 {worst:.3e}"


# =====================================================================================================================
# driver level: DDPM_model._train_one_epoch with Adam, two fresh models and a second process
# =====================================================================================================================
def test_train_epoch_reproducible_across_models_and_processes(nat):
    from tests import _det_driver as dd
    m1, l1, h1 = dd.run(True)
    m2, l2, h2 = dd.run(True)
    sd1, sd2 = m1.denoiser.state_dict(), m2.denoiser.state_dict()
    assert sd1.keys() == sd2.keys()
    for k in sd1:
        assert torch.equal(sd1[k], sd2[k]), k
    assert l1 == l2 and h1 == h2
    env = dict(os.environ, CUBLAS_WORKSPACE_CONFIG=":4096:8")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "_det_driver.py")], cwd=ROOT, env=env,
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = [x for x in out.stdout.splitlines() if x.startswith("SHA ")][-1].split()
    assert line[1] == h1, "another process trained to different parameters"
    assert float.fromhex(line[3]) == l1[0]


def test_train_epochs_flag_off_still_learn(nat):
    from tests import _det_driver as dd
    _, losses, _ = dd.run(False, epochs=3)
    print(f"flag off: epoch losses {losses}")
    assert all(torch.isfinite(torch.tensor(losses)))
    assert losses[-1] < losses[0], losses
