"""GPU parity of the native training forward/backward (SURVEY.md §8 a7): the product UNet under
autograd (cm_unet_train_forward / cm_unet_backward through the C ABI) against (a) the CPU oracle's
autograd on identical weights, t, eps — per-parameter-tensor gradients — and (b) the golden
loss / gradient norms / random projections generated from the unmodified reference.

Tolerances (BASELINE.json north_star: "training loss and gradients within 1e-3"; SURVEY.md §8d): loss
relative error <= 1e-3; global gradient-vector rel-L2 <= GRAD_TOL = 1e-3; EVERY parameter tensor rel-L2 <=
TENSOR_TOL = 1e-3.  No exceptions are needed: the training forward multiplies hi|lo fp16 activation pairs
(cm_unet_config.train_act_terms = 2) and the data-gradient convs hi|lo dOut pairs (dgrad_terms = 2), which
took the worst tensor from 2.6e-3 (round 1, single fp16 operands: the error was the forward's activation
rounding propagating into every deep-layer gradient -- shown by the CPU emulation in
profiles/r2_train_grad_parity.txt) to 5.8e-4 / 3.4e-4 / 3.2e-4 on the three cases below (measured on B200).
"""
import pytest
import torch
import torch.nn.functional as F

from oracle import ddpm_oracle as do
from oracle import unet_oracle as uo
from tests._util import build_unet, load_golden, rel_l2, structure

pytestmark = pytest.mark.gpu

LOSS_TOL = 1e-3
GRAD_TOL = 1e-3
TENSOR_TOL = 1e-3
# name (regex) -> (bound, why): empty -- every tensor meets TENSOR_TOL (see the module docstring)
TENSOR_EXCEPTIONS = {}


@pytest.fixture(scope="module", autouse=True)
def _no_device_errors():
    import crowdmod_ddpm_4d_b200._native as n
    yield
    assert n.lib().cm_device_error() == 0, "a kernel reported a protocol error"


def _oracle_grads(meta, a, t, eps, dropout=None):
    net = build_unet(meta)
    sd = {k: v.detach().clone().requires_grad_(v.dtype.is_floating_point and "time_blocks.0" not in k)
          for k, v in net.state_dict().items()}
    s = do.schedule(meta["T"], meta["scale"])
    den = lambda x, tt, p: uo.unet_forward(sd, x, tt, p, drop_masks=dropout, **structure(meta))
    loss = do.train_loss(den, s, a["future"], a["past"], t, eps)
    loss.backward()
    return loss.item(), {k: v.grad for k, v in sd.items() if v.grad is not None}, s


def _native_grads(meta, a, t, eps, s, dropout=None):
    net = build_unet(meta).cuda().train()
    if dropout is not None:
        net._injected_dropout = list(dropout.values())     # plan order == insertion order below
    x_t = do.q_sample(s, a["future"], t, eps).cuda()
    pred = net(x_t, t.cuda(), a["past"].cuda())
    loss = F.mse_loss(pred, eps.cuda())
    loss.backward()
    torch.cuda.synchronize()
    return loss.item(), {k: p.grad.cpu() for k, p in net.named_parameters() if p.grad is not None}, net


def _compare(lo, go, ln, gn):
    assert abs(ln - lo) <= LOSS_TOL * abs(lo), f"loss {ln} vs oracle {lo}"
    assert set(go) == set(gn), f"gradient key mismatch: {set(go) ^ set(gn)}"
    num = sum((gn[k].double() - go[k].double()).pow(2).sum().item() for k in go)
    den = sum(go[k].double().pow(2).sum().item() for k in go)
    worst = sorted(((rel_l2(gn[k], go[k]), k) for k in go), reverse=True)
    print("global grad rel-L2 = %.3e; worst tensors: %s" % ((num / den) ** 0.5,
          ", ".join("%s %.2e" % (k, e) for e, k in worst[:6])))
    assert (num / den) ** 0.5 <= GRAD_TOL
    import re
    for e, k in worst:
        # tensors whose gradient is numerically zero in the reference (e.g. k/q biases of the
        # attention softmax shift) are compared in absolute terms
        if go[k].double().norm().item() < 1e-9 * den ** 0.5:
            assert gn[k].double().norm().item() < 1e-6 * den ** 0.5, k
            continue
        bound = TENSOR_TOL
        for pat, (b, _why) in TENSOR_EXCEPTIONS.items():
            if re.fullmatch(pat, k):
                bound = b
        assert e <= bound, f"{k}: rel-L2 {e:.3e} > {bound:.1e}"


@pytest.mark.parametrize("name", ["train_small", "train_atc_b2"])
def test_train_step_vs_oracle_and_reference_golden(name):
    meta, a = load_golden(name)
    torch.manual_seed(meta["rng_seed"])
    t = torch.randint(0, meta["T"], (meta["B"],))
    eps = torch.randn_like(a["future"])
    lo, go, s = _oracle_grads(meta, a, t, eps)
    ln, gn, _ = _native_grads(meta, a, t, eps, s)
    _compare(lo, go, ln, gn)
    # golden: loss + per-tensor norms / random projections from the unmodified reference
    assert abs(ln - float(a["loss"])) <= LOSS_TOL * abs(float(a["loss"]))
    g = torch.Generator().manual_seed(meta["proj_seed"])
    for i, k in enumerate(meta["names"]):
        r = torch.randn(gn[k].shape, generator=g)
        n_ref, p_ref = float(a["grad_norms"][i]), float(a["grad_proj"][i])
        if n_ref < 1e-12:
            continue
        assert abs(gn[k].double().norm().item() - n_ref) <= TENSOR_TOL * n_ref, k
        assert abs((gn[k].double() * r.double()).sum().item() - p_ref) <= TENSOR_TOL * n_ref * r.norm().item(), k


def test_train_step_fresh_batch_b5_with_injected_dropout():
    """Odd batch (ragged tiles), mixed timesteps and Dropout3d masks injected into both sides."""
    meta, _ = load_golden("train_atc_b2")
    B = 5
    a = {"future": do.synthetic_macroprops(B, 3, 12, 36, 3, 77), "past": do.synthetic_macroprops(B, 3, 12, 36, 5, 78)}
    g = torch.Generator().manual_seed(9)
    t = torch.tensor([0, 3, 500, 998, 999])
    eps = torch.randn(a["future"].shape, generator=g)
    # one [B, C] keep-mask/(1-p) per ResnetBlock, plan order (ATC: couts below), p = 0.25
    blocks = [("encoder_blocks.0", 32), ("encoder_blocks.2", 64), ("encoder_blocks.4", 128),
              ("bottleneck_blocks.0", 128), ("bottleneck_blocks.1", 128), ("decoder_blocks.0", 128),
              ("decoder_blocks.1", 128), ("decoder_blocks.3", 64), ("decoder_blocks.4", 64),
              ("decoder_blocks.6", 32), ("decoder_blocks.7", 32)]
    masks = {k: (torch.rand(B, c, generator=g) >= 0.25).float() / 0.75 for k, c in blocks}
    lo, go, s = _oracle_grads(meta, a, t, eps, dropout=masks)
    ln, gn, _ = _native_grads(meta, a, t, eps, s, dropout=masks)
    _compare(lo, go, ln, gn)


def test_optimizer_step_repacks_weights_and_loss_decreases():
    """Three Adam steps through the reference-facing driver objects: the native caches must follow
    the in-place parameter updates (loss on a fixed batch goes down, parameters change)."""
    meta, a = load_golden("train_small")
    net = build_unet(meta).cuda().train()
    opt = torch.optim.Adam(net.parameters(), lr=1e-3)
    s = do.schedule(meta["T"], meta["scale"])
    torch.manual_seed(1)
    t = torch.randint(0, meta["T"], (meta["B"],))
    eps = torch.randn_like(a["future"])
    x_t = do.q_sample(s, a["future"], t, eps).cuda()
    losses = []
    for _ in range(4):
        loss = F.mse_loss(net(x_t, t.cuda(), a["past"].cuda()), eps.cuda())
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        losses.append(loss.item())
    assert all(torch.isfinite(torch.tensor(losses)))
    assert losses[-1] < losses[0], losses


def test_eval_forward_or_sampling_between_forward_and_backward_raises():
    """The activation arena is shared: a no_grad forward or a sampling call on the same geometry between a
    training forward and its backward would silently corrupt the gradients -> it must raise instead."""
    from crowdmod_ddpm_4d_b200.models.diffusion.ddpm import DDPM, ddpm_coefficients
    meta, a = load_golden("train_small")
    net = build_unet(meta).cuda().train()
    x = torch.randn(meta["B"], 3, meta["rows"], meta["cols"], meta["F"], device="cuda")
    t = torch.zeros(meta["B"], dtype=torch.long, device="cuda")
    p = a["past"].cuda()
    y = net(x, t, p)
    with torch.no_grad():
        net(x, t, p)
    with pytest.raises(RuntimeError):
        y.sum().backward()
    y = net(x, t, p)
    ts, coef = ddpm_coefficients(DDPM(timesteps=3, scale=0.5))
    net.sample_chain(p.contiguous(), x.clone(), ts, coef, mode=0, seed=1)
    with pytest.raises(RuntimeError):
        y.sum().backward()
    y = net(x, t, p)
    y.sum().backward()                                   # undisturbed pair still works
    torch.cuda.synchronize()


def test_in_place_parameter_surgery_needs_explicit_invalidate():
    """Writes through p.data do not bump _version: invalidate_native_cache() re-derives the packed weights."""
    meta, a = load_golden("unet_small_b3")
    net = build_unet(meta).cuda().eval()
    args = (a["future"].cuda(), a["t"].cuda(), a["past"].cuda())
    with torch.no_grad():
        e0 = net(*args).clone()
        net.first.weight.data.mul_(0.5)
        net.invalidate_native_cache()
        e1 = net(*args).clone()
        net.first.weight.mul_(2.0)                       # a tracked in-place update: picked up by itself
        e2 = net(*args).clone()
    assert not torch.equal(e0, e1)
    assert torch.allclose(e0, e2, rtol=1e-5, atol=1e-6)


def test_second_forward_invalidates_first_backward():
    meta, a = load_golden("train_small")
    net = build_unet(meta).cuda().train()
    x = torch.randn(meta["B"], 3, meta["rows"], meta["cols"], meta["F"], device="cuda")
    t = torch.zeros(meta["B"], dtype=torch.long, device="cuda")
    p = a["past"].cuda()
    y1 = net(x, t, p)
    y2 = net(x, t, p)
    y2.sum().backward()
    with pytest.raises(RuntimeError):
        y1.sum().backward()
