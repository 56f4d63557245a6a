"""Op-level parity of the fp32 kernels of the training backward (csrc/backward.cu) against float64 autograd of the
PyTorch ops they replace, plus three model-level properties of cm_unet_backward.

The model tests (test_gpu_train.py, test_gpu_wide.py, ...) bound every parameter gradient at rel-L2 1e-3, a bound set by
the fp16 operands of the convs.  The kernels here are plain fp32 arithmetic and sit within ~1e-6 of float64, so they are
checked at 1e-5 (and per (sample, group) where one bad group could hide in a global norm), at the launch geometries where
their chunking changes: B > 592 (one chunk per sample), pixel counts below 4 x chunks, C/4 > 256 (one thread per
channel quad), ragged pixel chunks.  Kernel inputs are exactly the reference's inputs (the fp16-rounded operands where a
kernel reads fp16); outputs are pre-filled with NaN so that an unwritten element fails.
"""
import ctypes as C
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

NAN = float("nan")


@pytest.fixture(scope="module")
def nat():
    import crowdmod_ddpm_4d_b200._native as n
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    n.lib()
    assert n.lib().cm_device_error() == 0
    yield n
    assert n.lib().cm_device_error() == 0, "a kernel left the device error flag set"


def rel_l2(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-300)).item()


def gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


# =====================================================================================================================
# GroupNorm(8) (+SiLU) (+Dropout3d scale) backward
# =====================================================================================================================
def gn_case(nat, B, pixels, c0, c1, silu, drop, draw, init, params_all=0, seed=0):
    g = gen(seed)
    C_ = c0 + c1
    s0 = torch.randn(B, pixels, c0, device="cuda", generator=g) * 1.5 + 0.3
    s1 = torch.randn(B, pixels, c1, device="cuda", generator=g) * 0.7 - 0.2 if c1 else None
    gamma = torch.randn(C_, device="cuda", generator=g)
    beta = torch.randn(C_, device="cuda", generator=g)
    dnorm = torch.randn(B, pixels, C_, device="cuda", generator=g)
    x64 = (torch.cat([s0, s1], dim=2) if c1 else s0).double()
    # the forward's statistics: float64 mean / rstd per (sample, group), rounded to fp32
    xg = x64.reshape(B, pixels, 8, C_ // 8)
    mean = xg.mean(dim=(1, 3))
    rstd = (xg.var(dim=(1, 3), unbiased=False) + 1e-5).rsqrt()
    stats = torch.stack([mean, rstd], dim=2).float().contiguous()          # [B][8][2]
    drop_ld, drop_off = C_ + 12, 8                                          # the scale sits inside a wider table
    table = None
    if drop:
        table = torch.full((B, drop_ld), NAN, device="cuda")
        table[:, drop_off:drop_off + C_] = (torch.rand(B, C_, device="cuda", generator=g) >= 0.25).float() / 0.75
    raw = torch.randn(B, pixels, C_, device="cuda", generator=g) if draw else None
    init0, init1 = (1, 1) if init == 1 else (0, 0) if init == 0 else (0, 1)
    prev0 = torch.randn(B, pixels, c0, device="cuda", generator=g)
    prev1 = torch.randn(B, pixels, c1, device="cuda", generator=g) if c1 else None
    d0 = torch.full_like(s0, NAN) if init0 else prev0.clone()
    d1 = (torch.full_like(s1, NAN) if init1 else prev1.clone()) if c1 else None
    dgamma = torch.full((C_,), NAN, device="cuda")
    dbeta = torch.full((C_,), NAN, device="cuda")

    def run(d0, d1, dgamma, dbeta):
        nat.check(nat.lib().cm_op_gn_backward(
            nat.ptr(s0), c0, nat.ptr(s1), c1, nat.ptr(gamma), nat.ptr(beta), nat.ptr(stats), nat.ptr(dnorm),
            nat.ptr(raw), None if table is None else C.c_void_p(table.data_ptr() + 4 * drop_off), drop_ld, B, pixels, silu,
            nat.ptr(d0), init0, nat.ptr(d1), init1, nat.ptr(dgamma), nat.ptr(dbeta), params_all,
            nat.current_stream()))

    run(d0, d1, dgamma, dbeta)
    # reference: float64 autograd of F.group_norm -> F.silu -> x dropout scale
    x2 = x64.clone().requires_grad_(True)
    ga2 = gamma.double().requires_grad_(True)
    be2 = beta.double().requires_grad_(True)
    y2 = F.group_norm(x2.permute(0, 2, 1), 8, ga2, be2, 1e-5).permute(0, 2, 1)
    if silu:
        y2 = F.silu(y2)
    if drop:
        y2 = y2 * table[:, None, drop_off:drop_off + C_].double()
    y2.backward(dnorm.double())
    dx = x2.grad
    if draw:
        dx = dx + raw.double()
    ref0, ref1 = dx[..., :c0], dx[..., c0:]
    if not init0:
        ref0 = ref0 + prev0.double()
    if c1 and not init1:
        ref1 = ref1 + prev1.double()
    return dict(d0=d0, d1=d1, dgamma=dgamma, dbeta=dbeta, ref0=ref0, ref1=ref1, rdgamma=ga2.grad, rdbeta=be2.grad,
                dx_ref=dx, run=run, B=B, pixels=pixels, C=C_)


def check_gn(r, c1):
    got = torch.cat([r["d0"], r["d1"]], dim=2) if c1 else r["d0"]
    ref = torch.cat([r["ref0"], r["ref1"]], dim=2) if c1 else r["ref0"]
    assert not torch.isnan(got).any(), "unwritten dx elements"
    e_dx = rel_l2(got, ref)
    e_dg = rel_l2(r["dgamma"], r["rdgamma"])
    e_db = rel_l2(r["dbeta"], r["rdbeta"])
    # one bad (sample, group) must not hide in the global norm: rel-L2 of every group of the gradient itself
    B, P, C_ = r["B"], r["pixels"], r["C"]
    err = (got.double() - ref).reshape(B, P, 8, C_ // 8)
    den = r["dx_ref"].reshape(B, P, 8, C_ // 8).pow(2).sum(dim=(1, 3)).sqrt()
    per_group = (err.pow(2).sum(dim=(1, 3)).sqrt() / den.clamp_min(1e-300)).max().item()
    print(f"GN dx {e_dx:.2e} dgamma {e_dg:.2e} dbeta {e_db:.2e} worst group {per_group:.2e}")
    assert e_dx <= 1e-5, f"dx rel-L2 {e_dx:.3e}"
    assert per_group <= 2e-5, f"worst (sample, group) rel-L2 {per_group:.3e}"
    assert e_dg <= 1e-5, f"dgamma rel-L2 {e_dg:.3e}"
    assert e_db <= 1e-5, f"dbeta rel-L2 {e_db:.3e}"


GN_CASES = [
    # (B, pixels, c0, c1, silu, drop, draw, init)
    (2, 3456, 32, 0, 1, 1, 0, 1),       # ATC full resolution, Dropout3d normalize_2
    (5, 777, 64, 0, 1, 0, 1, 0),        # ragged chunks, raw-output gradient, accumulate
    (1, 7, 96, 0, 0, 1, 0, 1),          # single source with 12-channel groups, pixels < 4 x chunks
    (64, 54, 128, 0, 1, 1, 1, 1),       # training batch of 64 at the coarse level
    (3, 432, 128, 64, 1, 0, 0, 2),      # decoder concat, init0 = 0 / init1 = 1
    (2, 54, 96, 32, 1, 1, 0, 1),        # concat, dropout scale of the second source
    (2, 54, 32, 96, 1, 1, 1, 0),
    (2, 54, 100, 28, 1, 1, 0, 1),       # a group straddles the two sources
    (3, 13, 36, 28, 0, 1, 0, 2),
    (2, 3, 256, 0, 1, 0, 1, 1),
    (600, 3, 512, 0, 1, 1, 0, 1),       # B > 592: one chunk per sample
    (600, 1, 64, 32, 1, 0, 0, 0),
    (2, 54, 1024, 0, 1, 1, 0, 1),       # Q = 256: the widest 256-thread sweep
    (1, 54, 1024, 1024, 1, 1, 1, 2),    # C = 2048: T = Q = 512
    (1, 3456, 32, 32, 0, 0, 0, 0),
    (5, 1, 64, 0, 1, 1, 0, 1),          # one pixel per sample
]


@pytest.mark.parametrize("case", GN_CASES, ids=lambda c: "B%d_p%d_c%d+%d_s%d_d%d_r%d_i%d" % c)
def test_gn_backward_vs_float64_autograd(nat, case):
    B, pixels, c0, c1, silu, drop, draw, init = case
    r = gn_case(nat, B, pixels, c0, c1, silu, drop, draw, init)
    check_gn(r, c1)
    # the sums have a fixed order: a second run (into fresh outputs when the first one overwrote) is bit-identical
    if init == 1:
        again0 = torch.full_like(r["d0"], NAN)
        again1 = torch.full_like(r["d1"], NAN) if c1 else None
        dg, db = torch.full_like(r["dgamma"], NAN), torch.full_like(r["dbeta"], NAN)
        r["run"](again0, again1, dg, db)
        assert torch.equal(again0, r["d0"]), "GroupNorm backward is not deterministic"
        if c1:
            assert torch.equal(again1, r["d1"])
        assert torch.equal(dg, r["dgamma"]) and torch.equal(db, r["dbeta"])


@pytest.mark.parametrize("case", [(2, 3456, 32, 0, 1, 1, 0, 1), (3, 432, 128, 64, 1, 0, 0, 2),
                                  (600, 3, 512, 0, 1, 1, 0, 1), (1, 54, 1024, 1024, 1, 1, 1, 1)],
                         ids=lambda c: "B%d_p%d_c%d+%d_s%d_d%d_r%d_i%d" % c)
def test_gn_backward_params_through_table(nat, case):
    """dgamma / dbeta through gn_bwd_params_all_kernel, the route cm_unet_backward takes (one launch per plan)."""
    B, pixels, c0, c1, silu, drop, draw, init = case
    r = gn_case(nat, B, pixels, c0, c1, silu, drop, draw, init, params_all=1)
    check_gn(r, c1)


# =====================================================================================================================
# dOut preparation (cast_colsum) and the bias-gradient reductions
# =====================================================================================================================
CAST_CASES = [
    # (B, pixels, C, dup)
    (2, 3456, 32, 2), (5, 777, 64, 1), (1, 7, 4, 2), (64, 54, 128, 2), (600, 3, 12, 1), (600, 54, 96, 2),
    (2, 54, 1024, 2), (1, 13, 2048, 2), (3, 1, 2048, 1), (1, 3456, 256, 2),
]


@pytest.mark.parametrize("case", CAST_CASES, ids=lambda c: "B%d_p%d_C%d_dup%d" % c)
@pytest.mark.parametrize("acc_init", [1, 0])
def test_cast_colsum(nat, case, acc_init):
    B, pixels, C_, dup = case
    g = gen(3)
    src = torch.randn(B, pixels, C_, device="cuda", generator=g) * 40.0
    src[0, 0, 0] = 1e-6                                    # an fp16 subnormal
    dst = torch.full((B, pixels, dup * C_), NAN, device="cuda").half()
    prev = torch.randn(B, pixels, C_, device="cuda", generator=g)
    acc = torch.full_like(src, NAN) if acc_init else prev.clone()
    ld = C_ + 8                                            # colsum rows wider than C: the guard columns stay put
    colsum0 = torch.randn(B, ld, device="cuda", generator=g)
    colsum = colsum0.clone()
    nat.check(nat.lib().cm_op_cast_colsum(nat.ptr(src), nat.ptr(dst), dup, nat.ptr(acc), acc_init, nat.ptr(colsum), ld,
                                          B, pixels, C_, nat.current_stream()))
    assert nat.lib().cm_device_error() == 0
    hi = dst[..., :C_]
    assert torch.equal(hi, src.half()), "fp16 operand != src.half()"
    if dup == 2:
        lo = dst[..., C_:]
        assert torch.equal(lo, (src - hi.float()).half()), "lo term != fp16(src - hi)"
        err = (hi.double() + lo.double() - src.double()).abs()
        assert (err <= 2.0 ** -22 * src.double().abs() + 2.0 ** -25).all(), "hi + lo does not reproduce src"
    if acc_init:
        assert torch.equal(acc, src)
    else:
        assert torch.equal(acc, prev + src)
    ref = colsum0.double()[:, :C_] + src.double().sum(dim=1)
    scale = colsum0.double()[:, :C_].abs() + src.double().abs().sum(dim=1)
    worst = ((colsum[:, :C_].double() - ref).abs() / scale).max().item()
    print(f"colsum worst |err| / sum|x| = {worst:.2e}")
    assert worst <= 1e-6, f"column sums off by {worst:.3e} of the absolute sum"
    assert torch.equal(colsum[:, C_:], colsum0[:, C_:]), "colsum wrote past C"


def test_cast_colsum_without_optional_outputs(nat):
    """dst16 only (the dgrad-only route of cm_op_conv3d_dgrad_f32), and colsum only."""
    g = gen(4)
    B, pixels, C_ = 3, 100, 64
    src = torch.randn(B, pixels, C_, device="cuda", generator=g)
    dst = torch.full((B, pixels, C_), NAN, device="cuda").half()
    nat.check(nat.lib().cm_op_cast_colsum(nat.ptr(src), nat.ptr(dst), 1, None, 0, None, 0, B, pixels, C_,
                                          nat.current_stream()))
    assert torch.equal(dst, src.half())
    colsum = torch.zeros(B, C_, device="cuda")
    nat.check(nat.lib().cm_op_cast_colsum(nat.ptr(src), None, 1, None, 0, nat.ptr(colsum), C_, B, pixels, C_,
                                          nat.current_stream()))
    assert ((colsum.double() - src.double().sum(1)).abs() <= 1e-6 * src.double().abs().sum(1)).all()


def test_cast_colsum_saturation_sets_flag_301(nat):
    """A loss-scaled gradient beyond the fp16 range is clamped to +-65504 and reported once through the device error
    flag (the kernel's designed error path: it neither traps nor writes inf)."""
    assert nat.lib().cm_device_error() == 0
    g = gen(5)
    B, pixels, C_ = 2, 54, 64
    src = torch.randn(B, pixels, C_, device="cuda", generator=g)
    src[1, 17, 5] = 1e5
    src[0, 3, 60] = -7e4
    dst = torch.zeros(B, pixels, 2 * C_, device="cuda", dtype=torch.half)
    nat.check(nat.lib().cm_op_cast_colsum(nat.ptr(src), nat.ptr(dst), 2, None, 0, None, 0, B, pixels, C_,
                                          nat.current_stream()))
    assert nat.lib().cm_device_error() == 301
    assert nat.lib().cm_device_error() == 0, "reading the flag clears it"
    assert dst[1, 17, 5].item() == 65504.0 and dst[0, 3, 60].item() == -65504.0
    clamped = src.clamp(-65504.0, 65504.0)
    assert torch.equal(dst[..., :C_], clamped.half())
    assert torch.equal(dst[..., C_:], (clamped - dst[..., :C_].float()).half())


@pytest.mark.parametrize("B", [1, 5, 8, 9, 64, 600])
def test_rowsum_all_vs_float64(nat, B):
    """Every conv's bias gradient in one launch: table entries with row strides wider than C, C not a multiple of 32
    and C > 32 (several 32-channel passes), batch not a multiple of the 8 batch slices."""
    g = gen(6)
    spec = [(32, 32), (64, 96), (3, 8), (200, 256), (1, 1), (130, 130)]     # (C, row stride)
    offs, o = [], 0
    for c, ld in spec:
        offs.append(o)
        o += B * ld
    base = torch.randn(o, device="cuda", generator=g)
    gsize = sum(c for c, _ in spec) + 8 * len(spec)
    grads = torch.full((gsize,), NAN, device="cuda")
    tab, go = [], 0
    for (c, ld), so in zip(spec, offs):
        tab.append((so, ld, c, go))
        go += c + 8
    t = np.ascontiguousarray(np.array(tab, dtype=np.int64))
    nat.check(nat.lib().cm_op_rowsum_all(nat.ptr(base), t.ctypes.data_as(C.POINTER(C.c_int64)), len(tab), B,
                                         nat.ptr(grads), nat.current_stream()))
    for (c, ld), (so, _, _, gofs) in zip(spec, tab):
        rows = base[so:so + B * ld].reshape(B, ld)[:, :c].double()
        ref = rows.sum(0)
        got = grads[gofs:gofs + c].double()
        assert ((got - ref).abs() <= 1e-6 * rows.abs().sum(0)).all(), (c, ld)
        assert torch.isnan(grads[gofs + c:gofs + c + 8]).all(), "rowsum_all wrote past C"


# =====================================================================================================================
# final conv backward
# =====================================================================================================================
def final_case(nat, B, H, W, P, F_, cin, cout, hilo, packed, scale, seed=7):
    g = gen(seed)
    L = P + F_
    a32 = torch.randn(B, L, H, W, cin, device="cuda", generator=g)
    hi = a32.half()
    if hilo:
        lo = (a32 - hi.float()).half()
        act16 = torch.cat([hi, lo], dim=-1).contiguous()
        act_val = hi.double() + lo.double()
    else:
        act16 = hi.contiguous()
        act_val = hi.double()
    w = torch.randn(cout, cin, 3, 3, 3, device="cuda", generator=g) / (27 * cin) ** 0.5
    deps = torch.randn(B, cout, H, W, F_, device="cuda", generator=g) * 1e-3
    dact = torch.full((B, L, H, W, cin), NAN, device="cuda")
    dw = torch.full_like(w, NAN)
    db = torch.full((cout,), NAN, device="cuda")
    d16 = torch.full((B, L, H, W, 32), NAN, device="cuda").half() if packed else None
    nat.check(nat.lib().cm_op_final_conv_backward(
        nat.ptr(deps), scale, nat.ptr(act16), 2 * cin if hilo else 0, cin if hilo else 0, nat.ptr(w), nat.ptr(dact),
        nat.ptr(dw), nat.ptr(db), B, H, W, L, P, cin, cout, nat.ptr(d16), nat.current_stream()))
    # reference: the final conv in the API layout [B, C, H, W, L] (unet.py:121,165-167), only future frames kept
    x = act_val.permute(0, 4, 2, 3, 1).contiguous().requires_grad_(True)
    w64 = w.double().requires_grad_(True)
    b64 = torch.zeros(cout, dtype=torch.float64, device="cuda", requires_grad=True)
    out = F.conv3d(x, w64, b64, padding=1)[..., P:]
    out.backward(deps.double())
    inv = 1.0 / scale
    return dict(dact=dact.permute(0, 4, 2, 3, 1).double() * inv, dw=dw.double() * inv, db=db.double() * inv,
                rdact=x.grad, rdw=w64.grad, rdb=b64.grad, d16=d16, deps=deps, L=L)


FINAL_CASES = [
    # (B, H, W, P, F, cin, cout, hilo)
    (2, 12, 36, 5, 3, 32, 3, 1),        # ATC
    (1, 28, 24, 8, 8, 64, 4, 1),        # HERMES grid, 16 frames
    (3, 2, 3, 2, 1, 32, 1, 0),          # tiny: edge taps everywhere
    (2, 2, 3, 5, 3, 64, 2, 0),
    (1, 12, 36, 2, 1, 64, 3, 1),
]
PACKED_CASES = [
    (2, 12, 36, 5, 3, 32, 3, 1),
    (2, 12, 36, 5, 3, 96, 3, 1),
    (1, 28, 24, 8, 8, 128, 4, 1),
    (2, 12, 36, 5, 3, 256, 1, 1),
    (3, 2, 3, 2, 1, 128, 2, 1),
    (1, 2, 3, 8, 8, 96, 4, 0),
]
# dw of the packed route, rel-L2 against float64 (about twice the 2.2e-4 .. 3.0e-4 measured on a B200 at cin 32 .. 256;
# test_final_conv_backward_packed says where it comes from)
PACKED_DW_BOUND = 6e-4


@pytest.mark.parametrize("case", FINAL_CASES, ids=lambda c: "B%d_%dx%d_P%d_F%d_ci%d_co%d_hl%d" % c)
@pytest.mark.parametrize("scale", [2.0 ** 9, 2.0 ** -5])
def test_final_conv_backward_simt(nat, case, scale):
    B, H, W, P, F_, cin, cout, hilo = case
    r = final_case(nat, B, H, W, P, F_, cin, cout, hilo, False, scale)
    for k in ("dact", "dw", "db"):
        assert not torch.isnan(r[k]).any(), f"unwritten {k}"
    e = {k: rel_l2(r[k], r["r" + k]) for k in ("dact", "dw", "db")}
    print("final SIMT " + " ".join(f"{k} {v:.2e}" for k, v in e.items()))
    for k, v in e.items():
        assert v <= 1e-5, f"{k} rel-L2 {v:.3e}"


@pytest.mark.parametrize("case", PACKED_CASES, ids=lambda c: "B%d_%dx%d_P%d_F%d_ci%d_co%d_hl%d" % c)
def test_final_conv_backward_packed(nat, case):
    """The final conv backward as the training backward runs it for base != 64: dact and db from the fp32 kernels
    (1e-5), dw from the conv weight gradient over two fp16 operands.  One is the single fp16 term of d_eps * S that
    pack_final_dout_kernel writes, the other the hi halves of the hi|lo activation rows.  Each carries 2^-11 relative
    rounding.  Measured on a B200 (1000 W): 2.2e-4 rel-L2 from the d_eps term alone (the case with plain fp16
    activations, which the reference sees unrounded too) and 2.9e-4 .. 3.0e-4 with hi|lo activations at cin 32, 96, 128
    and 256.  That is under a third of the 1e-3 the model tests allow per parameter tensor, and a lo term for d_eps
    would leave the activation share (~2e-4), so the route keeps one term and the bound sits at about twice the
    measured error."""
    B, H, W, P, F_, cin, cout, hilo = case
    scale = 2.0 ** 11
    r = final_case(nat, B, H, W, P, F_, cin, cout, hilo, True, scale)
    for k in ("dact", "dw", "db"):
        assert not torch.isnan(r[k]).any(), f"unwritten {k}"
    e = {k: rel_l2(r[k], r["r" + k]) for k in ("dact", "dw", "db")}
    print("final packed " + " ".join(f"{k} {v:.2e}" for k, v in e.items()))
    assert e["dact"] <= 1e-5 and e["db"] <= 1e-5, e
    assert e["dw"] <= PACKED_DW_BOUND, f"packed dw rel-L2 {e['dw']:.3e}"
    # the packed operand: d_eps * S in columns 0 .. cout-1 of the future frames, zero everywhere else
    d16 = r["d16"].float()
    want = torch.zeros_like(d16)
    want[:, P:, :, :, :cout] = (r["deps"] * scale).permute(0, 4, 2, 3, 1).half().float()
    assert torch.equal(d16, want), "packed dOut operand differs from fp16(d_eps * S) at its place"


# =====================================================================================================================
# first conv weight gradient (SIMT kernel, base 64)
# =====================================================================================================================
FIRST_CASES = [
    # (B, H, W, P, F, cin, cout): B * L * H * W pixels around multiples of the 192-pixel chunk
    (2, 12, 36, 5, 3, 3, 64),           # ATC, 36 chunks
    (1, 28, 24, 8, 8, 4, 32),           # HERMES, 56 chunks
    (1, 2, 3, 16, 15, 3, 64),           # 186 = one partial chunk
    (4, 2, 3, 5, 3, 4, 64),             # 192 = one full chunk
    (3, 2, 3, 6, 5, 3, 32),             # 198 = one chunk + 6
    (1, 28, 24, 2, 1, 4, 64),           # 2016 = 10.5 chunks
]


@pytest.mark.parametrize("case", FIRST_CASES, ids=lambda c: "B%d_%dx%d_P%d_F%d_ci%d_co%d" % c)
def test_first_conv_wgrad(nat, case):
    B, H, W, P, F_, cin, cout = case
    g = gen(8)
    L = P + F_
    x = torch.randn(B, cin, H, W, F_, device="cuda", generator=g)
    past = torch.randn(B, cin, H, W, P, device="cuda", generator=g)
    dout = torch.randn(B, L, H, W, cout, device="cuda", generator=g)
    dw = torch.full((cout, cin, 3, 3, 3), NAN, device="cuda")
    db = torch.full((cout,), NAN, device="cuda")
    nat.check(nat.lib().cm_op_first_conv_wgrad(nat.ptr(x), nat.ptr(past), nat.ptr(dout), nat.ptr(dw), nat.ptr(db),
                                               B, H, W, P, F_, cin, cout, nat.current_stream()))
    inp = torch.cat([past, x], dim=-1).double()
    w64 = torch.zeros(cout, cin, 3, 3, 3, dtype=torch.float64, device="cuda", requires_grad=True)
    b64 = torch.zeros(cout, dtype=torch.float64, device="cuda", requires_grad=True)
    F.conv3d(inp, w64, b64, padding=1).backward(dout.double().permute(0, 4, 2, 3, 1))
    e_w, e_b = rel_l2(dw, w64.grad), rel_l2(db, b64.grad)
    print(f"first conv dw {e_w:.2e} db {e_b:.2e}")
    assert e_w <= 1e-5 and e_b <= 1e-5, (e_w, e_b)


# =====================================================================================================================
# time-embedding MLP backward
# =====================================================================================================================
@pytest.fixture(scope="module")
def atc_block_channels():
    """Output channels of every ResnetBlock of the ATC plan (base 32), plan order, from the native plan itself."""
    from crowdmod_ddpm_4d_b200.models.backbones.unet_autograd import dropout_layout
    from tests._util import build_unet, load_golden
    meta, _ = load_golden("train_atc_b2")
    net = build_unet(meta).cuda()
    layout, ld = dropout_layout(net._plan(meta["rows"], meta["cols"], meta["P"], meta["F"]))
    assert layout[0][0] == 0 and all(a[0] + a[1] == b[0] for a, b in zip(layout, layout[1:]))
    assert ld == layout[-1][0] + layout[-1][1]
    return [ch for _, ch in layout]


@pytest.mark.parametrize("base", [32, 64, 128])
@pytest.mark.parametrize("B", [1, 5, 64])
@pytest.mark.parametrize("gap", [0, 8])
def test_temb_backward_vs_float64_autograd(nat, atc_block_channels, base, B, gap):
    """Linear(base, E) -> SiLU -> Linear(E, E) (embeddings.py:22-34) and every block's dense_1(SiLU(.)) (layers.py:35,
    62), E = 4 base.  gap > 0 leaves padding columns between the blocks of dtemb (c >= couts[k]), filled with garbage
    that must not reach any gradient."""
    g = gen(9)
    E = 4 * base
    couts = [ch * base // 32 for ch in atc_block_channels]
    offs, o = [], 0
    for c in couts:
        offs.append(o)
        o += c + gap
    ld = o
    nb = len(couts)
    e = torch.randn(B, base, device="cuda", generator=g)
    w1 = torch.randn(E, base, device="cuda", generator=g) / base ** 0.5
    b1 = torch.randn(E, device="cuda", generator=g) * 0.1
    w2 = torch.randn(E, E, device="cuda", generator=g) / E ** 0.5
    b2 = torch.randn(E, device="cuda", generator=g) * 0.1
    wd = [torch.randn(c, E, device="cuda", generator=g) / E ** 0.5 for c in couts]
    dtemb = torch.randn(B, ld, device="cuda", generator=g)
    mask = torch.zeros(ld, dtype=torch.bool, device="cuda")
    for c, of in zip(couts, offs):
        mask[of:of + c] = True
    dtemb[:, ~mask] = 1e30
    # forward in float64; the kernels get the pre-activations rounded to fp32, as the training forward saved them
    E64 = e.double()
    W1 = w1.double().requires_grad_(True)
    B1 = b1.double().requires_grad_(True)
    W2 = w2.double().requires_grad_(True)
    B2 = b2.double().requires_grad_(True)
    WD = [w.double().requires_grad_(True) for w in wd]
    BD = [torch.zeros(c, dtype=torch.float64, device="cuda", requires_grad=True) for c in couts]
    h1 = E64 @ W1.T + B1
    s1 = F.silu(h1)
    s1.retain_grad()
    h2 = s1 @ W2.T + B2
    s2 = F.silu(h2)
    s2.retain_grad()
    loss = sum((F.linear(s2, wk, bk) * dtemb[:, of:of + c].double()).sum() for wk, bk, of, c in zip(WD, BD, offs, couts))
    loss.backward()
    h1f, h2f = h1.detach().float().contiguous(), h2.detach().float().contiguous()
    gsize = sum(c * E + c for c in couts) + 64 * nb
    dense = torch.full((gsize,), NAN, device="cuda")
    goff_w, goff_b, p = [], [], 0
    for c in couts:
        goff_w.append(p)
        p += c * E + 32
        goff_b.append(p)
        p += c + 32
    outs = {k: torch.full(s, NAN, device="cuda") for k, s in
            (("dw1", (E, base)), ("db1", (E,)), ("dw2", (E, E)), ("db2", (E,)), ("ds1", (B, E)), ("ds2", (B, E)))}
    wd_ptrs = (C.c_void_p * nb)(*[w.data_ptr() for w in wd])
    a_couts = (C.c_int32 * nb)(*couts)
    a_offs = (C.c_int32 * nb)(*offs)
    a_gw = (C.c_int64 * nb)(*goff_w)
    a_gb = (C.c_int64 * nb)(*goff_b)
    nat.check(nat.lib().cm_op_temb_backward(
        nat.ptr(e), nat.ptr(h1f), nat.ptr(h2f), nat.ptr(dtemb), ld, B, base, E, nat.ptr(w2), wd_ptrs, a_couts, a_offs,
        nb, nat.ptr(dense), a_gw, a_gb, nat.ptr(outs["dw1"]), nat.ptr(outs["db1"]), nat.ptr(outs["dw2"]),
        nat.ptr(outs["db2"]), nat.ptr(outs["ds1"]), nat.ptr(outs["ds2"]), nat.current_stream()))
    refs = {"dw1": W1.grad, "db1": B1.grad, "dw2": W2.grad, "db2": B2.grad, "ds1": s1.grad, "ds2": s2.grad}
    errs = {k: rel_l2(outs[k], refs[k]) for k in refs}
    for k, c in enumerate(couts):
        errs[f"wd{k}"] = rel_l2(dense[goff_w[k]:goff_w[k] + c * E].view(c, E), WD[k].grad)
        errs[f"bd{k}"] = rel_l2(dense[goff_b[k]:goff_b[k] + c], BD[k].grad)
    worst = max(errs.items(), key=lambda kv: kv[1])
    print(f"temb worst {worst[0]} {worst[1]:.2e}")
    for k, v in errs.items():
        assert v <= 1e-5, f"{k} rel-L2 {v:.3e}"


# =====================================================================================================================
# loss scale
# =====================================================================================================================
def expected_scale(m, target=64.0):
    if m == 0.0 or not math.isfinite(m):
        return 1.0
    q = float(np.float32(target) / np.float32(m))            # the kernel divides in fp32
    e = math.frexp(q)[1] - 1
    return 2.0 ** max(-60, min(60, e))


def loss_scale(nat, x):
    out = torch.full((2,), NAN, device="cuda")
    nat.check(nat.lib().cm_op_loss_scale(nat.ptr(x), x.numel(), 64.0, nat.ptr(out), nat.current_stream()))
    return out[0].item(), out[1].item()


@pytest.mark.parametrize("e", [-70, -66, -40, -7, -1, 0, 1, 5, 6, 7, 30, 63, 66, 70])
def test_loss_scale_power_of_two(nat, e):
    g = gen(10)
    for mant in (1.0, 1.5, 1.999):
        m = float(np.float32(mant * 2.0 ** e))
        x = torch.rand(100003, device="cuda", generator=g) * m * 0.9
        x[31337] = -m                                         # the maximum is a negative element
        S, inv = loss_scale(nat, x)
        want = expected_scale(m)
        assert S == want, (m, S, want)
        assert S * inv == 1.0 and inv == 1.0 / want
        if abs(math.log2(want)) < 60:
            assert 32.0 <= m * S <= 64.0, m * S


def test_loss_scale_special_values(nat):
    assert loss_scale(nat, torch.zeros(5000, device="cuda")) == (1.0, 1.0)
    x = torch.randn(5000, device="cuda", generator=gen(11))
    base = expected_scale(x.abs().max().item())
    assert loss_scale(nat, x)[0] == base
    y = x.clone()
    y[123] = float("inf")
    assert loss_scale(nat, y) == (1.0, 1.0)
    y[123] = -float("inf")
    assert loss_scale(nat, y) == (1.0, 1.0)
    y[123] = float("nan")
    assert loss_scale(nat, y)[0] == base, "a NaN must not change the scale of the finite part"


def test_loss_scale_large_n(nat):
    """absmax over 2^24 + 3 elements: grid-stride loop, warp reduction and one atomicMax per warp."""
    n = (1 << 24) + 3
    x = torch.rand(n, device="cuda", generator=gen(12)) * 0.001
    x[n - 1] = -3.0                                          # the very last element carries the maximum
    assert loss_scale(nat, x) == (16.0, 1.0 / 16.0)
    x[n - 1] = 0.0
    x[7] = 5e-3
    assert loss_scale(nat, x)[0] == expected_scale(5e-3)


# =====================================================================================================================
# model-level properties of cm_unet_backward
# =====================================================================================================================
def _net_and_inputs(name, B, seed):
    from oracle import ddpm_oracle as do
    from tests._util import build_unet, load_golden
    meta, a = load_golden(name)
    net = build_unet(meta).cuda().eval()     # eval: no dropout drawn; parameters still require grad -> native training
    g = torch.Generator().manual_seed(seed)
    shp_f = (B, 3, meta["rows"], meta["cols"], meta["F"])
    shp_p = (B, 3, meta["rows"], meta["cols"], meta["P"])
    x = do.synthetic_macroprops(B, 3, meta["rows"], meta["cols"], meta["F"], seed) if B != meta["B"] else a["future"]
    past = do.synthetic_macroprops(B, 3, meta["rows"], meta["cols"], meta["P"], seed + 1) if B != meta["B"] else a["past"]
    assert tuple(x.shape) == shp_f and tuple(past.shape) == shp_p
    t = torch.randint(0, meta["T"], (B,), generator=g)
    d_eps = torch.randn(shp_f, generator=g) * 1e-4
    return meta, net, x.cuda(), t.cuda(), past.cuda(), d_eps.cuda()


def _flat_grad(net, x, t, past, d_eps):
    out = net(x, t, past)
    out.backward(d_eps)
    torch.cuda.synchronize()
    return net._last_flat_grad.clone()


@pytest.mark.parametrize("name", ["train_small", "train_atc_b2"])
def test_backward_loss_scale_invariance(nat, name):
    """d_eps x 2^k moves the device-chosen loss scale S by 2^-k, so d_eps * S -- everything the backward computes --
    is unchanged and the unscaled gradient is exactly 2^k times the k = 0 gradient.  A path that skips the scale or the
    unscale, or reads d_eps without S (the final conv kernels read scale_dev; the time-MLP tail must run before
    scale_inplace) is off by a power of two.  The backward's float atomics (weight-gradient epilogues, channel sums)
    make run-to-run differences in the last bits, so the comparison is at the level of that noise."""
    meta, net, x, t, past, d_eps = _net_and_inputs(name, 3 if name == "train_small" else 2, 21)
    g0 = _flat_grad(net, x, t, past, d_eps)
    g0b = _flat_grad(net, x, t, past, d_eps)
    noise = rel_l2(g0b, g0)
    worst = 0.0
    for k in (-30, -10, 10, 30):
        gk = _flat_grad(net, x, t, past, d_eps * 2.0 ** k)
        assert torch.isfinite(gk).all()
        e = rel_l2(gk * 2.0 ** -k, g0)
        worst = max(worst, e)
        bitwise = torch.equal(gk * 2.0 ** -k, g0)
        print(f"{name} k={k}: rel-L2 {e:.2e} (run-to-run {noise:.2e}, bit-identical {bitwise})")
        assert e <= 1e-6, f"k={k}: gradient is not 2^k times the k=0 gradient (rel-L2 {e:.3e})"
    assert nat.lib().cm_device_error() == 0


def test_train_step_batch_1_vs_oracle():
    """B = 1 (one sample: every chunking falls to its single-sample geometry) against the CPU oracle at the bounds of
    test_gpu_train.py."""
    from oracle import ddpm_oracle as do
    from tests._util import load_golden
    from tests.test_gpu_train import _compare, _native_grads, _oracle_grads
    meta, _ = load_golden("train_atc_b2")
    a = {"future": do.synthetic_macroprops(1, 3, 12, 36, 3, 31), "past": do.synthetic_macroprops(1, 3, 12, 36, 5, 32)}
    t = torch.tensor([417])
    eps = torch.randn(a["future"].shape, generator=torch.Generator().manual_seed(33))
    lo, go, s = _oracle_grads(meta, a, t, eps)
    ln, gn, _ = _native_grads(meta, a, t, eps, s)
    _compare(lo, go, ln, gn)


def test_gradient_batch_permutation_equivariance(nat):
    """The parameter gradient is a sum over the batch: permuting (x, t, eps, past, dropout masks) only reorders that
    sum."""
    from crowdmod_ddpm_4d_b200.models.backbones.unet_autograd import dropout_layout
    meta, net, x, t, past, d_eps = _net_and_inputs("train_atc_b2", 5, 41)
    layout, _ = dropout_layout(net._plan(meta["rows"], meta["cols"], meta["P"], meta["F"]))
    g = torch.Generator().manual_seed(42)
    masks = [((torch.rand(5, ch, generator=g) >= 0.25).float() / 0.75).cuda() for _, ch in layout]
    net._injected_dropout = masks
    g0 = _flat_grad(net, x, t, past, d_eps)
    perm = torch.tensor([3, 0, 4, 2, 1], device="cuda")
    net._injected_dropout = [m[perm] for m in masks]
    g1 = _flat_grad(net, x[perm].contiguous(), t[perm].contiguous(), past[perm].contiguous(), d_eps[perm].contiguous())
    from crowdmod_ddpm_4d_b200.models.backbones.unet_autograd import grad_layout
    plan = net._plan(meta["rows"], meta["cols"], meta["P"], meta["F"])
    offs, total = grad_layout(plan)
    bounds = list(offs) + [total]
    worst = max(rel_l2(g1[a:b], g0[a:b]) if g0[a:b].abs().max() > 0 else 0.0 for a, b in zip(bounds, bounds[1:]))
    print(f"batch permutation: global {rel_l2(g1, g0):.2e}, worst tensor {worst:.2e}")
    assert worst <= 1e-6, f"worst parameter tensor rel-L2 {worst:.3e}"
