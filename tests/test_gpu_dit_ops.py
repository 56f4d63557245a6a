"""Op-level parity of the DiT4D_V4 sampling kernels (csrc/dit.cu) and of the in-kernel Philox noise stream.

The model tests (test_gpu_dit.py, test_gpu_attn_long.py) bound the DiT's eps at rel-L2 1e-3 and its chains at 5e-3: a
wrong LayerNorm epsilon, a gate read from the wrong sample or an un-patch order that is wrong only for t_patch > 1 can
hide inside those bounds.  Here every kernel runs alone, through the cm_op_dit_* entry points (which launch through the
same enqueue functions as cm_dit_forward / cm_dit_sample), against a float64 restatement of the reference op:

* gather kernels (patchify, un-patch) and the fp32 position add: bit-exact;
* LayerNorm + AdaLN modulate and temporal attention, fp16 outputs: one fp16 ulp of the float64 value (fp32 arithmetic
  is ~1e-6 relative, an fp16 ulp 2^-11 relative);
* the tcgen05 GEMM with the DiT's epilogue fusions: rel-L2 2e-5, the bound of the hi|lo conv tests;
* the reverse-step update: a few fp32 ulps of its largest term.

Kernel inputs are exactly what the kernel reads (fp16-rounded where it reads fp16); outputs are pre-filled with NaN so
that an unwritten element fails.  The Philox4x32-10 + Box-Muller stream is restated in numpy (checked against the
Random123 known-answer vectors) and pinned for both backbones; the DiT's AdaLN table is compared with the per-sample
forward at every table chunk edge.
"""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

NAN = float("nan")


@pytest.fixture(scope="module")
def nat():
    import crowdmod_ddpm_4d_b200._native as n
    torch.backends.cuda.matmul.allow_tf32 = False
    n.lib()
    assert n.lib().cm_device_error() == 0
    yield n
    assert n.lib().cm_device_error() == 0, "a kernel left the device error flag set"


def gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def rel_l2(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-300)).item()


def ulp16(v):
    """Spacing of fp16 at |v| (subnormal spacing 2^-24 below 2^-14)."""
    a = v.double().abs().clamp_min(2.0 ** -14)
    return torch.exp2(torch.floor(torch.log2(a)) - 10)


def fp16_close(got16, ref64, extra=0.0):
    """Every element within one fp16 ulp (+ extra) of the float64 value; returns the share equal to fp16(ref)."""
    g = got16.double()
    assert not torch.isnan(g).any(), "unwritten or NaN output elements"
    err = (g - ref64).abs()
    tol = ulp16(torch.maximum(g.abs(), ref64.abs())) + extra
    bad = err > tol
    assert not bad.any(), f"{int(bad.sum())} elements beyond one fp16 ulp; worst excess {(err - tol).max().item():.3e}"
    return (got16 == ref64.half()).double().mean().item()


# =====================================================================================================================
# patch embedding operand and positional embeddings
# =====================================================================================================================
def patch_matrix(past, future, p, pt):
    """Rows (b, slot, ph, pw), columns (c, dt, dy, dx): the unfold behind Conv3d(kernel = stride = (pt, p, p))."""
    x = torch.cat([past, future], dim=4)                                      # [B][C][H][W][T]
    B, Cc, H, W, T = x.shape
    x = x.reshape(B, Cc, H // p, p, W // p, p, T // pt, pt)                  # b c ph dy pw dx slot dt
    return x.permute(0, 6, 2, 4, 1, 7, 3, 5).reshape(B * (T // pt) * (H // p) * (W // p), Cc * pt * p * p)


@pytest.mark.gpu
@pytest.mark.parametrize("B,Cc,H,W,P,Fr,p,pt,extra_pad", [
    (3, 3, 12, 36, 5, 3, 4, 2, 0),     # the ATC geometry at t_patch 2: slot 2 straddles past (t=4) and future (t=5)
    (2, 4, 12, 36, 5, 3, 4, 4, 0),     # slot 1 = past frame 4 + future frames 0..2
    (2, 3, 8, 12, 4, 4, 2, 1, 0),      # K = 12 -> Kpad 32: 20 pad columns
    (5, 1, 4, 6, 6, 2, 2, 4, 0),       # K = 16, slot 1 straddles
    (1, 2, 8, 8, 3, 5, 4, 1, 32),      # K = 32 with 32 more pad columns
])
def test_patchify_bit_exact(nat, B, Cc, H, W, P, Fr, p, pt, extra_pad):
    """A16 = fp16 of the unfolded patch matrix of cat(past, future) along time, Conv3d weight order (c, dt, dy, dx);
    columns K .. Kpad-1 exactly 0.  Pure gather + round-to-nearest: bit-exact."""
    g = gen(1)
    past = torch.randn(B, Cc, H, W, P, device="cuda", generator=g) + 10.0     # past and future distinguishable
    fut = torch.randn(B, Cc, H, W, Fr, device="cuda", generator=g)
    K = Cc * pt * p * p
    kpad = (K + 31) // 32 * 32 + extra_pad
    rows = B * ((P + Fr) // pt) * (H // p) * (W // p)
    a16 = torch.full((rows, kpad), NAN, device="cuda", dtype=torch.float16)
    nat.check(nat.lib().cm_op_dit_patchify(nat.ptr(fut), nat.ptr(past), B, Cc, H, W, P, Fr, p, pt, kpad, nat.ptr(a16),
                                           nat.current_stream()))
    ref = patch_matrix(past, fut, p, pt).half()
    assert torch.equal(a16[:, :K], ref)
    assert torch.equal(a16[:, K:], torch.zeros_like(a16[:, K:])), "pad columns must be written as 0"


@pytest.mark.gpu
@pytest.mark.parametrize("B,Tp,Ns,D", [(3, 4, 27, 256), (1, 8, 6, 32), (5, 2, 168, 128), (7, 3, 1, 96)])
def test_add_pos_bit_exact(nat, B, Tp, Ns, D):
    """x += spatial[s] then + temporal[slot] in fp32, in that order (DiT4D_V4.py:329-346), with temporal_pos_embed
    holding more slots than Tp.  Bit-exact."""
    g = gen(2)
    rows = B * Tp * Ns
    x = torch.randn(rows, D, device="cuda", generator=g)
    sp = torch.randn(Ns, D, device="cuda", generator=g) * 0.02
    tp = torch.randn(Tp + 3, D, device="cuda", generator=g) * 0.02
    ref = ((x.reshape(B, Tp, Ns, D) + sp[None, None]) + tp[None, :Tp, None]).reshape(rows, D)
    nat.check(nat.lib().cm_op_dit_add_pos(nat.ptr(x), nat.ptr(sp), nat.ptr(tp), rows, Tp, Ns, D, nat.current_stream()))
    assert torch.equal(x, ref)


# =====================================================================================================================
# LayerNorm + AdaLN modulate -> fp16
# =====================================================================================================================
def ln_mod_case(nat, D, rows, rows_per_sample, per_sample, seed, x=None, zero_mod=False):
    g = gen(seed)
    nsamp = (rows + rows_per_sample - 1) // rows_per_sample
    if x is None:
        x = torch.randn(rows, D, device="cuda", generator=g) * 1.7 + 0.4
    # the vectors sit inside a wider row, scale before shift, as the blocks' chunk(9) layout does
    ld = 3 * D + 8
    off_shift, off_scale = D + 4, 4
    mods = torch.full((nsamp if per_sample else 1, ld), NAN, device="cuda")
    mods[:, off_shift:off_shift + D] = 0.0 if zero_mod else torch.randn(mods.shape[0], D, device="cuda", generator=g)
    mods[:, off_scale:off_scale + D] = 0.0 if zero_mod else torch.randn(mods.shape[0], D, device="cuda", generator=g) * 0.5
    out = torch.full((rows, D), NAN, device="cuda", dtype=torch.float16)
    nat.check(nat.lib().cm_op_dit_ln_mod(nat.ptr(x), nat.ptr(mods), ld if per_sample else 0, off_shift, off_scale,
                                         rows_per_sample, rows, D, nat.ptr(out), nat.current_stream()))
    b = torch.arange(rows, device="cuda") // rows_per_sample if per_sample else torch.zeros(rows, dtype=torch.long,
                                                                                             device="cuda")
    shift = mods[b, off_shift:off_shift + D].double()
    scale = mods[b, off_scale:off_scale + D].double()
    n = F.layer_norm(x.double(), (D,), eps=1e-6)
    ref = n * (1.0 + scale) + shift                                                # oracle/dit_oracle.py _ln / _mod
    terms = (n * (1.0 + scale)).abs() + shift.abs()
    return out, ref, shift, scale, terms


@pytest.mark.gpu
@pytest.mark.parametrize("D", [32, 96, 128, 256, 512])
@pytest.mark.parametrize("rows,rows_per_sample,per_sample", [(323, 27, True), (1001, 168, True), (13, 5, True),
                                                              (205, 41, False)])
def test_ln_mod_vs_float64(nat, D, rows, rows_per_sample, per_sample):
    """LayerNorm(eps 1e-6, no affine) * (1 + scale[b]) + shift[b] -> fp16, b = row / rows_per_sample (ld_mods = the row
    width) or one vector for all rows (ld_mods = 0, sampling).  Row counts are not multiples of the 8 warps of a block
    and rows_per_sample splits blocks between samples; D = 32 and 96 leave lanes idle.  Bound: every element within
    one fp16 ulp of the float64 value plus 2^-20 of |LN(x) (1 + scale)| + |shift|, and >= 99 % equal to its
    round-to-nearest.  The fp32 normalisation is ~1e-6 relative, 2^-11 below an fp16 ulp, except where the modulated
    sum cancels toward 0: there an fp16 ulp is tiny and the terms' fp32 error (measured on a B200: up to 1e-7 beyond
    one ulp) dominates."""
    out, ref, _, _, terms = ln_mod_case(nat, D, rows, rows_per_sample, per_sample, seed=D + rows)
    share = fp16_close(out, ref, extra=2.0 ** -20 * terms)
    print(f"ln_mod D={D} rows={rows}: {share:.4%} equal to fp16(ref)")
    assert share >= 0.99


@pytest.mark.gpu
@pytest.mark.parametrize("D", [96, 256])
def test_ln_mod_edge_rows(nat, D):
    """Rows that pin the statistics: mean 1e3 with std 1 (a one-pass E[x^2] - mean^2 variance in fp32 loses the
    variance to cancellation: ~1e-1 relative); variance ~1e-8 with the modulation off (the output scales as
    1/sqrt(var + eps): eps 1e-5 instead of 1e-6 shrinks it by 3.2x); all-zero rows, whose output is exactly
    fp16(shift).  Bounds as test_ln_mod_vs_float64, except that the mean-1e3 rows get 2e-3 * |1 + scale| more: the
    fp32 partial sums of those rows reach 2.6e5 (D = 256), where an fp32 ulp is 2^-6, so their mean is exact to
    ~1e-4 only.  A one-pass variance is off by ~1e-1 there."""
    g = gen(7)
    rows = 3 * 9
    x = torch.empty(rows, D, device="cuda")
    x[0:9] = 1000.0 + torch.randn(9, D, device="cuda", generator=g)
    x[9:18] = 1e-4 * torch.randn(9, D, device="cuda", generator=g)
    x[18:27] = 0.0
    for zero_mod in (False, True):
        out, ref, shift, scale, terms = ln_mod_case(nat, D, rows, 9, True, seed=3, x=x, zero_mod=zero_mod)
        fp16_close(out[:9], ref[:9], extra=2e-3 * (1.0 + scale[:9]).abs() + 2.0 ** -20 * terms[:9])
        fp16_close(out[9:18], ref[9:18], extra=2.0 ** -20 * terms[9:18])
        assert torch.equal(out[18:], shift[18:].half()), "an all-zero row must give fp16(shift) exactly"


# =====================================================================================================================
# temporal cross-attention
# =====================================================================================================================
@pytest.mark.gpu
@pytest.mark.parametrize("B,Tp,qs,Ns,dh,heads,span", [
    (1, 1, 0, 27, 96, 1, 1.0),        # 27 warps: not a multiple of 8
    (2, 2, 1, 168, 32, 4, 1.0),
    (3, 4, 2, 27, 40, 4, 60.0),
    (2, 4, 0, 1, 64, 3, 1.0),
    (2, 8, 3, 27, 128, 2, 60.0),
    (1, 8, 7, 168, 8, 4, 100.0),
    (5, 8, 0, 1, 32, 16, 1.0),
    (3, 6, 2, 27, 64, 2, 60.0),
    (1, 2, 0, 27, 128, 1, 1.0),
])
def test_tattn_vs_float64(nat, B, Tp, qs, Ns, dh, heads, span):
    """Slots [qs, Tp) of every (sample, spatial patch) query all Tp slots of that patch, per head (dit_oracle.block
    step 2): float64 softmax(q k^T / sqrt(dh)) v.  `span` scales q and k so that the scores reach about +-span
    (+-100 overflows exp() in fp32 without the max subtraction).  Bound: one fp16 ulp of the output plus 1e-4 of the
    largest |v|: fp32 scores of magnitude up to 100 carry ~1e-5 absolute error, which moves every softmax weight by
    ~1e-5 relative."""
    D = dh * heads
    g = gen(Tp * 100 + dh)
    qkv = torch.randn(B, Tp, Ns, 3 * D, device="cuda", generator=g)
    if span > 1:
        qkv[..., :2 * D] *= (span / 3) ** 0.5          # scores with std span / 3
    nq = Tp - qs
    ctx = torch.full((B, nq, Ns, D), NAN, device="cuda", dtype=torch.float16)
    nat.check(nat.lib().cm_op_dit_tattn(nat.ptr(qkv), nat.ptr(ctx), B, Tp, Ns, D, heads, qs, nat.current_stream()))
    t = qkv.double().reshape(B, Tp, Ns, 3, heads, dh)
    q = t[:, qs:, :, 0].permute(0, 2, 3, 1, 4)                 # [B][Ns][heads][nq][dh]
    k = t[:, :, :, 1].permute(0, 2, 3, 1, 4)
    v = t[:, :, :, 2].permute(0, 2, 3, 1, 4)
    s = q @ k.transpose(-1, -2) / dh ** 0.5
    ref = (torch.softmax(s, dim=-1) @ v).permute(0, 3, 1, 2, 4).reshape(B, nq, Ns, D)
    print(f"tattn Tp={Tp} qs={qs} dh={dh}: max |score| {s.abs().max().item():.1f}")
    fp16_close(ctx, ref, extra=1e-4 * v.abs().max().item())


# =====================================================================================================================
# tcgen05 GEMM with the DiT epilogue fusions
# =====================================================================================================================
def linear_case(nat, nb, pps, cin, cout, act=0, gate=None, rmap=None, seed=0):
    g = gen(seed)
    M = nb * pps
    a16 = (torch.randn(M, cin, device="cuda", generator=g)).half()
    w = torch.randn(cout, cin, device="cuda", generator=g) * cin ** -0.5
    bias = torch.randn(cout, device="cuda", generator=g) * 0.1
    v64 = a16.double() @ w.double().t() + bias.double()
    return a16, w, bias, v64


@pytest.mark.gpu
@pytest.mark.parametrize("nb,pps,cin,cout", [(1, 12, 256, 256), (3, 27, 128, 384), (5, 168, 256, 1024), (64, 12, 1024, 256),
                                             (2, 504, 512, 96), (7, 27, 1024, 128)])
def test_linear_plain_and_gelu(nat, nb, pps, cin, cout):
    """out32 = A.W^T + b on fp16 A and fp32 W (packed hi|lo), against float64 on the same fp16 A: rel-L2 <= 2e-5 (the
    hi|lo conv tests' bound) overall and <= 1e-4 per row (a row's error is the same fp32-accumulation noise over cout
    elements instead of all of them; 5x the overall bound covers the worst of up to 3.5e3 rows).  act = 1 (mlp.0 +
    GELU): out16 = fp16(exact-erf GELU), within one fp16 ulp plus 1e-5 of max |v| (the GEMM's own error)."""
    a16, w, bias, v64 = linear_case(nat, nb, pps, cin, cout, seed=nb + cin)
    out = torch.full((nb * pps, cout), NAN, device="cuda")
    nat.check(nat.lib().cm_op_dit_linear(nat.ptr(a16), nb, pps, cin, nat.ptr(w), nat.ptr(bias), cout, 0, None, 0, 0, 0,
                                         nat.ptr(out), None, nat.current_stream()))
    e = rel_l2(out, v64)
    rows = ((out.double() - v64).norm(dim=1) / v64.norm(dim=1)).max().item()
    print(f"linear nb={nb} pps={pps} cin={cin} cout={cout}: rel-L2 {e:.2e}, worst row {rows:.2e}")
    assert e <= 2e-5 and rows <= 1e-4
    o16 = torch.full((nb * pps, cout), NAN, device="cuda", dtype=torch.float16)
    nat.check(nat.lib().cm_op_dit_linear(nat.ptr(a16), nb, pps, cin, nat.ptr(w), nat.ptr(bias), cout, 1, None, 0, 0, 0,
                                         None, nat.ptr(o16), nat.current_stream()))
    fp16_close(o16, F.gelu(v64), extra=1e-5 * v64.abs().max().item())


@pytest.mark.gpu
@pytest.mark.parametrize("nb,pps,cin,cout,rmap,per_sample", [
    (3, 27, 128, 128, None, True),          # M = 81: one tile, three samples
    (5, 27, 256, 256, None, False),         # gate_ld = 0 (sampling)
    (2, 12, 512, 256, None, True),
    (64, 12, 1024, 128, None, True),        # 768 rows, tiles straddle samples
    (4, 168 * 3, 256, 256, (168 * 8, 168 * 5), True),   # temporal out-projection, Tp 8 / nq 3, Ns 168
    (3, 27 * 2, 256, 256, (27 * 4, 27 * 2), False),     # Tp 4 / nq 2 (the ATC plan), sampling gate
    (7, 27, 128, 128, (27 * 2, 27), True),              # Tp 2 / nq 1
])
def test_linear_gated_residual(nat, nb, pps, cin, cout, rmap, per_sample):
    """x[orow] += gate[b] * (A.W^T + b) in place (the out-projections and mlp.3 with AdaLN-Zero gates): gate rows at
    a block offset inside per-sample rows of width gate_ld (other columns NaN), or one row for all (gate_ld = 0).
    With rmap, GEMM row m of sample b = m / pps lands at b*rmap_out + rmap_off + (m - b*pps); every other row (the
    past slots) must be bit-unchanged.  Bound: rel-L2 <= 2e-5 of the update, as test_linear_plain_and_gelu."""
    a16, w, bias, v64 = linear_case(nat, nb, pps, cin, cout, seed=pps + cout)
    g = gen(11)
    rows_out = nb * (rmap[0] if rmap else pps)
    x0 = torch.randn(rows_out, cout, device="cuda", generator=g)
    gate_ld, goff = 9 * cout, 5 * cout
    gt = torch.full((nb if per_sample else 1, gate_ld), NAN, device="cuda")
    gt[:, goff:goff + cout] = torch.randn(gt.shape[0], cout, device="cuda", generator=g)
    x = x0.clone()
    nat.check(nat.lib().cm_op_dit_linear(nat.ptr(a16), nb, pps, cin, nat.ptr(w), nat.ptr(bias), cout, 0,
                                         C.c_void_p(gt.data_ptr() + 4 * goff), gate_ld if per_sample else 0,
                                         rmap[0] if rmap else 0, rmap[1] if rmap else 0, nat.ptr(x), None,
                                         nat.current_stream()))
    m = torch.arange(nb * pps, device="cuda")
    b = m // pps
    orow = b * rmap[0] + rmap[1] + (m - b * pps) if rmap else m
    gate = gt[b if per_sample else torch.zeros_like(b), goff:goff + cout].double()
    upd = gate * v64
    ref = x0.double().clone()
    ref[orow] += upd
    e = ((x.double() - ref).norm() / upd.norm()).item()
    print(f"gated linear nb={nb} pps={pps} rmap={rmap}: rel-L2 of the update {e:.2e}")
    assert e <= 2e-5
    untouched = torch.ones(rows_out, dtype=torch.bool, device="cuda")
    untouched[orow] = False
    assert torch.equal(x[untouched], x0[untouched]), "rows outside the remapped block changed"


# =====================================================================================================================
# un-patch + reverse-step update
# =====================================================================================================================
def unpatch_ref(out, B, Cc, H, W, P, Fr, p, pt):
    """PatchUnEmbed4D + slice to the future frames (dit_oracle.dit_forward lines 99-102)."""
    Tp, hp, wp = (P + Fr) // pt, H // p, W // p
    o = out[:, :pt * Cc * p * p].reshape(B, Tp, hp, wp, pt, Cc, p, p).permute(0, 5, 1, 4, 2, 6, 3, 7)
    o = o.reshape(B, Cc, Tp * pt, H, W).permute(0, 1, 3, 4, 2)
    return o[..., P:].contiguous()


def run_unpatch(nat, out, ld, geo, eps_out=None, x=None, coef=None, nsteps=0, step=0, mode=0, noise=None, history=None):
    B, Cc, H, W, P, Fr, p, pt = geo
    nat.check(nat.lib().cm_op_dit_unpatch_step(nat.ptr(out), ld, B, Cc, H, W, P, Fr, p, pt, nat.ptr(eps_out), nat.ptr(x),
                                               nat.ptr(coef), nsteps, step, mode, nat.ptr(noise), 0, 0,
                                               nat.ptr(history), nat.current_stream()))


GEOS = [(3, 3, 12, 36, 5, 3, 4, 4), (2, 3, 8, 12, 4, 4, 4, 2), (2, 4, 12, 36, 5, 3, 4, 1), (3, 2, 4, 8, 3, 5, 2, 4)]


@pytest.mark.gpu
@pytest.mark.parametrize("geo", GEOS)
def test_unpatch_eps_bit_exact(nat, geo):
    """eps_out = the future frames of the un-patched FinalLayer output, column ((dt*C + c)*p + dy)*p + dx, read from
    rows of stride ld > t_patch*C*p*p (the extra columns hold NaN): a pure gather, bit-exact."""
    B, Cc, H, W, P, Fr, p, pt = geo
    rows = B * ((P + Fr) // pt) * (H // p) * (W // p)
    nout = pt * Cc * p * p
    ld = nout + 32
    out = torch.full((rows, ld), NAN, device="cuda")
    out[:, :nout] = torch.randn(rows, nout, device="cuda", generator=gen(5))
    eps = torch.full((B, Cc, H, W, Fr), NAN, device="cuda")
    run_unpatch(nat, out, ld, geo, eps_out=eps)
    assert torch.equal(eps, unpatch_ref(out, *geo))


def update_ref(x, eps, z, cf, mode):
    """DDPM.step (ddpm.py:25-38) / DDIM eq. 12 (:262-265) + Sparsity sign guidance on channel 0 (guidance.py:4-8), in
    float64.  Returns (x_next, the magnitude of its largest terms) for the fp32 bound."""
    x, eps, z, cf = x.double(), eps.double(), z.double(), [float(c) for c in cf]
    if mode == 0:
        xn = cf[0] * (x - cf[1] * eps) + cf[2] * z
        mag = abs(cf[0]) * (x.abs() + abs(cf[1]) * eps.abs()) + abs(cf[2]) * z.abs()
    else:
        x0 = (x - cf[0] * eps) / cf[1]
        xn = cf[2] * x0 + cf[3] * eps + cf[4] * z
        mag = abs(cf[2]) * (x.abs() + abs(cf[0]) * eps.abs()) / abs(cf[1]) + abs(cf[3]) * eps.abs() + abs(cf[4]) * z.abs()
    if cf[5] != 0.0:
        xn[:, 0] -= cf[5] * torch.sign(xn[:, 0])
        mag[:, 0] += abs(cf[5])
    return xn, mag


@pytest.mark.gpu
@pytest.mark.parametrize("geo", GEOS[:3])
@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("guided", [False, True])
def test_unpatch_step_update(nat, geo, mode, guided):
    """Step `step` of a 4-step chain with injected noise and a distinct random coefficient row per step (a row
    mix-up fails): x in place, history slot step+1 written, every other slot bit-untouched; with coef[5] != 0 the
    sign guidance applies to channel 0 only.  Bound per element: 8 fp32 ulps (2^-24 each) of the sum of the
    magnitudes of the update's terms (five roundings)."""
    B, Cc, H, W, P, Fr, p, pt = geo
    g = gen(17 + mode)
    rows = B * ((P + Fr) // pt) * (H // p) * (W // p)
    nout = pt * Cc * p * p
    out = torch.randn(rows, nout, device="cuda", generator=g)
    nsteps, step = 4, 2
    coef = torch.rand(nsteps, 8, device="cuda", generator=g) + 0.25
    if not guided:
        coef[:, 5] = 0.0
    shape = (B, Cc, H, W, Fr)
    x0 = torch.randn(shape, device="cuda", generator=g)
    noise = torch.randn(nsteps, *shape, device="cuda", generator=g)
    hist0 = torch.randn(nsteps + 1, *shape, device="cuda", generator=g)
    x, hist = x0.clone(), hist0.clone()
    eps = torch.full(shape, NAN, device="cuda")
    run_unpatch(nat, out, nout, geo, eps_out=eps, x=x, coef=coef, nsteps=nsteps, step=step, mode=mode, noise=noise,
                history=hist)
    e = unpatch_ref(out, *geo)
    assert torch.equal(eps, e)
    ref, mag = update_ref(x0, e, noise[step], coef[step].tolist(), mode)
    err = (x.double() - ref).abs()
    assert (err <= 8 * 2.0 ** -24 * mag).all(), f"worst {(err / mag).max().item() * 2 ** 24:.1f} fp32 ulps of the terms"
    assert torch.equal(hist[step + 1], x)
    keep = [i for i in range(nsteps + 1) if i != step + 1]
    assert torch.equal(hist[keep], hist0[keep])


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1])
def test_unpatch_step_zero_noise_coef_and_sign_of_zero(nat, mode):
    """A step whose noise coefficient is 0 (coef[2] in DDPM, coef[4] in DDIM) must not read its noise slice (NaN
    here), while the other steps' slices and the other coefficient hold finite values; x_next == 0 exactly keeps its
    sign guidance at 0 (sign(0) = 0).  The first step maps x to itself (DDPM {1, 0, 0}; DDIM {0, 1, 1, 0, 0}), so
    x = 0 entries stay exactly 0."""
    geo = (2, 3, 8, 12, 4, 4, 4, 2)
    B, Cc, H, W, P, Fr, p, pt = geo
    g = gen(23)
    rows = B * ((P + Fr) // pt) * (H // p) * (W // p)
    out = torch.randn(rows, pt * Cc * p * p, device="cuda", generator=g)
    shape = (B, Cc, H, W, Fr)
    coef = torch.rand(2, 8, device="cuda", generator=g) + 0.25
    if mode == 0:
        coef[0, :3] = torch.tensor([1.0, 0.0, 0.0])
        coef[0, 4] = 1.0                 # DDIM's noise coefficient: must be ignored in DDPM mode
    else:
        coef[0, :5] = torch.tensor([0.0, 1.0, 1.0, 0.0, 0.0])
    coef[0, 5] = 0.3
    noise = torch.randn(2, *shape, device="cuda", generator=g)
    noise[0] = NAN
    x0 = torch.randn(shape, device="cuda", generator=g)
    x0[:, :, :, :6] = 0.0
    x = x0.clone()
    run_unpatch(nat, out, pt * Cc * p * p, geo, x=x, coef=coef, nsteps=2, step=0, mode=mode, noise=noise)
    ref = x0.clone()
    ref[:, 0] -= 0.3 * torch.sign(ref[:, 0])
    assert not torch.isnan(x).any(), "the step read the noise slice of a zero noise coefficient"
    assert torch.equal(x, ref)


# =====================================================================================================================
# Philox4x32-10 + Box-Muller noise of production sampling
# =====================================================================================================================
M0, M1, W0, W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """Random123 Philox4x32-10 on numpy arrays of 32-bit words (carried in uint64)."""
    c = [np.asarray(v, dtype=np.uint64) & MASK for v in ctr]
    k0, k1 = (np.asarray(v, dtype=np.uint64) & MASK for v in key)
    for _ in range(10):
        p0 = np.uint64(M0) * c[0]
        p1 = np.uint64(M1) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & MASK, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & MASK]
        k0 = (k0 + np.uint64(W0)) & MASK
        k1 = (k1 + np.uint64(W1)) & MASK
    return c


def test_philox_restatement_known_answers():
    """The numpy restatement reproduces the Random123 known-answer vectors of philox4x32_10."""
    cases = [((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
             ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
             ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
              (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))]
    for ctr, key, want in cases:
        assert tuple(int(v) for v in philox4x32_10(ctr, key)) == want


def philox_noise(n, Cc, H, W, Fr, nsteps, seed, sample_offset):
    """z[step][b][c][y][x][f] of the sampling kernels: counter (gp_lo, gp_hi, step, 0) with gp = (sample_offset + b) *
    H*W*F + (y*W + x)*F + f, key (seed_lo, seed_hi); u = ((a >> 8) + 0.5) * 2^-24; channel c takes normal c of
    (r cos, r sin) of words (0, 1) then (2, 3).  Float64 Box-Muller on the exact u."""
    plane = H * W * Fr
    b = np.arange(n, dtype=np.uint64)[:, None]
    gp = (np.uint64(sample_offset) + b) * np.uint64(plane) + np.arange(plane, dtype=np.uint64)[None, :]
    out = np.empty((nsteps, n, Cc, plane))
    for s in range(nsteps):
        w = philox4x32_10((gp & MASK, gp >> np.uint64(32), np.full_like(gp, s), np.zeros_like(gp)),
                          (seed & 0xFFFFFFFF, seed >> 32))
        u = [((v >> np.uint64(8)).astype(np.float64) + 0.5) * 2.0 ** -24 for v in w]
        r0, r1 = np.sqrt(-2 * np.log(u[0])), np.sqrt(-2 * np.log(u[2]))
        z = [r0 * np.cos(2 * np.pi * u[1]), r0 * np.sin(2 * np.pi * u[1]), r1 * np.cos(2 * np.pi * u[3]),
             r1 * np.sin(2 * np.pi * u[3])]
        for c in range(Cc):
            out[s, :, c] = z[c]
    return torch.from_numpy(out.reshape(nsteps, n, Cc, H, W, Fr))


def noise_chain(net, n, Cc, H, W, P, Fr, nsteps, mode, seed, offset):
    """A chain whose every step returns exactly its noise: mode 0 {0, 0, 1, ...}, mode 1 {0, 1, 0, 0, 1, ...}."""
    coef = torch.zeros(nsteps, 8)
    if mode == 0:
        coef[:, 2] = 1.0
    else:
        coef[:, 1] = 1.0
        coef[:, 4] = 1.0
    ts = torch.arange(nsteps, 0, -1, dtype=torch.int32) * 7
    g = torch.Generator().manual_seed(4)
    past = torch.randn(n, Cc, H, W, P, generator=g).cuda()
    x = torch.randn(n, Cc, H, W, Fr, generator=g).cuda()
    hist = torch.full((nsteps + 1, n, Cc, H, W, Fr), NAN, device="cuda")
    hist[0] = x
    net.sample_chain(past, x, ts, coef, mode=mode, seed=seed, sample_offset=offset, history=hist)
    torch.cuda.synchronize()
    assert torch.equal(hist[-1], x)
    return hist[1:].cpu()


def small_unet(Cc):
    from crowdmod_ddpm_4d_b200.models.backbones.unet import UNet
    torch.manual_seed(0)
    return UNet(input_channels=Cc, output_channels=Cc, num_res_blocks=2, base_channels=32, base_channels_multiples=[1, 2],
                apply_attention=[True, True], dropout_rate=0.0, time_multiple=4, condition="Past").cuda().eval()


def small_dit(Cc, H, W, P, Fr):
    from crowdmod_ddpm_4d_b200.models.backbones.DiT4D_V4 import DiT4D_V4
    torch.manual_seed(0)
    p = 4 if Cc == 3 else 2                        # t_patch * C * p^2 must be a multiple of 32
    return DiT4D_V4(input_channels=Cc, output_channels=Cc, grid_rows=H, grid_cols=W, past_len=P, future_len=Fr,
                    t_patch_size=2, patch_size=p, hidden_size=64, depth=1, num_heads=2, time_multiple=2).cuda().eval()


@pytest.mark.gpu
@pytest.mark.parametrize("Cc,mode,nsteps", [(3, 0, 5), (4, 1, 4), (4, 0, 6), (3, 1, 4)])
def test_philox_stream_pinned_for_both_backbones(nat, Cc, mode, nsteps):
    """Every z of a UNet and of a DiT chain against the numpy restatement, with a seed whose two 32-bit halves are
    both nonzero and a sample_offset that makes gp cross 2^32 inside the batch.  Box-Muller runs on __logf /
    __sincosf in the kernels, so the bound is max |dz| <= 1e-3 and median |dz| <= 1e-6 (any counter or key fault
    gives O(1) errors; measured on a B200 at 1000 W: max 1.9e-6, median 1.4e-7).  Steps must differ from each other, and the
    two backbones must draw bit-identical noise for the same geometry, seed and offset."""
    n, H, W, P, Fr = 5, 4, 4, 2, 2
    seed = 0x9E3779B97F4A7C15
    plane = H * W * Fr
    offset = (1 << 32) // plane - 2                  # samples offset .. offset+4: gp crosses 2^32 at sample 2
    assert offset * plane < 1 << 32 < (offset + n) * plane
    ref = philox_noise(n, Cc, H, W, Fr, nsteps, seed, offset)
    zs = {}
    for name, net in (("unet", small_unet(Cc)), ("dit", small_dit(Cc, H, W, P, Fr))):
        z = noise_chain(net, n, Cc, H, W, P, Fr, nsteps, mode, seed, offset)
        d = (z.double() - ref).abs()
        print(f"{name} C={Cc} mode={mode}: max |dz| {d.max().item():.2e}, median {d.median().item():.2e}")
        assert d.max().item() <= 1e-3 and d.median().item() <= 1e-6
        for s in range(1, nsteps):
            assert (z[s] != z[s - 1]).all(), "a step repeated the previous step's noise"
        zs[name] = z
    assert torch.equal(zs["unet"], zs["dit"]), "the DiT draws differently from the UNet"


# =====================================================================================================================
# per-timestep tables of sampling against the per-sample conditioning of the forward
# =====================================================================================================================
TABLE_TS = [0, 1, 127, 128, 255, 256, 895, 896, 998, 999]


def table_vs_forward(net, past, x, ts):
    """One step with coef {1, 1, 0, ...} returns x - eps(x, t) with the conditioning from the sampling table; eps from
    it against net(x, t, past), whose conditioning is computed per sample.  Returns the worst per-sample rel-L2."""
    coef = torch.zeros(1, 8)
    coef[0, :2] = 1.0
    worst = 0.0
    for t in ts:
        y = x.clone()
        net.sample_chain(past, y, torch.tensor([t], dtype=torch.int32), coef, mode=0, noise=torch.zeros_like(x)[None])
        with torch.no_grad():
            eps = net(x, torch.full((x.shape[0],), t, dtype=torch.long, device="cuda"), past)
        e_chain = x.double() - y.double()
        for b in range(x.shape[0]):
            worst = max(worst, rel_l2(e_chain[b], eps[b]))
    return worst


@pytest.mark.gpu
def test_dit_mods_table_every_chunk_edge(nat):
    """The DiT's AdaLN vectors of sampling come from mods_table, built in chunks of 128 timesteps (the last chunk of a
    1000-step table holds 104); the forward computes them per sample.  At t on both sides of every chunk edge the
    two eps agree to rel-L2 1e-5 per sample: they differ only in GEMM row position, and the chain's x - eps adds one
    fp32 rounding of x (measured on a B200: 5.9e-8)."""
    from tests._util import build_dit, load_golden
    meta, _ = load_golden("dit_small_b3")
    net, _ = build_dit(meta)
    net = net.cuda().eval()
    kw = meta["kw"]
    g = torch.Generator().manual_seed(8)
    n = 3
    past = torch.randn(n, 3, kw["grid_rows"], kw["grid_cols"], kw["past_len"], generator=g).cuda()
    x = torch.randn(n, 3, kw["grid_rows"], kw["grid_cols"], kw["future_len"], generator=g).cuda()
    worst = table_vs_forward(net, past, x, TABLE_TS)
    print(f"DiT mods table vs per-sample conditioning: worst per-sample eps rel-L2 {worst:.2e}")
    assert worst <= 1e-5


@pytest.mark.gpu
def test_dit_forward_tp8_nq3_vs_oracle(nat):
    """A configuration no golden reaches: 4 channels, patch 4, t_patch 1, past 5, future 3 on the ATC grid, so Tp = 8
    (the temporal kernel's limit), three query slots and Ns = 27.  eps against dit_oracle at rel-L2 1e-3, the model
    tests' bound."""
    from crowdmod_ddpm_4d_b200.models.backbones.DiT4D_V4 import DiT4D_V4
    from oracle import dit_oracle as dto
    torch.manual_seed(3)
    kw = dict(input_channels=4, output_channels=4, grid_rows=12, grid_cols=36, past_len=5, future_len=3, t_patch_size=1,
              patch_size=4, hidden_size=128, depth=2, num_heads=4, time_multiple=4)
    net = DiT4D_V4(**kw)
    sd = dto.randomize_zero_init({k: v.detach().clone() for k, v in net.state_dict().items()}, 3)
    net.load_state_dict(sd)
    net = net.cuda().eval()
    g = torch.Generator().manual_seed(6)
    B = 3
    fut = torch.randn(B, 4, 12, 36, 3, generator=g)
    past = torch.randn(B, 4, 12, 36, 5, generator=g)
    t = torch.tensor([3, 500, 999])
    with torch.no_grad():
        ref = dto.dit_forward(sd, fut, t, past, patch=4, t_patch=1, heads=4, depth=2)
        eps = net(fut.cuda(), t.cuda(), past.cuda()).cpu()
    e = rel_l2(eps, ref)
    print(f"DiT Tp=8 nq=3: eps rel-L2 vs oracle {e:.2e}")
    assert e <= 1e-3
