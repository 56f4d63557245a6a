"""Op-level parity of the UNet forward's fused epilogues (GPU), each launched through the function the model calls,
against float64 PyTorch:

* conv epilogue (cm_op_conv3d_epi -> conv_run_prepare / conv_run_enqueue): time-embedding rows (one table row *t_dev for
  the batch, or one row per sample), bias2, residual, fp16 hi|lo outputs, on every kernel that takes a time embedding
  (conv_umma non-split and split-K, conv_plane, conv_res32);
* the training forward's hi|lo operand pairs (lo_from / lo_from_x): fed the pair of an UNROUNDED fp32 activation the
  conv must match float64 on that fp32 tensor to fp32 accumulation order;
* the GroupNorm records of the plane / res32 epilogues and gn_apply2 merging them (cm_op_gn), the GroupNorm's training
  outputs (stats, Dropout3d scale, hi|lo pairs) on its three routes, and a residual stream with a DC offset;
* the production first conv (pack_first_input_enqueue + the padded weights on the plane / res32 kernel), the UNet's
  fused reverse step (final_conv_kernel) and the time-embedding table (temb_kernel).

Every output starts NaN-filled.  Shapes follow the UNet layers (ATC 12 x 36, HERMES-CR-120 28 x 24, ETH-UCY 8 x 12 at
level 0, 8 frames).  Bounds are stated next to each test with the worst value measured on a B200.
"""
import ctypes as C

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
    return n


def gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def rel_l2(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


def hilo(x32):
    """fp16 hi | lo pair of an fp32 tensor along the last dim: hi = fp16(x), lo = fp16(x - hi)."""
    hi = x32.half()
    return torch.cat([hi, (x32 - hi.float()).half()], dim=-1)


def out_grid(mode, D, H, W):
    if mode == 1:
        return (D - 1) // 2 + 1, (H - 1) // 2 + 1, (W - 1) // 2 + 1
    if mode == 2:
        return 2 * D, 2 * H, 2 * W
    return D, H, W


def conv64(mode, x, w, extra=None, wx=None):
    """float64 conv of channels-last x [B, D, H, W, C] -> [B, od, oh, ow, cout] (weights over the activation dims)."""
    x = x.double().permute(0, 4, 1, 2, 3)
    w = w.double()
    if mode == 0:
        y = F.conv3d(x, w, padding=1)
    elif mode == 1:
        y = F.conv3d(x, w, stride=2, padding=1)
    elif mode == 2:
        y = F.conv3d(F.interpolate(x, scale_factor=2, mode="nearest"), w, padding=1)
    else:
        y = F.conv3d(x, w)
    if extra is not None:
        y = y + F.conv3d(extra.double().permute(0, 4, 1, 2, 3), wx.double()[:, :, None, None, None])
    return y.permute(0, 2, 3, 4, 1)


# =====================================================================================================================
# conv epilogue
# =====================================================================================================================
def run_conv(nat, mode, B, D, H, W, cin, cout, cx=0, impl=0, dup=1, temb=None, bias2=False, resid=0.0, out16=False,
             lo=False, rec=False, seed=0, dc=0.0):
    """One conv through cm_op_conv3d_epi.  temb: None, ("row", t) = row t of a table for the whole batch (t through
    device memory), "sample" = one distinct row per sample.  resid: scale of a random residual (0: none); dc: a DC
    offset added to it.  dup = 2: the operands are the hi|lo pairs of unrounded fp32 activations.  Returns a dict with
    the outputs and the float64 reference (over the fp32 activations for dup = 2, the fp16 ones otherwise)."""
    g = gen(seed)
    od, oh, ow = out_grid(mode, D, H, W)
    k = 1 if mode == 3 else 3
    a32 = torch.randn(B, D, H, W, cin, device="cuda", generator=g)
    w = torch.randn(cout, cin, k, k, k, device="cuda", generator=g) / (cin * k ** 3) ** 0.5
    x32 = wx = None
    if cx:
        x32 = torch.randn(B, od, oh, ow, cx, device="cuda", generator=g)
        wx = torch.randn(cout, cx, device="cuda", generator=g) / cx ** 0.5
    if dup == 2:
        a16, x16, a_ref, x_ref = hilo(a32), (hilo(x32) if cx else None), a32, x32
    else:
        a16, x16 = a32.half(), (x32.half() if cx else None)
        a_ref, x_ref = a16, x16
    e = nat.ConvEpilogue()
    keep = {}
    bias = torch.randn(cout, device="cuda", generator=g)
    e.bias = bias.data_ptr()
    add = bias.double()[None, None, None, None, :].expand(B, 1, 1, 1, cout)
    if bias2:
        b2 = torch.randn(cout, device="cuda", generator=g)
        keep["b2"] = b2
        e.bias2 = b2.data_ptr()
        add = add + b2.double()
    trow = None
    if temb is not None:
        ld = cout + 32
        rows = 5 if temb != "sample" else B
        # large and distinct per row: a wrong row is off by O(10) against outputs of O(1)
        tab = torch.randn(rows, ld, device="cuda", generator=g) * 4 + torch.arange(rows, device="cuda")[:, None] * 3.0
        keep["tab"] = tab
        e.temb, e.temb_ld = tab.data_ptr(), ld
        if temb == "sample":
            e.temb_bstride = ld
            trow = tab[:, :cout].double()[:, None, None, None, :]
        else:
            t = temb[1]
            td = torch.tensor([t], dtype=torch.int32, device="cuda")
            keep["t"] = td
            e.t_dev = td.data_ptr()
            trow = tab[t, :cout].double()[None, None, None, None, :]
        add = add + trow
    res = None
    if resid:
        res = torch.randn(B, od, oh, ow, cout, device="cuda", generator=g) * resid + dc
        e.resid = res.data_ptr()
    out32 = torch.full((B, od, oh, ow, cout), NAN, device="cuda")
    e.out32 = out32.data_ptr()
    o16 = None
    if out16:
        o16 = torch.full((B, od, oh, ow, cout * (2 if lo else 1)), NAN, device="cuda").half()
        e.out16 = o16.data_ptr()
        if lo:
            e.out16_ld, e.out16_lo = 2 * cout, cout
    if dup == 2:
        e.lo_from, e.lo_from_x = cin, cx
    recb = None
    if rec:
        units_max = B * D * H
        recb = torch.full((units_max * cout * 4,), NAN, device="cuda")
        e.stats_rec = recb.data_ptr()
    geom = (C.c_int32 * 4)()
    nat.check(nat.lib().cm_op_conv3d_epi(mode, nat.ptr(a16), B, D, H, W, cin, nat.ptr(x16), cx, dup, nat.ptr(w),
                                         nat.ptr(wx), cout, 2, C.byref(e), impl, geom, nat.current_stream()))
    torch.cuda.synchronize()
    assert nat.lib().cm_device_error() == 0
    ref = conv64(mode, a_ref, w, x_ref, wx) + add
    if res is not None:
        ref = ref + res.double()
    r = dict(out32=out32, out16=o16, ref=ref, geom=tuple(geom), rec=recb, shape=(B, od, oh, ow, cout))
    if rec:
        u = r["geom"][0]
        r["rec"] = recb[:B * u * cout * 4].reshape(B, u, cout, 4)
    return r


def unit_view(x, geom):
    """[B, D, H, W, C] -> [B, units, rows of a unit, C] in the records' unit order."""
    units, nvalid, R, HB = geom
    B, D, H, W, Cc = x.shape
    v = x.reshape(B, D // R, R, H // HB, HB, W, Cc).permute(0, 1, 3, 2, 4, 5, 6)
    v = v.reshape(B, units, R * HB * W, Cc)
    assert v.shape[2] == nvalid
    return v


# (mode, B, D, H, W, cin, cout, cx, impl, temb, bias2, resid) -- the kernel each case reaches is noted
EPI_CASES = [
    (0, 4, 8, 12, 36, 32, 32, 0, 0, "sample", True, True),         # conv_umma non-split (108 M tiles), per-sample rows
    (0, 4, 8, 12, 36, 32, 32, 0, 0, ("row", 3), True, False),      # conv_umma non-split, sampling row t = 3
    (0, 32, 4, 6, 18, 64, 64, 32, 0, "sample", True, True),        # conv_umma non-split, level 1 + match_input slab
    (0, 2, 3, 9, 2, 256, 128, 0, 0, "sample", True, True),         # conv_umma split-K (decoder_blocks.0.conv_1)
    (0, 2, 3, 9, 2, 256, 128, 0, 0, ("row", 4), True, True),       # split-K, sampling row t = 4
    (0, 2, 8, 12, 36, 64, 32, 0, 2, "sample", True, False),        # conv_plane, per-sample rows
    (0, 2, 8, 12, 36, 64, 32, 0, 2, ("row", 2), False, True),      # conv_plane, sampling row
    (0, 40, 8, 12, 36, 32, 32, 0, 2, "sample", True, True),        # conv_plane, more units than SMs (cv per unit)
    (0, 3, 4, 6, 18, 128, 64, 64, 2, "sample", True, False),       # conv_plane, level 1, 2 N tiles
    (0, 2, 8, 12, 36, 32, 32, 0, 3, ("row", 3), True, True),       # conv_res32, sampling row t = 3
    (0, 40, 8, 12, 36, 32, 32, 64, 3, "sample", True, True),       # conv_res32, per-sample rows, many units per CTA
    (0, 3, 8, 28, 24, 32, 32, 0, 3, "sample", False, True),        # conv_res32 at HERMES-CR-120 level 0
]


@pytest.mark.parametrize("case", EPI_CASES, ids=lambda c: "m%d_B%d_%dx%dx%d_ci%d_co%d_x%d_impl%d_%s_b2%d_r%d" % (
    c[:9] + ("t%d" % c[9][1] if isinstance(c[9], tuple) else c[9], c[10], c[11])))
def test_conv_epilogue_temb_bias2_resid(nat, case):
    """Time-embedding row (sampling: row *t_dev with t != 0; training: row b per sample), bias2 and residual against
    float64.  Bound: rel-L2 2e-5 (fp16 activations, hi+lo weights: fp32 accumulation order only), as
    test_gpu_ops.py.  The temb rows differ by O(10) per sample: any wrong row is O(1) relative."""
    mode, B, D, H, W, cin, cout, cx, impl, temb, b2, resid = case
    r = run_conv(nat, mode, B, D, H, W, cin, cout, cx, impl, temb=temb, bias2=b2, resid=1.0 if resid else 0.0,
                 out16=True)
    assert not torch.isnan(r["out32"]).any()
    e = rel_l2(r["out32"], r["ref"])
    print(f"rel-L2 {e:.2e}")
    assert e <= 2e-5
    assert torch.equal(r["out16"], r["out32"].half())


@pytest.mark.parametrize("case", [
    (1, 2, 8, 12, 36, 32, 32, 0),       # encoder_blocks.1.downsample (stride 2)
    (1, 3, 4, 6, 18, 64, 64, 0),        # encoder_blocks.3.downsample
    (2, 2, 3, 9, 2, 128, 128, 0),       # decoder_blocks.2.upsample (8 phase convs, scatter)
    (2, 1, 4, 6, 18, 64, 64, 0),        # decoder_blocks.5.upsample
], ids=lambda c: "m%d_B%d_%dx%dx%d_ci%d_co%d_x%d" % c)
def test_conv_scatter_and_stride2_resid_hilo_out(nat, case):
    """The UpSample scatter and the stride-2 conv as the training forward runs them: hi|lo operand pairs, a residual,
    fp16 hi|lo outputs (the model gives them no time embedding).  rel-L2 2e-5 against float64 on the unrounded fp32
    activations; hi == fp16(out32) and lo == fp16(out32 - hi) bit for bit."""
    mode, B, D, H, W, cin, cout, cx = case
    r = run_conv(nat, mode, B, D, H, W, cin, cout, cx, 0, dup=2, bias2=True, resid=1.0, out16=True, lo=True)
    e = rel_l2(r["out32"], r["ref"])
    print(f"rel-L2 {e:.2e}")
    assert e <= 2e-5
    o, c = r["out32"], cout
    assert torch.equal(r["out16"][..., :c], o.half())
    assert torch.equal(r["out16"][..., c:], (o - o.half().float()).half())


# (mode, B, D, H, W, cin, cout, cx, impl)
HILO_CASES = [
    (0, 3, 3, 9, 2, 128, 128, 64, 0),    # conv_umma: encoder_blocks.4.conv_2 + match_input slab (split-K)
    (0, 32, 4, 6, 18, 64, 64, 32, 0),    # conv_umma non-split + slab
    (3, 3, 3, 9, 2, 128, 384, 0, 0),     # attention in_proj (1x1x1)
    (0, 2, 8, 12, 36, 32, 32, 96, 2),    # conv_plane: decoder_blocks.6.conv_2 + match_input (3 slabs)
    (0, 2, 4, 6, 18, 128, 64, 64, 2),    # conv_plane, level 1 + 2 slabs
    (0, 1, 4, 6, 18, 192, 64, 0, 2),     # conv_plane, R = 2 planes per unit
]


@pytest.mark.parametrize("case", HILO_CASES, ids=lambda c: "m%d_B%d_%dx%dx%d_ci%d_co%d_x%d_impl%d" % c)
def test_hilo_operands_exact_to_fp32(nat, case):
    """The training forward's hi|lo operand pairs of an UNROUNDED fp32 activation (main source and the 1x1x1 slab):
    with lo_from / lo_from_x the kernel skips only the lo x lo_w product (2^-22), so the conv matches float64 on the
    fp32 tensor to fp32 accumulation order.  Bound rel-L2 2e-5 (dropping hi x lo_w as well costs ~2.4e-4; fp16-rounded
    operands ~3e-4).  hi|lo outputs bit-exact against out32."""
    mode, B, D, H, W, cin, cout, cx, impl = case
    r = run_conv(nat, mode, B, D, H, W, cin, cout, cx, impl, dup=2, temb="sample" if mode == 0 else None, resid=1.0,
                 out16=True, lo=True)
    e = rel_l2(r["out32"], r["ref"])
    print(f"rel-L2 {e:.2e}")
    assert e <= 2e-5
    o = r["out32"]
    assert torch.equal(r["out16"][..., :cout], o.half())
    assert torch.equal(r["out16"][..., cout:], (o - o.half().float()).half())


# =====================================================================================================================
# GroupNorm records (plane / res32 epilogues)
# =====================================================================================================================
REC_CASES = [
    (2, 8, 12, 36, 32, 32, 0, 3),        # res32, ATC level 0 (HB = 3)
    (150, 8, 12, 36, 32, 32, 0, 3),      # res32, many units per persistent CTA
    (1, 3, 12, 36, 32, 32, 0, 3),        # res32, odd depth
    (5, 8, 8, 12, 32, 32, 32, 3),        # res32, ETH-UCY level 0 + slab
    (2, 8, 12, 36, 64, 32, 0, 2),        # plane
    (1, 4, 6, 18, 192, 64, 0, 2),        # plane, R = 2 planes per unit
    (3, 3, 12, 36, 64, 32, 0, 2),        # plane, odd depth and batch
    (40, 8, 12, 36, 32, 32, 0, 2),       # plane, several units per persistent CTA
    (2, 4, 6, 18, 128, 64, 64, 2),       # plane, level 1, 2 N tiles
]


def check_records(r):
    """shift == out32 at the unit's first row (bit for bit); sum / sum of squares of (out32 - shift) over the unit's rows
    within 1e-5 of sum |.| / sum (.)^2 in float64, plus the rounding of the stored values: the kernels sum the values
    before the column constants (bias + temb) are added, and out32 and the shift each carry one rounding of that
    addition, up to 2^-24 |out32| (measured on a B200: 1.8e-5 of sum |.| from rounding alone where temb rows reach
    450); the fourth field 0."""
    rec = r["rec"]
    assert not torch.isnan(rec).any(), "unwritten records"
    ov = unit_view(r["out32"], r["geom"])                       # [B, U, n, C]
    shift = rec[..., 0]
    assert torch.equal(shift, ov[:, :, 0, :]), "record shift is not the unit's first value"
    d = ov.double() - shift.double()[:, :, None, :]
    rnd = (ov.double().abs() + shift.double().abs()[:, :, None, :]) * 2.0 ** -24   # per-element rounding bound
    s1, a1, s2 = d.sum(2), d.abs().sum(2), (d * d).sum(2)
    t1 = 1e-5 * a1 + rnd.sum(2)
    t2 = 1e-5 * s2 + 2 * (d.abs() * rnd).sum(2) + (rnd * rnd).sum(2)
    e1 = ((rec[..., 1].double() - s1).abs() / t1.clamp_min(1e-30)).max().item()
    e2 = ((rec[..., 2].double() - s2).abs() / t2.clamp_min(1e-30)).max().item()
    print(f"records: worst sum err {e1:.2f}, sumsq err {e2:.2f} of their bounds")
    assert e1 <= 1.0 and e2 <= 1.0
    assert (rec[..., 3] == 0).all()


@pytest.mark.parametrize("case", REC_CASES, ids=lambda c: "B%d_%dx%dx%d_ci%d_co%d_x%d_impl%d" % c)
def test_conv_records(nat, case):
    B, D, H, W, cin, cout, cx, impl = case
    r = run_conv(nat, 0, B, D, H, W, cin, cout, cx, impl, temb="sample", bias2=True, resid=1.0, rec=True)
    units, nvalid, R, HB = r["geom"]
    print(f"geometry: {units} units of {R} x {HB} rows")
    assert units == (D // R) * (H // HB) and nvalid == R * HB * W
    assert rel_l2(r["out32"], r["ref"]) <= 2e-5
    check_records(r)


# =====================================================================================================================
# GroupNorm: three routes, training outputs
# =====================================================================================================================
def gn_ref(x, gamma, beta, silu, drop):
    """float64 GroupNorm(8) over [B, pixels, C] (+SiLU) (*drop [B][C]); also (mean, rstd) [B, 8, 2]."""
    B, P, Cc = x.shape
    xd = x.double()
    grp = xd.reshape(B, P, 8, Cc // 8)
    mean = grp.mean(dim=(1, 3))
    var = grp.var(dim=(1, 3), unbiased=False)
    rstd = 1.0 / torch.sqrt(var + 1e-5)
    y = F.group_norm(xd.permute(0, 2, 1), 8, gamma.double(), beta.double(), 1e-5).permute(0, 2, 1)
    if silu:
        y = F.silu(y)
    if drop is not None:
        y = y * drop.double()[:, None, :]
    return y, torch.stack([mean, rstd], dim=-1), var.sqrt()


def run_gn(nat, src0, src1, gamma, beta, silu=1, dup=1, drop=None, recs=(None, None), stats=True, raw=True):
    B, P, c0 = src0.shape
    c1 = src1.shape[2] if src1 is not None else 0
    Cc = c0 + c1
    a = nat.GnArgs()
    a.src0, a.c0 = src0.data_ptr(), c0
    if src1 is not None:
        a.src1, a.c1 = src1.data_ptr(), c1
    a.gamma, a.beta, a.B, a.pixels, a.eps, a.silu = gamma.data_ptr(), beta.data_ptr(), B, P, 1e-5, silu
    if drop is not None:
        a.drop_scale, a.drop_ld = drop.data_ptr(), drop.shape[1]
    out = torch.full((B, P, dup * Cc), NAN, device="cuda").half()
    a.out_norm16, a.dup = out.data_ptr(), dup
    rw = None
    if raw:
        rw = torch.full((B, P, dup * Cc), NAN, device="cuda").half()
        a.out_raw16 = rw.data_ptr()
    st = None
    if stats:
        st = torch.full((B, 8, 2), NAN, device="cuda")
        a.stats = st.data_ptr()
    for i, rr in enumerate(recs):
        if rr is not None:
            setattr(a, "rec%d" % i, rr[0].data_ptr())
            setattr(a, "rec%d_units" % i, rr[1][0])
            setattr(a, "rec%d_nvalid" % i, rr[1][1])
    nl = C.c_int32(0)
    nat.check(nat.lib().cm_op_gn(C.byref(a), C.byref(nl), nat.current_stream()))
    torch.cuda.synchronize()
    return out, rw, st, nl.value


def check_gn(out, rw, st, x, gamma, beta, silu, dup, drop, tag=""):
    """dup = 1: the fp16 bounds of test_gpu_ops.py::test_gn_silu (rel-L2 4e-4, max 2e-3 of max(1, |ref|)); dup = 2:
    hi + lo within rel-L2 1e-5.  stats: mean within 1e-6 of the group's standard deviation (+ four fp32 ulps of the
    mean), rstd within 1e-5 relative.  raw: the fp16 copy (dup = 2: hi | lo pair) bit for bit."""
    ref, sref, sd = gn_ref(x, gamma, beta, silu, drop)
    Cc = x.shape[2]
    if dup == 2:
        got = out[..., :Cc].double() + out[..., Cc:].double()
        e = rel_l2(got, ref)
        print(f"{tag} dup=2 rel-L2 {e:.2e}")
        assert e <= 1e-5
    else:
        e = rel_l2(out.float(), ref)
        m = (out.double() - ref).abs().max().item()
        print(f"{tag} dup=1 rel-L2 {e:.2e}, max {m:.2e}")
        assert e <= 4e-4
        assert m <= 2e-3 * max(1.0, ref.abs().max().item())
    if st is not None:
        em = ((st[..., 0].double() - sref[..., 0]).abs() / (1e-6 * sd + 2.0 ** -21 * sref[..., 0].abs())).max().item()
        er = ((st[..., 1].double() - sref[..., 1]).abs() / sref[..., 1]).max().item()
        print(f"{tag} stats: mean err {em:.2f} of its bound, rstd rel err {er:.2e}")
        assert em <= 1.0 and er <= 1e-5
    if rw is not None:
        assert torch.equal(rw, hilo(x) if dup == 2 else x.half())


# (B, pixels, c0, c1, expected launches): gn_small (one CTA per sample) and gn_stats2 + gn_apply2
ROUTES = {
    "small": (3, 54, 128, 0, 1),            # encoder_blocks.4 GroupNorm (3 x 9 x 2 pixels)
    "small_concat": (2, 54, 128, 128, 1),   # decoder_blocks.0: skip concat
    "stats2": (2, 3456, 32, 32, 2),         # decoder_blocks.7 at ATC level 0 (8 x 12 x 36)
    "stats2_hermes": (1, 5376, 64, 32, 2),  # HERMES-CR-120 level 0, 96 channels
}


@pytest.mark.parametrize("route", sorted(ROUTES))
@pytest.mark.parametrize("dup", [1, 2])
@pytest.mark.parametrize("drop", [False, True])
def test_gn_routes_training_outputs(nat, route, dup, drop):
    """gn_small / gn_stats2 + gn_apply2 with the training forward's outputs: (mean, rstd), the Dropout3d scale (after
    the SiLU), hi|lo pairs for out_norm and out_raw.  The launch count identifies the route."""
    B, P, c0, c1, launches = ROUTES[route]
    g = gen(7)
    s0 = torch.randn(B, P, c0, device="cuda", generator=g) * 2 + 0.5
    s1 = torch.randn(B, P, c1, device="cuda", generator=g) * 0.5 - 1.0 if c1 else None
    Cc = c0 + c1
    gamma = torch.randn(Cc, device="cuda", generator=g)
    beta = torch.randn(Cc, device="cuda", generator=g)
    ds = None
    if drop:
        ds = torch.full((B, Cc + 32), NAN, device="cuda")
        ds[:, :Cc] = (torch.rand(B, Cc, device="cuda", generator=g) > 0.2).float() / 0.8
    out, rw, st, nl = run_gn(nat, s0, s1, gamma, beta, 1, dup, ds)
    assert nl == launches
    x = torch.cat([s0, s1], dim=2) if c1 else s0
    check_gn(out, rw, st, x, gamma, beta, 1, dup, ds[:, :Cc] if drop else None, route)


def conv_out_with_records(nat, B, cin, impl, seed, temb="sample", dc=0.0, resid=1.0, geo=(8, 12, 36)):
    D, H, W = geo
    r = run_conv(nat, 0, B, D, H, W, cin, 32, 0, impl, temb=temb, bias2=True, resid=resid, rec=True, seed=seed, dc=dc)
    return r


@pytest.mark.parametrize("src", ["res32", "plane", "concat"])
@pytest.mark.parametrize("dup", [1, 2])
@pytest.mark.parametrize("drop", [False, True])
def test_gn_from_records(nat, src, dup, drop):
    """gn_apply2 from the producing convs' records (no statistics pass: one launch): one conv's records, or a skip concat
    whose sources come from conv_res32 (units of 3 rows) and conv_plane (its own unit geometry).  Against float64
    F.group_norm of the convs' fp32 outputs; bounds of check_gn."""
    B = 3
    parts = []
    if src in ("res32", "concat"):
        parts.append(conv_out_with_records(nat, B, 32, 3, 1))
    if src in ("plane", "concat"):
        parts.append(conv_out_with_records(nat, B, 64, 2, 2))
    if src == "concat":
        print("unit geometries:", parts[0]["geom"], parts[1]["geom"])
    xs = [p["out32"].reshape(B, -1, 32) for p in parts]
    recs = [(p["rec"], p["geom"]) for p in parts] + [None]
    g = gen(9)
    Cc = 32 * len(xs)
    gamma = torch.randn(Cc, device="cuda", generator=g)
    beta = torch.randn(Cc, device="cuda", generator=g)
    ds = (torch.rand(B, Cc, device="cuda", generator=g) > 0.2).float() / 0.8 if drop else None
    out, rw, st, nl = run_gn(nat, xs[0], xs[1] if len(xs) > 1 else None, gamma, beta, 1, dup, ds, recs=recs[:2])
    assert nl == 1
    x = torch.cat(xs, dim=2)
    check_gn(out, rw, st, x, gamma, beta, 1, dup, ds, src)


@pytest.mark.parametrize("impl", [3, 2], ids=["res32", "plane"])
@pytest.mark.parametrize("k", [0, 30, 100, 1000])
def test_gn_records_dc_offset(nat, impl, k):
    """A residual stream k * sigma + N(0, sigma^2) shared by every channel: the GroupNorm from the records must meet the
    bound the statistics route meets on the same data (check_gn, dup = 1).  The records' shift is the unit's first
    value, so their sums do not cancel; with a shift of bias + temb far from the data, sum((v - s)^2) - sum(v - s)^2 / n
    lost k^2 * 2^-24 of the unit variance (median 0.12 at k = 1000)."""
    B = 2
    r = conv_out_with_records(nat, B, 32 if impl == 3 else 64, impl, 11, dc=float(k))
    x = r["out32"].reshape(B, -1, 32)
    g = gen(12)
    gamma = torch.rand(32, device="cuda", generator=g) + 0.5
    beta = torch.randn(32, device="cuda", generator=g)
    a, _, _, n_stats = run_gn(nat, x, None, gamma, beta, 0, 1, stats=False, raw=False)
    assert n_stats == 2
    check_gn(a, None, None, x, gamma, beta, 0, 1, None, f"stats route k={k}")
    b, _, st, n_rec = run_gn(nat, x, None, gamma, beta, 0, 1, recs=[(r["rec"], r["geom"]), None], raw=False)
    assert n_rec == 1
    check_gn(b, None, st, x, gamma, beta, 0, 1, None, f"records route k={k}")


# =====================================================================================================================
# production first conv
# =====================================================================================================================
@pytest.mark.parametrize("geo", [(2, 12, 36, 5, 3), (1, 28, 24, 5, 3), (3, 8, 12, 4, 4)], ids=["atc", "hermes", "eth"])
@pytest.mark.parametrize("cin", [1, 3, 4])
@pytest.mark.parametrize("dup", [1, 2])
def test_first_conv_packed(nat, geo, cin, dup):
    """pack_first_input_enqueue -> the conv over the weights zero-padded to 32 input channels (res32 for dup = 1, plane
    for dup = 2), as the model runs UNet.first.  Against float64 F.conv3d on cat(past, future): dup = 2 on the fp32
    input (rel-L2 2e-5), dup = 1 on its fp16 rounding (2e-5).  The packed operand is bit-exact (hi | lo halves, zero
    channels), and its records feed encoder_blocks.0's GroupNorm (check_gn)."""
    B, H, W, P, Fu = geo
    cout = 32
    g = gen(13)
    x = torch.randn(B, cin, H, W, Fu, device="cuda", generator=g) * 2
    past = torch.randn(B, cin, H, W, P, device="cuda", generator=g) * 2
    w = torch.randn(cout, cin, 3, 3, 3, device="cuda", generator=g) / (27 * cin) ** 0.5
    b = torch.randn(cout, device="cuda", generator=g)
    L = P + Fu
    out = torch.full((B, L, H, W, cout), NAN, device="cuda")
    in16 = torch.full((B, L, H, W, 32 * dup), NAN, device="cuda").half()
    rec = torch.full((B * L * H * cout * 4,), NAN, device="cuda")
    geom = (C.c_int32 * 4)()
    nat.check(nat.lib().cm_op_first_conv_packed(nat.ptr(x), nat.ptr(past), nat.ptr(w), nat.ptr(b), B, H, W, P, Fu, cin,
                                                cout, dup, nat.ptr(out), nat.ptr(in16), nat.ptr(rec), geom,
                                                nat.current_stream()))
    torch.cuda.synchronize()
    assert nat.lib().cm_device_error() == 0
    xin = torch.cat([past, x], dim=4)                                    # [B, cin, H, W, L]
    xcl = xin.permute(0, 4, 2, 3, 1)                                     # [B, L, H, W, cin]
    want16 = torch.zeros(B, L, H, W, 32 * dup, device="cuda").half()
    want16[..., :cin] = xcl.half()
    if dup == 2:
        want16[..., 32:32 + cin] = (xcl - xcl.half().float()).half()
    assert torch.equal(in16, want16)
    xr = xin if dup == 2 else xin.half().float()
    ref = F.conv3d(xr.double(), w.double(), b.double(), padding=1).permute(0, 4, 2, 3, 1)
    e = rel_l2(out, ref)
    print(f"first conv rel-L2 {e:.2e}, geometry {tuple(geom)}")
    assert e <= 2e-5
    units = geom[0]
    assert units > 0
    r = dict(out32=out, rec=rec[:B * units * cout * 4].reshape(B, units, cout, 4), geom=tuple(geom))
    check_records(r)
    gamma = torch.rand(cout, device="cuda", generator=g) + 0.5
    beta = torch.randn(cout, device="cuda", generator=g)
    xs = out.reshape(B, -1, cout)
    o, rw, st, nl = run_gn(nat, xs, None, gamma, beta, 1, dup, recs=[(r["rec"], r["geom"]), None])
    assert nl == 1
    check_gn(o, rw, st, xs, gamma, beta, 1, dup, None, "encoder_blocks.0 GroupNorm")


# =====================================================================================================================
# final conv + reverse step
# =====================================================================================================================
def update_ref(x, eps, z, cf, mode):
    """DDPM.step / DDIM eq. 12 + sign guidance on channel 0 in float64 (as test_gpu_dit_ops.py), with the magnitude of
    the update's terms."""
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


def run_final(nat, act16, act_ld, act_lo, w, b, geo, x=None, coef=None, nsteps=0, step=0, mode=0, noise=None, seed=0,
              offset=0, history=None):
    B, H, W, P, Fu, cin, cout = geo
    eps = torch.full((B, cout, H, W, Fu), NAN, device="cuda")
    nat.check(nat.lib().cm_op_final_conv_step(nat.ptr(act16), act_ld, act_lo, nat.ptr(w), nat.ptr(b), nat.ptr(eps), B, H,
                                              W, P + Fu, P, cin, cout, nat.ptr(x), nat.ptr(coef), nsteps, step, mode,
                                              nat.ptr(noise), seed, offset, nat.ptr(history), nat.current_stream()))
    torch.cuda.synchronize()
    return eps


FINAL_GEOS = [(2, 12, 36, 5, 3, 32, 3), (1, 8, 12, 4, 4, 64, 4), (3, 4, 4, 2, 2, 32, 2)]


@pytest.mark.parametrize("geo", FINAL_GEOS, ids=lambda g: "B%d_%dx%d_P%dF%d_ci%d_co%d" % g)
@pytest.mark.parametrize("mode", [0, 1], ids=["ddpm", "ddim"])
@pytest.mark.parametrize("guided", [False, True])
@pytest.mark.parametrize("philox", [False, True])
def test_final_conv_step(nat, geo, mode, guided, philox):
    """final_conv_kernel's fused reverse step: eps against float64 F.conv3d on the hi|lo activation pair (act_lo,
    rows of 2*cin + 32: rel-L2 1e-5); x_next against the float64 update of the kernel's own eps within 8 fp32 ulps of
    the update's terms (injected noise) or + 1e-4 of the noise term (Philox: Box-Muller on fast intrinsics, pinned by
    test_gpu_dit_ops.py); history slot step + 1 written, every other slot untouched; guidance on channel 0 only."""
    from tests.test_gpu_dit_ops import philox_noise
    B, H, W, P, Fu, cin, cout = geo
    L = P + Fu
    g = gen(19 + mode)
    a32 = torch.randn(B, L, H, W, cin, device="cuda", generator=g)
    ld = 2 * cin + 32
    act = torch.full((B, L, H, W, ld), NAN, device="cuda").half()
    act[..., :2 * cin] = hilo(a32)
    w = torch.randn(cout, cin, 3, 3, 3, device="cuda", generator=g) / (27 * cin) ** 0.5
    b = torch.randn(cout, device="cuda", generator=g)
    nsteps, step = 4, 2
    coef = torch.rand(nsteps, 8, device="cuda", generator=g) + 0.25
    if not guided:
        coef[:, 5] = 0.0
    shape = (B, cout, H, W, Fu)
    x0 = torch.randn(shape, device="cuda", generator=g)
    seed, offset = 0x9E3779B97F4A7C15, 7
    if philox:
        noise = None
        z = philox_noise(B, cout, H, W, Fu, nsteps, seed, offset)[step].cuda()
    else:
        noise = torch.randn(nsteps, *shape, device="cuda", generator=g)
        z = noise[step]
    hist0 = torch.randn(nsteps + 1, *shape, device="cuda", generator=g)
    x, hist = x0.clone(), hist0.clone()
    eps = run_final(nat, act, ld, cin, w, b, geo, x, coef, nsteps, step, mode, noise, seed, offset, hist)
    ref_eps = F.conv3d(a32.double().permute(0, 4, 2, 3, 1), w.double(), b.double(), padding=1)[..., P:]
    assert rel_l2(eps, ref_eps) <= 1e-5
    ref, mag = update_ref(x0, eps, z, coef[step].tolist(), mode)
    cz = float(coef[step, 2] if mode == 0 else coef[step, 4])
    tol = 8 * 2.0 ** -24 * mag + (cz * 1e-4 if philox else 0.0)
    err = (x.double() - ref).abs()
    print(f"worst {(err / mag).max().item() * 2 ** 24:.1f} fp32 ulps of the terms")
    assert (err <= tol).all()
    assert torch.equal(hist[step + 1], x)
    keep = [i for i in range(nsteps + 1) if i != step + 1]
    assert torch.equal(hist[keep], hist0[keep])


@pytest.mark.parametrize("mode", [0, 1], ids=["ddpm", "ddim"])
def test_final_conv_zero_noise_coef(nat, mode):
    """A step whose noise coefficient is 0 must not read its noise slice (NaN here); the step maps x to itself (DDPM
    {1, 0, 0}, DDIM {0, 1, 1, 0, 0}) plus the sign guidance on channel 0, exactly."""
    geo = (2, 8, 12, 4, 4, 32, 3)
    B, H, W, P, Fu, cin, cout = geo
    g = gen(23)
    act = torch.randn(B, P + Fu, H, W, cin, device="cuda", generator=g).half()
    w = torch.randn(cout, cin, 3, 3, 3, device="cuda", generator=g) / (27 * cin) ** 0.5
    b = torch.randn(cout, device="cuda", generator=g)
    coef = torch.rand(2, 8, device="cuda", generator=g) + 0.25
    if mode == 0:
        coef[0, :3] = torch.tensor([1.0, 0.0, 0.0])
        coef[0, 4] = 1.0                 # DDIM's noise coefficient: ignored in DDPM mode
    else:
        coef[0, :5] = torch.tensor([0.0, 1.0, 1.0, 0.0, 0.0])
    coef[0, 5] = 0.3
    shape = (B, cout, H, W, Fu)
    noise = torch.randn(2, *shape, device="cuda", generator=g)
    noise[0] = NAN
    x0 = torch.randn(shape, device="cuda", generator=g)
    x0[:, :, :, :4] = 0.0
    x = x0.clone()
    run_final(nat, act, 0, 0, w, b, geo, x, coef, 2, 0, mode, noise)
    ref = x0.clone()
    ref[:, 0] -= 0.3 * torch.sign(ref[:, 0])
    assert not torch.isnan(x).any(), "the step read the noise slice of a zero noise coefficient"
    assert torch.equal(x, ref)


# =====================================================================================================================
# time-embedding MLP: the sampling table and the per-sample rows
# =====================================================================================================================
def temb_setup(base=32, E=128, couts=(32, 64, 128, 96), seed=29, T=1000):
    g = gen(seed)
    p = dict(table=torch.randn(T, base, device="cuda", generator=g),
             w1=torch.randn(E, base, device="cuda", generator=g) / base ** 0.5,
             b1=torch.randn(E, device="cuda", generator=g),
             w2=torch.randn(E, E, device="cuda", generator=g) / E ** 0.5,
             b2=torch.randn(E, device="cuda", generator=g))
    p["wd"] = [torch.randn(c, E, device="cuda", generator=g) / E ** 0.5 for c in couts]
    p["bd"] = [torch.randn(c, device="cuda", generator=g) for c in couts]
    offs, o = [], 0
    for c in couts:
        offs.append(o)
        o += c
    p["offs"], p["couts"], p["ld"], p["base"], p["E"] = offs, list(couts), o + 8, base, E
    return p


def temb_ref(p, t):
    """float64 Linear -> SiLU -> Linear, then SiLU -> each block's dense_1; also e, h1, h2."""
    d = {k: v.double() for k, v in p.items() if isinstance(v, torch.Tensor)}
    e = d["table"][t]
    h1 = e @ d["w1"].T + d["b1"]
    h2 = F.silu(h1) @ d["w2"].T + d["b2"]
    outs = [F.silu(h2) @ wd.double().T + bd.double() for wd, bd in zip(p["wd"], p["bd"])]
    return torch.cat(outs, dim=1), e, h1, h2


def run_temb(nat, p, t, rows, saves=False):
    nb = len(p["couts"])
    out = torch.full((rows, p["ld"]), NAN, device="cuda")
    se = sh1 = sh2 = None
    if saves:
        se = torch.full((rows, p["base"]), NAN, device="cuda")
        sh1 = torch.full((rows, p["E"]), NAN, device="cuda")
        sh2 = torch.full((rows, p["E"]), NAN, device="cuda")
    wd = (C.c_void_p * nb)(*[x.data_ptr() for x in p["wd"]])
    bd = (C.c_void_p * nb)(*[x.data_ptr() for x in p["bd"]])
    couts = (C.c_int32 * nb)(*p["couts"])
    offs = (C.c_int32 * nb)(*p["offs"])
    nat.check(nat.lib().cm_op_temb(nat.ptr(p["table"]), nat.ptr(p["w1"]), nat.ptr(p["b1"]), nat.ptr(p["w2"]),
                                   nat.ptr(p["b2"]), wd, bd, couts, offs, nb, p["base"], p["E"], nat.ptr(t), rows,
                                   nat.ptr(out), p["ld"], nat.ptr(se), nat.ptr(sh1), nat.ptr(sh2), nat.current_stream()))
    torch.cuda.synchronize()
    return out, se, sh1, sh2


def test_temb_sampling_table(nat):
    """The sampling table (t = NULL, one row per timestep, as cm_unet_pack(build_time_table=1) builds it): rows t = 0, 1,
    127, 128, 255, 256, 998, 999 within rel 1e-5 (per row) of the float64 MLP; the padding columns stay untouched."""
    p = temb_setup()
    out, _, _, _ = run_temb(nat, p, None, 1000)
    n = sum(p["couts"])
    assert torch.isnan(out[:, n:]).all()
    for t in (0, 1, 127, 128, 255, 256, 998, 999):
        ref, _, _, _ = temb_ref(p, torch.tensor([t]))
        e = rel_l2(out[t, :n], ref[0])
        assert e <= 1e-5, f"row {t}: rel {e:.2e}"


def test_temb_per_sample_with_saves(nat):
    """The per-sample rows of a training batch (distinct t, out of order) and the saved e (bit-exact table rows), h1,
    h2 (the pre-activations, rel 1e-5)."""
    p = temb_setup(base=64, E=256, couts=(64, 128, 256), seed=31)
    t = torch.tensor([999, 0, 500, 17, 256, 1, 998], dtype=torch.int64, device="cuda")
    out, se, sh1, sh2 = run_temb(nat, p, t, len(t), saves=True)
    n = sum(p["couts"])
    ref, e, h1, h2 = temb_ref(p, t)
    assert torch.equal(se, p["table"][t])
    for name, got, want in (("out", out[:, :n], ref), ("h1", sh1, h1), ("h2", sh2, h2)):
        for r in range(len(t)):
            er = rel_l2(got[r], want[r])
            assert er <= 1e-5, f"{name} row {r}: rel {er:.2e}"
