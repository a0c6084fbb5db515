"""-m gpu: every kernel of the stage-1 decoder launched alone, in both operand types (bf16, and fp32 rounded to TF32),
at every shape the two decoders of oracle/s1_oracle.py launch (IMAGENET_S1, the stage 1 of all shipped YAMLs, and
TINY_S1) plus the edges where a kernel's indexing changes, against an fp64 restatement of the same operation on the same
operands.  The hooks (hq_debug_s1_*) run the host functions the decode calls, so the launch geometry is the decoder's.

Sentinels.  Every output buffer is larger than the tensor the launch owns and is filled with a NaN bit pattern first;
whatever the kernel must not write has to hold the pattern afterwards, bit for bit.  Inputs that are read only in the
interior (GroupNorm, resample, attention) carry NaN in their padding border, so a border read shows up as a NaN.

Borders.  Every writer of a convolution operand (GroupNorm, resample, quant) writes +0 at every border position: the
activation buffers are reused across resolutions and a 3x3 tap reads the border as the convolution's zero padding."""
import math

import pytest
import torch
from torch.nn import functional as F

from oracle import s1_oracle as S1
from tests import tf32_emulation as T

pytestmark = pytest.mark.gpu

PAT = {torch.bfloat16: 0x7FA5, torch.float32: 0x7FA5A5A5}        # NaN bit patterns
DTYPES = [pytest.param(torch.bfloat16, id="bf16"), pytest.param(torch.float32, id="tf32")]
MANT = {torch.bfloat16: 7, torch.float32: 10}                      # explicit mantissa bits of the operand type
EXTRA = 4096                                                       # sentinel elements past every output tensor
TILES = (0, 32, 64, 128, 256)
DEV = "cuda"


# ------------------------------------------------------------------------------------------------
# shapes: every launch of the decode, from the oracle's decoder plan
# ------------------------------------------------------------------------------------------------
def _launches(cfg):
    """dict of the decode's launches for `cfg`, in decode order, duplicates removed:
    conv (res, Cin, Cout, k, mode, in-place residual), norm (res, C, swish), resample (res, C, up), attn (res, C),
    quant (E, hb, n_embed)."""
    lat, E = cfg.latent_res, cfg.embed_dim
    top = cfg.ch * cfg.ch_mult[-1]
    out = {"conv": [], "norm": [], "resample": [], "attn": [], "quant": [(E, lat, cfg.n_embed)]}

    def add(kind, item):
        if item not in out[kind]:
            out[kind].append(item)

    def resblock(r, cin, cout):
        add("norm", (r, cin, 1))
        add("conv", (r, cin, cout, 3, 0, False))
        add("norm", (r, cout, 1))
        if cin != cout:
            add("resample", (r, cin, 1))                               # operand copy of x for nin_shortcut
            add("conv", (r, cin, cout, 1, 0, False))
        add("conv", (r, cout, cout, 3, 0, True))                       # conv2 + the residual, in place

    def attnblock(r, c):
        add("norm", (r, c, 0))
        add("conv", (r, c, 3 * c, 1, 1, False))                       # fused q | k | v
        add("attn", (r, c))
        add("conv", (r, c, c, 1, 0, True))                             # proj_out + x, in place

    add("conv", (lat, 2 * E, cfg.z_channels, 1, 0, False))             # post_quant_conv_b
    add("resample", (lat, cfg.z_channels, 1))
    add("conv", (lat, cfg.z_channels, top, 3, 0, False))               # conv_in
    resblock(lat, top, top)
    attnblock(lat, top)
    resblock(lat, top, top)
    for _, blocks, up_ch, r in S1.decoder_plan(cfg):
        for cin, cout, has_attn in blocks:
            resblock(r, cin, cout)
            if has_attn:
                attnblock(r, cout)
        add("resample", (r, up_ch, 2))
        add("conv", (2 * r, up_ch, up_ch, 3, 0, False))                # upsample conv
    add("norm", (cfg.resolution, cfg.ch * cfg.ch_mult[0], 1))          # norm_out
    add("conv", (cfg.resolution, cfg.ch * cfg.ch_mult[0], cfg.out_ch, 3, 2, False))   # conv_out, image mode
    return out


def _all(kind):
    seen = []
    for cfg in (S1.TINY_S1, S1.IMAGENET_S1):
        for item in _launches(cfg)[kind]:
            if item not in seen:
                seen.append(item)
    return seen


def test_shape_lists_cover_both_decoders():
    """The lists below are derived, not copied: check them against the parameter shapes of both decoders."""
    for cfg in (S1.TINY_S1, S1.IMAGENET_S1):
        shapes = S1.param_shapes(cfg)
        L = _launches(cfg)
        convs = {(cin, cout, k) for _, cin, cout, k, mode, _ in L["conv"] if mode != 1}
        want = {(s[1], s[0], s[2]) for n, s in shapes.items() if n.endswith(".weight") and len(s) == 4
                and not n.endswith((".q.weight", ".k.weight", ".v.weight"))}
        assert convs == want
        norms = {c for _, c, _ in L["norm"]}
        assert norms == {s[0] for n, s in shapes.items() if ".norm" in n and n.endswith(".weight")}
        assert len(L["attn"]) == 1 and L["quant"] == [(cfg.embed_dim, cfg.latent_res, cfg.n_embed)]
    assert (16, 512) in _all("attn") and (4, 128) in _all("attn")
    assert (256, 128, 128, 3, 0, False) in _all("conv")                # 521 row blocks at B = 2


# ------------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------------
def _round(t, dt):
    """fp32 -> the operand type as the kernels round: bf16 nearest-even, or fp32 rounded to TF32 (ties away)."""
    return t.to(torch.bfloat16) if dt == torch.bfloat16 else T.round_tf32(t)


def _bits(t):
    return t.view(torch.int16) if t.dtype == torch.bfloat16 else t.view(torch.int32)


def _sentinel(shape, dt):
    """(buffer, view): a NaN-patterned buffer EXTRA elements longer than the tensor `shape` it starts with."""
    n = math.prod(shape)
    idt = torch.int16 if dt == torch.bfloat16 else torch.int32
    buf = torch.full((n + EXTRA,), PAT[dt], dtype=idt, device=DEV).view(dt)
    return buf, buf[:n].view(shape)


def _assert_tail(buf, n, what):
    assert bool((_bits(buf[n:]) == PAT[buf.dtype]).all()), f"{what}: wrote past the output tensor"


def _border(B, Hp):
    m = torch.ones(B, Hp, Hp, dtype=torch.bool, device=DEV)
    m[:, 1:-1, 1:-1] = False
    return m


def _padded(interior, fill=float("nan")):
    """[B, r, r, C] -> [B, r+2, r+2, C] with `fill` in the border."""
    B, r, _, C = interior.shape
    x = torch.full((B, r + 2, r + 2, C), fill, dtype=interior.dtype, device=DEV)
    x[:, 1:-1, 1:-1] = interior
    return x


def _ulp(ref, dt):
    """One ulp of the operand type at |ref| (normal range)."""
    e = torch.floor(torch.log2(ref.abs().clamp_min(2.0 ** -126)))
    return torch.exp2(e - MANT[dt])


def _assert_within(got, ref, bound, what):
    err = (got.double() - ref).abs()
    bad = ~(err <= bound)
    if bool(bad.any()):
        i = tuple(bad.nonzero()[0].tolist())
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} out of bound; first at {i}: got "
                             f"{float(got[i])!r} ref {float(ref[i])!r} bound {float(bound[i] if torch.is_tensor(bound) else bound):.3g}")


# ------------------------------------------------------------------------------------------------
# 1. convolutions: every (res, Cin, Cout, k, mode, residual) the decoders launch, at every tile width
# ------------------------------------------------------------------------------------------------
CONV_CASES = _all("conv")


def _conv_id(c):
    res, cin, cout, k, mode, inplace = c
    return f"r{res}_{cin}to{cout}_k{k}_m{mode}" + ("_resid" if inplace else "")


@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("res,Cin,Cout,k,mode,inplace", CONV_CASES, ids=[_conv_id(c) for c in CONV_CASES])
def test_conv_against_fp64_at_every_tile(dt, res, Cin, Cout, k, mode, inplace):
    """B = 2.  Reference: fp64 conv2d of the same operands (A as stored, the weights rounded as the decoder packs them).
    Bound: fp32 accumulation of exact products, 1e-5 of sum |a w| (+ |residual|) + 1e-6 |y| + 1e-7, plus one rounding to
    bf16 (2^-8 |y|) for the bf16 q | k | v.  Every tile width gives the planner's result bit for bit; at res 256 the
    upsample convolution has 521 row blocks, several tiles per CTA pair at every width (the TMEM accumulator handoff)."""
    from hqtransformer_b200.stage1 import debug_s1_conv
    B, Hp = 2, res + 2
    g = torch.Generator(device=DEV).manual_seed(Cin * 7 + Cout + k + res)
    A = torch.zeros(B, Hp, Hp, Cin, device=DEV, dtype=dt)
    A[:, 1:-1, 1:-1, :] = _round(torch.randn(B, res, res, Cin, generator=g, device=DEV), dt)
    W = torch.randn(Cout, Cin, k, k, generator=g, device=DEV) / (Cin * k * k) ** 0.5
    bias = 0.1 * torch.randn(Cout, generator=g, device=DEV)
    rw = (lambda w: w.to(torch.bfloat16).float()) if dt == torch.bfloat16 else T.round_tf32
    y, scale = T.conv_fp64(A.float(), W, bias, k, round_weight=rw)
    resid = torch.randn(B, res, res, Cout, generator=g, device=DEV) if inplace else None
    bound = 1e-5 * scale + 1e-6 * y.abs() + 1e-7
    if resid is not None:
        r = resid.permute(0, 3, 1, 2).double()
        y = y + r
        bound = bound + 1e-5 * r.abs()
    del scale
    if mode == 1 and dt == torch.bfloat16:
        bound = 1.01 * bound + 2.0 ** -8 * y.abs()
    out_dt = dt if mode == 1 else torch.float32
    first = None
    for tile in TILES:
        shape = (B, Cout, res, res) if mode == 2 else (B, Hp, Hp, Cout)
        buf, out = _sentinel(shape, out_dt)
        if resid is not None:
            out[:, 1:-1, 1:-1, :] = resid
        debug_s1_conv(A, W, bias, out, mode, resid=out if inplace else None, tile=tile)
        _assert_tail(buf, out.numel(), f"tile {tile}")
        if mode == 2:
            got = out
        else:
            assert bool((_bits(out[_border(B, Hp)]) == PAT[out_dt]).all()), f"tile {tile}: wrote a padding position"
            got = out[:, 1:-1, 1:-1, :].permute(0, 3, 1, 2)
        assert bool(torch.isfinite(got).all()), f"tile {tile}: interior not fully written"
        _assert_within(got, y, bound, f"tile {tile}")
        if mode == 1 and dt == torch.float32:                          # q | k | v stay UNROUNDED fp32
            assert float(((got.contiguous().view(torch.int32) & 0x1FFF) != 0).float().mean()) > 0.9
        if first is None:
            first = got.clone()
        else:
            assert torch.equal(_bits(got.contiguous()), _bits(first.contiguous())), f"tile {tile} differs from the planner's"


def test_debug_conv_rejects_bad_plans():
    """In both operand types: tile widths the planner never picks, Cin not a multiple of 64, and Cout % 4 != 0 in the
    modes that store 4-wide vectors per row (the vectors of the next row would be misaligned)."""
    import hqtransformer_b200 as H
    from hqtransformer_b200.stage1 import debug_s1_conv
    W, b = torch.zeros(64, 64, 3, 3, device=DEV), torch.zeros(64, device=DEV)
    out = torch.zeros(1, 6, 6, 64, device=DEV)
    for dt in (torch.bfloat16, torch.float32):
        A = torch.zeros(1, 6, 6, 64, device=DEV, dtype=dt)
        for tile in (16, 48, 288):
            with pytest.raises(H.HQError):
                debug_s1_conv(A, W, b, out, 0, tile=tile)
        with pytest.raises(H.HQError):                               # Cin must be a multiple of 64
            debug_s1_conv(torch.zeros(1, 6, 6, 32, device=DEV, dtype=dt), torch.zeros(64, 32, 3, 3, device=DEV), b, out, 0)
        for mode in (0, 1):                                          # Cout % 4
            o = torch.zeros(1, 6, 6, 62, device=DEV, dtype=dt if mode == 1 else torch.float32)
            with pytest.raises(H.HQError):
                debug_s1_conv(A, torch.zeros(62, 64, 1, 1, device=DEV), torch.zeros(62, device=DEV), o, mode)


# ------------------------------------------------------------------------------------------------
# 2. GroupNorm (+ swish)
# ------------------------------------------------------------------------------------------------
def _swish64(v):
    return v / (1.0 + torch.exp(-v))


def _gn_stats64(x_int):
    """fp64 (mean, rstd) per image and group of the interior [B, r, r, C]: [B, 32] each (eps 1e-6, layers.py:17-21)."""
    B, r, _, C = x_int.shape
    v = x_int.double().reshape(B, r * r, 32, C // 32)
    mean = v.mean(dim=(1, 3))
    var = ((v - mean[:, None, :, None]) ** 2).mean(dim=(1, 3))
    return mean, 1.0 / torch.sqrt(var + 1e-6)


def _gn_apply64(x_int, stat, gamma, beta, swish):
    """fp64 (x - mean_f) rstd_f gamma + beta (+ swish) with the kernel's own fp32 statistics, and the scale of the fp32
    rounding errors of that expression: |(x - mean) rstd gamma| + |beta|."""
    B, r, _, C = x_int.shape
    cg = C // 32
    m = stat[..., 0].double().repeat_interleave(cg, dim=1)[:, None, None, :]
    rs = stat[..., 1].double().repeat_interleave(cg, dim=1)[:, None, None, :]
    t = (x_int.double() - m) * rs * gamma.double()
    pre = t + beta.double()
    return (_swish64(pre) if swish else pre), t.abs() + beta.double().abs()


def _gn_run(dt, x_int, gamma, beta, swish):
    from hqtransformer_b200.stage1 import debug_s1_groupnorm
    B, r, _, C = x_int.shape
    x = _padded(x_int)
    buf, out = _sentinel((B, r + 2, r + 2, C), dt)
    stat = torch.full((B, 32, 2), float("nan"), device=DEV)
    debug_s1_groupnorm(x, gamma, beta, out, swish=bool(swish), stat_out=stat)
    _assert_tail(buf, out.numel(), "GroupNorm")
    return out, stat


def _gn_check_apply(dt, x_int, out, stat, gamma, beta, swish, what):
    """Border exactly +0; interior within one ulp of the operand type of the fp64 apply with the kernel's statistics,
    plus 4 fp32 roundings of the terms (times 1.1, the largest slope of swish), 1e-5 relative for swish_f's fast
    exponential and division, and 1e-35 absolute: __fdividef returns 0 once 1 + e^-v exceeds 2^126 (v < -87.3), where
    swish(v) is below 2e-36."""
    B, r, _, C = x_int.shape
    assert bool((_bits(out[_border(B, r + 2)]) == 0).all()), f"{what}: border not +0"
    ref, terms = _gn_apply64(x_int, stat, gamma, beta, swish)
    bound = _ulp(ref, dt) + 1.1 * 4 * 2.0 ** -24 * terms + 1e-5 * ref.abs() + 1e-35
    _assert_within(out[:, 1:-1, 1:-1, :], ref, bound, what)


def _gn_input(B, r, C, g, ratio=None):
    """x = mu + sigma z per (image, group): sigma in [0.5, 1.5); mu = ratio * sigma (random sign), or 2 N(0, 1) if no
    ratio is given.  Different in every image and group, so a group boundary or an image index that is off shows."""
    z = torch.randn(B, r, r, C, generator=g, device=DEV)
    sigma = 0.5 + torch.rand(B, 1, 1, 32, generator=g, device=DEV)
    if ratio is None:
        mu = 2 * torch.randn(B, 1, 1, 32, generator=g, device=DEV)
    else:
        mu = ratio * sigma * torch.where(torch.rand(B, 1, 1, 32, generator=g, device=DEV) < 0.5, -1.0, 1.0)
    cg = C // 32
    return mu.repeat_interleave(cg, dim=3) + sigma.repeat_interleave(cg, dim=3) * z


def _gn_affine(C, g):
    return 1.0 + 0.3 * torch.randn(C, generator=g, device=DEV), 0.2 * torch.randn(C, generator=g, device=DEV)


# (res, C, swish) of both decoders, and the edges: C = 32 / 96 / 160 (1, 3 and 5 channels per group: the per-lane group
# path of the apply kernel), C = 1024 (one pixel lane per CTA in the statistics kernel), res = 100 (a 200-pixel decoder
# with 2 levels: 64 slices of 2 rows, slices 50 .. 63 get no rows)
GN_CASES = _all("norm") + [(8, 32, 1), (8, 96, 1), (8, 160, 0), (8, 1024, 1), (100, 128, 1)]


@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("res,C,swish", GN_CASES, ids=[f"r{r}_C{c}_sw{s}" for r, c, s in GN_CASES])
def test_groupnorm_against_fp64(dt, res, C, swish):
    """B = 2.  Statistics against fp64 (eps 1e-6): mean within 1e-6 sigma; rstd within 2e-6 relative (inputs with
    |mu| <= 6 sigma; fp32 per-thread partials).  The apply against fp64 with the kernel's own statistics (see
    _gn_check_apply)."""
    g = torch.Generator(device=DEV).manual_seed(res * 1031 + C + swish)
    x_int = _gn_input(2, res, C, g)
    gamma, beta = _gn_affine(C, g)
    out, stat = _gn_run(dt, x_int, gamma, beta, swish)
    mean, rstd = _gn_stats64(x_int)
    assert bool(((stat[..., 0].double() - mean).abs() <= 1e-6 / rstd).all()), "mean"
    assert bool(((stat[..., 1].double() / rstd - 1).abs() <= 2e-6).all()), "rstd"
    _gn_check_apply(dt, x_int, out, stat, gamma, beta, swish, f"GroupNorm r{res} C{C}")


# bars on the relative error of rstd and on |mean error| / sigma by mu / sigma.  Largest errors measured on an NVIDIA B200
# (1000 W power limit) over both shapes: rstd 5.3e-8, 1.2e-6, 1.14e-4; mean 3.2e-9, 5.9e-7, 5.9e-6.  The bar at 100 is
# 2^-12 relative, half a TF32 ulp at the top of a binade: the rounding the tf32 decoder gives the GroupNorm output anyway.
GN_OFFSET_BARS = {0: (4e-7, 2e-7), 10: (5e-6, 2e-6), 100: (2.0 ** -12, 2e-5)}


@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("ratio", sorted(GN_OFFSET_BARS))
@pytest.mark.parametrize("res,C", [(16, 512), (256, 128)])
def test_groupnorm_statistics_of_offset_inputs(dt, ratio, res, C):
    """x = mu + sigma z with mu / sigma = 0, 10, 100 in every group.  The statistics kernel forms var = E[x^2] - mean^2
    from fp32 per-thread partial sums, so the relative error of rstd grows with (mu / sigma)^2: the bars are
    GN_OFFSET_BARS, set from the errors a B200 shows (printed).  The apply is checked as in test_groupnorm_against_fp64."""
    g = torch.Generator(device=DEV).manual_seed(ratio * 7 + res)
    x_int = _gn_input(2, res, C, g, ratio=float(ratio))
    gamma, beta = _gn_affine(C, g)
    out, stat = _gn_run(dt, x_int, gamma, beta, 1)
    mean, rstd = _gn_stats64(x_int)
    e_mean = float(((stat[..., 0].double() - mean).abs() * rstd).max())
    e_rstd = float((stat[..., 1].double() / rstd - 1).abs().max())
    print(f"\n[GroupNorm offset] mu/sigma {ratio} res {res} C {C}: |dmean|/sigma {e_mean:.2e}, |drstd|/rstd {e_rstd:.2e}")
    rstd_bar, mean_bar = GN_OFFSET_BARS[ratio]
    assert e_rstd <= rstd_bar and e_mean <= mean_bar, (e_rstd, e_mean)
    _gn_check_apply(dt, x_int, out, stat, gamma, beta, 1, f"GroupNorm mu/sigma {ratio}")


@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("C", [64, 128])
def test_groupnorm_swish_function_accuracy(dt, C):
    """Dense sweep of the swish pre-activation over [-90, 90]: x uniform in each group, gamma = 52 (|x - mean| rstd
    reaches sqrt 3), beta spread over [0, 0.25); 2 x 64 x 64 x C points, against fp64 swish of the fp64 apply with the
    kernel's statistics (the bound of _gn_check_apply).  C = 64 takes the per-lane group path (2 channels per group)."""
    g = torch.Generator(device=DEV).manual_seed(C)
    x_int = 2 * torch.rand(2, 64, 64, C, generator=g, device=DEV) - 1
    gamma = torch.full((C,), 52.0, device=DEV)
    beta = torch.arange(C, device=DEV, dtype=torch.float32) * (0.25 / C)
    out, stat = _gn_run(dt, x_int, gamma, beta, 1)
    ref, _ = _gn_apply64(x_int, stat, gamma, beta, 0)
    assert float(ref.min()) < -85 and float(ref.max()) > 85
    _gn_check_apply(dt, x_int, out, stat, gamma, beta, 1, "swish sweep")


@pytest.mark.parametrize("dt", DTYPES)
def test_groupnorm_is_deterministic_and_per_image(dt):
    """The last slice CTA of an image (ticket counter) sums the slices in a fixed order: repeated calls give the same bits,
    and image b gives the same bits alone as inside a batch of 5."""
    g = torch.Generator(device=DEV).manual_seed(5)
    x_int = _gn_input(5, 64, 256, g)
    gamma, beta = _gn_affine(256, g)
    out, stat = _gn_run(dt, x_int, gamma, beta, 1)
    out2, stat2 = _gn_run(dt, x_int, gamma, beta, 1)
    assert torch.equal(_bits(out), _bits(out2)) and torch.equal(_bits(stat), _bits(stat2))
    for b in (0, 3):
        o1, s1 = _gn_run(dt, x_int[b:b + 1].contiguous(), gamma, beta, 1)
        assert torch.equal(_bits(o1[0]), _bits(out[b])) and torch.equal(_bits(s1[0]), _bits(stat[b])), b


# ------------------------------------------------------------------------------------------------
# 3. resample: nearest 2x (upsample conv input) and the up = 1 operand copy - exact
# ------------------------------------------------------------------------------------------------
RESAMPLE_CASES = _all("resample")


@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("res,C,up", RESAMPLE_CASES, ids=[f"r{r}_C{c}_up{u}" for r, c, u in RESAMPLE_CASES])
def test_resample_is_exact(dt, res, C, up):
    """The interior equals F.interpolate(x, nearest) rounded to the operand type bit for bit (up = 1: the rounded copy);
    the border is +0; B = 3."""
    from hqtransformer_b200.stage1 import debug_s1_resample
    B = 3
    g = torch.Generator(device=DEV).manual_seed(res * 13 + C + up)
    x_int = torch.randn(B, res, res, C, generator=g, device=DEV) * torch.exp(torch.randn(B, 1, 1, C, generator=g, device=DEV))
    ro = up * res
    buf, out = _sentinel((B, ro + 2, ro + 2, C), dt)
    debug_s1_resample(_padded(x_int), out, up)
    _assert_tail(buf, out.numel(), "resample")
    assert bool((_bits(out[_border(B, ro + 2)]) == 0).all()), "border not +0"
    want = F.interpolate(x_int.permute(0, 3, 1, 2), scale_factor=float(up), mode="nearest").permute(0, 2, 3, 1)
    assert torch.equal(_bits(out[:, 1:-1, 1:-1, :].contiguous()), _bits(_round(want.contiguous(), dt)))


# ------------------------------------------------------------------------------------------------
# 4. quant: codebook gather + PixelShuffle + concat - exact
# ------------------------------------------------------------------------------------------------
QUANT_CASES = _all("quant")


@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("E,hb,n_embed", QUANT_CASES, ids=[f"E{e}_hb{h}_n{n}" for e, h, n in QUANT_CASES])
def test_quant_is_exact(dt, E, hb, n_embed):
    """The oracle's own expression cat([pixel_shuffle(E_t[code_t]), E_b[code_b]]) rounded to the operand type, bit for
    bit, with codes 0 and n_embed - 1 among them; the border is +0; B = 3."""
    from hqtransformer_b200.stage1 import debug_s1_quant
    B = 3
    g = torch.Generator(device=DEV).manual_seed(E + hb)
    E_t = torch.randn(n_embed, 4 * E, generator=g, device=DEV)
    E_b = torch.randn(n_embed, E, generator=g, device=DEV)
    ct = torch.randint(0, n_embed, (B, hb // 2, hb // 2), generator=g, device=DEV)
    cb = torch.randint(0, n_embed, (B, hb, hb), generator=g, device=DEV)
    ct[0, 0, 0], ct[1, -1, -1], cb[0, 0, 0], cb[2, -1, 0] = 0, n_embed - 1, n_embed - 1, 0
    buf, out = _sentinel((B, hb + 2, hb + 2, 2 * E), dt)
    debug_s1_quant(ct, cb, E_t, E_b, out)
    _assert_tail(buf, out.numel(), "quant")
    assert bool((_bits(out[_border(B, hb + 2)]) == 0).all()), "border not +0"
    want = torch.cat([F.pixel_shuffle(E_t[ct].permute(0, 3, 1, 2), 2), E_b[cb].permute(0, 3, 1, 2)], dim=1)
    want = _round(want.permute(0, 2, 3, 1).contiguous(), dt)
    assert torch.equal(_bits(out[:, 1:-1, 1:-1, :].contiguous()), _bits(want))


# ------------------------------------------------------------------------------------------------
# 5. AttnBlock core
# ------------------------------------------------------------------------------------------------
# the decoders' (res, C), then (8, 256); (12, 384): N = 144, a partial 32-key chunk and a partial 64-key V tile, and
# C = 384 takes the generic index split of the tensor-core kernel's tile loader; (2, 128) and (32, 128): N = 4 and
# N = 1024, where the decoder takes the CUDA-core kernel
ATTN_CASES = _all("attn") + [(8, 256), (12, 384), (2, 128), (32, 128)]
# near-uniform scores, or peaked: q . k C^-1/2 ~ N(0, 30^2), so exp() overflows fp32 without the max subtraction
REGIMES = {"uniform": 0.1, "peaked": 30.0 ** 0.5}


def _attn_variants():
    out = []
    for res, C in ATTN_CASES:
        for regime in REGIMES:
            out += [pytest.param(torch.bfloat16, 0, res, C, regime, id=f"bf16_mma_r{res}_C{C}_{regime}"),
                    pytest.param(torch.bfloat16, 1, res, C, regime, id=f"bf16_simt_r{res}_C{C}_{regime}"),
                    pytest.param(torch.float32, 0, res, C, regime, id=f"tf32_r{res}_C{C}_{regime}")]
    return out


@pytest.mark.parametrize("dt,variant,res,C,regime", _attn_variants())
def test_attention_against_fp64(dt, variant, res, C, regime):
    """B = 2.  Reference: fp64 softmax(q k^T C^-1/2) v of the same q / k / v (bf16, or unrounded fp32 for tf32).  With
    A = sum_j p_j |v_jc| and ds = 2^-22 sqrt(C) max_j sum_c |q_c k_jc| C^-1/2 (fp32 score accumulation, which moves each
    p_j by at most 2 ds relative), the bound is (2 ds + 2^-22 sqrt(N)) A, plus:
      bf16, tensor-core kernel (variant 0 where the decoder takes it): 2^-8 A - P is rounded to bf16 before P V, which
      the reference does not do - plus one bf16 ulp of the result;
      bf16, CUDA-core kernel: one bf16 ulp of the result;
      tf32 (the CUDA-core kernel in fp32): one TF32 ulp of round_tf32(reference), against which it is compared.
    The output's border is never written: it keeps the NaN pattern."""
    from hqtransformer_b200.stage1 import debug_s1_attention
    B, N, Hp = 2, res * res, res + 2
    g = torch.Generator(device=DEV).manual_seed(res * 31 + C + len(regime))
    s = REGIMES[regime]
    q = s * torch.randn(B, N, C, generator=g, device=DEV)
    k = s * torch.randn(B, N, C, generator=g, device=DEV)
    v = torch.randn(B, N, C, generator=g, device=DEV)
    qkv_int = torch.cat([q, k, v], dim=2).to(dt).reshape(B, res, res, 3 * C)
    qkv = _padded(qkv_int)
    buf, out = _sentinel((B, Hp, Hp, C), dt)
    debug_s1_attention(qkv, out, variant)
    _assert_tail(buf, out.numel(), "attention")
    assert bool((_bits(out[_border(B, Hp)]) == PAT[dt]).all()), "wrote a border position"
    q, k, v = (t.double() for t in qkv_int.reshape(B, N, 3 * C).split(C, dim=2))
    scale = C ** -0.5
    p = torch.softmax(q @ k.transpose(1, 2) * scale, dim=-1)
    ref = p @ v
    a = p @ v.abs()
    ds = 2.0 ** -22 * math.sqrt(C) * ((q.abs() @ k.abs().transpose(1, 2)).amax(dim=-1, keepdim=True) * scale)
    bound = (2 * ds + 2.0 ** -22 * math.sqrt(N)) * a
    mma = variant == 0 and dt == torch.bfloat16 and N % 16 == 0 and N <= 256 and C % 128 == 0 and C <= 512
    if dt == torch.float32:
        ref = T.round_tf32(ref.float()).double()
    if mma:
        bound = bound + 2.0 ** -8 * a
    bound = bound + _ulp(ref, dt)
    got = out[:, 1:-1, 1:-1, :].reshape(B, N, C)
    _assert_within(got, ref, bound, f"attention {'mma' if mma else 'simt'} r{res} C{C} {regime}")


@pytest.mark.parametrize("dt", DTYPES)
def test_debug_hooks_reject_bad_arguments(dt):
    """Each hook refuses what its kernels do not take, with HQ_ERR_INVALID and no launch (the tensors are large enough
    for the shapes passed)."""
    import hqtransformer_b200 as H
    from hqtransformer_b200 import stage1 as HS
    one = torch.ones(1024, device=DEV)
    for C in (48, 2048):                                             # GroupNorm: C % 32, C <= 1024
        x = torch.zeros(1, 6, 6, C, device=DEV)
        with pytest.raises(H.HQError):
            HS.debug_s1_groupnorm(x, one.repeat(2)[:C].contiguous(), one.repeat(2)[:C].contiguous(),
                                  torch.zeros(1, 6, 6, C, device=DEV, dtype=dt), swish=True)
    x = torch.zeros(1, 6, 6, 64, device=DEV)
    with pytest.raises(H.HQError):                                   # swish is 0 or 1
        HS._s1_call(HS._lib.load(), "hq_debug_s1_groupnorm", (x,), HS._s1_prec(x.to(dt)), x.data_ptr(),
                          one.data_ptr(), one.data_ptr(), torch.zeros(1, 6, 6, 64, device=DEV, dtype=dt).data_ptr(),
                          1, 4, 64, 2, None)
    for up, C in ((3, 64), (0, 64), (2, 6)):                         # resample: up in {1, 2}, C % 4
        x = torch.zeros(1, 6, 6, C, device=DEV)
        with pytest.raises(H.HQError):
            HS.debug_s1_resample(x, torch.zeros(1, 4 * 3 + 2, 4 * 3 + 2, C, device=DEV, dtype=dt), up)
    codes = torch.zeros(1, 4, 4, dtype=torch.int64, device=DEV)
    with pytest.raises(H.HQError):                                   # quant: the bottom grid side is even
        HS.debug_s1_quant(codes[:, :2, :2].contiguous(), codes[:, :3, :3].contiguous(), torch.zeros(4, 256, device=DEV),
                          torch.zeros(4, 64, device=DEV), torch.zeros(1, 5, 5, 128, device=DEV, dtype=dt))
    for res, C, variant in ((4, 12, 0), (4, 128, 2), (64, 512, 1)):  # attention: C % 8, variant, 32 (C + N) <= 96 KB
        qkv = torch.zeros(1, res + 2, res + 2, 3 * C, device=DEV, dtype=dt)
        with pytest.raises(H.HQError):
            HS.debug_s1_attention(qkv, torch.zeros(1, res + 2, res + 2, C, device=DEV, dtype=dt), variant)
