"""-m gpu: the fp16 engine (HQ_PREC_F16, `precision="fp16"`): the bf16 engine's kernels and rounding points with IEEE fp16
as the 2-byte type - the reference's own autocast format.

Kernel level (hq_debug_gemm_epi / hq_debug_attention / hq_debug_layernorm), against fp64 restatements of the same
operation on the same fp16 operands: bars as in test_gpu_epilogues.py with half an fp16 ulp (2^-11 |ref|) for fp16
outputs; NaN-filled oversized outputs; bit-identical results over every tile plan, ring depth and M.  Sampling loop: the
fp16-emulating oracle (tests/fp16_emulation.py), the reference-made fp32 goldens, the fp16 engine's error against fp32 at most half the
bf16 engine's on the same inputs, and the invariances the project claims for the bf16 engine.  Logit bars hold ~3x headroom
over the values measured on one NVIDIA B200 (1000 W power limit), which the tests print."""
from dataclasses import replace

import numpy as np
import pytest
import torch

from hqtransformer_b200 import engine as E
from oracle import hq_oracle as O
from tests import fp16_emulation as F
from tests.helpers import build_model, cfg_from_meta, load_golden
from tests.test_gpu_epilogues import (LN_MAPS, QKV_PATHS, SPLIT_SHAPES, _acc_bound, _assert_close, _gelu64, _ln_ref, _m_sweep,
                                      _operands, _plans)
from tests.test_gpu_fused_sampler import _chi2_ok, _softmax

pytestmark = pytest.mark.gpu

F16 = torch.float16
PAT_F16 = 0x7E5A                      # fp16 NaN
PAT32 = 0x7FA5A5A5                    # fp32 NaN
HALF_ULP = 2.0 ** -11                 # half an fp16 ulp, relative
GREEDY = dict(top_k_top=1, top_p_top=1.0, top_k_bot=1, top_p_bot=1.0, softmax_temperature=[1.0, 1.0])
STOCH = dict(top_k_top=50, top_p_top=0.9, top_k_bot=50, top_p_bot=0.9, softmax_temperature=[0.9, 0.9])


def _sentinel(shape, dtype):
    if dtype == F16:
        return torch.full(shape, PAT_F16, dtype=torch.int16, device="cuda").view(F16)
    return torch.full(shape, PAT32, dtype=torch.int32, device="cuda").view(torch.float32)


def _bits(t):
    return t.view(torch.int16) if t.dtype == F16 else t.view(torch.int32)


def _assert_sentinel(t, keep, what):
    b = _bits(t)[keep]
    pat = PAT_F16 if t.dtype == F16 else PAT32
    bad = (b != pat).nonzero()
    assert bad.numel() == 0, f"{what}: {bad.shape[0]} sentinel elements overwritten"


def _bound(ref, K, out_f16, slope=1.0):
    b = slope * _acc_bound(ref, K)
    return b + HALF_ULP * ref.abs() if out_f16 else b


# ------------------------------------------------------------------------------------------------
# GEMM epilogues at kernel level
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D", [128, 1536])
@pytest.mark.parametrize("name,rpb,t_stride,t0,mode1", QKV_PATHS, ids=[p[0] for p in QKV_PATHS])
def test_fp16_qkv_epilogue(name, rpb, t_stride, t0, mode1, D):
    """q -> [M, D], k / v -> cache row (m / rpb) * t_stride + t0 + m % rpb, + bias, fp16; every plan bit-identical."""
    N = 2 * D if mode1 else 3 * D
    off = D if mode1 else 0
    ms = _m_sweep(rpb)
    Mmax = ms[0]
    A, W, g = _operands(Mmax, N, D, F16, D * 7 + rpb * 131 + t_stride + t0, w_rows=3 * D)
    bias = torch.randn(N, generator=g, device="cuda")
    ref_all = A.double() @ W[off:off + N].double().t() + bias.double()
    mpad = (Mmax + 255) // 256 * 256 + 256
    kv_rows = mpad * t_stride + t_stride
    first = None
    for M in ms:
        m = torch.arange(M, device="cuda")
        slot = (m // rpb) * t_stride + t0 + m % rpb
        snap = None
        for tile, ks1 in _plans(N):
            what = f"fp16 QKV D={D} rpb={rpb} t_stride={t_stride} t0={t0} M={M} tile={tile} ks1={ks1}"
            q = _sentinel((mpad, D), F16)
            kc = _sentinel((kv_rows, D), F16)
            vc = _sentinel((kv_rows, D), F16)
            vdup = _sentinel((mpad, D), F16) if mode1 else None
            E.debug_gemm_epi(A[:M].contiguous(), W, E.EPI_QKV, N=N, w_row_off=off, tile=tile, ks1=ks1, bias=bias,
                             q=None if mode1 else q, kdst=kc, vdst=vc, vdup=vdup, D=D, sec0=1 if mode1 else 0, rpb=rpb,
                             t_stride=t_stride, t0=t0)
            bufs = [kc, vc] + ([vdup] if mode1 else [q])
            if snap is not None:
                for a, b in zip(bufs, snap):
                    assert torch.equal(_bits(a), _bits(b)), f"{what}: differs bitwise from tile={_plans(N)[0]}"
                continue
            snap = bufs
            got = torch.cat(([] if mode1 else [q[:M]]) + [kc[slot], vc[slot]], dim=1)
            _assert_close(got, ref_all[:M], _bound(ref_all[:M], D, True), what)
            written = torch.zeros(kv_rows, dtype=torch.bool, device="cuda")
            written[slot] = True
            _assert_sentinel(kc, ~written, what + " k cache outside the slots")
            _assert_sentinel(vc, ~written, what + " v cache outside the slots")
            if mode1:
                assert torch.equal(_bits(vdup[:M]), _bits(vc[slot])), what + ": vdup != v"
                _assert_sentinel(vdup[M:], slice(None), what + " vdup rows >= M")
            else:
                _assert_sentinel(q[M:], slice(None), what + " q rows >= M")
            if first is None:
                first = got
            else:
                assert torch.equal(_bits(got), _bits(first[:M])), f"{what}: rows differ bitwise from the M={Mmax} launch"


def _rowwise(epi, N, K, seed):
    ms = _m_sweep()
    Mmax = ms[0]
    A, W, g = _operands(Mmax, N, K, F16, seed)
    bias = torch.randn(N, generator=g, device="cuda")
    acc = A.double() @ W.double().t() + bias.double()
    mpad = (Mmax + 255) // 256 * 256 + 256
    x0 = torch.randn(Mmax, N, generator=g, device="cuda")
    if epi == E.EPI_RESID:
        ref_all, out_dt, slope = x0.double() + acc, torch.float32, 1.0
    else:
        ref_all, out_dt, slope = _gelu64(acc), F16, 1.13
    first = None
    for M in ms:
        snap = None
        for tile, ks1 in _plans(N):
            what = f"fp16 {'RESID' if epi == E.EPI_RESID else 'GELU'} N={N} K={K} M={M} tile={tile} ks1={ks1}"
            buf = _sentinel((mpad, N), out_dt)
            if epi == E.EPI_RESID:
                buf[:M] = x0[:M]
                E.debug_gemm_epi(A[:M].contiguous(), W, epi, tile=tile, ks1=ks1, bias=bias, x=buf)
            else:
                E.debug_gemm_epi(A[:M].contiguous(), W, epi, tile=tile, ks1=ks1, bias=bias, out=buf)
            if snap is not None:
                assert torch.equal(_bits(buf), _bits(snap)), f"{what}: differs bitwise from tile={_plans(N)[0]}"
                continue
            snap = buf
            _assert_close(buf[:M], ref_all[:M], _bound(ref_all[:M], K, out_dt == F16, slope), what)
            _assert_sentinel(buf[M:], slice(None), what + " rows >= M")
            if first is None:
                first = buf[:M]
            else:
                assert torch.equal(_bits(buf[:M]), _bits(first[:M])), f"{what}: rows differ bitwise from the M={Mmax} launch"


@pytest.mark.parametrize("D", [128, 1536])
@pytest.mark.parametrize("kind", ["proj", "fc2", "fc1_gelu"])
def test_fp16_resid_and_gelu_epilogues(kind, D):
    if kind == "fc1_gelu":
        _rowwise(E.EPI_GELU, 4 * D, D, seed=D + 3)
    else:
        _rowwise(E.EPI_RESID, D, D if kind == "proj" else 4 * D, seed=D + 11)


def test_fp16_gelu_function_accuracy():
    """The 2-byte engines' GELU on 327 680 exactly set pre-activations in [-12, 12], fp16 output: |got - gelu(v)| <= half
    an fp16 ulp of gelu(v) + 5e-7 (the approximation's absolute error is ~4.3e-7)."""
    rows, cols = 640, 512
    v = torch.linspace(-12.0, 12.0, rows, device="cuda").to(torch.bfloat16).float()     # exact in fp16 as well
    b = torch.arange(cols, device="cuda", dtype=torch.float64).mul(0.0625 / cols).float()
    A = torch.zeros(rows, 64, device="cuda", dtype=F16)
    A[:, 0] = v.to(F16)
    W = torch.zeros(cols, 64, device="cuda", dtype=F16)
    W[:, 0] = 1.0
    pre = (v[:, None] + b[None, :]).double()
    out = _sentinel((rows + 128, cols), F16)
    E.debug_gemm_epi(A, W, E.EPI_GELU, bias=b, out=out)
    ref = _gelu64(pre)
    err = (out[:rows].double() - ref).abs()
    print(f"fp16 GELU: max |got - gelu| {err.max():.3e}, max in units of half an fp16 ulp "
          f"{(err / (HALF_ULP * ref.abs() + 5e-7)).max():.3f}")
    _assert_close(out[:rows], ref, HALF_ULP * ref.abs() + 5e-7, "fp16 GELU")
    _assert_sentinel(out[rows:], slice(None), "rows >= M")


@pytest.mark.parametrize("N,K", SPLIT_SHAPES)
@pytest.mark.parametrize("M", [100, 300])
def test_fp16_splitk_partials_each_slice(N, K, M):
    A, W, _ = _operands(M, N, K, F16, seed=N + K + M)
    kb = K // 64
    ldo = N + 32
    mpad = (M + 255) // 256 * 256 + 64
    stride = mpad * ldo
    plans = _plans(N) if M > 128 else [p for p in _plans(N) if p[0] <= 0]
    for S in [s for s in range(1, 7) if kb % s == 0]:
        ks = K // S
        refs = [A[:, s * ks:(s + 1) * ks].double() @ W[:, s * ks:(s + 1) * ks].double().t() for s in range(S)]
        snap = None
        for tile, ks1 in plans:
            what = f"fp16 F32 N={N} K={K} M={M} splits={S} tile={tile} ks1={ks1}"
            outf = _sentinel((S + 1, mpad, ldo), torch.float32)
            E.debug_gemm_epi(A, W, E.EPI_F32, tile=tile, ks1=ks1, outf=outf, ldo=ldo, splits=S, split_stride=stride)
            if snap is not None:
                assert torch.equal(_bits(outf), _bits(snap)), f"{what}: differs bitwise from tile={plans[0]}"
                continue
            snap = outf
            for s in range(S):
                _assert_close(outf[s, :M, :N], refs[s], _acc_bound(refs[s], ks), f"{what} slice {s}")
            keep = torch.ones(outf.shape, dtype=torch.bool, device="cuda")
            keep[:S, :M, :N] = False
            _assert_sentinel(outf, keep, what + " outside [splits, M, N]")


def test_fp16_plain_gemm_every_tile():
    """hq_debug_gemm at fp16: every tile width and both single-CTA kernels give the same bits, within the fp32 bar."""
    A, W, _ = _operands(300, 768, 512, F16, seed=4)
    ref = A.double() @ W.double().t()
    first = None
    for tile in (0, 32, 64, 96, 128, 192, 256, -64, -128):
        got = E.debug_gemm(A, W, tile=tile)
        if first is None:
            _assert_close(got, ref, _acc_bound(ref, 512), f"fp16 GEMM tile={tile}")
            first = got
        else:
            assert torch.equal(got, first), f"tile {tile} differs bitwise"


# ------------------------------------------------------------------------------------------------
# decode attention and LayerNorm
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_keys", [1, 7, 8, 9, 32, 33, 127])
@pytest.mark.parametrize("n_heads", [6, 24])
def test_fp16_decode_attention_vs_fp64(n_keys, n_heads):
    """hq_debug_attention at fp16 (the persistent mma.sync kernel and the scalar one) against fp64 softmax attention of the
    same fp16 q / K / V; bar: half an fp16 ulp of the output plus 1e-4 (the fp16 head / tail weight
    split and fp32 accumulation; measured: the output rounding alone, <= 9.8e-4 at values up to ~2).  A second launch (the ticket counter re-armed by the first) gives the same bits."""
    B, T = 37, 128
    D = n_heads * 64
    g = torch.Generator(device="cuda").manual_seed(n_keys * 13 + n_heads)
    q = (torch.randn(B, D, generator=g, device="cuda") * 2).to(F16)
    K = (torch.randn(B, T, D, generator=g, device="cuda") * 2).to(F16)
    V = torch.randn(B, T, D, generator=g, device="cuda").to(F16)
    qh = q.double().view(B, n_heads, 64)
    Kh = K.double()[:, :n_keys].view(B, n_keys, n_heads, 64)
    Vh = V.double()[:, :n_keys].view(B, n_keys, n_heads, 64)
    s = torch.einsum("bhd,bthd->bht", qh, Kh) / 8.0
    ref = torch.einsum("bht,bthd->bhd", torch.softmax(s, -1), Vh).reshape(B, D)
    outs = []
    for variant in (0, 0, 1):
        got = E.debug_attention(q, K, V, n_keys, variant=variant)
        err = (got.double() - ref).abs()
        print(f"fp16 attention keys={n_keys} heads={n_heads} variant={variant}: max err {err.max():.3e}")
        _assert_close(got, ref, HALF_ULP * ref.abs() + 1e-4, f"fp16 attention keys={n_keys} variant={variant}")
        outs.append(got)
    assert torch.equal(outs[0], outs[1]), "repeated launches differ"


@pytest.mark.parametrize("D", [384, 1536, 2048])
@pytest.mark.parametrize("name,rows,in_group,in_mul,in_off,out_mul", LN_MAPS[:3], ids=[m[0] for m in LN_MAPS[:3]])
def test_fp16_layernorm_with_splitk_fold(name, rows, in_group, in_mul, in_off, out_mul, D):
    """fp16 LayerNorm output with 0..6 folded split-K partial sums; the fold written back bit for bit as a host restatement."""
    g = torch.Generator(device="cuda").manual_seed(D + rows)
    r = torch.arange(rows, device="cuda")
    in_row = (r // in_group) * in_mul + in_off + r % in_group
    x_rows = int(in_row.max()) + 1 + in_mul + 3
    x0 = torch.randn(x_rows, D, generator=g, device="cuda") * 2.0 + 0.5
    gamma = torch.randn(D, generator=g, device="cuda") * 0.5 + 1.0
    beta = torch.randn(D, generator=g, device="cuda") * 0.1
    fold_stride = x_rows * D + 64
    parts = torch.randn(7 * fold_stride, generator=g, device="cuda") * 0.5
    fbias = torch.randn(D, generator=g, device="cuda") * 0.3
    out_rows = rows * out_mul + 8
    written = torch.zeros(out_rows, dtype=torch.bool, device="cuda")
    written[r * out_mul] = True
    for n_fold in range(7):
        what = f"fp16 LN {name} D={D} n_fold={n_fold}"
        x = x0.clone()
        out = _sentinel((out_rows, D), F16)
        E.debug_layernorm(x, gamma, beta, out, rows, in_group=in_group, in_mul=in_mul, in_off=in_off, out_mul=out_mul,
                          fold=parts if n_fold else None, n_fold=n_fold, fold_stride=fold_stride,
                          fold_bias=fbias if n_fold else None)
        want = x0.clone()
        if n_fold:
            p = [parts[s * fold_stride:s * fold_stride + x_rows * D].view(x_rows, D)[in_row] for s in range(n_fold)]
            a = p[0].clone()
            for s in range(1, n_fold):
                a = a + p[s]
            want[in_row] = x0[in_row] + (fbias + a)
        assert torch.equal(_bits(x), _bits(want)), f"{what}: x differs bitwise from the fold restatement"
        ref = _ln_ref(want[in_row].double(), gamma.double(), beta.double(), None)
        _assert_close(out[r * out_mul], ref, 2e-5 * max(ref.abs().max().item(), 1.0) + HALF_ULP * ref.abs(), what)
        _assert_sentinel(out, ~written, what + " out rows not written")


# ------------------------------------------------------------------------------------------------
# the sampling loop
# ------------------------------------------------------------------------------------------------
def _golden(name):
    g, meta = load_golden(name)
    cfg = cfg_from_meta(meta)
    return g, meta, cfg, O.make_params(cfg, seed=meta["seed"], init=meta["init"])


@pytest.mark.parametrize("name", ["tiny_cls_greedy.npz", "small_cls_greedy.npz", "asym_cls_greedy.npz"])
def test_fp16_step_logits_vs_oracle_reference_and_bf16(name):
    """Teacher-forced logits of the fp16 engine: (a) against the fp16-emulating oracle, (b) against the reference-made fp32
    logits, (c) on the same inputs, its max-abs error against the fp32 oracle at most half the bf16 engine's.
    Measured on one B200: (a) max <= 1.1e-3, mean <= 1.5e-4; (b) max <= 1.2e-3, mean <= 2.0e-4; (c) ratio 0.12-0.15."""
    import hqtransformer_b200 as H
    g, meta, cfg, P = _golden(name)
    labels, ct, cb = torch.from_numpy(g["labels"]), torch.from_numpy(g["codes_top"]), torch.from_numpy(g["codes_bot"])
    m16 = build_model(cfg, P, precision="fp16")
    lg = H.step_logits(m16, labels, ct, cb, use_fp16=True).cpu()
    emu = F.step_logits(P, cfg, labels, ct, cb)
    d = (lg - emu).abs()
    want = torch.from_numpy(g["logits"])
    d2 = (lg[:, meta["logit_positions"]] - want).abs()
    ref = O.step_logits(P, cfg, labels, ct, cb)
    e16 = (lg - ref).abs().max().item()
    lgb = H.step_logits(build_model(cfg, P, precision="bf16"), labels, ct, cb, use_fp16=True).cpu()
    eb = (lgb - ref).abs().max().item()
    print(f"{name}: fp16 vs fp16-emulating oracle max {d.max():.3e} mean {d.mean():.3e}; vs reference fp32 max "
          f"{d2.max():.3e} mean {d2.mean():.3e}; max-abs vs fp32: fp16 {e16:.3e} bf16 {eb:.3e} (ratio {e16 / eb:.3f})")
    assert d.max() <= 4e-3 and d.mean() <= 5e-4, (d.max(), d.mean())
    assert d2.max() <= 5e-3 and d2.mean() <= 1e-3, (d2.max(), d2.mean())
    assert e16 <= 0.5 * eb, (e16, eb)


def test_fp16_greedy_margin_aware():
    """Every greedy disagreement with the fp32 reference sits where the reference's top-1 / top-2 margin is below the
    fp16 logit error bar (measured: 1280 of 1280 decisions agree)."""
    import hqtransformer_b200 as H
    g, meta, cfg, P = _golden("small_cls_greedy.npz")
    labels, ct, cb = torch.from_numpy(g["labels"]), torch.from_numpy(g["codes_top"]), torch.from_numpy(g["codes_bot"])
    lg = H.step_logits(build_model(cfg, P, precision="fp16"), labels, ct, cb, use_fp16=True).cpu()
    ref = O.step_logits(P, cfg, labels, ct, cb)
    bad = lg.argmax(-1) != ref.argmax(-1)
    top2 = ref.topk(2, dim=-1).values
    margin = top2[..., 0] - top2[..., 1]
    print(f"fp16 greedy agreement {(~bad).float().mean():.5f} ({int(bad.sum())} flips of {bad.numel()}); largest margin "
          f"among flips {margin[bad].max().item() if bad.any() else 0:.3e}")
    assert (~bad).float().mean() > 0.99
    assert not bad.any() or margin[bad].max() < 0.02


def test_fp16_text_prefix_logits():
    import hqtransformer_b200 as H
    g, meta, cfg, P = _golden("asym_txt_greedy.npz")
    ids, ctg, cbg = torch.from_numpy(g["text_ids"]), torch.from_numpy(g["codes_top"]), torch.from_numpy(g["codes_bot"])
    lg = H.step_logits(build_model(cfg, P, precision="fp16"), ids, ctg, cbg, use_fp16=True).cpu()
    emu = F.step_logits(P, cfg, ids, ctg, cbg)
    d = (lg - emu).abs()
    print(f"text: fp16 vs fp16-emulating oracle max {d.max():.3e} mean {d.mean():.3e}")
    assert d.max() <= 4e-3 and d.mean() <= 5e-4, (d.max(), d.mean())


@pytest.mark.parametrize("kw,B", [(dict(model_type="top2bot"), 5), (dict(model_type="bidirectional"), 5),
                                  (dict(model_type="bidirectional", embedding_type="reduce", position_embedding="2d"), 150),
                                  (dict(model_type="top2bot"), 140)])
def test_fp16_variant_step_logits_vs_oracle(kw, B):
    import hqtransformer_b200 as H
    cfg = replace(O.SMALL, **kw)
    P = O.make_params(cfg, seed=9, init="rich")
    S = 4
    g = torch.Generator().manual_seed(1)
    cond = torch.randint(0, cfg.n_classes, (B,), generator=g) if cfg.cond == "cls" else None
    ct = torch.randint(0, cfg.vocab_top, (B, S), generator=g)
    cb = torch.randint(0, cfg.vocab_bot, (B, S, 4), generator=g)
    emu = F.step_logits(P, cfg, cond, ct, cb)
    lg = H.step_logits(build_model(cfg, P, precision="fp16", max_batch=B, max_seq_len=S), cond, ct, cb, use_fp16=True).cpu()
    d = (lg - emu).abs()
    print(f"{kw} B={B}: fp16 vs fp16-emulating oracle max {d.max():.3e} mean {d.mean():.3e}")
    assert d.max() <= 4e-3 and d.mean() <= 5e-4, (d.max(), d.mean())


@pytest.mark.parametrize("B", [4, 20])
def test_fp16_level3_step_logits_vs_oracle(B):
    import hqtransformer_b200 as H
    from oracle import hq3_oracle as O3
    from tests.test_gpu_level3 import _model
    cfg = O3.SMALL3
    P = O3.make_params(cfg, seed=7)
    S = 3
    g = torch.Generator().manual_seed(B)
    labels = torch.randint(0, cfg.n_classes, (B,), generator=g)
    given = torch.stack([torch.randint(0, cfg.vocab_sizes[0 if j == 0 else (1 if j < 5 else 2)], (B, S), generator=g)
                         for j in range(21)], dim=-1)
    codes = [given[:, :, 0], given[:, :, 1:5].contiguous(), given[:, :, 5:].contiguous()]
    _, emu = F.sample3(P, cfg, labels, B, max_seq_len=S, given=given, return_logits=True)
    m = _model(cfg, P, "fp16", B, max_seq_len=S)
    assert set(m._engines) == {"fp16"}
    lg = H.step_logits3(m, labels, codes, use_fp16=True).cpu()
    d = (lg - emu).abs()
    print(f"3-level B={B}: fp16 vs fp16-emulating oracle max {d.max():.3e} mean {d.mean():.3e}")
    assert d.max() <= 4e-3 and d.mean() <= 5e-4, (d.max(), d.mean())
    ct, cm, cb = H.sampling_hqtransformer(m, B, labels, top_k=[50, 50, 50], top_p=[0.9, 0.9, 0.9], use_fp16=True,
                                          max_seq_len=S, is_tqdm=False, seed=3)
    ct2, cm2, cb2 = H.sampling_hqtransformer(m, B, labels, top_k=[50, 50, 50], top_p=[0.9, 0.9, 0.9], use_fp16=True,
                                             max_seq_len=S, is_tqdm=False, seed=3)
    assert torch.equal(ct, ct2) and torch.equal(cm, cm2) and torch.equal(cb, cb2)


def test_fp16_deterministic_and_launch_mode_invariant():
    import hqtransformer_b200 as H
    g, meta, cfg, P = _golden("small_cls_greedy.npz")
    labels = torch.arange(300) % cfg.n_classes
    kw = dict(use_fp16=True, max_seq_len=16, is_tqdm=False, seed=7, **STOCH)
    base = build_model(cfg, P, precision="fp16", max_batch=300, use_cuda_graph=False, use_pdl=False)
    ct0, cb0 = H.sampling_ihqgpt(base, 300, labels, **kw)
    model = build_model(cfg, P, precision="fp16", max_batch=300, use_cuda_graph=True, use_pdl=True)
    for _ in range(3):
        ct, cb = H.sampling_ihqgpt(model, 300, labels, **kw)
        assert torch.equal(ct, ct0) and torch.equal(cb, cb0)


@pytest.mark.parametrize("cuts", [(0, 19, 37), (0, 1, 36, 37), (0, 150, 300)])
def test_fp16_results_do_not_depend_on_how_the_batch_is_cut(cuts):
    import hqtransformer_b200 as H
    cfg = O.SMALL
    P = O.make_params(cfg, seed=5, init="rich")
    B = cuts[-1]
    labels = torch.randint(0, cfg.n_classes, (B,), generator=torch.Generator().manual_seed(0)).cuda()
    model = build_model(cfg, P, precision="fp16", max_batch=B, max_seq_len=16)
    for kw in (dict(top_k_top=1, top_k_bot=1), STOCH):
        ct, cb = H.sampling_ihqgpt(model, B, labels, max_seq_len=16, is_tqdm=False, use_fp16=True, seed=3, **kw)
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            ct_s, cb_s = H.sampling_ihqgpt(model, hi - lo, labels[lo:hi], max_seq_len=16, is_tqdm=False, use_fp16=True,
                                           seed=3, row_offset=lo, **kw)
            assert torch.equal(ct_s, ct[lo:hi]) and torch.equal(cb_s, cb[lo:hi]), (lo, hi, kw)


def test_fp16_shared_text_prefix_equals_per_row_prefill():
    import hqtransformer_b200 as H
    cfg = replace(O.ASYM, cond="txt")
    P = O.make_params(cfg, seed=6, init="rich")
    ids = torch.randint(0, cfg.vocab_txt, (1, cfg.ctx_len_txt), generator=torch.Generator().manual_seed(3)).repeat(7, 1)
    model = build_model(cfg, P, precision="fp16", max_batch=7, max_seq_len=6)
    for kw in (dict(top_k_top=1, top_k_bot=1), dict(top_k_top=20, top_k_bot=30, softmax_temperature=[0.9, 1.1])):
        a = H.sampling_ihqgpt(model, 7, ids, max_seq_len=6, is_tqdm=False, use_fp16=True, seed=5, shared_prefix=False, **kw)
        b = H.sampling_ihqgpt(model, 7, ids, max_seq_len=6, is_tqdm=False, use_fp16=True, seed=5, shared_prefix=True, **kw)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def test_fp16_sampling_step_api_matches_full_loop():
    import hqtransformer_b200 as H
    g, meta, cfg, P = _golden("tiny_cls_greedy.npz")
    model = build_model(cfg, P, precision="fp16")
    labels = torch.from_numpy(g["labels"])
    want_t, want_b = H.sampling_ihqgpt(model, len(labels), labels, use_fp16=True, max_seq_len=64, is_tqdm=False, **GREEDY)
    sos = P["sos.weight"][labels].unsqueeze(1).cuda()
    codes_top = codes_bot = past = None
    for cnt in range(64):
        if codes_top is None:
            ct_ = cb_ = pos_ = None
        else:
            ct_ = codes_top[:, cnt - 1:cnt]
            cb_ = codes_bot[:, cnt - 1, :]
            pos_ = H.get_positional_encoding(codes_top, mode="1d")[:, cnt - 1:cnt]
        code_top, code_bot, present = model.sampling_step(sos=sos, codes_t=ct_, codes_b=cb_, pos_codes=pos_, use_fp16=True,
                                                          past=past, **GREEDY)
        past = [present] if past is None else past + [present]
        codes_top = code_top if codes_top is None else torch.cat([codes_top, code_top], 1)
        codes_bot = code_bot if codes_bot is None else torch.cat([codes_bot, code_bot], 1)
    assert torch.equal(codes_top.cpu(), want_t.cpu()) and torch.equal(codes_bot.cpu(), want_b.cpu())


def test_fp16_fused_head_sampler_follows_the_engines_own_logits():
    """The head GEMM that draws in its epilogue, at fp16: the top-code frequencies over 16384 rows match softmax(z / T) of
    the same engine's teacher-forced logits (chi-square, 5 sigma)."""
    import hqtransformer_b200 as H
    cfg = O.SMALL
    P = O.make_params(cfg, seed=21, init="rich")
    B, T = 16384, 0.8
    model = build_model(cfg, P, precision="fp16", max_batch=B, max_seq_len=1)
    labels = torch.full((B,), 3, dtype=torch.int64)
    ct, _ = H.sampling_ihqgpt(model, B, labels, use_fp16=True, max_seq_len=1, is_tqdm=False, seed=5, softmax_temperature=[T, 1.0])
    lg = H.step_logits(model, labels[:4], torch.zeros(4, 1, dtype=torch.int64), torch.zeros(4, 1, 4, dtype=torch.int64),
                       use_fp16=True)
    pr = _softmax(lg[0, 0, 0, :cfg.vocab_top].cpu().numpy(), T)
    ok, info = _chi2_ok(np.bincount(ct[:, 0].cpu().numpy(), minlength=cfg.vocab_top).astype(np.float64), pr, B)
    assert ok, info


# ------------------------------------------------------------------------------------------------
# full size and API
# ------------------------------------------------------------------------------------------------
def test_fp16_l12_bounded_sample_and_b256_determinism():
    """ImageNet L12 (D = 1536, 12 + 4 layers, V = 8192): 2 images x 2 positions against the fp32 and the fp16-emulating
    oracle (measured: max 3.2e-3 / mean 5.4e-4 and 2.6e-3 / 4.5e-4); B = 256 stochastic sampling twice, bit-identical."""
    import hqtransformer_b200 as H
    cfg = O.IMAGENET_L12
    P = O.make_params(cfg, seed=0, init="reference")
    g = torch.Generator().manual_seed(1)
    labels = torch.randint(0, cfg.n_classes, (2,), generator=g)
    ct = torch.randint(0, cfg.vocab_top, (2, 2), generator=g)
    cb = torch.randint(0, cfg.vocab_bot, (2, 2, 4), generator=g)
    model = build_model(cfg, P, precision="fp16", max_batch=256)
    lg = H.step_logits(model, labels, ct, cb, use_fp16=True).cpu()
    ref = O.step_logits(P, cfg, labels, ct, cb)
    emu = F.step_logits(P, cfg, labels, ct, cb)
    d, de = (lg - ref).abs(), (lg - emu).abs()
    print(f"L12 fp16: vs fp32 oracle max {d.max():.3e} mean {d.mean():.3e}; vs fp16-emulating oracle max {de.max():.3e} "
          f"mean {de.mean():.3e}")
    assert d.max() <= 1e-2 and d.mean() <= 2e-3
    assert de.max() <= 1e-2 and de.mean() <= 2e-3
    B = 256
    lab = torch.randint(0, cfg.n_classes, (B,), generator=g)
    kw = dict(top_k_top=2048, top_p_top=0.95, top_k_bot=2048, top_p_bot=0.95, softmax_temperature=[0.95, 0.95],
              use_fp16=True, max_seq_len=64, is_tqdm=False, seed=11)
    a = H.sampling_ihqgpt(model, B, lab, **kw)
    b = H.sampling_ihqgpt(model, B, lab, **kw)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def test_fp16_api_builds_no_bf16_engine_and_ignores_use_chain():
    import hqtransformer_b200 as H
    cfg = O.SMALL
    P = O.make_params(cfg, seed=2, init="rich")
    model = build_model(cfg, P, precision="fp16", max_batch=200, max_seq_len=4, use_chain=True)
    labels = torch.arange(200) % cfg.n_classes
    H.sampling_ihqgpt(model, 200, labels, use_fp16=True, max_seq_len=4, is_tqdm=False, seed=1)
    assert set(model._engines) == {"fp16"}
    assert model.engine().chain_launches == 0
    with pytest.raises(ValueError, match="precision"):
        build_model(cfg, P, precision="fp8")
    # the bf16-built model is unchanged: use_fp16=True is its bf16 engine
    mb = build_model(cfg, P, precision="bf16", max_seq_len=4)
    H.sampling_ihqgpt(mb, 2, labels[:2], use_fp16=True, max_seq_len=4, is_tqdm=False, seed=1)
    assert set(mb._engines) == {"bf16"}
