"""-m gpu: the fused GEMM epilogues (QKV scatter into the KV cache, residual add, GELU, split-K fp32 partial sums) and the
LayerNorm that folds the split-K partial sums back into the residual stream, each launched alone through the production
templates (hq_debug_gemm_epi / hq_debug_layernorm) and compared with an fp64 restatement of the same operation on the
same bf16 / fp32 inputs.

Bars.  acc_bound = 2e-5 * max(|ref|max, 1) * sqrt(K / 64) + 1e-5 is the fp32-accumulation bound of the plain GEMM tests
(test_gpu_kernels.py); bf16 outputs add half a bf16 ulp, 2^-8 |ref|; the fp32 CUDA-core engine gets 1e-5 * max(|ref|, 1).

Sentinels.  Every output buffer is larger than the region the launch may write and is filled with a NaN bit pattern first;
afterwards everything outside that region must still hold the pattern, bit for bit.  The margins are wide enough that a
wrong row or cache-slot index lands inside the allocation, where it shows up as a clobbered sentinel.

Invariance.  For a fixed epilogue and split, the tile width, the kernel (CTA pair or single CTA) and the ring-stage depth
(one or two k-blocks per stage) must not change a single output bit, and rows [0, r) of a launch with M = r must equal
those rows of the largest launch: per-row results that do not depend on the batch (resid_splits in engine.cu)."""
import math

import pytest
import torch

from hqtransformer_b200 import engine as E

pytestmark = pytest.mark.gpu

PAT16 = 0x7FA5            # bf16 NaN
PAT32 = 0x7FA5A5A5        # fp32 NaN
TILES = (0, 32, 64, 96, 128, 192, 256, -64, -128)
M_SWEEP = (1, 5, 127, 128, 129, 256, 300, 513)
SQRT1_2 = 0.70710678118654752440


def _sentinel(shape, dtype):
    if dtype == torch.bfloat16:
        return torch.full(shape, PAT16, dtype=torch.int16, device="cuda").view(torch.bfloat16)
    return torch.full(shape, PAT32, dtype=torch.int32, device="cuda").view(torch.float32)


def _bits(t):
    return t.view(torch.int16) if t.dtype == torch.bfloat16 else t.view(torch.int32)


def _pat(t):
    return PAT16 if t.dtype == torch.bfloat16 else PAT32


def _assert_sentinel(t, keep, what):
    """Elements where `keep` is True must still hold the NaN pattern."""
    b = _bits(t)[keep]
    bad = (b != _pat(t)).nonzero()
    assert bad.numel() == 0, f"{what}: {bad.shape[0]} sentinel elements overwritten"


def _plans(N, bf16=True):
    """Every (tile, ks1) the hook accepts for N: all CTA-pair widths dividing N, the engine's choice, both single-CTA
    kernels; one and two k-blocks per ring stage."""
    if not bf16:
        return [(0, False)]
    out = []
    for t in TILES:
        ok = N % t == 0 if t > 0 else (N % 128 == 0 if t == -128 else N % 64 == 0)
        if ok:
            out += [(t, False), (t, True)]
    return out


def _m_sweep(rpb=1):
    return sorted({max(rpb, (m + rpb - 1) // rpb * rpb) for m in M_SWEEP}, reverse=True)


def _acc_bound(ref, K):
    return 2e-5 * max(ref.abs().max().item(), 1.0) * math.sqrt(K / 64) + 1e-5


def _assert_close(got, ref, bound, what):
    """got [M, N] vs fp64 ref elementwise against `bound` (scalar or tensor); names the first failing row and column."""
    err = (got.double() - ref).abs()
    bad = ~(err <= bound)
    if bad.any():
        r, c = bad.nonzero()[0].tolist()
        b = bound[r, c].item() if torch.is_tensor(bound) else bound
        raise AssertionError(f"{what}: {int(bad.sum())} elements out of bound; first at row {r} col {c}: "
                             f"got {got[r, c].item()!r} ref {ref[r, c].item()!r} bound {b:.3g}")


def _bound(ref, K, out_bf16, bf16_engine, slope=1.0):
    """acc_bound (times the largest slope of the epilogue function) plus half a bf16 ulp for bf16 outputs; the fp32
    CUDA-core engine's bar for fp32 engines."""
    if not bf16_engine:
        return 1e-5 * max(ref.abs().max().item(), 1.0)
    b = slope * _acc_bound(ref, K)
    return b + 2.0 ** -8 * ref.abs() if out_bf16 else b


def _gelu64(v):
    """x * Phi(x) in fp64 (erfc form: no cancellation for x << 0)."""
    return v * 0.5 * torch.special.erfc(-v * SQRT1_2)


def _operands(M, N, K, dt, seed, w_rows=None, scale=0.05):
    g = torch.Generator(device="cuda").manual_seed(seed)
    A = torch.randn(M, K, generator=g, device="cuda").to(dt)
    W = (torch.randn(w_rows or N, K, generator=g, device="cuda") * scale).to(dt)
    return A, W, g


# ------------------------------------------------------------------------------------------------
# EPI_QKV: every (rows per image, cache stride, first slot, section) the sampler passes to run_block
# ------------------------------------------------------------------------------------------------
TC = 127          # spatial cache of a text model: T0 = 64 prefix tokens + 63 image positions
QKV_PATHS = [     # name, rpb, t_stride, t0, depth pass 0 (k and v only: sec0 = 1, N = 2D, W rows from D, vdup)
    ("spatial_first", 1, TC, 0, False),
    ("spatial_mid", 1, TC, 70, False),
    ("spatial_last", 1, TC, TC - 1, False),
    ("text_prefill", 64, TC, 0, False),
    ("depth_pass0", 1, 5, 0, True),
    ("depth_pass1", 4, 5, 1, False),
] + [(f"top2bot_slot{c}", 1, 5, c, False) for c in range(5)] + [
    ("bidirectional", 5, 5, 0, False),
    ("level3_pass0", 1, 21, 0, True),
    ("level3_pass1", 4, 21, 1, False),
    ("level3_pass2", 16, 21, 5, False),
]


def _qkv_case(D, rpb, t_stride, t0, mode1, dt, seed):
    bf = dt == torch.bfloat16
    N = 2 * D if mode1 else 3 * D
    off = D if mode1 else 0
    ms = _m_sweep(rpb)
    Mmax = ms[0]
    A, W, g = _operands(Mmax, N, D, dt, seed, w_rows=3 * D)
    bias = torch.randn(N, generator=g, device="cuda")
    ref_all = A.double() @ W[off:off + N].double().t() + bias.double()
    mpad = (Mmax + 255) // 256 * 256 + 256
    # a row index computed as if rpb were 1 still lands inside: mpad * t_stride rows
    kv_rows = mpad * t_stride + t_stride
    first = None
    for M in ms:
        m = torch.arange(M, device="cuda")
        slot = (m // rpb) * t_stride + t0 + m % rpb
        ref = ref_all[:M]
        snap = None
        for tile, ks1 in _plans(N, bf):
            what = f"QKV D={D} rpb={rpb} t_stride={t_stride} t0={t0} sec0={int(mode1)} M={M} tile={tile} ks1={ks1}"
            q = _sentinel((mpad, D), dt)
            kc = _sentinel((kv_rows, D), dt)
            vc = _sentinel((kv_rows, D), dt)
            vdup = _sentinel((mpad, D), dt) if mode1 else None
            E.debug_gemm_epi(A[:M].contiguous(), W, E.EPI_QKV, N=N, w_row_off=off, tile=tile, ks1=ks1, bias=bias,
                             q=None if mode1 else q, kdst=kc, vdst=vc, vdup=vdup, D=D, sec0=1 if mode1 else 0, rpb=rpb,
                             t_stride=t_stride, t0=t0)
            bufs = [kc, vc] + ([vdup] if mode1 else [q])
            if snap is not None:
                for name, a, b in zip(("k cache", "v cache", "vdup" if mode1 else "q"), bufs, snap):
                    assert torch.equal(_bits(a), _bits(b)), f"{what}: {name} differs bitwise from tile={_plans(N, bf)[0]}"
                continue
            snap = bufs
            secs = ([] if mode1 else [q[:M]]) + [kc[slot], vc[slot]]
            got = torch.cat(secs, dim=1)
            _assert_close(got, ref, _bound(ref, D, True, bf), what)
            written = torch.zeros(kv_rows, dtype=torch.bool, device="cuda")
            written[slot] = True
            _assert_sentinel(kc, ~written, what + " k cache outside slots t0..t0+rpb-1")
            _assert_sentinel(vc, ~written, what + " v cache outside slots t0..t0+rpb-1")
            if mode1:
                assert torch.equal(_bits(vdup[:M]), _bits(vc[slot])), what + ": vdup != v"
                _assert_sentinel(vdup[M:], slice(None), what + " vdup rows >= M")
            else:
                _assert_sentinel(q[M:], slice(None), what + " q rows >= M")
            if first is None:
                first = got
            else:
                assert torch.equal(_bits(got), _bits(first[:M])), f"{what}: rows differ bitwise from the M={Mmax} launch"


@pytest.mark.parametrize("D", [128, 384, 1536])
@pytest.mark.parametrize("name,rpb,t_stride,t0,mode1", QKV_PATHS, ids=[p[0] for p in QKV_PATHS])
def test_qkv_epilogue_scatters_into_the_cache_slots(name, rpb, t_stride, t0, mode1, D):
    """q -> [M, D], k / v -> cache row (m / rpb) * t_stride + t0 + m % rpb, + bias, bf16; every tile plan bit-identical."""
    _qkv_case(D, rpb, t_stride, t0, mode1, torch.bfloat16, seed=D * 7 + rpb * 131 + t_stride + t0)


@pytest.mark.parametrize("name,rpb,t_stride,t0,mode1", QKV_PATHS, ids=[p[0] for p in QKV_PATHS])
def test_qkv_epilogue_fp32_engine(name, rpb, t_stride, t0, mode1):
    _qkv_case(128, rpb, t_stride, t0, mode1, torch.float32, seed=rpb * 17 + t_stride + t0)


# ------------------------------------------------------------------------------------------------
# EPI_RESID and EPI_GELU over every tile plan and M
# ------------------------------------------------------------------------------------------------
def _rowwise_case(epi, N, K, dt, seed, ms=None, plans=None, bias_fn=None):
    bf = dt == torch.bfloat16
    ms = ms or _m_sweep()
    Mmax = ms[0]
    A, W, g = _operands(Mmax, N, K, dt, seed)
    bias = bias_fn(N) if bias_fn else torch.randn(N, generator=g, device="cuda")
    acc = A.double() @ W.double().t() + bias.double()
    mpad = (Mmax + 255) // 256 * 256 + 256
    x0 = torch.randn(Mmax, N, generator=g, device="cuda")
    if epi == E.EPI_RESID:
        ref_all, out_dt, slope = x0.double() + acc, torch.float32, 1.0
    else:
        ref_all, out_dt, slope = _gelu64(acc), dt, 1.13      # |gelu'| <= 1.13: the accumulation error, carried through
    first = None
    for M in ms:
        ref = ref_all[:M]
        snap = None
        for tile, ks1 in plans or _plans(N, bf):
            what = f"{'RESID' if epi == E.EPI_RESID else 'GELU'} N={N} K={K} M={M} tile={tile} ks1={ks1}"
            buf = _sentinel((mpad, N), out_dt)
            if epi == E.EPI_RESID:
                buf[:M] = x0[:M]
                E.debug_gemm_epi(A[:M].contiguous(), W, epi, tile=tile, ks1=ks1, bias=bias, x=buf)
            else:
                E.debug_gemm_epi(A[:M].contiguous(), W, epi, tile=tile, ks1=ks1, bias=bias, out=buf)
            if snap is not None:
                assert torch.equal(_bits(buf), _bits(snap)), f"{what}: differs bitwise from tile={(plans or _plans(N, bf))[0]}"
                continue
            snap = buf
            _assert_close(buf[:M], ref, _bound(ref, K, out_dt == torch.bfloat16, bf, slope), what)
            _assert_sentinel(buf[M:], slice(None), what + " rows >= M")
            if first is None:
                first = buf[:M]
            else:
                assert torch.equal(_bits(buf[:M]), _bits(first[:M])), f"{what}: rows differ bitwise from the M={Mmax} launch"


@pytest.mark.parametrize("D", [128, 384, 1536])
@pytest.mark.parametrize("kind", ["proj", "fc2"])
def test_resid_epilogue_adds_into_x(kind, D):
    """x += A W^T + bias on the fp32 residual stream (proj [D, D], fc2 [D, 4D])."""
    K = D if kind == "proj" else 4 * D
    _rowwise_case(E.EPI_RESID, D, K, torch.bfloat16, seed=D + K)


@pytest.mark.parametrize("D", [128, 384, 1536])
def test_gelu_epilogue(D):
    """out = gelu(A W^T + bias) in bf16 (fc1 [4D, D])."""
    _rowwise_case(E.EPI_GELU, 4 * D, D, torch.bfloat16, seed=D + 3)


@pytest.mark.parametrize("epi", [E.EPI_RESID, E.EPI_GELU])
def test_resid_and_gelu_epilogues_fp32_engine(epi):
    _rowwise_case(epi, 512 if epi == E.EPI_GELU else 384, 384, torch.float32, seed=epi + 40)


def test_persistent_gemm_reloads_the_bias_of_every_tile():
    """More tiles than the 74 CTA pairs (1024 x 6144, tile 64: 384 tiles), so every pair runs several tiles: the bias
    refill of each tile and the double-buffered accumulator's phase.  The bias takes a different value in every column
    of a tile width (a stale or shifted bias would be off by >= 0.1)."""
    def column_bias(N):
        n = torch.arange(N, device="cuda")
        return ((n * 37) % 101).float() * 0.1 - 5.0
    _rowwise_case(E.EPI_GELU, 6144, 1536, torch.bfloat16, seed=9, ms=[1024], plans=[(64, False), (64, True), (32, False)],
                  bias_fn=column_bias)


def test_persistent_qkv_launch_with_many_tiles():
    """QKV at M = 1024, N = 3 * 1536 with tile 64: 288 tiles over at most 74 CTA pairs."""
    D, M, N = 1536, 1024, 4608
    A, W, g = _operands(M, N, D, torch.bfloat16, seed=21)
    n = torch.arange(N, device="cuda")
    bias = ((n * 37) % 101).float() * 0.1 - 5.0
    ref = A.double() @ W.double().t() + bias.double()
    q = _sentinel((M + 256, D), torch.bfloat16)
    kc = _sentinel(((M + 256) * 5, D), torch.bfloat16)
    vc = _sentinel(((M + 256) * 5, D), torch.bfloat16)
    E.debug_gemm_epi(A, W, E.EPI_QKV, tile=64, bias=bias, q=q, kdst=kc, vdst=vc, D=D, sec0=0, rpb=4, t_stride=5, t0=1)
    m = torch.arange(M, device="cuda")
    slot = (m // 4) * 5 + 1 + m % 4
    got = torch.cat([q[:M], kc[slot], vc[slot]], dim=1)
    _assert_close(got, ref, _bound(ref, D, True, True), "QKV M=1024 tile=64")
    written = torch.zeros(kc.shape[0], dtype=torch.bool, device="cuda")
    written[slot] = True
    _assert_sentinel(kc, ~written, "k cache")
    _assert_sentinel(vc, ~written, "v cache")
    _assert_sentinel(q[M:], slice(None), "q rows >= M")


# ------------------------------------------------------------------------------------------------
# GELU as a function: the pre-activation is set exactly, the dense sweep separates approximations
# ------------------------------------------------------------------------------------------------
def _gelu_function_inputs(dt, rows=640, cols=512):
    """K = 64, A row m = [v_m, 0, ...], W row n = [1, 0, ...], bias b_n: the accumulator is v_m exactly and the
    pre-activation is float32(v_m + b_n).  v_m: bf16 values spread over [-12, 12]; b_n: [0, 1/16) (the widest bf16
    spacing there), so the rows * cols points cover the range densely."""
    v = torch.linspace(-12.0, 12.0, rows, device="cuda").to(torch.bfloat16).float()
    b = torch.arange(cols, device="cuda", dtype=torch.float64).mul(0.0625 / cols).float()
    A = torch.zeros(rows, 64, device="cuda", dtype=dt)
    A[:, 0] = v.to(dt)
    W = torch.zeros(cols, 64, device="cuda", dtype=dt)
    W[:, 0] = 1.0
    pre = (v[:, None] + b[None, :]).double()        # float32 sum, exactly as the epilogue forms it
    return A, W, b, pre


def test_gelu_bf16_engine_function_accuracy():
    """The bf16 engine's GELU (Abramowitz & Stegun 7.1.26 erfc, gelu_bf16out) on 327 680 pre-activations in [-12, 12]:
    |got - gelu(v)| <= half a bf16 ulp of gelu(v) + 5e-7, an absolute bar: the approximation's error is at most ~4.3e-7
    absolute, and for v < -6 (|gelu| < 1e-8) it is many bf16 ulps relative.  On a CPU restatement this bar passes the
    code as written and fails a 4th-digit change of one coefficient (0.254829592 -> 0.2549) and the tanh form."""
    A, W, b, pre = _gelu_function_inputs(torch.bfloat16)
    out = _sentinel((A.shape[0] + 128, W.shape[0]), torch.bfloat16)
    E.debug_gemm_epi(A, W, E.EPI_GELU, bias=b, out=out)
    ref = _gelu64(pre)
    got = out[:A.shape[0]]
    _assert_close(got, ref, 2.0 ** -8 * ref.abs() + 5e-7, "bf16 GELU")
    _assert_sentinel(out[A.shape[0]:], slice(None), "rows >= M")


def test_gelu_fp32_engine_function_accuracy():
    """The fp32 engine's exact GELU, 0.5 v (1 + erff(v / sqrt 2)): within 2e-6 relative + 1e-7, plus what erff's
    documented 2-ulp error becomes where erf is close to -1 and 1 + erf cancels: 2 * 2^-24 absolute, times 0.5 |v|."""
    A, W, b, pre = _gelu_function_inputs(torch.float32)
    out = _sentinel((A.shape[0] + 128, W.shape[0]), torch.float32)
    E.debug_gemm_epi(A, W, E.EPI_GELU, bias=b, out=out)
    ref = _gelu64(pre)
    _assert_close(out[:A.shape[0]], ref, 2e-6 * ref.abs() + 1e-7 + pre.abs() * 2.0 ** -24, "fp32 GELU")


# ------------------------------------------------------------------------------------------------
# EPI_F32 split-K: every slice against the product over its own K range
# ------------------------------------------------------------------------------------------------
SPLIT_SHAPES = [(1536, 1536), (1536, 6144), (256, 1024), (384, 1152)]   # (N, K): proj / fc2 at D = 1536, SMALL fc2, odd slices


@pytest.mark.parametrize("N,K", SPLIT_SHAPES)
@pytest.mark.parametrize("M", [100, 300])
def test_splitk_partials_each_slice(N, K, M):
    """Slice s of an S-way split writes the product over k in [s K / S, (s + 1) K / S) to outf + s * split_stride, for
    every S in 1..6 dividing K / 64 (K = 1152: 18 k-blocks, slices of 18, 9, 6 and 3 - odd counts take the one-k-block
    ring), on the single-CTA kernel (M = 100) and the CTA pair (M = 300: the second CTA's rows).  Slices are checked one
    by one (a sum would not see two swapped slices); per split, all tile plans agree bit for bit."""
    A, W, _ = _operands(M, N, K, torch.bfloat16, seed=N + K + M)
    kb = K // 64
    ldo = N + 32                     # columns N .. ldo - 1 are never written
    mpad = (M + 255) // 256 * 256 + 64
    stride = mpad * ldo
    for S in [s for s in range(1, 7) if kb % s == 0]:
        ks = K // S
        refs = [A[:, s * ks:(s + 1) * ks].double() @ W[:, s * ks:(s + 1) * ks].double().t() for s in range(S)]
        snap = None
        plans = _plans(N) if M > 128 else [p for p in _plans(N) if p[0] <= 0]
        for tile, ks1 in plans:
            what = f"F32 N={N} K={K} M={M} splits={S} tile={tile} ks1={ks1}"
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


# ------------------------------------------------------------------------------------------------
# LayerNorm with the split-K fold
# ------------------------------------------------------------------------------------------------
T0 = 64
LN_MAPS = [   # name, rows, in_group, in_mul, in_off, out_mul
    ("rows", 37, 1, 1, 0, 1),
    ("bidirectional_top", 13, 1, 5, 0, 1),
    ("bidirectional_bottom", 52, 4, 5, 1, 1),
    ("ln_f_text_prefill", 6, 1, T0, T0 - 1, 1),
    ("ln_f_bidirectional", 13, 1, 1, 0, 5),
    ("ln_f_text_bidirectional", 6, 1, T0, T0 - 1, 5),
]


def _ln_ref(x, g, b, add):
    m = x.mean(-1, keepdim=True)
    var = ((x - m) ** 2).mean(-1, keepdim=True)
    y = (x - m) / torch.sqrt(var + 1e-5) * g + b
    return y + add if add is not None else y


@pytest.mark.parametrize("D", [128, 384, 1536, 2048])
@pytest.mark.parametrize("name,rows,in_group,in_mul,in_off,out_mul", LN_MAPS, ids=[m[0] for m in LN_MAPS])
def test_layernorm_folds_splitk_partials(name, rows, in_group, in_mul, in_off, out_mul, D):
    """x[in_row] += fold_bias + (p0 + p1 + ... + p(n-1)), summed left to right in fp32, written back bit for bit as a host
    float32 restatement of that order; then out[r * out_mul] = LN(x[in_row]) * gamma + beta (+ add) against fp64 LN of
    the updated row.  n_fold 0..6 covers both instantiations (<= 3 and <= 6 partial sums); D = 2048 takes the strided
    path.  Rows of x that are not mapped, and rows of out that are not written, must not change."""
    g = torch.Generator(device="cuda").manual_seed(D + rows * 7 + in_mul)
    r = torch.arange(rows, device="cuda")
    in_row = (r // in_group) * in_mul + in_off + r % in_group
    x_rows = int(in_row.max()) + 1 + in_mul + 3         # mapped rows plus rows that must stay untouched
    x0 = torch.randn(x_rows, D, generator=g, device="cuda") * 2.0 + 0.5
    gamma = torch.randn(D, generator=g, device="cuda") * 0.5 + 1.0
    beta = torch.randn(D, generator=g, device="cuda") * 0.1
    add = torch.randn(D, generator=g, device="cuda")
    fold_stride = x_rows * D + 64
    parts = torch.randn(7 * fold_stride, generator=g, device="cuda") * 0.5
    fbias = torch.randn(D, generator=g, device="cuda") * 0.3
    unmapped = torch.ones(x_rows, dtype=torch.bool, device="cuda")
    unmapped[in_row] = False
    out_rows = rows * out_mul + 8
    written = torch.zeros(out_rows, dtype=torch.bool, device="cuda")
    written[r * out_mul] = True
    for n_fold in range(7):
        for out_dt in (torch.bfloat16, torch.float32):
            for with_add in (False, True):
                what = f"LN {name} D={D} n_fold={n_fold} out={str(out_dt)[6:]} add={with_add}"
                x = x0.clone()
                out = _sentinel((out_rows, D), out_dt)
                E.debug_layernorm(x, gamma, beta, out, rows, add=add if with_add else None, in_group=in_group,
                                  in_mul=in_mul, in_off=in_off, out_mul=out_mul,
                                  fold=parts if n_fold else None, n_fold=n_fold, fold_stride=fold_stride,
                                  fold_bias=fbias if n_fold else None)
                want = x0.clone()
                if n_fold:
                    p = [parts[s * fold_stride:s * fold_stride + x_rows * D].view(x_rows, D)[in_row] for s in range(n_fold)]
                    a = p[0].clone()
                    for s in range(1, n_fold):
                        a = a + p[s]
                    want[in_row] = x0[in_row] + (fbias + a)
                bad = (_bits(x) != _bits(want)).any(-1).nonzero()
                assert bad.numel() == 0, f"{what}: x rows {bad.flatten()[:8].tolist()} differ bitwise from the fold restatement"
                assert torch.equal(_bits(x[unmapped]), _bits(x0[unmapped])), f"{what}: unmapped x rows changed"
                ref = _ln_ref(want[in_row].double(), gamma.double(), beta.double(), add.double() if with_add else None)
                bound = 2e-5 * max(ref.abs().max().item(), 1.0)
                if out_dt == torch.bfloat16:
                    bound = bound + 2.0 ** -8 * ref.abs()
                _assert_close(out[r * out_mul], ref, bound, what)
                _assert_sentinel(out, ~written, what + " out rows not written")


def test_debug_hooks_reject_what_the_engine_never_launches():
    """Invalid plans are refused rather than run: a split that does not divide the k-blocks, a tile width that does not
    divide N, split-K outside EPI_F32, a QKV cache slot past t_stride, a fold without partial sums."""
    from hqtransformer_b200._lib import HQError
    A, W, _ = _operands(64, 384, 320, torch.bfloat16, seed=1)
    outf = torch.empty(4, 64, 384, device="cuda")
    x = torch.zeros(64, 384, device="cuda")
    with pytest.raises(HQError, match="splits"):
        E.debug_gemm_epi(A, W, E.EPI_F32, outf=outf, ldo=384, splits=2, split_stride=64 * 384)      # 5 k-blocks
    with pytest.raises(HQError, match="tile"):
        E.debug_gemm_epi(A, W, E.EPI_F32, tile=256, outf=outf, ldo=384)
    with pytest.raises(HQError, match="split-K"):
        E.debug_gemm_epi(A[:, :256].contiguous(), W[:, :256].contiguous(), E.EPI_RESID, x=x, splits=2)
    kc = torch.empty(64 * 5, 128, device="cuda", dtype=torch.bfloat16)
    with pytest.raises(HQError, match="QKV"):
        E.debug_gemm_epi(A, W, E.EPI_QKV, q=kc, kdst=kc, vdst=kc, D=128, rpb=4, t_stride=5, t0=2)
    with pytest.raises(HQError, match="fold"):
        E.debug_layernorm(x, x[0], x[0], x, 4, n_fold=2)
