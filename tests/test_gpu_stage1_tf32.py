"""-m gpu: the tf32 stage-1 decoder (precision="tf32", HQ_PREC_TF32): whole decodes against the fp32 oracle, its TF32
emulation (tests/tf32_emulation.py) and the oracle run with PyTorch's own cuDNN TF32 convolutions on the GPU.  Its kernels
one by one: tests/test_gpu_stage1_kernels.py."""
import os

import pytest
import torch

from oracle import s1_oracle as S1
from tests import tf32_emulation as T
from tests.helpers import load_golden

pytestmark = pytest.mark.gpu


def _decoder(cfg, P, max_batch, precision="tf32"):
    import hqtransformer_b200 as H
    dec = H.HQVAEDecoder(embed_dim=cfg.embed_dim, n_embed=cfg.n_embed, z_channels=cfg.z_channels, resolution=cfg.resolution,
                         ch=cfg.ch, ch_mult=cfg.ch_mult, num_res_blocks=cfg.num_res_blocks,
                         attn_resolutions=cfg.attn_resolutions, out_ch=cfg.out_ch, max_batch=max_batch, precision=precision)
    dec.load_state_dict(P, strict=True)
    return dec


def _codes(cfg, B, seed):
    g = torch.Generator().manual_seed(seed)
    h = cfg.latent_res // 2
    return (torch.randint(0, cfg.n_embed, (B, h, h), generator=g),
            torch.randint(0, cfg.n_embed, (B, 2 * h, 2 * h), generator=g))


def _pix8(x):
    return torch.round(torch.clamp(x * 0.5 + 0.5, 0, 1) * 255)


def _report(name, got, ref):
    e = (got - ref).abs()
    eq8 = float((_pix8(got) == _pix8(ref)).float().mean())
    print(f"\n[tf32 stage 1] {name}: max-abs {float(e.max()):.3e} mean-abs {float(e.mean()):.3e} 8-bit equal {eq8:.4f}")
    return float(e.max()), float(e.mean()), eq8


# ---- 2. / 3. whole decodes ----------------------------------------------------------------------------------------------
def _check_fp32_bars(m):
    assert m[0] <= 1e-2 and m[1] <= 1e-3 and m[2] >= 0.90, m


def test_tf32_decode_tiny_golden():
    """The reference-made golden (unmodified decode_code, CPU fp32) and the TF32-emulating oracle."""
    g, meta = load_golden("s1_tiny_decode.npz")
    cfg = S1.S1Config.from_dict(meta["config"])
    P = S1.make_params(cfg, seed=meta["seed"])
    ct, cb = torch.from_numpy(g["code_t"]), torch.from_numpy(g["code_b"])
    got = _decoder(cfg, P, max_batch=4).decode_code(ct, cb).cpu()
    assert torch.isfinite(got).all()
    _check_fp32_bars(_report("tiny golden vs fp32", got, torch.from_numpy(g["pixels"])))
    m = _report("tiny golden vs tf32 emulation", got, T.decode_code(P, cfg, ct, cb))
    assert m[0] <= 5e-3 and m[1] <= 5e-4, m


def test_tf32_decode_full_size_vs_oracle():
    """The shipped HQ-VAE decoder (256 x 256, ch 128, ch_mult [1,2,4,4], attention at 16 x 16) on two images."""
    cfg = S1.IMAGENET_S1
    P = S1.make_params(cfg, seed=2)
    ct, cb = _codes(cfg, 2, 5)
    got = _decoder(cfg, P, max_batch=2).decode_code(ct, cb).cpu()
    _check_fp32_bars(_report("full size vs fp32", got, S1.decode_code(P, cfg, ct, cb)))
    m = _report("full size vs tf32 emulation", got, T.decode_code(P, cfg, ct, cb))
    assert m[0] <= 5e-3 and m[1] <= 5e-4, m


def test_tf32_decode_vs_pytorch_cudnn_tf32_on_the_gpu():
    """The oracle's ops run by PyTorch on this GPU under its defaults (cuDNN convolutions in TF32, bmm in fp32): what the
    reference's decode_code computes there."""
    cfg = S1.IMAGENET_S1
    P = S1.make_params(cfg, seed=2)
    ct, cb = _codes(cfg, 4, 9)
    dev = torch.device("cuda", 0)
    saved = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = True, False
    try:
        ref = S1.decode_code({k: v.to(dev) for k, v in P.items()}, cfg, ct.to(dev), cb.to(dev)).cpu()
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved
    got = _decoder(cfg, P, max_batch=4).decode_code(ct, cb).cpu()
    _check_fp32_bars(_report("full size vs PyTorch cuDNN TF32", got, ref))


# ---- 4. determinism and batching ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,max_batch", [(1, 1), (5, 2), (7, 8)])
def test_tf32_decode_batches_and_chunks(B, max_batch):
    cfg = S1.TINY_S1
    P = S1.make_params(cfg, seed=3)
    ct, cb = _codes(cfg, B, B)
    dec = _decoder(cfg, P, max_batch=max_batch)
    a = dec.decode_code(ct, cb)
    assert torch.equal(a, dec.decode_code(ct, cb))
    single = dec.decode_code(ct[B - 1:], cb[B - 1:])
    assert torch.equal(single[0], a[B - 1])
    got = a.cpu()
    _check_fp32_bars(_report(f"tiny B={B} max_batch={max_batch} vs fp32", got, S1.decode_code(P, cfg, ct, cb)))
    emu = T.decode_code(P, cfg, ct, cb)
    m = _report(f"tiny B={B} max_batch={max_batch} vs tf32 emulation", got, emu)
    # on these images the emulation bars (5e-3 / 5e-4) are at the floor any fp32 accumulation order reaches: the same
    # emulation with fp64 between the rounding points lands about as far away (mean 4.9e-4, max 3.3e-3 - 4.1e-3)
    floor = _report("  tf32 emulation, fp64 vs fp32 accumulation", T.decode_code(P, cfg, ct, cb, accumulate=torch.float64), emu)
    assert m[0] <= max(5e-3, 1.5 * floor[0]) and m[1] <= max(5e-4, 1.5 * floor[1]), (m, floor)


# ---- 5. range: activations beyond fp16's 65504 --------------------------------------------------------------------------
def test_tf32_decode_keeps_the_fp32_range():
    cfg = S1.TINY_S1
    P = S1.make_params(cfg, seed=4)
    for name in ("quantize_t.embedding", "quantize_b.embedding"):
        P[name] = P[name] * 3e5
    assert float(P["quantize_b.embedding"].abs().max()) > 65504       # the gathered conv input itself overflows fp16
    ct, cb = _codes(cfg, 3, 11)
    got = _decoder(cfg, P, max_batch=4).decode_code(ct, cb).cpu()
    assert torch.isfinite(got).all()
    want = S1.decode_code(P, cfg, ct, cb)
    e = (got - want).abs()
    print(f"\n[tf32 stage 1] scaled codebook: max |out| {float(want.abs().max()):.3f} max-abs {float(e.max()):.3e} "
          f"mean-abs {float(e.mean()):.3e}")
    assert float(e.max()) <= 1e-2 * float(want.abs().max()) and float(e.mean()) <= 1e-3 * float(want.abs().mean())


# ---- 6. API -------------------------------------------------------------------------------------------------------------
def test_image_gpt2_sample_with_tf32_stage1_and_hq_create_rejects_tf32():
    import ctypes as C
    import hqtransformer_b200 as H
    from hqtransformer_b200 import _lib
    path = os.path.join(os.path.dirname(H.__file__), "configs", "imagenet_l12.yaml")
    model = H.ImageGPT2.from_config(path, with_stage1=True, stage1_max_batch=4, stage1_precision="tf32", device=0,
                                    precision="bf16", max_batch=4).eval()
    assert model.stage1.precision == "tf32"
    px = model.sample(cls_idx=7, top_k=256, num_candidates=4, is_tqdm=False)
    assert tuple(px.shape) == (4, 3, 256, 256) and float(px.min()) >= 0.0 and float(px.max()) <= 1.0
    lib = _lib.load()
    cfg = _lib.HQConfig(embed_dim=64, n_heads=1, n_layers=1, n_layers_depth=1, vocab_top=64, vocab_bot=64, n_classes=4,
                        ctx_len_img=4, cond_kind=_lib.HQ_COND_CLS, precision=_lib.HQ_PREC_TF32, max_seq_len=4)
    ctx = C.c_void_p()
    assert lib.hq_create(C.byref(cfg), 0, 1, C.byref(ctx)) == 1 and not ctx.value   # HQ_ERR_INVALID
    assert b"stage-1" in lib.hq_last_error(None)
