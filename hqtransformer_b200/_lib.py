"""ctypes binding of libhqgraft.so (include/hqgraft.h).  No fallback: a missing or stale library is an error."""
from __future__ import annotations

import ctypes as C
import os

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG_DIR, "libhqgraft.so")
ABI_VERSION = 9

HQ_OK = 0
HQ_COND_CLS, HQ_COND_TXT, HQ_COND_UNCOND = 0, 1, 2
HQ_PREC_BF16, HQ_PREC_FP32, HQ_PREC_F16, HQ_PREC_TF32 = 0, 1, 2, 3
HQ_PREC = {"bf16": HQ_PREC_BF16, "fp32": HQ_PREC_FP32, "fp16": HQ_PREC_F16}
HQ_F32, HQ_BF16, HQ_F16 = 0, 1, 2
HQ_MODEL = {"parallel": 0, "top2bot": 1, "bidirectional": 2}
HQ_EMB = {"transformer1": 0, "reduce": 1}
HQ_POS = {"1d": 0, "2d": 1}


class HQConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "embed_dim", "n_heads", "n_layers", "n_layers_depth", "vocab_top", "vocab_bot", "vocab_txt", "n_classes",
        "ctx_len_img", "ctx_len_txt", "cond_kind", "precision", "max_seq_len", "use_cuda_graph", "use_pdl", "use_chain", "model_type", "embedding_kind",
        "position_kind", "code_levels", "vocab_mid", "fuse_head_sampler")]


class HQSamplingParams(C.Structure):
    _fields_ = [("top_k_top", C.c_int32), ("top_k_bot", C.c_int32),
                ("top_p_top", C.c_float), ("top_p_bot", C.c_float),
                ("temperature_top", C.c_float), ("temperature_bot", C.c_float),
                ("seed", C.c_uint64), ("row_offset", C.c_uint64),
                ("top_k_mid", C.c_int32), ("top_p_mid", C.c_float), ("temperature_mid", C.c_float), ("reserved", C.c_int32)]


class HQRunArgs(C.Structure):
    _fields_ = [("batch", C.c_int32), ("seq_len", C.c_int32), ("pos_begin", C.c_int32), ("pos_end", C.c_int32),
                ("cond", C.c_void_p), ("sos", C.c_void_p), ("given_top", C.c_void_p), ("given_bot", C.c_void_p),
                ("codes_top", C.c_void_p), ("codes_bot", C.c_void_p), ("logits", C.c_void_p),
                ("sampling", HQSamplingParams), ("codes_mid", C.c_void_p), ("given_mid", C.c_void_p),
                ("shared_prefix", C.c_int32), ("prefix_len", C.c_int32)]


class HQDebugEpi(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "epi", "tile", "ks1", "D", "sec0", "rpb", "t_stride", "t0", "w_row_off", "ldo", "splits", "reserved")] + \
        [("split_stride", C.c_uint64)] + \
        [(n, C.c_void_p) for n in ("bias", "q", "kdst", "vdst", "vdup", "x", "out", "outf")]


class HQS1Config(C.Structure):
    _fields_ = [("embed_dim", C.c_int32), ("n_embed", C.c_int32), ("z_channels", C.c_int32), ("resolution", C.c_int32),
                ("ch", C.c_int32), ("ch_mult", C.c_int32 * 8), ("n_levels", C.c_int32), ("num_res_blocks", C.c_int32),
                ("attn_resolution", C.c_int32), ("out_ch", C.c_int32), ("precision", C.c_int32)]


# every symbol include/hqgraft.h declares: name -> (restype, argtypes)
PROTOTYPES = {
    "hq_abi_version": (C.c_int, []),
    "hq_last_error": (C.c_char_p, [C.c_void_p]),
    "hq_create": (C.c_int, [C.POINTER(HQConfig), C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "hq_destroy": (C.c_int, [C.c_void_p]),
    "hq_reserve_batch": (C.c_int, [C.c_void_p, C.c_int]),
    "hq_max_batch": (C.c_int, [C.c_void_p]),
    "hq_load_param": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int, C.POINTER(C.c_int64), C.c_int, C.c_int]),
    "hq_params_complete": (C.c_int, [C.c_void_p]),
    "hq_run": (C.c_int, [C.c_void_p, C.POINTER(HQRunArgs), C.c_void_p]),
    "hq_run_host": (C.c_int, [C.c_void_p, C.POINTER(HQRunArgs)]),
    "hq_last_launch_count": (C.c_int64, [C.c_void_p]),
    "hq_device_bytes": (C.c_size_t, [C.c_void_p]),
    "hq_chain_launch_count": (C.c_int64, [C.c_void_p]),
    "hq_debug_gemm": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                             C.c_void_p]),
    "hq_debug_gemm_epi": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                    C.POINTER(HQDebugEpi), C.c_void_p]),
    "hq_debug_layernorm": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                     C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_size_t, C.c_void_p,
                                     C.c_void_p]),
    "hq_debug_philox": (C.c_int, [C.c_uint64, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "hq_debug_sample": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_int, C.c_float, C.c_uint64, C.c_uint64,
                                  C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "hq_debug_attention": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                     C.c_int, C.c_int, C.c_void_p]),
    "hq_debug_attention_prefix": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                            C.c_int, C.c_int, C.c_void_p]),
    "hq_debug_attention_phases": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_uint64), C.c_int,
                                            C.POINTER(C.c_int), C.c_void_p]),
    "hq_debug_chain_phases": (C.c_int, [C.c_void_p, C.POINTER(HQRunArgs), C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_uint64),
                                        C.c_int, C.POINTER(C.c_int)]),
    "hq_bench_attention": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float), C.c_void_p]),
    "hq_trace_run": (C.c_int, [C.c_void_p, C.POINTER(HQRunArgs), C.c_void_p, C.POINTER(C.c_uint64), C.c_char_p, C.c_int,
                               C.POINTER(C.c_int)]),
    "hq_debug_gemm_phases": (C.c_int, [C.c_void_p, C.POINTER(HQRunArgs), C.c_void_p, C.c_int, C.POINTER(C.c_uint64), C.c_int,
                                       C.POINTER(C.c_uint64), C.c_char_p, C.c_int, C.POINTER(C.c_int)]),
    "hq_bench_gemm_shape": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float),
                                      C.POINTER(C.c_float), C.c_void_p]),
    "hq_bench_gemm": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float), C.c_void_p]),
    "hq_s1_create": (C.c_int, [C.POINTER(HQS1Config), C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "hq_s1_destroy": (C.c_int, [C.c_void_p]),
    "hq_s1_last_error": (C.c_char_p, [C.c_void_p]),
    "hq_s1_device_bytes": (C.c_size_t, [C.c_void_p]),
    "hq_s1_load_param": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int, C.POINTER(C.c_int64), C.c_int, C.c_int]),
    "hq_s1_params_complete": (C.c_int, [C.c_void_p]),
    "hq_s1_decode_codes": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "hq_s1_reserve_grid": (C.c_int, [C.c_void_p, C.c_int]),
    "hq_s1_decode_codes_grid": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "hq_s1_last_conv_flops": (C.c_double, [C.c_void_p]),
    "hq_debug_s1_conv": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                   C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "hq_debug_s1_groupnorm": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                        C.c_int, C.c_void_p, C.c_void_p]),
    "hq_debug_s1_resample": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "hq_debug_s1_quant": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                    C.c_int, C.c_int, C.c_void_p]),
    "hq_debug_s1_attention": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
}

_lib = None


class HQError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Loads libhqgraft.so, binds every prototype and checks the ABI version."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python hqtransformer_b200/build.py` "
            "(hqtransformer_b200 has no CPU or PyTorch fallback path)")
    path = LIB_PATH
    if os.environ.get("HQ_DEBUG", "0") not in ("", "0") and os.environ.get("HQGRAFT_LIB"):
        path = os.environ["HQGRAFT_LIB"]          # experiments only: an instrumented twin of the library (build.py --phase-stamps)
    lib = C.CDLL(path)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    got = lib.hq_abi_version()
    if got != ABI_VERSION:
        raise ImportError(f"libhqgraft.so ABI version {got} != binding version {ABI_VERSION}: rebuild the library")
    _lib = lib
    return lib


def check(rc: int, ctx=None, what: str = "") -> None:
    if rc != HQ_OK:
        msg = load().hq_last_error(ctx)
        raise HQError(f"{what or 'libhqgraft'} failed (status {rc}): {msg.decode() if msg else '?'}")


def check_s1(rc: int, ctx, lib, what: str = "") -> None:
    if rc != HQ_OK:
        msg = lib.hq_s1_last_error(ctx)
        raise HQError(f"{what or 'libhqgraft stage 1'} failed (status {rc}): {msg.decode() if msg else '?'}")
