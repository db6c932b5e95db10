"""ctypes binding of the C ABI in include/twb200.h (libtwb200.so, built by build.py).

There is no CPU fallback: if the library is missing or no B200 is visible the calls raise.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TWB200_LIB", os.path.join(HERE, "libtwb200.so"))   # TWB200_LIB: probe builds (tools/probes)

TW_OK, TW_E_INVALID, TW_E_CUDA, TW_E_NOMEM, TW_E_UNSUPPORTED, TW_E_SHAPE, TW_E_STATE = 0, -1, -2, -3, -4, -5, -6
TW_F32, TW_BF16, TW_I16, TW_I32 = 0, 1, 2, 3

# every symbol include/twb200.h declares (tests check the library exports each one)
EXPORTS = [
    "tw_abi_version", "tw_ctx_create", "tw_ctx_destroy", "tw_last_error", "tw_launch_count", "tw_logmel",
    "tw_model_load", "tw_model_free", "tw_model_bytes", "tw_model_get_desc", "tw_workspace_bytes", "tw_encode", "tw_decode_greedy", "tw_transcribe_host",
    "tw_last_stage_ms", "tw_debug_gemm", "tw_profile", "tw_debug_set_pdl", "tw_debug_set_row_budgets", "tw_decoder_logits", "tw_debug_attention", "tw_debug_self_attention_paged",
    "tw_debug_decode_attention", "tw_debug_encoder_attention", "tw_debug_self_attention", "tw_debug_gemm_grouped",
    "tw_debug_absorbed_attention", "tw_pipeline_enable", "tw_pipeline_resize", "tw_pipeline_info", "tw_pipeline_stage_ms", "tw_pipeline_encode", "tw_pipeline_encode_at", "tw_pipeline_decode",
    "tw_debug_select_steps", "tw_debug_kv_append", "tw_debug_self_attention_step", "tw_debug_decode_attention_step",
    "tw_debug_layernorm", "tw_debug_cross_kv", "tw_debug_read_stage1", "tw_debug_decode_taps", "tw_debug_decoder_logits_taps",
    "tw_decode_greedy_rows", "tw_transcribe_host_rows", "tw_pipeline_decode_rows", "tw_debug_select_steps_rows", "tw_detect_language",
]


class ModelDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in
                ("d_model", "ffn", "heads", "enc_layers", "dec_layers", "n_mel", "vocab", "max_target", "dtype", "max_batch")]


class Weight(C.Structure):
    _fields_ = [("name", C.c_char_p), ("ptr", C.c_void_p), ("dtype", C.c_int32), ("numel", C.c_int64)]


class Rules(C.Structure):
    _fields_ = [("suppress", C.POINTER(C.c_int32)), ("n_suppress", C.c_int32),
                ("begin_suppress", C.POINTER(C.c_int32)), ("n_begin_suppress", C.c_int32),
                ("eos", C.c_int32), ("pad", C.c_int32), ("timestamp_begin", C.c_int32),
                ("no_timestamps", C.c_int32), ("max_initial_timestamp_index", C.c_int32)]


class PromptRows(C.Structure):
    _fields_ = [("prompts", C.POINTER(C.c_int32)), ("lang_ids", C.POINTER(C.c_int32)), ("n_lang", C.c_int32),
                ("out_lang", C.c_void_p)]


PROMPT_DETECT = -1       # at prompt index 1: detect the row's language there


class TwError(RuntimeError):
    pass


_lib = None


def load_library() -> C.CDLL:
    """Loads libtwb200.so; raises (loudly) when it has not been built — no fallback path exists."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise TwError(f"{LIB_PATH} is missing: build it with `python -m taiwan_whisper_b200.build` "
                      "(the B200 path has no CPU / PyTorch fallback)")
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    lib.tw_abi_version.restype = C.c_int
    lib.tw_ctx_create.argtypes = [C.c_int, C.POINTER(vp)]
    lib.tw_ctx_destroy.argtypes = [vp]
    lib.tw_ctx_destroy.restype = None
    lib.tw_last_error.argtypes = [vp]
    lib.tw_last_error.restype = C.c_char_p
    lib.tw_launch_count.argtypes = [vp]
    lib.tw_launch_count.restype = C.c_uint64
    lib.tw_logmel.argtypes = [vp, vp, C.c_int, i64, vp, C.c_int, C.c_int, vp, vp]
    lib.tw_model_load.argtypes = [vp, C.POINTER(ModelDesc), C.POINTER(Weight), C.c_size_t, C.POINTER(vp)]
    lib.tw_model_free.argtypes = [vp]
    lib.tw_model_free.restype = None
    lib.tw_model_bytes.argtypes = [vp]
    lib.tw_model_bytes.restype = C.c_size_t
    lib.tw_model_get_desc.argtypes = [vp, C.POINTER(ModelDesc)]
    lib.tw_workspace_bytes.argtypes = [C.POINTER(ModelDesc)]
    lib.tw_workspace_bytes.restype = C.c_size_t
    lib.tw_encode.argtypes = [vp, vp, C.c_int, vp, C.c_int, vp, vp]
    lib.tw_decode_greedy.argtypes = [vp, vp, C.c_int, C.POINTER(i32), C.c_int, C.POINTER(Rules), C.c_int, vp, vp, vp, vp,
                                     C.c_int, vp]
    lib.tw_transcribe_host.argtypes = [vp, vp, vp, C.c_int, C.POINTER(i32), C.c_int, C.POINTER(Rules), C.c_int, vp, vp, vp]
    lib.tw_last_stage_ms.argtypes = [vp, C.POINTER(C.c_float)]
    lib.tw_debug_decode_attention.argtypes = [vp, vp, i64, vp, i64, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp]
    lib.tw_debug_self_attention.argtypes = [vp, vp, i64, vp, i64, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp]
    lib.tw_debug_encoder_attention.argtypes = [vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp]
    lib.tw_debug_attention.argtypes = [vp, vp, i64, C.c_int, vp, i64, C.c_int, C.c_int, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                       C.c_int, C.c_int, vp]
    lib.tw_debug_self_attention_paged.argtypes = [vp, vp, i64, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp]
    lib.tw_decoder_logits.argtypes = [vp, vp, C.c_int, vp, C.c_int, vp, i64, vp]
    lib.tw_debug_set_row_budgets.argtypes = [vp, C.POINTER(C.c_int32), C.c_int]
    lib.tw_debug_set_pdl.argtypes = [C.c_int]
    lib.tw_debug_set_pdl.restype = None
    lib.tw_profile.argtypes = [vp, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_int), C.POINTER(C.c_double)]
    lib.tw_debug_gemm.argtypes = [vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, C.c_int, C.c_int, vp]
    lib.tw_debug_gemm_grouped.argtypes = [vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp]
    lib.tw_debug_absorbed_attention.argtypes = [vp, vp, vp, C.c_int, C.c_int, C.c_int, vp, vp, vp, C.c_int, vp]
    lib.tw_debug_select_steps.argtypes = [vp, vp, i64, C.c_int, C.POINTER(i32), C.c_int, C.POINTER(Rules), C.c_int, C.POINTER(i32), vp, vp,
                                          C.c_int, vp, vp, vp, vp, vp]
    lib.tw_debug_kv_append.argtypes = [vp, vp, vp, vp, vp, vp, vp, C.c_int, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp]
    lib.tw_debug_self_attention_step.argtypes = [vp, vp, i64, vp, i64, vp, C.c_int, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp]
    lib.tw_debug_decode_attention_step.argtypes = [vp, vp, i64, vp, i64, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, C.c_int, vp, vp]
    lib.tw_debug_layernorm.argtypes = [vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, vp]
    lib.tw_debug_cross_kv.argtypes = [vp, vp, C.c_int, C.c_int, vp]
    lib.tw_debug_read_stage1.argtypes = [vp, C.c_int, C.c_int, C.c_int, vp, C.c_int, vp, vp]
    lib.tw_debug_decode_taps.argtypes = [vp, vp, C.c_int, C.POINTER(i32), C.c_int, C.POINTER(Rules), C.c_int, vp, vp, vp, vp, C.c_int,
                                         vp, C.c_int, C.c_int, vp, C.c_int, vp]
    lib.tw_debug_decoder_logits_taps.argtypes = [vp, vp, C.c_int, vp, C.c_int, vp, i64, vp, vp]
    lib.tw_pipeline_enable.argtypes = [vp, C.c_int]
    lib.tw_pipeline_resize.argtypes = [vp, C.c_int]
    lib.tw_pipeline_stage_ms.argtypes = [vp, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_float)]
    lib.tw_pipeline_info.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.tw_pipeline_encode.argtypes = [vp, vp, vp, C.c_int, C.c_int]
    lib.tw_pipeline_encode_at.argtypes = [vp, vp, vp, C.c_int, C.c_int, C.c_int]
    lib.tw_pipeline_decode.argtypes = [vp, C.c_int, C.c_int, C.POINTER(i32), C.c_int, C.POINTER(Rules), C.c_int, vp, vp]
    rows = C.POINTER(PromptRows)
    lib.tw_decode_greedy_rows.argtypes = [vp, vp, C.c_int, rows, C.c_int, C.POINTER(Rules), C.c_int, vp, vp, vp, vp, C.c_int, vp]
    lib.tw_transcribe_host_rows.argtypes = [vp, vp, vp, C.c_int, rows, C.c_int, C.POINTER(Rules), C.c_int, vp, vp, vp]
    lib.tw_pipeline_decode_rows.argtypes = [vp, C.c_int, C.c_int, rows, C.c_int, C.POINTER(Rules), C.c_int, vp, vp]
    lib.tw_debug_select_steps_rows.argtypes = [vp, vp, i64, C.c_int, rows, C.c_int, C.POINTER(Rules), C.c_int, C.POINTER(i32), vp,
                                               vp, C.c_int, vp, vp, vp, vp, vp]
    lib.tw_detect_language.argtypes = [vp, vp, C.c_int, C.POINTER(i32), C.c_int, vp, vp]
    _lib = lib
    return lib


_EXC = {TW_E_INVALID: ValueError, TW_E_SHAPE: ValueError, TW_E_UNSUPPORTED: NotImplementedError,
        TW_E_NOMEM: MemoryError}


class Context:
    """One tw_ctx per device per process."""
    _by_device: dict = {}

    def __init__(self, device: int):
        self.lib = load_library()
        h = C.c_void_p()
        rc = self.lib.tw_ctx_create(device, C.byref(h))
        self.handle = h
        self.device = device
        if rc != TW_OK:
            msg = self.lib.tw_last_error(h).decode() if h else "tw_ctx_create failed"
            if h:
                self.lib.tw_ctx_destroy(h)
            self.handle = None
            raise _EXC.get(rc, TwError)(f"twb200: {msg}")

    @classmethod
    def get(cls, device: int) -> "Context":
        if device not in cls._by_device:
            cls._by_device[device] = Context(device)
        return cls._by_device[device]

    def check(self, rc: int):
        if rc != TW_OK:
            msg = self.lib.tw_last_error(self.handle).decode()
            raise _EXC.get(rc, TwError)(f"twb200: {msg}")

    def launch_count(self) -> int:
        return int(self.lib.tw_launch_count(self.handle))


def make_prompt_rows(prompts, lang_ids=None, out_lang=None):
    """Returns (PromptRows struct, keepalive, P) from per-row prompt lists of one length (PROMPT_DETECT at index 1 = detect);
    out_lang: address of the [B] int32 buffer for the languages, or None."""
    P = len(prompts[0])
    if any(len(p) != P for p in prompts):
        raise ValueError("every row's prompt must have the same length")
    flat = (C.c_int32 * (len(prompts) * P))(*[int(t) for p in prompts for t in p])
    langs = (C.c_int32 * max(1, len(lang_ids or ())))(*[int(t) for t in (lang_ids or ())])
    r = PromptRows(C.cast(flat, C.POINTER(C.c_int32)), C.cast(langs, C.POINTER(C.c_int32)) if lang_ids else None,
                   len(lang_ids or ()), out_lang)
    return r, (flat, langs), P


def make_rules(suppress, begin_suppress, eos, pad, timestamp_begin, no_timestamps, max_initial_ts):
    """Returns (Rules struct, keepalive) from python lists."""
    sup = (C.c_int32 * max(1, len(suppress)))(*suppress)
    beg = (C.c_int32 * max(1, len(begin_suppress)))(*begin_suppress)
    r = Rules(C.cast(sup, C.POINTER(C.c_int32)), len(suppress), C.cast(beg, C.POINTER(C.c_int32)), len(begin_suppress),
              eos, pad, -1 if timestamp_begin is None else timestamp_begin, no_timestamps,
              -1 if max_initial_ts is None else max_initial_ts)
    return r, (sup, beg)
