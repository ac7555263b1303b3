"""ctypes binding of libtwb200.so (C ABI: include/twb200.h).  Fails loudly when the library is
missing — there is no fallback implementation of any kernel."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# TWB200_LIB: another build of the same library (kernel A/B variants made by tools/build_variants.sh); the default is the
# in-tree library __graft_entry__.build() makes
LIB_PATH = os.environ.get("TWB200_LIB") or os.path.join(_HERE, "libtwb200.so")

c_void_p, c_int32, c_int64, c_float, c_size_t = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_size_t


class TwError(RuntimeError):
    pass


class GemmArgs(C.Structure):
    _fields_ = [
        ("a", c_void_p), ("a_row_stride", c_int64), ("a_batch_stride", c_int64), ("a_rows", c_int32),
        ("a_row_off", c_void_p), ("w", c_void_p), ("batches", c_int32), ("rows", c_int32),
        ("n", c_int32), ("k", c_int32), ("bias", c_void_p), ("act", c_int32), ("resid", c_void_p),
        ("resid_ld", c_int64), ("resid_batch_rows", c_int64), ("out", c_void_p), ("out_f32", c_int32),
        ("out_ld", c_int64), ("out_batch_rows", c_int64), ("out_row_off", c_int32), ("out_mode", c_int32),
    ]


class SkinnyArgs(C.Structure):
    _fields_ = [("w", c_void_p), ("x", c_void_p), ("ldx", c_int32), ("bias", c_void_p), ("batch", c_int32),
                ("n", c_int32), ("k", c_int32), ("ln_gamma", c_void_p), ("ln_beta", c_void_p), ("ln_out_bf16", c_void_p),
                ("ln_counter", c_void_p), ("ln_part_out", c_void_p), ("x_bf16_out", c_void_p), ("ln_stats_out", c_void_p),
                ("ln_stats_in", c_void_p), ("ln_c", c_void_p)]


class FlacInfo(C.Structure):
    _fields_ = [("sample_rate", c_int32), ("channels", c_int32), ("bits_per_sample", c_int32), ("max_block", c_int32),
                ("total_samples", c_int64), ("md5", C.c_uint8 * 16)]


class BeamConfig(C.Structure):
    _fields_ = [(n, c_int32) for n in ("num_beams", "vocab", "max_length", "prompt_len", "eos", "pad", "no_timestamps",
                                       "max_initial_ts", "timestamps", "track_indices")] + [("length_penalty", c_float)]


class BeamState(C.Structure):
    _fields_ = [(n, c_void_p) for n in ("hist", "fin", "run_score", "fin_score", "fin_flag", "fin_len", "gram",
                                        "improvable", "hits_all", "ctrl")]


class Grammar(C.Structure):
    _fields_ = [(n, c_int32) for n in ("eos", "pad", "no_timestamps", "ts_begin", "vocab", "lang_first", "lang_last",
                                       "max_initial_ts", "begin_index")]


class RowState(C.Structure):
    _fields_ = [(n, c_int32) for n in ("pos", "finished", "last_ts", "text_lo", "ts_lo", "ts_hi", "begin", "mode")]


# name -> (restype, argtypes); mirrors include/twb200.h one to one (tests/test_abi.py checks it)
SIGNATURES = {
    "tw_last_error": (C.c_char_p, []),
    "tw_abi_version": (C.c_int, []),
    "tw_logmel_tables_bytes": (c_size_t, []),
    "tw_logmel_scratch_bytes": (c_size_t, [c_int32]),
    "tw_logmel_init": (C.c_int, [c_void_p, c_void_p]),
    "tw_logmel": (C.c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int32, c_void_p, c_void_p, c_void_p,
                            c_int64, c_int32, c_void_p]),
    "tw_logmel_long": (C.c_int, [c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                 c_int64, c_int32, c_void_p]),
    "tw_logmel_init_n": (C.c_int, [c_void_p, c_void_p, c_int32]),
    "tw_logmel_n": (C.c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int32, c_void_p, c_void_p, c_void_p,
                              c_int64, c_int32, c_int32, c_void_p]),
    "tw_logmel_long_n": (C.c_int, [c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_int64, c_int32, c_int32, c_void_p]),
    "tw_layernorm": (C.c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_float, c_void_p]),
    "tw_gemm_bf16": (C.c_int, [C.POINTER(GemmArgs), c_void_p]),
    "tw_attention_enc": (C.c_int, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int64, c_void_p]),
    "tw_set_pdl": (C.c_int, [c_int32]),
    "tw_set_cross_attn_stream": (C.c_int, [c_int32]),
    "tw_cross_attn_plan": (C.c_int, [c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p]),
    "tw_dec_embed": (C.c_int, [c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_void_p,
                               c_void_p, c_void_p, c_void_p]),
    "tw_dec_linear": (C.c_int, [C.POINTER(SkinnyArgs), c_int32, c_void_p, c_int32, c_void_p]),
    "tw_dec_qkv": (C.c_int, [C.POINTER(SkinnyArgs), c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_void_p]),
    "tw_dec_self_attn": (C.c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_int32, c_int32,
                                   c_void_p]),
    "tw_dec_cross_attn": (C.c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int32,
                                    c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p]),
    "tw_dec_lmhead_parts": (c_int32, [c_int32]),
    "tw_dec_max_rows": (c_int32, []),
    "tw_dec_lmhead": (C.c_int, [C.POINTER(SkinnyArgs), C.POINTER(Grammar), c_void_p, c_void_p, c_void_p, c_void_p,
                                c_void_p, c_void_p, c_void_p]),
    "tw_dec_finalize": (C.c_int, [c_void_p, c_void_p, c_int32, c_void_p, c_int32, c_void_p, c_void_p, c_void_p,
                                  C.POINTER(Grammar), c_int32, c_void_p]),
    "tw_attention_enc_set_trace": (C.c_int, [c_void_p]),
    "tw_shift_frames": (C.c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int64,
                                  c_int32, c_void_p]),
    "tw_logmel_long_multi": (C.c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_void_p, c_void_p, c_void_p,
                                       c_int32, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_void_p]),
    "tw_gather_frames": (C.c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_int64, c_int32,
                                   c_void_p]),
    "tw_resample": (C.c_int, [c_void_p, c_int32, c_int32, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_int32, c_int32,
                              c_int32, c_void_p]),
    "tw_prefill_embed": (C.c_int, [c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_int32, c_void_p]),
    "tw_prefill_kv_store": (C.c_int, [c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_int32, c_int32, c_void_p]),
    "tw_prefill_self_attn": (C.c_int, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p]),
    "tw_prefill_cross_attn": (C.c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p,
                                        c_int32, c_int32, c_int32, c_int32, c_void_p]),
    "tw_dec_align_tap": (C.c_int, [c_void_p, c_int32, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_void_p, c_void_p,
                                   c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p]),
    "tw_align_matrix": (C.c_int, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32,
                                  c_void_p, c_void_p, c_void_p]),
    "tw_dtw_token_frames": (C.c_int, [c_void_p, c_int64, c_int32, c_int32, c_void_p]),
    "tw_dtw_token_frames_batch": (C.c_int, [c_void_p, c_int64, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_int32]),
    "tw_flac_info_read": (C.c_int, [c_void_p, c_int64, c_void_p]),
    "tw_flac_decode": (C.c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p]),
    "tw_beam_record_width": (c_int32, [C.POINTER(BeamConfig)]),
    "tw_beam_step": (C.c_int, [C.POINTER(BeamConfig), C.POINTER(BeamState), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                               c_void_p, c_void_p, c_int32, c_void_p, c_int32, c_int32, c_void_p, c_int32, c_int32, c_int32,
                               c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_void_p]),
    "tw_beam_step_host": (C.c_int, [C.POINTER(BeamConfig), C.POINTER(BeamState), c_void_p, c_int32, c_void_p, c_void_p,
                                    c_void_p, c_void_p, c_int32]),
    # host-only: (tw_asr_window*, n, tw_asr_config*, out_tokens, cap, offsets, t0, t1, lang, max_chunks, n_chunks*, flags*)
    "tw_decode_asr": (C.c_int, [c_void_p, c_int32, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p,
                                c_int32, c_void_p, c_void_p]),
}

_lib = None


def load() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise TwError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  turbo-whisper-workspace_b200 has no CPU or PyTorch fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        if lib.tw_abi_version() != 1:
            raise TwError("libtwb200.so ABI version mismatch")
        _lib = lib
    return _lib


_SYNC_CHECK = bool(os.environ.get("TWB200_SYNC_CHECK"))   # debug: synchronise after every call so a device fault names its kernel


def check(status: int, what: str = "") -> None:
    if status != 0:
        msg = load().tw_last_error().decode("utf-8", "replace")
        raise TwError(f"{what or 'libtwb200'} failed (status {status}): {msg}")
    if _SYNC_CHECK:
        import torch
        try:
            torch.cuda.synchronize()
        except Exception as e:  # noqa: BLE001
            raise TwError(f"device fault detected after {what or 'a libtwb200 call'}: {e}") from e
