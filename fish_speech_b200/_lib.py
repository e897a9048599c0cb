"""ctypes binding of include/fishb200.h.  Fails loudly when the CUDA library is absent."""
from __future__ import annotations

import ctypes as C
from pathlib import Path

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "libfishb200.so"


class FsbError(RuntimeError):
    pass


class LmConfig(C.Structure):
    _fields_ = [(n, C.c_int) for n in (
        "dim", "n_layer", "n_head", "n_kv_head", "head_dim", "intermediate",
        "fast_dim", "n_fast_layer", "fast_n_head", "fast_n_kv_head", "fast_head_dim", "fast_intermediate",
        "vocab_size", "codebook_size", "num_codebooks",
        "semantic_begin_id", "semantic_end_id", "im_end_id")] + [("norm_eps", C.c_float)] + [
        (n, C.c_int) for n in (
            "qk_norm", "fast_qk_norm", "scale_codebook_embeddings", "norm_fastlayer_input",
            "max_batch", "kv_len", "max_rows", "max_frames", "debug")]


class LmLayer(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "d_attn_norm", "d_wqkv", "d_bqkv", "d_q_norm", "d_k_norm", "d_wo", "d_bo", "d_ffn_norm", "d_w13", "d_w2")]


class LmWeights(C.Structure):
    _fields_ = [
        ("d_embeddings", C.c_void_p), ("d_codebook_embeddings", C.c_void_p), ("d_norm", C.c_void_p),
        ("d_head", C.c_void_p), ("head_rows", C.c_int), ("d_freqs", C.c_void_p),
        ("layers", C.POINTER(LmLayer)),
        ("d_fast_embeddings", C.c_void_p), ("d_fast_norm", C.c_void_p), ("d_fast_output", C.c_void_p),
        ("d_fast_freqs", C.c_void_p), ("d_fast_proj_w", C.c_void_p), ("d_fast_proj_b", C.c_void_p),
        ("fast_layers", C.POINTER(LmLayer)),
    ]


class Sampling(C.Structure):
    _fields_ = [("temperature", C.c_float), ("top_p", C.c_float), ("top_k", C.c_int),
                ("seed", C.c_ulonglong)]


class SlotCtlArgs(C.Structure):
    """fsb_op_slot_ctl (include/fishb200.h)."""
    _fields_ = [("state", C.c_void_p), ("limit", C.c_void_p), ("temperature", C.c_void_p), ("top_p", C.c_void_p),
                ("top_k", C.c_void_p), ("seed", C.c_void_p), ("n_out", C.c_void_p)]


class SampleArgs(C.Structure):
    """fsb_op_sample_args (include/fishb200.h)."""
    _fields_ = [("ws", C.c_void_p), ("nparts", C.c_void_p), ("tiles", C.c_int), ("max_parts", C.c_int),
                ("n", C.c_int), ("rows", C.c_int), ("temperature", C.c_float), ("top_p", C.c_float),
                ("top_k", C.c_int), ("slow", C.c_int), ("n_sem", C.c_int), ("sem_begin", C.c_int),
                ("im_end_id", C.c_int), ("codebook_size", C.c_int), ("use_ras", C.c_int),
                ("ras_window", C.c_void_p), ("ras_update", C.c_int), ("seed", C.c_ulonglong),
                ("rng_offset", C.c_void_p), ("draw_id", C.c_int), ("cur_tok", C.c_void_p), ("cb_index", C.c_int),
                ("num_cb", C.c_int), ("logits_out", C.c_void_p), ("finished", C.c_void_p),
                ("row_slot", C.c_void_p), ("noise_u", C.c_void_p), ("noise_draws", C.c_int),
                ("noise_ld", C.c_int), ("ctl", SlotCtlArgs)]


_lib = None


def exported_symbols() -> list[str]:
    """Every function include/fishb200.h declares (checked by the CPU test-suite)."""
    import re

    hdr = (_HERE.parent / "include" / "fishb200.h").read_text()
    return sorted(set(re.findall(r"\b(fsb_[a-z0-9_]+)\s*\(", hdr)))


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise FsbError(
            f"{LIB_PATH} is missing: build it with `python -m fish_speech_b200.csrc.build` "
            "(there is no CPU / eager fallback for the hot path)")
    L = C.CDLL(str(LIB_PATH))
    L.fsb_last_error.restype = C.c_char_p
    L.fsb_launch_count.restype = C.c_longlong
    vp, i32 = C.c_void_p, C.c_int
    L.fsb_device_info.argtypes = [C.POINTER(i32)] * 3
    L.fsb_memcpy_d2h.argtypes = [vp, vp, C.c_size_t, vp]
    L.fsb_memcpy_h2d.argtypes = [vp, vp, C.c_size_t, vp]
    L.fsb_lm_create.argtypes = [C.POINTER(LmConfig), C.POINTER(LmWeights), C.POINTER(vp)]
    L.fsb_lm_destroy.argtypes = [vp]
    L.fsb_lm_destroy.restype = None
    L.fsb_lm_prefill.argtypes = [vp, vp, vp, vp, i32, vp, vp, i32, i32, C.POINTER(Sampling), vp]
    L.fsb_lm_decode.argtypes = [vp, i32, i32, C.POINTER(Sampling), i32, vp]
    L.fsb_lm_reset.argtypes = [vp, vp]
    L.fsb_lm_set_context_bound.argtypes = [vp, i32]
    L.fsb_lm_set_slot_control.argtypes = [vp, i32]
    L.fsb_lm_buffer.argtypes = [vp, C.c_char_p, C.POINTER(vp), C.POINTER(C.c_size_t)]
    L.fsb_lm_set_sampler_noise.argtypes = [vp, vp, i32, i32]
    L.fsb_lm_copy_kv.argtypes = [vp, i32, i32, i32, vp]
    L.fsb_lm_repeat_step_gemm.argtypes = [vp, i32, i32, i32, vp]
    L.fsb_lm_trace_frame.argtypes = [vp, i32, C.POINTER(Sampling), vp, i32, vp, i32, vp]
    L.fsb_lm_trace_step_gemms.argtypes = [vp, vp, i32, C.POINTER(i32), vp]
    L.fsb_lm_bench_gemms.argtypes = [vp, i32, C.POINTER(C.c_double), C.POINTER(i32), vp]
    f32p, i32p, ll = C.c_void_p, C.POINTER(C.c_int), C.c_longlong
    L.fsb_conv_gemm.argtypes = [vp, i32, i32, i32, i32, ll, vp, i32, i32, i32, i32p, i32, vp, vp, vp, i32, vp, vp, vp,
                                vp, i32, vp]
    L.fsb_linear_f32.argtypes = [vp, i32, i32, vp, i32, vp, vp]
    L.fsb_codebook_sum.argtypes = [vp, vp, vp, i32, i32, i32, i32, vp, vp]
    L.fsb_dwconv_ln.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, i32, C.c_float, vp, vp]
    L.fsb_final_conv_tanh.argtypes = [vp, vp, C.c_float, i32, i32, i32, i32, vp, vp]
    L.fsb_first_conv.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, i32, vp, vp, vp]
    L.fsb_snake.argtypes = [vp, vp, vp, ll, i32, vp, vp]
    L.fsb_vq_encode.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp, vp]
    L.fsb_resid_scale_norm.argtypes = [vp, i32, vp, vp, vp, vp, vp, i32, i32, C.c_float, i32, vp]
    L.fsb_qkv_rope.argtypes = [vp, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, i32, vp]
    L.fsb_res_unit_supported.argtypes = [i32]
    L.fsb_res_unit.argtypes = [vp, vp, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.fsb_op_res_unit_trace.argtypes = [vp]
    L.fsb_op_attn_score_chunk.argtypes = [i32]
    L.fsb_window_attn.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, vp, vp]
    L.fsb_swiglu_f32.argtypes = [vp, i32, i32, vp, vp]
    L.fsb_op_gemm.argtypes = [vp, vp, vp, i32, i32, i32, i32, i32, vp]
    L.fsb_op_step_gemm.argtypes = [vp, i32, i32, vp, i32, i32, vp, i32, vp, C.c_float, i32, i32, vp, C.c_size_t,
                                   vp, i32p, i32p, i32p, vp]
    L.fsb_op_step_finalize.argtypes = [i32, vp, vp, i32, i32, i32, i32, i32, vp, vp, vp, vp, vp, i32, vp]
    L.fsb_op_attn_decode.argtypes = [vp, vp, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32,
                                     i32, i32, i32, C.c_float, vp]
    L.fsb_op_sample.argtypes = [C.POINTER(SampleArgs), vp]
    L.fsb_op_frame_end.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, C.POINTER(SlotCtlArgs), vp]
    _lib = L
    return L


def check(rc: int) -> None:
    if rc != 0:
        raise FsbError(lib().fsb_last_error().decode("utf-8", "replace"))


def launch_count() -> int:
    return int(lib().fsb_launch_count())
