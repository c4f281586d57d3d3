"""ctypes binding of libwenet_b200.so (include/wenet_b200.h).

The product path has NO CPU fallback: if the shared library is missing, or no CUDA device is
present, the compute entry points raise.  `load()` never silently substitutes anything.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("WENET_B200_LIB") or os.path.join(_HERE, "lib", "libwenet_b200.so")

_lib = None

c_i32p = C.POINTER(C.c_int32)
c_f32p = C.POINTER(C.c_float)
vp = C.c_void_p
i64 = C.c_int64
i32 = C.c_int
f32 = C.c_float
sz = C.c_size_t


class WbModelConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "input_dim", "d_model", "heads", "ffn_dim", "enc_layers", "cnn_kernel", "cnn_causal",
        "cnn_norm", "vocab", "dec_layers", "rdec_layers", "dec_heads", "dec_ffn_dim", "max_pos",
        "has_cmvn", "precise")] + [("ln_eps", C.c_float), ("dec_ln_eps", C.c_float)] + [(n, C.c_int32) for n in (
        "arch", "dec_flavor", "dec_max_len")]


class WbContextGraph(C.Structure):
    _fields_ = [("num_nodes", C.c_int32)] + [(n, C.c_void_p) for n in (
        "child_off", "child_tok", "child_node", "fail", "token", "node_score", "token_score", "output_score")]


# name -> (restype, argtypes); mirrors include/wenet_b200.h one to one
_PROTOS = {
    "wb_last_error": (C.c_char_p, []),
    "wb_version": (C.c_char_p, []),
    "wb_launch_count": (C.c_ulonglong, []),
    "wb_set_sm_reserve": (None, [i32]),
    "wb_prof_enable": (None, [i32]),
    "wb_prof_reset": (None, []),
    "wb_prof_num_tags": (i32, []),
    "wb_prof_tag_name": (C.c_char_p, [i32]),
    "wb_prof_collect": (i32, [vp, vp, vp]),
    "wb_fbank_create": (i32, [C.POINTER(vp), i32, i32, i32, f32, vp, vp]),
    "wb_fbank_destroy": (None, [vp]),
    "wb_fbank_forward": (i32, [vp, vp, i32, i64, vp, i32, f32, vp, i64, i32, vp]),
    "wb_model_create": (i32, [C.POINTER(vp), C.POINTER(WbModelConfig)]),
    "wb_model_destroy": (None, [vp]),
    "wb_model_set_tensor": (i32, [vp, C.c_char_p, vp, i32, i64]),
    "wb_model_finalize": (i32, [vp, vp]),
    "wb_encoder_workspace_bytes": (sz, [vp, i32, vp]),
    "wb_encoder_out_rows": (i64, [i32, vp]),
    "wb_encoder_forward": (i32, [vp, vp, i64, vp, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, sz, vp]),
    "wb_encoder_chunk_workspace_bytes": (sz, [vp, i32, i32]),
    "wb_encoder_forward_chunk": (i32, [vp, vp, i32, i32, i32, vp, i32, vp, vp, vp, vp,
                                        C.POINTER(C.c_int), C.POINTER(C.c_int), vp, sz, vp]),
    "wb_encoder_forward_chunk_static": (i32, [vp, vp, i32, vp, i32, vp, i32, vp, vp, vp, vp, vp, sz, vp]),
    "wb_encoder_chunk_batch_workspace_bytes": (sz, [vp, i32, i32, i32]),
    "wb_encoder_forward_chunk_batch": (i32, [vp, vp, i32, i32, vp, i32, vp, i32, vp, vp, vp, vp, C.POINTER(C.c_int),
                                              C.POINTER(C.c_int), vp, sz, vp]),
    "wb_encoder_forward_chunk_batch_static": (i32, [vp, vp, i32, i32, vp, i32, vp, i32, vp, vp, vp, vp, vp, sz, vp]),
    "wb_unpack_rows": (i32, [vp, vp, vp, i32, i32, i32, vp, i64, vp]),
    "wb_ctc_logprobs": (i32, [vp, vp, i64, i32, f32, vp, i64, i32, vp, vp, vp]),
    "wb_ctc_topk": (i32, [vp, vp, i64, i32, f32, vp, i64, i32, vp, vp, vp]),
    "wb_ctc_greedy_search": (i32, [vp, i32, vp, vp, i32, i32, vp, i32, vp, vp]),
    "wb_prefix_beam_workspace_bytes": (sz, [i32, i32, i32]),
    "wb_ctc_prefix_beam_search": (i32, [vp, vp, i32, vp, vp, i32, i32, i32, i32, vp, vp, vp, vp, vp,
                                         vp, sz, vp]),
    "wb_ctc_prefix_beam_search_ctx": (i32, [vp, vp, i32, vp, vp, i32, i32, i32, i32, C.POINTER(WbContextGraph), vp, vp, vp,
                                             vp, vp, vp, sz, vp]),
    "wb_rescoring_workspace_bytes": (sz, [vp, i64, i64]),
    "wb_attention_rescoring": (i32, [vp, vp, i64, vp, vp, i32, i32, vp, vp, vp, vp, vp, i32, i32, f32,
                                      f32, vp, vp, vp, vp, vp, sz, vp]),
    "wb_gemm_diag": (i32, [vp, i32]),
    "wb_attention_rescoring_dev": (i32, [vp, vp, i64, vp, vp, i32, i32, vp, vp, vp, vp, vp, i32, i32, f32,
                                          f32, vp, vp, vp, vp, vp, sz, vp]),
    "wb_prefix_share_tables": (i32, [i32, i32, i32, vp, vp, vp, vp, i32, vp, vp, vp, vp, vp, vp]),
    "wb_decoder_logprobs": (i32, [vp, vp, i64, vp, vp, i32, i32, vp, vp, vp, vp, i32, i32, i32, vp, vp,
                                   i64, vp, sz, vp]),
    "wb_attention_beam_workspace_bytes": (sz, [vp, i64, i32, i32, i32]),
    "wb_attention_beam_search": (i32, [vp, vp, i64, vp, vp, i32, i32, vp, i32, i32, i32, f32, vp, i32, vp, vp, vp, vp, sz, vp]),
    "wb_logmel_create": (i32, [C.POINTER(vp), i32, i32, i32, vp, vp]),
    "wb_logmel_destroy": (None, [vp]),
    "wb_logmel_forward": (i32, [vp, vp, i64, vp, i32, vp, i64, i32, vp, vp]),
    "wb_whisper_encoder_out_rows": (i64, [i32, vp, i32]),
    "wb_whisper_encoder_workspace_bytes": (sz, [vp, i32, vp, i32]),
    "wb_whisper_encoder_forward": (i32, [vp, vp, i64, vp, i32, i32, vp, vp, vp, vp, vp, sz, vp]),
    "wb_op_attention_beam_step": (i32, [vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp]),
    "wb_op_gemm": (i32, [vp, i64, vp, i32, i32, i32, vp, i32, f32, vp, i64, i32, vp]),
    "wb_op_gemm_resid_splitk": (i32, [vp, i64, vp, i32, i32, i32, vp, f32, vp, i64, vp]),
    "wb_op_gemm_resid_ln": (i32, [vp, i64, vp, i32, i32, i32, vp, f32, vp, i64, vp, vp, vp, vp, f32, vp, i64, vp]),
    "wb_op_layernorm": (i32, [vp, i64, i32, i32, vp, vp, f32, vp, i64, i32, vp, i64, vp]),
    "wb_op_cast_bf16": (i32, [vp, i64, i32, i32, vp, i64, i32, vp]),
    "wb_op_attention": (i32, [vp, i64, i64, i32, vp, i64, i64, i32, vp, i64, i64, i32, vp, i32, vp, vp,
                               vp, vp, i32, i32, i32, i32, i32, f32, vp, i64, i32, i32, vp]),
    "wb_op_relpos_kprep": (i32, [vp, i64, vp, vp, vp, vp, i32, i32, vp, i64, vp, vp]),
    "wb_op_dwconv": (i32, [vp, i64, vp, vp, vp, i32, i32, i32, i32, i32, i32, vp, vp, i32, vp, vp, f32,
                            vp, i32, vp, i64, vp]),
    "wb_op_logsoftmax_topk": (i32, [vp, i64, i32, i32, i32, f32, i32, vp, vp, vp]),
    "wb_op_lse_topk_sliced": (i32, [vp, i64, i32, i32, i32, i32, vp, vp, vp, sz, vp]),
    "wb_op_lse_topk": (i32, [vp, i64, i32, i32, i32, f32, i32, vp, vp, vp]),
    "wb_op_attention_ex": (i32, [vp, i64, i64, i32, vp, i64, i64, i32, vp, i64, i64, i32, vp, i32, vp, vp,
                                  vp, vp, i32, i32, i32, i32, i32, f32, vp, i64, i32, i32, i32, i32, vp, vp, vp]),
    "wb_op_lse_parts": (i32, [i32, i32]),
    "wb_op_gemm_lse_partials": (i32, [vp, i64, vp, i32, i32, i32, vp, vp, vp]),
    "wb_op_lse_target_logprob": (i32, [vp, i32, vp, i64, vp, i32, vp, vp, vp, i32, i32, vp, vp]),
    "wb_op_embed_tokens": (i32, [vp, vp, i32, i32, vp, vp, f32, vp, vp]),
    "wb_op_rescore_combine": (i32, [vp, vp, vp, vp, vp, vp, i32, vp, f32, f32, vp, vp, vp]),
    "wb_op_dec_self_attn_step": (i32, [vp, vp, vp, i32, i32, i32, i32, i32, f32, vp, vp]),
}

EXPORTED_SYMBOLS = tuple(sorted(_PROTOS))


class WbError(RuntimeError):
    pass


def lib_available() -> bool:
    return os.path.exists(LIB_PATH)


def load():
    """dlopen the in-tree library (building it is `python -m wenet_b200.build`)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise WbError(
            "libwenet_b200.so not found at %s — build it with `python -m wenet_b200.build` "
            "(there is no CPU fallback)" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _PROTOS.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().wb_last_error()
        raise WbError("%s failed (%d): %s" % (what or "wenet_b200 call", rc,
                                               msg.decode() if msg else "?"))


def ptr(t):
    """device/host pointer of a torch tensor or numpy array (None -> NULL)."""
    if t is None:
        return None
    if hasattr(t, "data_ptr"):
        return C.c_void_p(t.data_ptr())
    return C.c_void_p(t.ctypes.data)


def cur_stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
