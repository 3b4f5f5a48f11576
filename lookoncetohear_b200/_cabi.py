"""ctypes binding of include/lookonce_b200.h.  The only compute entry into the product.

There is no fallback: if the shared library is missing or fails to load, importing the engine
raises.  (Build it with ``python -m lookoncetohear_b200.build`` or ``__graft_entry__.build()``.)
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "liblookonce_b200.so")

c_void_pp = ctypes.POINTER(ctypes.c_void_p)
c_float_p = ctypes.POINTER(ctypes.c_float)


class SepConfig(ctypes.Structure):
    """l2h_sep_config (configs/tsh.json model_params)."""
    _fields_ = [(n, ctypes.c_int32) for n in (
        "stft_chunk_size", "stft_pad_size", "embed_dim", "num_ch", "D", "L", "I", "J", "B", "H",
        "local_atten_len", "use_attn", "lookahead", "chunk_causal", "num_src")]


class EmbedConfig(ctypes.Structure):
    """l2h_embed_config (configs/embed.json model_params)."""
    _fields_ = [(n, ctypes.c_int32) for n in ("embed_dim", "num_ch", "n_fft", "stride", "num_blocks")]


_lib = None

_SIGS = {
    "l2h_abi_version": (ctypes.c_int, []),
    "l2h_last_error": (ctypes.c_char_p, []),
    "l2h_sep_create": (ctypes.c_int, [ctypes.POINTER(SepConfig), c_void_pp]),
    "l2h_sep_destroy": (ctypes.c_int, [ctypes.c_void_p]),
    "l2h_sep_load_weight": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_void_p, ctypes.c_int64]),
    "l2h_sep_weights_expected": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int32),
                                               ctypes.POINTER(ctypes.c_int32)]),
    "l2h_sep_commit_weights": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p]),
    "l2h_sep_state_bytes": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int32, ctypes.POINTER(ctypes.c_size_t)]),
    "l2h_sep_state_init": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p]),
    "l2h_sep_state_layout": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int64),
                                           ctypes.POINTER(ctypes.c_int64)]),
    "l2h_sep_state_offsets": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int64), ctypes.c_int32]),
    "l2h_sep_workspace_bytes": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_uint32,
                                              ctypes.POINTER(ctypes.c_size_t)]),
    "l2h_sep_forward": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64,
                                      ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                      ctypes.c_int64, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32,
                                      ctypes.c_int32, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_uint32,
                                      ctypes.c_void_p]),
    "l2h_sep_stream_host": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p,
                                          ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32,
                                          ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p,
                                          ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]),
    "l2h_sep_stream_dev": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p,
                                         ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32,
                                         ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p, ctypes.c_size_t,
                                         ctypes.c_void_p]),
    "l2h_sep_profile": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p,
                                      ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32,
                                      ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int32,
                                      ctypes.POINTER(ctypes.c_char_p), ctypes.POINTER(ctypes.c_float),
                                      ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int32),
                                      ctypes.c_void_p]),
    "l2h_sep_stream_workspace_bytes": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32,
                                                     ctypes.POINTER(ctypes.c_size_t)]),
    "l2h_sep_set_option": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_int32]),
    "l2h_sep_pipeline_frames": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int32)]),
    "l2h_sep_tap_info": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32,
                                       ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int32)]),
    "l2h_sep_launches_per_forward": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int32,
                                                   ctypes.POINTER(ctypes.c_int32)]),
    "l2h_sep_weight_info": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int32, ctypes.POINTER(ctypes.c_char_p),
                                          ctypes.POINTER(ctypes.c_int64)]),
    "l2h_sep_launch_count": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int64), ctypes.c_int32]),
    "l2h_sep_trace_start": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int32]),
    "l2h_sep_trace_read": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.POINTER(ctypes.c_int32)]),
    "l2h_eval_metrics": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32,
                                       ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p,
                                       ctypes.c_void_p]),
    "l2h_eval_binaural_workspace_bytes": (ctypes.c_int, [ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                                                        ctypes.POINTER(ctypes.c_size_t)]),
    "l2h_eval_binaural": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                                        ctypes.c_int32, ctypes.c_double, ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p,
                                        ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]),
    "l2h_render_binaural": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32,
                                          ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p,
                                          ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "l2h_embed_create": (ctypes.c_int, [ctypes.POINTER(EmbedConfig), c_void_pp]),
    "l2h_embed_destroy": (ctypes.c_int, [ctypes.c_void_p]),
    "l2h_embed_set_option": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_int32]),
    "l2h_embed_load_weight": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_void_p, ctypes.c_int64]),
    "l2h_embed_weights_expected": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int32),
                                                 ctypes.POINTER(ctypes.c_int32)]),
    "l2h_embed_commit_weights": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p]),
    "l2h_embed_workspace_bytes": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32,
                                                ctypes.POINTER(ctypes.c_size_t)]),
    "l2h_embed_max_batch": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int32, ctypes.POINTER(ctypes.c_int32)]),
    "l2h_embed_forward": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32,
                                        ctypes.c_int32, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]),
}


def lib():
    """Load (once) and return the shared library; raises if it is absent -- no CPU fallback."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not built: run `python -m lookoncetohear_b200.build` "
                "(the engine has no fallback path)")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(L, name)          # AttributeError if the symbol is missing
            fn.restype, fn.argtypes = res, args
        if L.l2h_abi_version() != 1:
            raise RuntimeError("liblookonce_b200.so ABI version mismatch")
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise RuntimeError(f"lookonce_b200 error {rc}: {lib().l2h_last_error().decode()}")


def declared_symbols():
    return sorted(_SIGS)
