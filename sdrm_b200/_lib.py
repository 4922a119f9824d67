"""ctypes binding of libsdrm_b200.so (the C ABI declared in include/sdrm_b200.h).

There is no CPU fallback: if the shared library is missing or a call fails, this raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SDRM_B200_LIB") or os.path.join(_HERE, "csrc", "libsdrm_b200.so")   # override: tuning builds only

_lib = None

# name -> (restype, argtypes); must list every symbol include/sdrm_b200.h declares
_P = C.c_void_p
SIGNATURES = {
    "sdrm_version": (C.c_int, []),
    "sdrm_last_error": (C.c_char_p, []),
    "sdrm_create": (C.c_int, [C.POINTER(_P), C.c_int]),
    "sdrm_destroy": (C.c_int, [_P]),
    "sdrm_denoiser_pack": (C.c_int, [_P] + [_P] * 11 + [C.c_int] * 4 + [C.c_float, _P]),
    "sdrm_decoder_pack": (C.c_int, [_P] + [_P] * 4 + [C.c_int] * 3 + [_P]),
    "sdrm_sample_workspace_bytes": (C.c_size_t, [_P, C.c_int64]),
    "sdrm_sample": (C.c_int, [_P, C.c_int64, C.c_int64, _P, _P, C.c_uint64, _P, _P, C.c_int64, _P, _P, _P, _P,
                              C.c_size_t, _P]),
    "sdrm_sample_bf16": (C.c_int, [_P, C.c_int64, C.c_int64, _P, _P, C.c_uint64, _P, _P, C.c_int64, _P, _P, _P, _P,
                                   C.c_size_t, _P]),
    "sdrm_last_launch_count": (C.c_int, [_P]),
    "sdrm_check_device_error": (C.c_int, [_P, _P]),
    "sdrm_probe_linear_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int, C.c_int]),
    "sdrm_set_option": (C.c_int, [_P, C.c_int, C.c_int64]),
    "sdrm_last_cluster_size": (C.c_int, [_P]),
    "sdrm_last_resident_mode": (C.c_int, [_P]),
    "sdrm_last_split_size": (C.c_int, [_P]),
    "sdrm_layer_geometry": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "sdrm_resident_ctas": (C.c_int, [_P, C.c_int]),
    "sdrm_probe_linear": (C.c_int, [_P, _P, _P, _P, C.c_int64, C.c_int, C.c_int, C.c_int, _P, C.c_size_t, _P]),
    "sdrm_topk": (C.c_int, [_P, C.c_int64, C.c_int, C.c_int64, C.c_int, _P, _P, _P]),
    "sdrm_topk_f64": (C.c_int, [_P, C.c_int64, C.c_int, C.c_int64, C.c_int, _P, _P, _P]),
    "sdrm_recall_ndcg_at_k": (C.c_int, [_P, C.c_int, C.c_int, _P, C.c_int64, C.c_int, C.c_int64, _P, _P, _P, _P]),
    "sdrm_noise_inputs": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int, C.c_float, C.c_double, C.c_uint64, C.c_int64,
                                    _P, _P, _P, _P, _P, _P, _P, _P]),
    "sdrm_loss_stats": (C.c_int, [_P, _P, _P, _P, C.c_int64, C.c_double, _P, _P]),
    "sdrm_encode_csr": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int, _P, _P, C.c_int, _P, _P]),
    "sdrm_multinomial_nll_fwd": (C.c_int, [_P, _P, C.c_int64, C.c_int, C.c_int64, C.c_int64, _P, _P, _P, _P]),
    "sdrm_multinomial_nll_bwd": (C.c_int, [_P, _P, C.c_int64, C.c_int, C.c_int64, C.c_int64, _P, _P, _P, C.c_float, _P, C.c_int64, _P]),
    "sdrm_key_histogram": (C.c_int, [_P, C.c_int64, C.c_int, C.c_int64, C.c_uint32, C.c_int, C.c_int, C.c_int, _P, _P]),
    "sdrm_threshold_pack": (C.c_int, [_P, C.c_int64, C.c_int, C.c_int64, C.c_double, C.c_int, _P, C.c_int64, _P, _P]),
    "sdrm_denoiser_train_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int, C.c_int, C.c_int]),
    "sdrm_denoiser_fwd": (C.c_int, [_P, _P, _P, C.c_int64, _P, C.c_int64, _P, _P, _P, _P, _P, _P, C.c_int64, C.c_int, C.c_int, C.c_int,
                                    C.c_int, _P, _P, C.c_size_t, _P]),
    "sdrm_denoiser_bwd": (C.c_int, [_P, _P, _P, _P, _P, C.c_int, _P, _P, _P, _P, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int,
                                    _P, _P, _P, _P, _P, _P, _P, _P, _P, C.c_size_t, _P]),
    "sdrm_train_check_device_error": (C.c_int, [_P, _P]),
    "sdrm_train_launch_count": (C.c_longlong, [C.c_int]),
    "sdrm_gemm_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int, C.c_int64, C.c_int]),
    "sdrm_gemm": (C.c_int, [_P, C.c_int64, C.c_int, _P, C.c_int64, C.c_int, _P, _P, C.c_int64, C.c_int64, C.c_int, C.c_int64, C.c_int,
                            C.c_int, _P, C.c_size_t, _P]),
    "sdrm_select_state_bytes": (C.c_size_t, []),
    "sdrm_select_begin": (C.c_int, [_P, C.c_uint64, C.c_uint64, _P]),
    "sdrm_select_histogram": (C.c_int, [_P, C.c_int64, C.c_int, C.c_int64, _P, C.c_int, _P, _P]),
    "sdrm_select_walk": (C.c_int, [_P, _P, C.c_int, C.c_double, C.c_int, _P]),
    "sdrm_select_threshold_pack": (C.c_int, [_P, C.c_int64, C.c_int, C.c_int64, _P, C.c_int, _P, C.c_int64, _P, _P]),
    "sdrm_key_histogram_bf16": (C.c_int, [_P, C.c_int64, C.c_int, C.c_int64, C.c_uint32, C.c_int, C.c_int, C.c_int, _P, _P]),
    "sdrm_threshold_pack_bf16": (C.c_int, [_P, C.c_int64, C.c_int, C.c_int64, C.c_double, C.c_int, _P, C.c_int64, _P, _P]),
    "sdrm_select_histogram_bf16": (C.c_int, [_P, C.c_int64, C.c_int, C.c_int64, _P, C.c_int, _P, _P]),
    "sdrm_select_walk_bf16": (C.c_int, [_P, _P, C.c_int, C.c_double, C.c_int, _P]),
    "sdrm_select_threshold_pack_bf16": (C.c_int, [_P, C.c_int64, C.c_int, C.c_int64, _P, C.c_int, _P, C.c_int64, _P, _P]),
    "sdrm_loss_grad_seeds": (C.c_int, [_P, _P, _P, _P, C.c_int64, C.c_double, _P, _P, _P, _P, _P, _P]),
}


OPT_CLUSTER, OPT_SUBTILES, OPT_GRID_LIMIT, OPT_NO_DISCARD, OPT_ENGINE, OPT_RESIDENT, OPT_NO_SPLIT, OPT_DEBUG_FLAGS, OPT_TRACE_BUFFER = 1, 2, 3, 4, 5, 6, 7, 100, 101   # enum sdrm_option


class SdrmError(RuntimeError):
    pass


def load():
    """Load the shared library once; raise loudly if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SdrmError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). There is no CPU fallback for the SDRM hot path.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        msg = load().sdrm_last_error().decode("utf-8", "replace")
        raise SdrmError(f"{what} failed ({rc}): {msg}")


def ptr(t):
    """Device pointer of a torch tensor (or None)."""
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


def stream_ptr(stream=None):
    import torch
    s = stream if stream is not None else torch.cuda.current_stream()
    return C.c_void_p(s.cuda_stream)
