"""ctypes binding of libuem_b200.so (the C-ABI declared in include/uem_b200.h).

There is deliberately no CPU or PyTorch fallback: if the shared library is missing, or a tensor is
not on a CUDA device, the call raises.
"""
import ctypes
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# UEM_B200_LIB: development override (A/B builds of the same ABI); the product default is the in-tree library
LIB_PATH = os.environ.get("UEM_B200_LIB") or os.path.join(_HERE, "libuem_b200.so")

_c = ctypes
_P = _c.c_void_p
_I = _c.c_int
_L = _c.c_int64
_F = _c.c_float

# name -> (restype, argtypes); mirrors include/uem_b200.h one to one
SIGNATURES = {
    "uem_last_error": (_c.c_char_p, []),
    "uem_version": (_I, []),
    "uem_set_device": (_I, [_I]),
    "uem_kernel_launches": (_L, []),
    "uem_profile_refine_events": (_I, [_P, _P]),
    "uem_set_option": (_I, [_c.c_char_p, _I]),
    "uem_softmax_conf_entropy_argmax_f32": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _F, _P, _P, _P, _P, _P]),
    "uem_entropy_uvem_weight_f32": (_I, [_P, _I, _I, _L, _F, _F, _F, _F, _F, _P, _P, _P]),
    "uem_uvem_weight_f32": (_I, [_P, _L, _F, _F, _F, _F, _F, _P, _P]),
    "uem_uvem_terms_f32": (_I, [_P, _P, _I, _I, _L, _F, _F, _F, _F, _F, _I, _L, _P, _P, _P, _P]),
    "uem_class_max_ws_bytes": (_L, [_I, _I, _L]),
    "uem_class_max_f32": (_I, [_P, _I, _I, _L, _P, _P, _P, _P, _P]),
    "uem_pseudo_select_f32": (_I, [_P, _P, _I, _I, _L, _F, _F, _L, _I, _P, _P]),
    "uem_i64_minmax": (_I, [_P, _L, _P, _P]),
    "uem_region_reduce_ws_bytes": (_L, [_I, _L, _I]),
    "uem_region_reduce_f32": (_I, [_P, _L, _L, _L, _P, _I, _L, _I, _L, _I, _P, _P, _P]),
    "uem_region_reduce_i64": (_I, [_P, _L, _L, _L, _P, _I, _L, _I, _L, _I, _P, _P, _P]),
    "uem_superpixel_expand_ws_bytes": (_L, [_I, _L, _I]),
    "uem_superpixel_expand_i64": (_I, [_P, _P, _I, _L, _I, _L, _L, _P, _P, _P]),
    "uem_downscale_label_i64": (_I, [_P, _I, _I, _I, _I, _I, _L, _F, _P, _P, _P]),
    "uem_pearson_ws_bytes": (_L, [_I, _I]),
    "uem_pearson_nchw_ws_bytes": (_L, [_I, _L, _I, _I]),
    "uem_pearson_dist_nchw_f32": (_I, [_P, _I, _I, _L, _P, _I, _F, _I, _P, _P, _P]),
    "uem_pearson_dist_rows_f32": (_I, [_P, _L, _I, _P, _I, _F, _P, _P, _P]),
    "uem_label_refine_ws_bytes": (_L, [_I, _I, _L, _I]),
    "uem_label_refine_f32": (_I, [_I, _P, _P, _P, _I, _I, _P, _P, _L, _P, _P, _I, _I, _I, _I, _F, _P, _P, _P, _P]),
    "uem_class_stats_bytes": (_L, [_I, _I]),
    "uem_select_entropy_stats_f32": (_I, [_P, _P, _I, _I, _L, _F, _F, _L, _P, _P, _P, _P, _P]),
    "uem_class_stats_decode_f32": (_I, [_P, _I, _I, _P, _P, _P]),
    "uem_mine_ws_bytes": (_L, [_I, _I, _I, _I, _I, _I, _I, _L]),
    "uem_mine_ws_stats_offset": (_L, [_I, _I, _I, _I, _I, _I, _I, _L]),
    "uem_mine_ws_maxid_offset": (_L, [_I, _I, _I, _I, _I, _I, _I, _L]),
    "uem_mine_region_phase_f32": (_I, [_P, _L, _P, _I, _I, _I, _I, _I, _I, _I, _F, _P, _P]),
    "uem_mine_region_phase_xchg_f32": (_I, [_P, _L, _P, _I, _I, _I, _I, _I, _I, _I, _F, _P, _P, _I, _I, _I, _I, _P, _P]),
    "uem_mine_proto_phase_f32": (_I, [_P, _I, _P, _I, _I, _I, _I, _I, _I, _L, _F, _P, _P]),
    "uem_mine_refine_select_f32": (_I, [_I, _P, _I, _P, _P, _P, _I, _I, _P, _L, _P, _P, _I, _I, _I, _I, _F, _F, _F, _F,
                                        _L, _P, _P, _P, _P, _P, _P, _P]),
    "uem_proto_weight_4pixel_f32": (_I, [_P, _I, _I, _P, _I, _I, _I, _I, _L, _F, _P, _P]),
    "uem_proto_accum_ws_bytes": (_L, [_I, _I, _I]),
    "uem_proto_accum_soft_ws_bytes": (_L, [_I, _I, _I, _I, _I]),
    "uem_proto_accum_nchw_f32": (_I, [_P, _I, _I, _L, _P, _I, _L, _P, _P, _P, _P]),
    "uem_proto_accum_soft_f32": (_I, [_P, _I, _I, _I, _I, _P, _I, _I, _I, _P, _P, _P]),
    "uem_proto_fold_finalize_ema_f32": (_I, [_P, _I, _I, _I, _P, _F, _F, _F, _P, _P]),
    "uem_proto_finalize_ema_f32": (_I, [_P, _P, _L, _P, _I, _I, _F, _F, _F, _P, _P, _P]),
    "uem_class_hist_i64": (_I, [_P, _L, _I, _L, _P, _P]),
    "uem_class_weight_lookup_f32": (_I, [_P, _L, _I, _L, _P, _P, _P]),
    "uem_hist_f32": (_I, [_P, _L, _I, _F, _F, _P, _P]),
    "uem_bucketize_f32": (_I, [_P, _L, _P, _I, _P, _P]),
    "uem_label_plus1_u8_i64": (_I, [_P, _L, _P, _P]),
    "uem_pcl_ws_bytes": (_L, [_I, _I, _L]),
    "uem_pcl_forward_f32": (_I, [_P, _I, _I, _L, _P, _I, _P, _L, _F, _P, _P, _P, _P]),
    "uem_pcl_backward_f32": (_I, [_P, _I, _I, _L, _I, _P, _P, _P, _P, _P]),
    "uem_pack_local_f64": (_I, [_P, _P, _P, _I, _I, _P, _P]),
    "uem_pack_local_partials_f64": (_I, [_P, _I, _I, _I, _P, _P, _P]),
    "uem_fold_gathered_f64": (_I, [_P, _I, _I, _I, _P, _P, _P, _P]),
    "uem_iast_hist_bytes": (_L, [_I]),
    "uem_iast_conf_hist_f32": (_I, [_P, _I, _I, _L, _P, _P]),
    "uem_iast_thresholds_f64": (_I, [_P, _I, _P, _c.c_double, _F, _P, _P, _P, _P]),
    "uem_iast_labels_u8": (_I, [_P, _I, _I, _L, _P, _P, _P]),
    "uem_window_accumulate_f32": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P]),
    "uem_window_average_f32": (_I, [_P, _P, _I, _I, _L, _P]),
    "uem_views_mean_f32": (_I, [_P, _I, _L, _P, _P]),
    "uem_xchg_region_bytes": (_L, [_I, _I, _I, _I]),
    "uem_xchg_send_f32": (_I, [_P, _I, _I, _I, _P, _P, _P, _I, _I, _I, _I, _P, _I, _P]),
    "uem_xchg_wait_maxid": (_I, [_P, _I, _I, _I, _I, _I, _P, _P]),
    "uem_xchg_fold_finalize_ema_f32": (_I, [_P, _I, _I, _I, _I, _I, _I, _P, _F, _F, _F, _P, _P, _P, _P, _P]),
    "uem_xchg_exchange_fold_ema_f32": (_I, [_P, _I, _I, _I, _P, _P, _I, _I, _I, _I, _P, _F, _F, _F, _P, _P, _P, _P, _P]),
    "uem_xchg_status": (_I, [_P, _P, _P]),
    "uem_peer_alloc": (_I, [_L, _P, _P]),
    "uem_peer_open": (_I, [_P, _P]),
    "uem_peer_close": (_I, [_P]),
    "uem_peer_free": (_I, [_P]),
    "uem_uvem_loss_forward_f32": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _P, _P, _P, _P]),
    "uem_uvem_loss_backward_ws_bytes": (_L, [_I, _I, _I, _I, _I]),
    "uem_uvem_loss_backward_f32": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P]),
    "uem_tile_gather": (_I, [_P, _P, _L, _I, _I, _I, _P, _P, _I, _I, _I, _P, _P, _P, _P]),
    "uem_label_gather_u8": (_I, [_P, _L, _I, _I, _P, _P, _P, _I, _I, _I, _P, _I, _I, _L, _F, _P, _P, _P]),
    "uem_image_gather_u8": (_I, [_P, _L, _I, _I, _I, _P, _P, _P, _I, _I, _I, _P, _P, _P]),
}

_lock = threading.Lock()
_lib = None


class UemLibraryError(RuntimeError):
    pass


def load():
    """Loads libuem_b200.so and binds every symbol of include/uem_b200.h.  Raises if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise UemLibraryError(
                "libuem_b200.so not found at %s: build it with `python -m uemda_b200.build` "
                "(there is no CPU / PyTorch fallback for the mining path)" % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        if lib.uem_version() != 1:
            raise UemLibraryError("libuem_b200.so ABI version %d != 1" % lib.uem_version())
        # UEM_B200_OPTS="name=value,...": development override of uem_set_option switches (A/B runs of whole test files)
        for kv in filter(None, os.environ.get("UEM_B200_OPTS", "").split(",")):
            name, _, val = kv.partition("=")
            if lib.uem_set_option(name.strip().encode(), int(val)) != 0:
                raise UemLibraryError(lib.uem_last_error().decode("utf-8", "replace"))
        _lib = lib
    return _lib


def check(rc):
    if rc != 0:
        raise UemLibraryError(load().uem_last_error().decode("utf-8", "replace"))


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise UemLibraryError("uemda_b200 runs on CUDA tensors only (got device %s); "
                                  "there is no CPU fallback for the mining path" % t.device)


def ptr(t):
    return None if t is None else _P(t.data_ptr())


def stream_of(t):
    return _P(torch.cuda.current_stream(t.device).cuda_stream)


_bound = threading.local()


def bind(t):
    """Make the tensor's device current for the library's (static) CUDA runtime."""
    idx = t.device.index if t.device.index is not None else torch.cuda.current_device()
    if getattr(_bound, "dev", None) != idx:
        check(load().uem_set_device(idx))
        _bound.dev = idx
    return load()


def workspace(nbytes, like):
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=like.device)


def f32c(t):
    """contiguous fp32 view/copy (inputs are never mutated)."""
    if t.dtype != torch.float32:
        t = t.float()
    return t if t.is_contiguous() else t.contiguous()


def i64c(t):
    if t.dtype != torch.int64:
        t = t.long()
    return t if t.is_contiguous() else t.contiguous()
