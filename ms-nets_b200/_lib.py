"""ctypes binding of libmsnets_b200.so (the C ABI in include/msnets_b200.h).

There is no CPU fallback: if the shared library is missing, or a compute entry
point is called without a CUDA device, an exception is raised.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmsnets_b200.so")

c_int, c_ll, c_float, c_size_t, c_void_p = (ctypes.c_int, ctypes.c_longlong, ctypes.c_float,
                                            ctypes.c_size_t, ctypes.c_void_p)


class MsParams(ctypes.Structure):
    """struct msn_ms_params (include/msnets_b200.h); defaults = cbmv_generator.py:434-462."""
    _fields_ = [("ndisp", c_int), ("censw", c_int), ("nccw", c_int), ("sadw", c_int),
                ("sobelw", c_int), ("board_h", c_int), ("board_w_left", c_int),
                ("board_w_right", c_int), ("cens_sigma", c_float), ("ncc_sigma", c_float),
                ("sad_sigma", c_float), ("lr", c_int), ("d_begin", c_int), ("d_count", c_int),
                ("row_begin", c_int), ("row_count", c_int)]


class SlabExchange(ctypes.Structure):
    """struct msn_slab_exchange (include/msnets_b200.h)."""
    _fields_ = [("tables", c_void_p * 8), ("world", c_int), ("rank", c_int), ("epoch", ctypes.c_uint),
                ("subs", c_int)]


class MsnetsError(RuntimeError):
    pass


_P = c_void_p  # every buffer crosses as a raw address
_SIGNATURES = {
    "msn_last_error": (ctypes.c_char_p, []),
    "msn_abi_version": (c_int, []),
    "msn_device_count": (c_int, [ctypes.POINTER(c_int)]),
    "msn_set_device": (c_int, [c_int]),
    "msn_initthreads": (c_int, [ctypes.POINTER(c_int)]),
    "msn_census_host": (c_int, [_P, _P, c_int, c_int, c_int, c_int, _P]),
    "msn_ncc_host": (c_int, [_P, _P, c_int, c_int, c_int, c_int, _P]),
    "msn_zsad_host": (c_int, [_P, _P, c_int, c_int, c_int, c_int, _P]),
    "msn_sobel_host": (c_int, [_P, c_int, c_int, _P]),
    "msn_sadsob_host": (c_int, [_P, _P, c_int, c_int, c_int, c_int, _P]),
    "msn_swap_axes_host": (c_int, [_P, c_int, c_int, c_int, _P]),
    "msn_swap_axes_back_host": (c_int, [_P, c_int, c_int, c_int, _P]),
    "msn_right_cost_host": (c_int, [_P, c_int, c_int, c_int, _P]),
    "msn_left_cost_host": (c_int, [_P, c_int, c_int, c_int, _P]),
    "msn_aml_host": (c_int, [_P, c_ll, c_int, c_float, _P]),
    "msn_pkrn_host": (c_int, [_P, c_ll, c_int, c_float, _P]),
    "msn_ms_params_default": (None, [ctypes.POINTER(MsParams)]),
    "msn_features_from_costs_host": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_float, c_float,
                                             c_float, c_int, _P]),
    "msn_ms_features_host": (c_int, [_P, _P, c_int, c_int, c_int, ctypes.POINTER(MsParams), _P]),
    "msn_ms_features_workspace_bytes": (c_size_t, [c_int, c_int, c_int, ctypes.POINTER(MsParams)]),
    "msn_ms_features_dev": (c_int, [_P, _P, c_int, c_int, c_int, ctypes.POINTER(MsParams), _P, _P,
                                    c_size_t, _P]),
    "msn_ms_features_bf16_dev": (c_int, [_P, _P, c_int, c_int, c_int, ctypes.POINTER(MsParams), _P, _P, c_size_t, _P]),
    "msn_set_aml_exact": (c_int, [c_int]),
    "msn_get_aml_exact": (c_int, []),
    "msn_profile_enable": (c_int, [c_int]),
    "msn_profile_read": (c_int, [ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double),
                                 ctypes.POINTER(ctypes.c_double), ctypes.POINTER(c_int)]),
    "msn_ms_slab_workspace_bytes": (c_size_t, [c_int, c_int, c_int, ctypes.POINTER(MsParams)]),
    "msn_ms_slab_phase_a_dev": (c_int, [_P, _P, c_int, c_int, c_int, ctypes.POINTER(MsParams), _P, _P,
                                        _P, _P, c_size_t, _P]),
    "msn_ms_slab_phase_b_dev": (c_int, [_P, _P, c_int, c_int, c_int, ctypes.POINTER(MsParams), _P, _P]),
    "msn_ms_slab_phase_c_dev": (c_int, [_P, _P, _P, c_int, c_int, c_int, ctypes.POINTER(MsParams), _P]),
    "msn_ms_slab_exchange_bytes": (c_size_t, [c_int, c_int, c_int, ctypes.POINTER(MsParams), c_int, c_int]),
    "msn_ms_slab_fused_workspace_bytes": (c_size_t, [c_int, c_int, c_int, ctypes.POINTER(MsParams)]),
    "msn_ms_slab_fused_dev": (c_int, [_P, _P, c_int, c_int, c_int, ctypes.POINTER(MsParams), _P, _P, _P, _P, _P, _P,
                                      c_size_t, _P]),
    "msn_wta_merge_dev": (c_int, [_P, _P, _P, c_int, c_ll, _P, _P, _P, _P]),
    "msn_ms_features_wta_dev": (c_int, [_P, _P, c_int, c_int, c_int, ctypes.POINTER(MsParams), _P, _P, _P, _P, _P,
                                        c_size_t, _P]),
    "msn_peer_alloc": (c_int, [c_size_t, ctypes.POINTER(c_void_p)]),
    "msn_peer_free": (c_int, [_P]),
    "msn_peer_export": (c_int, [_P, _P]),
    "msn_peer_open": (c_int, [_P, ctypes.POINTER(c_void_p)]),
    "msn_peer_close": (c_int, [_P]),
    "msn_rescale_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "msn_rescale_dev": (c_int, [_P, c_int, c_int, c_int, c_int, c_int, _P, c_int, _P, c_int, ctypes.c_double,
                                ctypes.c_double, _P, _P, c_size_t, _P]),
    "msn_rescale_host": (c_int, [_P, c_int, c_int, c_int, c_int, c_int, _P, c_int, _P, c_int, ctypes.c_double,
                                 ctypes.c_double, _P]),
    "msn_census_dev": (c_int, [_P, _P, c_int, c_int, c_int, c_int, _P, _P]),
    "msn_ncc_dev": (c_int, [_P, _P, c_int, c_int, c_int, c_int, _P, _P]),
    "msn_zsad_dev": (c_int, [_P, _P, c_int, c_int, c_int, c_int, _P, _P]),
    "msn_sobel_dev": (c_int, [_P, c_int, c_int, _P, _P]),
    "msn_sadsob_dev": (c_int, [_P, _P, c_int, c_int, c_int, c_int, _P, _P]),
    "msn_aml_dev": (c_int, [_P, c_ll, c_int, c_float, _P, _P]),
    "msn_pkrn_dev": (c_int, [_P, c_ll, c_int, c_float, _P, _P]),
    "msn_soft_argmin_dev": (c_int, [_P, c_int, c_int, c_int, c_int, _P, _P]),
    "msn_expect_disp_dev": (c_int, [_P, c_int, c_int, c_int, c_int, _P, _P]),
    "msn_soft_argmin_host": (c_int, [_P, c_int, c_int, c_int, c_int, _P]),
    "msn_soft_argmin_backward_dev": (c_int, [_P, _P, _P, c_int, c_int, c_int, c_int, _P, _P]),
    "msn_soft_argmin_partial_dev": (c_int, [_P, c_int, c_int, c_int, c_int, c_int, _P, _P]),
    "msn_soft_argmin_merge_dev": (c_int, [_P, c_int, c_int, c_int, c_int, _P, _P]),
    "msn_wta_dev": (c_int, [_P, c_ll, c_int, c_int, _P, _P, _P, _P]),
    "msn_wta_host": (c_int, [_P, c_ll, c_int, c_int, _P, _P, _P]),
    "msn_wta_keys_dev": (c_int, [_P, c_ll, c_int, c_int, c_int, _P, _P]),
    "msn_wta_unpack_dev": (c_int, [_P, c_ll, _P, _P, _P]),
    "msn_pkrn_conf_dev": (c_int, [_P, _P, c_ll, c_float, _P, _P]),
    "msn_lrc_dev": (c_int, [_P, c_int, c_int, c_int, c_int, _P, _P, _P, _P]),
    "msn_lrc_host": (c_int, [_P, c_int, c_int, c_int, c_int, _P, _P, _P]),
    "msn_concat_volume_dev": (c_int, [_P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P]),
    "msn_diff_volume_dev": (c_int, [_P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P]),
    "msn_concat_volume_backward_dev": (c_int, [_P, c_int, c_int, c_int, c_int, c_int, _P, _P, _P]),
    "msn_diff_volume_backward_dev": (c_int, [_P, c_int, c_int, c_int, c_int, c_int, _P, _P, _P]),
}
EXPORTS = tuple(sorted(_SIGNATURES))

_lib = None


def lib():
    """The loaded CDLL.  Raises MsnetsError (never falls back) if it is not built."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise MsnetsError(
                "%s is missing: build it with `python ms-nets_b200/csrc/build.py` "
                "(or __graft_entry__.build()); msnets_b200 has no CPU fallback" % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        if L.msn_abi_version() != 1:
            raise MsnetsError("libmsnets_b200.so ABI version mismatch")
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise MsnetsError(lib().msn_last_error().decode("utf-8", "replace"))


def device_count():
    n = c_int(0)
    check(lib().msn_device_count(ctypes.byref(n)))
    return n.value


def default_params(**overrides):
    p = MsParams()
    lib().msn_ms_params_default(ctypes.byref(p))
    for k, v in overrides.items():
        if not hasattr(p, k):
            raise TypeError("unknown msn_ms_params field %r" % k)
        setattr(p, k, v)
    return p
