"""ctypes binding of the C ABI (include/schnorr_b200.h).  Fails loudly when the CUDA library is
missing or cannot be built: there is no CPU fallback."""
import ctypes as C
import os

from . import build as _build

_LIB = None

_u8p = C.c_void_p
_sz = C.c_size_t

_SIGNATURES = {
    "schnorr_b200_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "schnorr_b200_params_pinned": (C.c_int, []),
    "schnorr_b200_params_provenance": (C.c_char_p, []),
    "schnorr_b200_create_multi": (C.c_int, [C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_void_p)]),
    "schnorr_b200_device_count": (C.c_int, [C.c_void_p]),
    "schnorr_b200_destroy": (None, [C.c_void_p]),
    "schnorr_b200_last_error": (C.c_char_p, [C.c_void_p]),
    "schnorr_b200_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "schnorr_b200_synchronize": (C.c_int, [C.c_void_p]),
    "schnorr_b200_launch_count": (C.c_uint64, [C.c_void_p]),
    "schnorr_b200_last_kernel_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "schnorr_b200_set_exact_only": (C.c_int, [C.c_void_p, C.c_int]),
    "schnorr_b200_last_exact_count": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64)]),
    "schnorr_b200_set_dist_threshold": (C.c_int, [C.c_void_p, _sz]),
    "schnorr_b200_set_one_threshold": (C.c_int, [C.c_void_p, _sz]),
    "schnorr_b200_set_batch_small_threshold": (C.c_int, [C.c_void_p, _sz]),
    "schnorr_b200_set_batch_dist_threshold": (C.c_int, [C.c_void_p, _sz]),
    "schnorr_b200_set_msm_geometry": (C.c_int, [C.c_void_p, C.c_int, C.c_uint]),
    "schnorr_b200_last_batch_plan": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_uint)]),
    "schnorr_b200_hash_messages": (C.c_int, [C.c_void_p, _sz] + [_u8p] * 5),
    "schnorr_b200_hash_messages_dev": (C.c_int, [C.c_void_p, _sz] + [_u8p] * 5),
    "schnorr_b200_verify_many": (C.c_int, [C.c_void_p, _sz] + [_u8p] * 6),
    "schnorr_b200_verify_many_dev": (C.c_int, [C.c_void_p, _sz] + [_u8p] * 6),
    "schnorr_b200_keyset_create": (C.c_int, [C.c_void_p, _sz, _u8p, _u8p, _u8p, C.POINTER(C.c_void_p)]),
    "schnorr_b200_keyset_destroy": (None, [C.c_void_p]),
    "schnorr_b200_keyset_append": (C.c_int, [C.c_void_p, C.c_void_p, _sz, _u8p, _u8p, _u8p]),
    "schnorr_b200_keyset_replace": (C.c_int, [C.c_void_p, C.c_void_p, _sz, _u8p, _u8p, _u8p, _u8p]),
    "schnorr_b200_keyset_remove": (C.c_int, [C.c_void_p, C.c_void_p, _sz, _u8p]),
    "schnorr_b200_set_keyset_block_threshold": (C.c_int, [C.c_void_p, _sz]),
    "schnorr_b200_keyset_debug_export": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, _sz, _sz] + [_u8p] * 6),
    "schnorr_b200_verify_registered_many": (C.c_int, [C.c_void_p, C.c_void_p, _sz] + [_u8p] * 5),
    "schnorr_b200_verify_registered_many_dev": (C.c_int, [C.c_void_p, C.c_void_p, _sz] + [_u8p] * 5),
    "schnorr_b200_keyset_lookup": (C.c_int, [C.c_void_p, C.c_void_p, _sz, _u8p, _u8p]),
    "schnorr_b200_keyset_lookup_dev": (C.c_int, [C.c_void_p, C.c_void_p, _sz, _u8p, _u8p]),
    "schnorr_b200_verify_keyed_registered_many": (C.c_int, [C.c_void_p, C.c_void_p, _sz] + [_u8p] * 4),
    "schnorr_b200_verify_keyed_registered_many_dev": (C.c_int, [C.c_void_p, C.c_void_p, _sz] + [_u8p] * 4),
    "schnorr_b200_verify_keyed_many":(C.c_int, [C.c_void_p, _sz] + [_u8p] * 4),
    "schnorr_b200_verify_keyed_many_dev": (C.c_int, [C.c_void_p, _sz] + [_u8p] * 4),
    "schnorr_b200_verify_batch": (C.c_int, [C.c_void_p, _sz] + [_u8p] * 6 + [C.POINTER(C.c_int), _u8p, _u8p]),
    "schnorr_b200_verify_batch_dev": (C.c_int, [C.c_void_p, _sz] + [_u8p] * 7),
    "schnorr_b200_locate_invalid": (C.c_int, [C.c_void_p, _sz] + [_u8p] * 7 + [C.POINTER(C.c_uint64)]),
    "schnorr_b200_locate_invalid_dev": (C.c_int, [C.c_void_p, _sz] + [_u8p] * 7),
    "schnorr_b200_verify_batch_registered": (C.c_int, [C.c_void_p, C.c_void_p, _sz] + [_u8p] * 5 + [C.POINTER(C.c_int), _u8p, _u8p]),
    "schnorr_b200_verify_batch_registered_dev": (C.c_int, [C.c_void_p, C.c_void_p, _sz] + [_u8p] * 6),
    "schnorr_b200_locate_invalid_registered": (C.c_int, [C.c_void_p, C.c_void_p, _sz] + [_u8p] * 6 + [C.POINTER(C.c_uint64)]),
    "schnorr_b200_verify_batch_keyed": (C.c_int, [C.c_void_p, _sz] + [_u8p] * 4 + [C.POINTER(C.c_int), _u8p, _u8p]),
    "schnorr_b200_verify_batch_keyed_dev": (C.c_int, [C.c_void_p, _sz] + [_u8p] * 5),
    "schnorr_b200_verify_batch_keyed_registered": (C.c_int, [C.c_void_p, C.c_void_p, _sz] + [_u8p] * 4
                                                   + [C.POINTER(C.c_int), _u8p, _u8p]),
    "schnorr_b200_verify_batch_keyed_registered_dev": (C.c_int, [C.c_void_p, C.c_void_p, _sz] + [_u8p] * 5),
    "schnorr_b200_locate_invalid_keyed": (C.c_int, [C.c_void_p, _sz] + [_u8p] * 5 + [C.POINTER(C.c_uint64)]),
    "schnorr_b200_locate_invalid_keyed_registered": (C.c_int, [C.c_void_p, C.c_void_p, _sz] + [_u8p] * 5
                                                     + [C.POINTER(C.c_uint64)]),
    "schnorr_b200_batch_randomizers": (C.c_int, [C.c_void_p, _sz, _u8p, C.c_uint64, _u8p]),
    "schnorr_b200_batch_randomizers_dev": (C.c_int, [C.c_void_p, _sz, _u8p, C.c_uint64, _u8p]),
    "schnorr_b200_verify_batch_seeded": (C.c_int, [C.c_void_p, _sz] + [_u8p] * 6 + [C.POINTER(C.c_int), _u8p, _u8p]),
    "schnorr_b200_verify_batch_registered_seeded": (C.c_int, [C.c_void_p, C.c_void_p, _sz] + [_u8p] * 5
                                                    + [C.POINTER(C.c_int), _u8p, _u8p]),
    "schnorr_b200_verify_batch_keyed_seeded": (C.c_int, [C.c_void_p, _sz] + [_u8p] * 4 + [C.POINTER(C.c_int), _u8p, _u8p]),
    "schnorr_b200_verify_batch_keyed_registered_seeded": (C.c_int, [C.c_void_p, C.c_void_p, _sz] + [_u8p] * 4
                                                          + [C.POINTER(C.c_int), _u8p, _u8p]),
    "schnorr_b200_locate_invalid_seeded": (C.c_int, [C.c_void_p, _sz] + [_u8p] * 7 + [C.POINTER(C.c_uint64)]),
    "schnorr_b200_locate_invalid_registered_seeded": (C.c_int, [C.c_void_p, C.c_void_p, _sz] + [_u8p] * 6
                                                      + [C.POINTER(C.c_uint64)]),
    "schnorr_b200_locate_invalid_keyed_seeded": (C.c_int, [C.c_void_p, _sz] + [_u8p] * 5 + [C.POINTER(C.c_uint64)]),
    "schnorr_b200_locate_invalid_keyed_registered_seeded": (C.c_int, [C.c_void_p, C.c_void_p, _sz] + [_u8p] * 5
                                                            + [C.POINTER(C.c_uint64)]),
    "schnorr_b200_last_batch_points": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64)]),
    "schnorr_b200_set_registered_batch_threshold": (C.c_int, [C.c_void_p, _sz]),
    "schnorr_b200_batch_partial_dev": (C.c_int, [C.c_void_p, _sz] + [_u8p] * 7),
    "schnorr_b200_batch_finish_dev": (C.c_int, [C.c_void_p, _sz, _u8p, _u8p]),
    "schnorr_b200_batch_finish": (C.c_int, [C.c_void_p, _sz, _u8p, C.POINTER(C.c_int), _u8p, _u8p]),
    "schnorr_b200_keygen": (C.c_int, [C.c_void_p, _sz] + [_u8p] * 3),
    "schnorr_b200_keygen_dev": (C.c_int, [C.c_void_p, _sz] + [_u8p] * 3),
    "schnorr_b200_sign_many": (C.c_int, [C.c_void_p, _sz] + [_u8p] * 7),
    "schnorr_b200_sign_many_dev": (C.c_int, [C.c_void_p, _sz] + [_u8p] * 7),
    "schnorr_b200_derive_master_keys": (C.c_int, [C.c_void_p, _sz, _u8p, _u8p, _u8p]),
    "schnorr_b200_derive_private_children": (C.c_int, [C.c_void_p, _sz, _u8p, _u8p, _u8p, _u8p]),
    "schnorr_b200_derive_public_children": (C.c_int, [C.c_void_p, _sz, _u8p, _u8p, _u8p, _u8p]),
    "schnorr_b200_decompress": (C.c_int, [C.c_void_p, _sz] + [_u8p] * 4),
    "schnorr_b200_compress": (C.c_int, [C.c_void_p, _sz] + [_u8p] * 3),
    "schnorr_b200_debug_field_ops": (C.c_int, [C.c_void_p, _sz, _u8p, _u8p, _u8p]),
    "schnorr_b200_debug_lazy_ops": (C.c_int, [C.c_void_p, _sz, _u8p, _u8p, _u8p]),
    "schnorr_b200_debug_fp_core": (C.c_int, [C.c_void_p, C.c_int, _sz, _u8p, _u8p]),
    "schnorr_b200_debug_verify_core": (C.c_int, [C.c_void_p, C.c_int, _sz] + [_u8p] * 5),
    "schnorr_b200_debug_verify_registered_core": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, _sz] + [_u8p] * 5),
    "schnorr_b200_imad_peak": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)


def library_path():
    return _build.SO


def lib():
    """Loads (building first if stale) schnorr-sig_b200/csrc/libschnorr_b200.so."""
    global _LIB
    if _LIB is None:
        so = _build.build()
        if not os.path.exists(so):
            raise RuntimeError("libschnorr_b200.so is missing and could not be built; there is no CPU fallback")
        L = C.CDLL(so)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(L, name)          # AttributeError here = ABI drift against include/schnorr_b200.h
            fn.restype = res
            fn.argtypes = args
        _LIB = L
    return _LIB
