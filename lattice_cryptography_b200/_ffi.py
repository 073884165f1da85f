"""ctypes binding of liblcb200.so (the C ABI declared in include/lcb200.h).

There is no CPU fallback: if the library has not been built (``python -c "import
__graft_entry__ as g; g.build()"`` or ``make -C lattice_cryptography_b200/csrc``) loading
fails loudly, and creating a context without an sm_100 GPU raises ``LcbError``.
"""
import ctypes
import os
from ctypes import (POINTER, Structure, c_char, c_char_p, c_int, c_int16, c_int32, c_int64, c_uint8, c_uint16,
                    c_void_p)

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('LCB200_LIB') or os.path.join(_PKG_DIR, 'liblcb200.so')
LCB_SALT_MAX = 32

LCB_OK = 0
LCB_ERR_INVALID = -1
LCB_ERR_CUDA = -2
LCB_ERR_NO_DEVICE = -3
LCB_ERR_NO_KEY_CH = -4
LCB_ERR_OOM = -5

LCB_CONTENT_VK = 0
LCB_CONTENT_ST = 1


class LcbError(RuntimeError):
    def __init__(self, status: int, what: str):
        super().__init__(f'lcb200 error {status}: {what}')
        self.status = status


class LcbScheme(Structure):
    """Mirror of `struct lcb_scheme` (include/lcb200.h)."""
    _fields_ = [
        ('sk_bd', c_int32), ('sk_wt', c_int32),
        ('ch_bd', c_int32), ('ch_wt', c_int32),
        ('ag_bd', c_int32), ('ag_wt', c_int32),
        ('wit_bd', c_int32), ('wit_wt', c_int32),
        ('sk_salt', c_char * LCB_SALT_MAX), ('ch_salt', c_char * LCB_SALT_MAX),
        ('ag_salt', c_char * LCB_SALT_MAX), ('wit_salt', c_char * LCB_SALT_MAX),
    ]


# name -> (restype, argtypes); every symbol include/lcb200.h declares
_P = c_void_p   # data pointers are passed as raw addresses (host or device)
PROTOTYPES = {
    'lcb_strerror': (c_char_p, [c_int]),
    'lcb_last_error': (c_char_p, [c_void_p]),
    'lcb_version': (c_int, []),
    'lcb_build_is_checked': (c_int, []),
    'lcb_checked_selftest': (c_int, [c_void_p]),
    'lcb_ctx_create': (c_int, [POINTER(c_void_p), c_int, c_int, c_int, c_int, c_int]),
    'lcb_ctx_destroy': (c_int, [c_void_p]),
    'lcb_ctx_set_stream': (c_int, [c_void_p, c_void_p]),
    'lcb_synchronize': (c_int, [c_void_p]),
    'lcb_ctx_root_of_unity': (c_int, [c_void_p]),
    'lcb_set_key_ch': (c_int, [c_void_p, _P]),
    'lcb_shake256_batch': (c_int, [c_void_p, _P, _P, c_int64, _P, c_int64]),
    'lcb_expand_seeds': (c_int, [c_void_p, _P, c_int64, c_int64, _P]),
    'lcb_hash2polyvec_batch': (c_int, [c_void_p, c_char_p, _P, _P, c_int64, c_int, c_int, c_int, _P, _P]),
    'lcb_ntt_fwd_batch': (c_int, [c_void_p, _P, c_int64, _P]),
    'lcb_ntt_inv_batch': (c_int, [c_void_p, _P, c_int64, _P]),
    'lcb_poly_mul_batch': (c_int, [c_void_p, _P, _P, c_int64, _P]),
    'lcb_ntt_reference_repr_batch': (c_int, [c_void_p, _P, c_int64, _P]),
    'lcb_lm_keygen_batch': (c_int, [c_void_p, POINTER(LcbScheme), _P, _P, c_int64, _P, _P, _P, _P]),
    'lcb_challenge_batch': (c_int, [c_void_p, POINTER(LcbScheme), _P, _P, c_int64, _P]),
    'lcb_lm_sign_batch': (c_int, [c_void_p, POINTER(LcbScheme), _P, _P, _P, c_int64, _P]),
    'lcb_lm_verify_batch': (c_int, [c_void_p, POINTER(LcbScheme), _P, _P, _P, _P, _P, c_int64, c_int, c_int, _P]),
    'lcb_pack_batch': (c_int, [c_void_p, _P, c_int64, c_int, c_int, _P, _P]),
    'lcb_unpack_batch': (c_int, [c_void_p, _P, c_int64, c_int, c_int, _P]),
    'lcb_lm_verify_packed_batch': (c_int, [c_void_p, POINTER(LcbScheme), _P, c_int, _P, _P, _P, c_int, c_int, c_int64,
                                           c_int, c_int, _P]),
    'lcb_lm_sign_packed_batch': (c_int, [c_void_p, POINTER(LcbScheme), _P, _P, _P, c_int64, c_int, c_int, _P, _P]),
    'lcb_lm_keygen_packed_batch': (c_int, [c_void_p, POINTER(LcbScheme), _P, _P, c_int64, c_int, c_int, _P, _P, c_int, _P]),
    'lcb_lm_sign_packed_sk_batch': (c_int, [c_void_p, POINTER(LcbScheme), _P, c_int, c_int, _P, _P, c_int64, c_int, c_int, _P,
                                            _P]),
    'lcb_adaptor_verify_packed_batch': (c_int, [c_void_p, POINTER(LcbScheme), _P, c_int, _P, _P, _P, c_int, c_int, _P, c_int,
                                                c_int64, c_int, c_int, _P]),
    'lcb_adaptor_adapt_packed_batch': (c_int, [c_void_p, _P, c_int, c_int, _P, c_int64, c_int, c_int, _P, _P]),
    'lcb_adaptor_extract_packed_batch': (c_int, [c_void_p, _P, c_int, c_int, _P, c_int, c_int, c_int64, _P]),
    'lcb_adaptor_witgen_packed_batch': (c_int, [c_void_p, POINTER(LcbScheme), _P, _P, c_int64, c_int, c_int, _P, _P, c_int,
                                                _P]),
    'lcb_adaptor_witness_verify_packed_batch': (c_int, [c_void_p, _P, c_int, c_int, _P, c_int, c_int64, c_int, c_int, _P]),
    'lcb_adaptor_adapt_packed_wit_batch': (c_int, [c_void_p, _P, c_int, c_int, _P, c_int, c_int, c_int64, c_int, c_int, _P,
                                                   _P]),
    'lcb_adaptor_extract_packed_wit_batch': (c_int, [c_void_p, _P, c_int, c_int, _P, c_int, c_int, c_int64, c_int, c_int,
                                                     _P, _P]),
    'lcb_content_str_batch': (c_int, [c_void_p, c_int, _P, c_int, c_int64, _P]),
    'lcb_challenge_inputs_batch': (c_int, [c_void_p, _P, _P, _P, _P, c_int64, _P, _P]),
    'lcb_aggregation_inputs_batch': (c_int, [c_void_p, _P, c_int64, _P, _P, _P, _P, _P]),
    'lcb_content_order_batch': (c_int, [c_void_p, _P, c_int64, _P, _P]),
    'lcb_gather_rows_batch': (c_int, [c_void_p, _P, c_int64, c_int64, _P, c_int64, _P]),
    'lcb_gather_ragged_batch': (c_int, [c_void_p, _P, _P, c_int64, _P, c_int64, _P, c_int64, _P]),
    'lcb_bklm_agg_coefs': (c_int, [c_void_p, POINTER(LcbScheme), _P, c_int64, c_int64, c_int64, _P]),
    'lcb_bklm_aggregate_partial': (c_int, [c_void_p, POINTER(LcbScheme), _P, _P, _P, c_int64, c_int64, c_int64, _P]),
    'lcb_bklm_aggregate_finish': (c_int, [c_void_p, _P, _P]),
    'lcb_bklm_aggverify_partial': (c_int, [c_void_p, POINTER(LcbScheme), _P, _P, _P, _P, _P, c_int64, c_int64,
                                           c_int64, _P]),
    'lcb_bklm_aggverify_finish': (c_int, [c_void_p, _P, _P, c_int64, c_int, c_int, c_int, _P]),
    'lcb_bklm_aggregate_batch': (c_int, [c_void_p, POINTER(LcbScheme), _P, c_int64, _P, _P, _P, _P]),
    'lcb_bklm_aggregate_verify_batch': (c_int, [c_void_p, POINTER(LcbScheme), _P, c_int64, _P, _P, _P, _P, _P, _P, c_int,
                                                c_int, c_int, _P]),
    'lcb_bklm_aggregate_packed_batch': (c_int, [c_void_p, POINTER(LcbScheme), _P, c_int64, _P, c_int, c_int, _P, _P, c_int,
                                                c_int, _P, _P]),
    'lcb_bklm_aggregate_verify_packed_batch': (c_int, [c_void_p, POINTER(LcbScheme), _P, c_int64, _P, c_int, _P, _P, _P, _P,
                                                       _P, c_int, c_int, c_int, c_int, c_int, _P]),
    'lcb_adaptor_witgen_batch': (c_int, [c_void_p, POINTER(LcbScheme), _P, _P, c_int64, _P, _P, _P]),
    'lcb_vec_add_batch': (c_int, [c_void_p, _P, _P, c_int64, _P]),
    'lcb_vec_sub_batch': (c_int, [c_void_p, _P, _P, c_int64, _P]),
    'lcb_adaptor_witness_verify_batch': (c_int, [c_void_p, _P, _P, c_int64, c_int, c_int, _P]),
    'lcb_mctx_create': (c_int, [POINTER(c_void_p), POINTER(c_int), c_int, c_int, c_int, c_int, c_int]),
    'lcb_mctx_destroy': (c_int, [c_void_p]),
    'lcb_mctx_ndev': (c_int, [c_void_p]),
    'lcb_mctx_ctx': (c_void_p, [c_void_p, c_int]),
    'lcb_mctx_last_error': (c_char_p, [c_void_p]),
    'lcb_mctx_set_key_ch': (c_int, [c_void_p, _P]),
    'lcb_mctx_lm_keygen_batch': (c_int, [c_void_p, POINTER(LcbScheme), _P, _P, c_int64, _P, _P, _P, _P]),
    'lcb_mctx_lm_sign_batch': (c_int, [c_void_p, POINTER(LcbScheme), _P, _P, _P, c_int64, _P]),
    'lcb_mctx_lm_verify_batch': (c_int, [c_void_p, POINTER(LcbScheme), _P, _P, _P, _P, _P, c_int64, c_int, c_int, _P]),
    'lcb_mctx_lm_verify_packed_batch': (c_int, [c_void_p, POINTER(LcbScheme), _P, c_int, _P, _P, _P, c_int, c_int, c_int64,
                                                c_int, c_int, _P]),
    'lcb_mctx_bklm_aggregate': (c_int, [c_void_p, POINTER(LcbScheme), _P, _P, c_int64, c_int64, _P]),
    'lcb_mctx_bklm_aggregate_verify': (c_int, [c_void_p, POINTER(LcbScheme), _P, _P, _P, _P, c_int64, c_int64, _P, c_int,
                                               c_int, c_int, _P]),
    'lcb_launch_count': (c_int64, [c_void_p]),
    'lcb_profile_enable': (c_int, [c_void_p, c_int]),
    'lcb_profile_reset': (c_int, [c_void_p]),
    'lcb_profile_read': (c_int, [c_void_p, c_char_p, POINTER(ctypes.c_double), POINTER(c_int64)]),
}

_lib = None


def load():
    """Load liblcb200.so and bind every prototype.  Raises if the library is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise LcbError(LCB_ERR_NO_DEVICE, f'{LIB_PATH} is not built; run __graft_entry__.build() '
                                          f'(there is no CPU fallback)')
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in PROTOTYPES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib
