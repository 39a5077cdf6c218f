"""ctypes binding of libplaysnark_b200.so (the C ABI in include/playsnark_b200.h).

The library is the product: there is no Python or CPU fallback.  Importing this module without the
built shared object, or creating a context without a CUDA device, raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# PLAYSNARK_B200_LIB may point at another nvcc build of the same library (kernel tuning experiments)
LIB_PATH = os.environ.get("PLAYSNARK_B200_LIB") or os.path.join(_HERE, "libplaysnark_b200.so")

PS_OK, PS_ERR_ARG, PS_ERR_LENGTH, PS_ERR_REMAINDER, PS_ERR_ENCODING, PS_ERR_CUDA, PS_ERR_ALLOC, PS_ERR_UNSUPPORTED = range(8)
PS_FMT_COMPRESSED, PS_FMT_AFFINE = 0, 1
PS_G1, PS_G2 = 1, 2

# every symbol include/playsnark_b200.h declares: (name, restype, argtypes)
_P = C.c_void_p
_B = C.c_char_p
_SZ = C.c_size_t
_I = C.c_int
SYMBOLS = [
    ("ps_strerror", C.c_char_p, [_I]),
    ("ps_version", C.c_char_p, []),
    ("ps_ctx_create", _I, [_I, C.POINTER(_P)]),
    ("ps_ctx_set_stream", _I, [_P, _P]),
    ("ps_ctx_set_option", _I, [_P, C.c_char_p, _I]),
    ("ps_ctx_sync", _I, [_P]),
    ("ps_ctx_destroy", None, [_P]),
    ("ps_launch_count", C.c_uint64, []),
    ("ps_bases_load", _I, [_P, _I, _B, _SZ, _I, _I, _I, C.POINTER(_P)]),
    ("ps_bases_len", _SZ, [_P]),
    ("ps_bases_info", _I, [_P, C.POINTER(C.c_int)]),
    ("ps_bases_free", None, [_P]),
    ("ps_bases_from_scalars", _I, [_P, _I, _B, _SZ, _I, _I, C.POINTER(_P)]),
    ("ps_bases_export", _I, [_P, _P, _SZ, _SZ, _I, _P]),
    ("ps_msm", _I, [_P, _P, _P, _SZ, _P]),
    ("ps_msm_rows", _I, [_P, _P, _P, _SZ, _SZ, _P]),
    ("ps_msm_device", _I, [_P, _P, _SZ, _P, _SZ, _P]),
    ("ps_msm_device_mont", _I, [_P, _P, _SZ, _P, _SZ, _P]),
    ("ps_msm_combine", _I, [_P, _I, _P, _SZ, _P]),
    ("ps_ntt_fr", _I, [_P, _P, C.c_uint, _I, _B]),
    ("ps_qap_load_dense", _I, [_P, _SZ, _SZ, _SZ, _B, _B, _B, _B, C.POINTER(_P)]),
    ("ps_qap_load_r1cs", _I, [_P, _SZ, _SZ, _SZ] + [_P] * 9 + [C.POINTER(_P)]),
    ("ps_qap_free", None, [_P]),
    ("ps_quotient", _I, [_P, _P, _P, _P, _P]),
    ("ps_g16_key_load", _I, [_P, _SZ, _SZ, _I] + [_B] * 9 + [C.POINTER(_P)]),
    ("ps_g16_key_free", None, [_P]),
    ("ps_g16_setup", _I, [_P, _P, _B, C.POINTER(_P), _P, _P]),
    ("ps_g16_key_export", _I, [_P, _P, _I] + [_P] * 9),
    ("ps_phgr13_setup", _I, [_P, _P, _B, C.POINTER(_P), _P, _P, _P, _P]),
    ("ps_phgr13_key_export", _I, [_P, _P, _I] + [_P] * 10),
    ("ps_g16_prove", _I, [_P, _P, _P, _P, _B, _B, _P, _P, _P, _P]),
    ("ps_g16_scalar_count", _SZ, [_P, _I]),
    ("ps_g16_key_bases", _P, [_P, _I]),
    ("ps_g16_scalars", _I, [_P, _P, _P, _P, _B, _B, _P, _P, _P]),
    ("ps_g16_msm_partials", _I, [_P, _P, _P, _P, _P, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t), _P]),
    ("ps_qap_aggregate_one", _I, [_P, _P, _P, _I, _P]),
    ("ps_g16_scalars_from_ab", _I, [_P, _P, _P, _P, _B, _B, _P, _P, _P, _P, _P]),
    ("ps_qap_interp_part", _I, [_P, _P, _P, _I, _SZ, _SZ, _P, _P, _P]),
    ("ps_qap_interp_part_dev", _I, [_P, _P, _P, _I, _SZ, _SZ, _P, _P, _P]),
    ("ps_fr_upload", _I, [_P, _P, _SZ, _P, _P]),
    ("ps_qap_interp_finish", _I, [_P, _P, _SZ, _P, _P]),
    ("ps_g16_scalars_ab", _I, [_P, _P, _B, _B, _P, _P, _P, _P, _P]),
    ("ps_g16_h_from_ab", _I, [_P, _P, _P, _P, _P]),
    ("ps_g16_combine", _I, [_P, _P, _SZ, _SZ, _P, _P, _P]),
    ("ps_host_alloc", _I, [_SZ, C.POINTER(_P)]),
    ("ps_host_free", None, [_P]),
    ("ps_phgr13_key_load", _I, [_P, _SZ, _SZ, _I] + [_B] * 10 + [C.POINTER(_P)]),
    ("ps_phgr13_key_free", None, [_P]),
    ("ps_phgr13_prove", _I, [_P, _P, _P, _P, _P, _P]),
    ("ps_pairing_check_batch", _I, [_P, _B, _B, C.POINTER(C.c_uint32), _SZ, _I, _P]),
    ("ps_g16_verify", _I, [_P, _B, _B, _B, _B, _B, _SZ, _B, _B, _B, _B, C.POINTER(C.c_int)]),
    ("ps_g16_verify_batch", _I, [_P, _B, _B, _B, _B, _B, _SZ, _SZ, _P, _P, _P, _P, _P, C.POINTER(C.c_int), _P]),
    ("ps_phgr13_verify", _I, [_P, _B, _B, _B, _B, _SZ, _B, _B, C.POINTER(C.c_int)]),
    ("ps_phgr13_verify_batch", _I, [_P, _B, _P, _P, _P, _SZ, _SZ, _P, _P, _P, C.POINTER(C.c_int), _P]),
    ("ps_mctx_create", _I, [C.POINTER(C.c_int), _I, C.POINTER(_P)]),
    ("ps_mctx_destroy", None, [_P]),
    ("ps_mctx_size", _I, [_P]),
    ("ps_mctx_ctx", _P, [_P, _I]),
    ("ps_mctx_set_option", _I, [_P, C.c_char_p, _I]),
    ("ps_mbases_load", _I, [_P, _I, _P, _SZ, _I, _I, _I, C.POINTER(_P)]),
    ("ps_mbases_from_scalars", _I, [_P, _I, _P, _SZ, _I, _I, C.POINTER(_P)]),
    ("ps_mbases_len", _SZ, [_P]),
    ("ps_mbases_free", None, [_P]),
    ("ps_mmsm", _I, [_P, _P, _P, _SZ, _P]),
    ("ps_mg16_key_load", _I, [_P, _SZ, _SZ, _I] + [_B] * 9 + [C.POINTER(_P)]),
    ("ps_mg16_key_free", None, [_P]),
    ("ps_mqap_load_r1cs", _I, [_P, _SZ, _SZ, _SZ] + [_P] * 9 + [C.POINTER(_P)]),
    ("ps_mqap_load_dense", _I, [_P, _SZ, _SZ, _SZ, _B, _B, _B, _B, C.POINTER(_P)]),
    ("ps_mqap_free", None, [_P]),
    ("ps_mg16_prove", _I, [_P, _P, _P, _P, _B, _B, _P, _P, _P]),
    ("ps_mg16_last_timeline", _I, [_P, _I, C.POINTER(C.c_float), _I, C.POINTER(C.c_int)]),
    ("ps_bench_intpipe", _I, [_P, _I, _I, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    ("ps_bench_fieldmul", _I, [_P, _I, _I, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    ("ps_last_msm_timing", _I, [_P, C.POINTER(C.c_float)]),
    ("ps_last_prove_timing", _I, [_P, C.POINTER(C.c_float)]),
    ("ps_last_verify_batch_timing", _I, [_P, C.POINTER(C.c_float)]),
]


class PlaysnarkError(RuntimeError):
    def __init__(self, status: int, msg: str):
        super().__init__("%s (status %d)" % (msg, status))
        self.status = status


def bind(path: str) -> C.CDLL:
    """Load a build of the C ABI and attach prototypes.  `path` is libplaysnark_b200.so for the
    product; tests may pass their host-emulation build explicitly (never done implicitly)."""
    if not os.path.exists(path):
        raise ImportError(
            "playsnark_b200: %s is missing -- build it with `python -c 'import __graft_entry__ as g; g.build()'`; "
            "there is no CPU fallback" % path)
    lib = C.CDLL(path)
    for name, res, args in SYMBOLS:
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    return lib


_lib = None


def load() -> C.CDLL:
    global _lib
    if _lib is None:
        _lib = bind(LIB_PATH)
    return _lib


def check(lib, status: int):
    if status != PS_OK:
        raise PlaysnarkError(status, lib.ps_strerror(status).decode())
