"""ctypes binding of include/qfall_b200.h.  There is NO CPU fallback: if the CUDA
library is missing or a call fails, an exception is raised."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libqfall_b200.so")

QF_OK, QF_ERR_INVALID, QF_ERR_CUDA, QF_ERR_NOT_IN_DOMAIN, QF_ERR_NO_KEY, QF_ERR_UNSUPPORTED, QF_ERR_NUMERIC = range(7)
QF_PSF_GPV, QF_PSF_PERTURBATION, QF_PSF_GPV_RING = 0, 1, 2
_STATUS = {0: "QF_OK", 1: "QF_ERR_INVALID", 2: "QF_ERR_CUDA", 3: "QF_ERR_NOT_IN_DOMAIN", 4: "QF_ERR_NO_KEY",
           5: "QF_ERR_UNSUPPORTED", 6: "QF_ERR_NUMERIC"}


class QfError(RuntimeError):
    def __init__(self, status, msg=""):
        super().__init__(f"{_STATUS.get(status, status)}: {msg}")
        self.status = status


class NotInDomain(QfError, AssertionError):
    """f_a on a sigma outside D_n -- the reference panics here (gpv.rs:191)."""


class QfParams(C.Structure):
    _fields_ = [("kind", C.c_int32), ("n", C.c_int64), ("k", C.c_int64), ("m_bar", C.c_int64), ("base", C.c_int64),
                ("q", C.c_uint64), ("s", C.c_double), ("r", C.c_double), ("norm_bound", C.c_uint64)]


_vp, _i64, _u64, _i32, _sz, _u32 = C.c_void_p, C.c_int64, C.c_uint64, C.c_int, C.c_size_t, C.c_uint32

# name -> (restype, argtypes); every symbol include/qfall_b200.h declares
SIGNATURES = {
    "qf_version": (C.c_char_p, []),
    "qf_ctx_create": (_i32, [C.POINTER(QfParams), _i32, C.POINTER(_vp)]),
    "qf_ctx_destroy": (None, [_vp]),
    "qf_last_error": (C.c_char_p, [_vp]),
    "qf_set_stream": (_i32, [_vp, _vp]),
    "qf_set_chunk": (_i32, [_vp, _i64]),
    "qf_synchronize": (_i32, [_vp]),
    "qf_launch_count": (_u64, [_vp]),
    "qf_profile": (_i32, [_vp, _i32]),
    "qf_profile_read": (_i32, [_vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_uint64),
                               C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_uint64)]),
    "qf_set_a": (_i32, [_vp, _vp]),
    "qf_set_trapdoor_perturbation": (_i32, [_vp, _vp, _vp, _vp, _vp]),
    "qf_set_tag": (_i32, [_vp, _vp, _vp]),
    "qf_gpv_set_tag": (_i32, [_vp, _vp, _vp, _vp]),
    "qf_set_tag_table": (_i32, [_vp, _vp, _i64]),
    "qf_set_f_a_tags": (_i32, [_vp, _vp, _i64, _vp]),
    "qf_set_tag_table_poly": (_i32, [_vp, _vp, _vp, _i64]),
    "qf_set_f_a_tags_poly": (_i32, [_vp, _vp, _vp, _i64, _vp]),
    "qf_compute_sqrt_sigma_2": (_i32, [_vp, _vp, _vp, _vp]),
    "qf_gen_short_basis": (_i32, [_vp, _vp, _vp]),
    "qf_gen_short_basis_tagged": (_i32, [_vp, _vp, _vp, _vp]),
    "qf_ring_gen_short_basis": (_i32, [_vp, _vp, _vp, _vp]),
    "qf_gso": (_i32, [_vp, _vp, _vp]),
    "qf_set_trapdoor_gpv": (_i32, [_vp, _vp, _vp]),
    "qf_ring_set_a": (_i32, [_vp, _vp]),
    "qf_trap_gen_from": (_i32, [_vp, _vp, _vp, _vp, _vp]),
    "qf_trap_gen": (_i32, [_vp, _u64, _vp, _vp]),
    "qf_ring_trap_gen_from": (_i32, [_vp, _vp, _vp, _vp, _vp]),
    "qf_f_a": (_i32, [_vp, _vp, _i64, _vp, _vp]),
    "qf_f_a_dev": (_i32, [_vp, _vp, _i64, _vp, _vp]),
    "qf_check_domain": (_i32, [_vp, _vp, _i64, _vp]),
    "qf_f_a_tagged": (_i32, [_vp, _vp, _vp, _i64, _vp, _vp]),
    "qf_f_a_tagged_dev": (_i32, [_vp, _vp, _vp, _i64, _vp, _vp]),
    "qf_ring_set_key_table": (_i32, [_vp, _vp, _i64]),
    "qf_ring_f_a_keyed": (_i32, [_vp, _vp, _vp, _i64, _vp, _vp]),
    "qf_ring_f_a_keyed_dev": (_i32, [_vp, _vp, _vp, _i64, _vp, _vp]),
    "qf_ring_f_a_keyed_packed": (_i32, [_vp, _vp, _vp, _i64, _i32, _i64, _vp, _vp]),
    "qf_ring_f_a_keyed_packed_dev": (_i32, [_vp, _vp, _vp, _i64, _i32, _i64, _vp, _vp]),
    "qf_ring_trap_gen_batch_from": (_i32, [_vp, _i64, _vp, _vp, _vp, _vp]),
    "qf_samp_d": (_i32, [_vp, _i64, _u64, _u64, _vp]),
    "qf_samp_d_dev": (_i32, [_vp, _i64, _u64, _u64, _vp]),
    "qf_samp_p": (_i32, [_vp, _vp, _i64, _u64, _u64, _vp]),
    "qf_samp_p_dev": (_i32, [_vp, _vp, _i64, _u64, _u64, _vp]),
    "qf_samp_p_i16": (_i32, [_vp, _vp, _i64, _u64, _u64, _vp]),
    "qf_samp_p_tagged": (_i32, [_vp, _vp, _vp, _i64, _u64, _u64, _vp]),
    "qf_samp_p_tagged_dev": (_i32, [_vp, _vp, _vp, _i64, _u64, _u64, _vp]),
    "qf_samp_p_offline": (_i32, [_vp, _i64, _u64, _u64]),
    "qf_samp_p_pool_info": (_i32, [_vp, _vp, _vp]),
    "qf_samp_p_online": (_i32, [_vp, _vp, _vp, _i64, _vp, _vp]),
    "qf_samp_p_online_dev": (_i32, [_vp, _vp, _vp, _i64, _vp, _vp]),
    "qf_f_a_i16": (_i32, [_vp, _vp, _i64, _vp, _vp]),
    "qf_narrow_i32_i16_dev": (_i32, [_vp, _vp, _sz, _vp, _vp]),
    "qf_domain_code_params": (_i32, [_vp, C.POINTER(_i32), C.POINTER(_i64)]),
    "qf_samp_p_packed": (_i32, [_vp, _vp, _vp, _i64, _u64, _u64, _i32, _i64, _vp, _vp]),
    "qf_f_a_packed": (_i32, [_vp, _vp, _vp, _i64, _i32, _i64, _vp, _vp]),
    "qf_domain_encode_dev": (_i32, [_vp, _i64, _i64, _i32, _i64, _vp, _vp, _vp]),
    "qf_domain_decode_dev": (_i32, [_vp, _i64, _i64, _i32, _i64, _vp, _vp, _vp]),
    "qf_randomized_nearest_plane_gadget": (_i32, [_vp, _vp, _i64, _u64, _u64, _vp]),
    "qf_compress_u16": (_i32, [_vp, _vp, _sz, _u32, _u32, _i32, _vp]),
    "qf_decompress_u16": (_i32, [_vp, _vp, _sz, _u32, _u32, _i32, _vp]),
    "qf_compress_i64": (_i32, [_vp, _vp, _sz, _u64, _u32, _i32, _vp]),
    "qf_decompress_i64": (_i32, [_vp, _vp, _sz, _u64, _u32, _i32, _vp]),
    "qf_compress_encode_u16": (_i32, [_vp, _vp, _sz, _u32, _u32, _i32, _i32, _vp]),
    "qf_decode_decompress_u16": (_i32, [_vp, _vp, _sz, _u32, _u32, _i32, _i32, _vp]),
    "qf_encode_digits": (_i32, [_vp, _vp, _sz, _u64, _u32, _i32, _i32, _vp]),
    "qf_decode_digits": (_i32, [_vp, _vp, _sz, _u64, _u32, _i32, _i32, _vp]),
    "qf_encode_bits_u16": (_i32, [_vp, _vp, _sz, _u32, _i32, _vp]),
    "qf_decode_bits_u16": (_i32, [_vp, _vp, _sz, _u32, _i32, _vp]),
    "qf_sample_z": (_i32, [_vp, _sz, C.c_double, _u64, _vp]),
    "qf_debug_gemm_i8": (_i32, [_vp, _vp, _i32, _i32, _i32, _i64, _i64, _i64, _u64, _vp]),
    "qf_probe_i8_peak": (_i32, [_i32, _i64, _i64, _i64, _i32, C.c_double, C.POINTER(C.c_double), C.POINTER(C.c_double),
                                C.POINTER(C.c_double)]),
    "qf_fill_uniform_modq_dev": (_i32, [_vp, _sz, _u64, _u64, _vp]),
}

_lib = None


def lib():
    """Load the CUDA library (building it is __graft_entry__.build()'s job)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: the CUDA extension was not built "
                "(run `python -m tools_b200.build`); there is no CPU fallback")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def ptr(a):
    """Host pointer of a C-contiguous numpy array, or a raw integer (device) pointer."""
    if a is None:
        return None
    if isinstance(a, (int, np.integer)):
        return C.c_void_p(int(a))
    assert a.flags["C_CONTIGUOUS"], "array must be C-contiguous"
    return C.c_void_p(a.ctypes.data)


class Context:
    """Owns one qf_ctx."""

    def __init__(self, kind, n, k, m_bar, base, q, s, r=1.0, norm_bound=0, device=0):
        self._h = _vp()
        self._lib = lib()
        p = QfParams(kind, n, k, m_bar, base, q, float(s), float(r), int(norm_bound))
        st = self._lib.qf_ctx_create(C.byref(p), device, C.byref(self._h))
        if st != QF_OK:
            self._h = _vp()
            raise QfError(st, "qf_ctx_create failed (is a CUDA device present?)")

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.qf_ctx_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def call(self, name, *args):
        st = getattr(self._lib, name)(self._h, *args)
        if st != QF_OK:
            msg = self._lib.qf_last_error(self._h).decode()
            if st == QF_ERR_NOT_IN_DOMAIN:
                raise NotInDomain(st, msg)
            raise QfError(st, msg)

    def status(self, name, *args):
        return getattr(self._lib, name)(self._h, *args)

    def launch_count(self):
        return int(self._lib.qf_launch_count(self._h))
