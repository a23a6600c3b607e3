"""ctypes binding of libcovest_b200.so (include/covest_b200.h).  This is the whole Python <-> native
boundary: plain pointers and sizes."""
import ctypes
import os

from . import build as _build

_lib = None

CVB_OK = 0
ABI_VERSION = 2  # CVB_ABI_VERSION of include/covest_b200.h this binding was written against
MODEL_BASIC, MODEL_REPEATS = 0, 1

c_double_p = ctypes.POINTER(ctypes.c_double)
c_int32_p = ctypes.POINTER(ctypes.c_int32)


class LibraryMissing(RuntimeError):
    pass


def load():
    """The loaded library.  Builds it first when the sources are newer and nvcc is present;
    raises LibraryMissing (never falls back to anything) when it cannot be had."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB_PATH
    if _build.is_stale():
        try:
            _build.build_library()
        except Exception as exc:  # no nvcc, or the compile failed
            if not os.path.exists(path):
                raise LibraryMissing(
                    'libcovest_b200.so is not built and could not be built (%s). Run '
                    '`python -m covest_b200.build` on a machine with nvcc; there is no CPU '
                    'implementation to fall back to.' % exc)
            import warnings
            warnings.warn('libcovest_b200.so is older than its sources and could not be rebuilt (%s); '
                          'using the existing binary if its ABI version matches' % exc)
    L = ctypes.CDLL(path)
    try:
        L.cvb_abi_version.restype = ctypes.c_int
        have = L.cvb_abi_version()
    except AttributeError:
        have = 1
    if have != ABI_VERSION:
        raise LibraryMissing('libcovest_b200.so has ABI version %d, this binding needs %d: rebuild it '
                             'with `python -m covest_b200.build --force`' % (have, ABI_VERSION))
    vp = ctypes.c_void_p
    i64 = ctypes.c_int64
    L.cvb_version.restype = ctypes.c_char_p
    L.cvb_last_error.restype = ctypes.c_char_p
    L.cvb_last_error.argtypes = [vp]
    L.cvb_ctx_create.restype = ctypes.c_int
    L.cvb_ctx_create.argtypes = [ctypes.c_int] * 5 + [c_int32_p, c_double_p, ctypes.c_double,
                                                      ctypes.c_double, c_double_p, c_double_p,
                                                      c_double_p, ctypes.c_int,
                                                      ctypes.POINTER(vp)]
    L.cvb_ctx_destroy.restype = None
    L.cvb_ctx_destroy.argtypes = [vp]
    L.cvb_loglik_batch.restype = ctypes.c_int
    L.cvb_loglik_batch.argtypes = [vp, i64, vp, vp, vp]
    L.cvb_probs_batch.restype = ctypes.c_int
    L.cvb_probs_batch.argtypes = [vp, i64, vp, ctypes.c_int, vp, vp, vp]
    L.cvb_topk.restype = ctypes.c_int
    L.cvb_topk.argtypes = [vp, i64, vp, vp, ctypes.c_int, vp, vp]
    L.cvb_loglik_topk.restype = ctypes.c_int
    L.cvb_loglik_topk.argtypes = [vp, i64, vp, vp, ctypes.c_int, vp, vp]
    L.cvb_lattice_eval.restype = ctypes.c_int
    L.cvb_lattice_eval.argtypes = [vp, c_int32_p, c_double_p, i64, i64, i64, i64, vp, ctypes.c_int,
                                   vp, vp]
    L.cvb_lattice_profile.restype = ctypes.c_int
    L.cvb_lattice_profile.argtypes = [vp, c_int32_p, c_double_p, i64, i64, i64, i64, ctypes.c_uint32, vp, vp]
    L.cvb_fp64_peak.restype = ctypes.c_int
    L.cvb_fp64_peak.argtypes = [vp, ctypes.c_int, ctypes.c_int, c_double_p]
    L.cvb_set_timing.restype = ctypes.c_int
    L.cvb_set_timing.argtypes = [vp, ctypes.c_int]
    L.cvb_last_kernel_ms.restype = ctypes.c_int
    L.cvb_last_kernel_ms.argtypes = [vp, c_double_p, ctypes.POINTER(ctypes.c_int)]
    L.cvb_set_path.restype = ctypes.c_int
    L.cvb_set_path.argtypes = [vp, ctypes.c_int]
    L.cvb_merge_rows.restype = ctypes.c_int
    L.cvb_merge_rows.argtypes = [vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, vp]
    L.cvb_last_path_info.restype = ctypes.c_int
    L.cvb_last_path_info.argtypes = [vp, c_double_p, ctypes.c_int]
    L.cvb_n_param.restype = ctypes.c_int
    L.cvb_n_param.argtypes = [vp]
    L.cvb_device_sm_count.restype = ctypes.c_int
    L.cvb_device_sm_count.argtypes = [vp]
    L.cvb_kmer_table_create.restype = ctypes.c_int
    L.cvb_kmer_table_create.argtypes = [ctypes.c_int, i64, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                        ctypes.POINTER(vp)]
    L.cvb_kmer_table_destroy.restype = None
    L.cvb_kmer_table_destroy.argtypes = [vp]
    L.cvb_kmer_last_error.restype = ctypes.c_char_p
    L.cvb_kmer_last_error.argtypes = [vp]
    L.cvb_kmer_clear.restype = ctypes.c_int
    L.cvb_kmer_clear.argtypes = [vp, vp]
    L.cvb_kmer_count.restype = ctypes.c_int
    L.cvb_kmer_count.argtypes = [vp, vp, i64, vp]
    L.cvb_kmer_stats.restype = ctypes.c_int
    L.cvb_kmer_stats.argtypes = [vp, vp, vp]
    L.cvb_kmer_histogram.restype = ctypes.c_int
    L.cvb_kmer_histogram.argtypes = [vp, i64, vp, vp]
    _lib = L
    return L


EXPORTS = ('cvb_ctx_create', 'cvb_ctx_destroy', 'cvb_last_error', 'cvb_loglik_batch',
           'cvb_probs_batch', 'cvb_topk', 'cvb_loglik_topk', 'cvb_lattice_eval', 'cvb_lattice_profile', 'cvb_fp64_peak', 'cvb_set_timing',
           'cvb_last_kernel_ms', 'cvb_set_path', 'cvb_merge_rows', 'cvb_last_path_info', 'cvb_n_param', 'cvb_device_sm_count', 'cvb_version',
           'cvb_abi_version', 'cvb_kmer_table_create', 'cvb_kmer_table_destroy', 'cvb_kmer_last_error',
           'cvb_kmer_clear', 'cvb_kmer_count', 'cvb_kmer_stats', 'cvb_kmer_histogram')
