"""ctypes binding of snarkvm_b200/libsnarkvm_b200.so (the C ABI in include/snarkvm_b200.h).

The library is the product: there is NO CPU fallback.  If the shared object is missing or a
symbol is absent, importing fails loudly; if a call returns a non-zero cudaError_t, CudaError
is raised (the Rust reference would fall back to its CPU path at this point —
algorithms/src/msm/variable_base/mod.rs:39-43 — this package never does).
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SNARKVM_B200_LIB") or os.path.join(_HERE, "libsnarkvm_b200.so")   # override: A/B builds

# every symbol include/snarkvm_b200.h declares
SYMBOLS = (
    "snarkvm_ntt", "snarkvm_polymul", "snarkvm_msm",
    "snarkvm_b200_version", "snarkvm_b200_launch_count", "snarkvm_b200_ntt_device",
    "snarkvm_b200_polymul_device", "snarkvm_b200_msm_plan", "snarkvm_b200_msm_device",
    "snarkvm_b200_msm_window_sums_device", "snarkvm_b200_xyzz_sum_ranks_device", "snarkvm_b200_msm_finish",
    "snarkvm_b200_kzg_commit_device", "snarkvm_b200_fr_from_mont_device", "snarkvm_b200_fr_to_mont_device",
    "snarkvm_b200_srs_decode_device", "snarkvm_b200_register_bases", "snarkvm_b200_unregister_bases", "snarkvm_b200_profile_enable", "snarkvm_b200_profile_collect", "snarkvm_b200_generate_bases_device",
    "snarkvm_b200_msm_precompute_device", "snarkvm_b200_msm_precomputed_free", "snarkvm_b200_msm_precomputed_info",
    "snarkvm_b200_msm_precomputed_device", "snarkvm_b200_kzg_commit_precomputed_device",
    "snarkvm_b200_kzg_commit_hiding_device", "snarkvm_b200_kzg_commit_batch_device", "snarkvm_b200_g1_ntt_device",
    "snarkvm_b200_fr_batch_inversion_and_mul_device", "snarkvm_b200_poly_divide_by_vanishing_device", "snarkvm_b200_poly_evaluate_device",
    "snarkvm_b200_poly_divide_by_linear_device", "snarkvm_b200_sparse_matvec_device",
    "snarkvm_b200_fr_vec_op_device", "snarkvm_b200_fr_vec_scalar_op_device", "snarkvm_b200_domain_elements_device",
    "snarkvm_b200_register_bases_precomputed",
    "snarkvm_b200_msm_batch_device", "snarkvm_b200_msm_window_sums_plan_device", "snarkvm_b200_kzg_commit_batch_hiding_device",
    "snarkvm_b200_kzg_commit_batch_precomputed_device", "snarkvm_b200_msm_scratch_stats", "snarkvm_b200_msm_set_scratch_limit", "snarkvm_b200_msm_window_sums_host", "snarkvm_b200_selftest_coop", "snarkvm_b200_msm_plan_levels", "snarkvm_b200_msm_g2", "snarkvm_b200_msm_g2_device", "snarkvm_b200_generate_bases_g2_device",
    "snarkvm_b200_sonic_commit_batch_device", "snarkvm_b200_generator_mul_device", "snarkvm_b200_selftest_host_copy",
    "snarkvm_b200_index_arithmetize_device",
)


class CudaError(RuntimeError):
    """Mirror of `cuda::Error` (algorithms/cuda/src/lib.rs:19): .code is the cudaError_t."""

    def __init__(self, code: int, message: str = ""):
        super().__init__(f"cuda error {code}: {message}")
        self.code = code
        self.message = message


class _RustError(ctypes.Structure):
    _fields_ = [("code", ctypes.c_int), ("message", ctypes.c_void_p)]


_lib = None
_libc = None


def lib():
    global _lib, _libc
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing — build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(snarkvm_b200 has no CPU fallback)")
    L = ctypes.CDLL(LIB_PATH)
    for s in SYMBOLS:
        if not hasattr(L, s):
            raise ImportError(f"{LIB_PATH} does not export {s}")
    vp, sz, u32, i32, u64 = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_uint32, ctypes.c_int, ctypes.c_uint64
    L.snarkvm_ntt.restype = _RustError
    L.snarkvm_ntt.argtypes = [vp, u32, i32, i32, i32]
    L.snarkvm_polymul.restype = _RustError
    L.snarkvm_polymul.argtypes = [vp, sz, vp, vp, sz, vp, vp, u32]
    L.snarkvm_msm.restype = _RustError
    L.snarkvm_msm.argtypes = [vp, vp, sz, vp, sz]
    L.snarkvm_b200_version.restype = ctypes.c_char_p
    L.snarkvm_b200_launch_count.restype = u64
    L.snarkvm_b200_ntt_device.argtypes = [vp, u32, i32, i32, i32, vp, vp]
    L.snarkvm_b200_polymul_device.argtypes = [vp, sz, vp, vp, sz, vp, vp, u32, vp]
    L.snarkvm_b200_msm_plan.argtypes = [sz, ctypes.POINTER(i32), ctypes.POINTER(i32), ctypes.POINTER(u32)]
    L.snarkvm_b200_msm_device.argtypes = [vp, vp, sz, vp, sz, vp]
    L.snarkvm_b200_msm_window_sums_device.argtypes = [vp, vp, sz, vp, sz, vp]
    L.snarkvm_b200_xyzz_sum_ranks_device.argtypes = [vp, vp, i32, i32, vp]
    L.snarkvm_b200_msm_finish.argtypes = [vp, vp, i32, i32]
    L.snarkvm_b200_kzg_commit_device.argtypes = [vp, vp, sz, vp, sz, vp]
    L.snarkvm_b200_fr_from_mont_device.argtypes = [vp, vp, sz, vp]
    L.snarkvm_b200_fr_to_mont_device.argtypes = [vp, vp, sz, vp]
    L.snarkvm_b200_srs_decode_device.argtypes = [vp, sz, vp, sz, vp, vp]
    L.snarkvm_b200_register_bases.argtypes = [vp, sz, sz]
    L.snarkvm_b200_unregister_bases.argtypes = [vp]
    L.snarkvm_b200_register_bases_precomputed.argtypes = [vp, sz, sz]
    L.snarkvm_b200_profile_enable.argtypes = [i32]
    L.snarkvm_b200_profile_collect.argtypes = [i32, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(u64)]
    L.snarkvm_b200_generate_bases_device.argtypes = [vp, sz, sz, u64, vp]
    L.snarkvm_b200_generate_bases_g2_device.argtypes = [vp, sz, sz, u64, vp]
    L.snarkvm_b200_msm_plan_levels.argtypes = [sz]
    L.snarkvm_b200_msm_g2_device.argtypes = [vp, vp, sz, vp, sz, vp]
    L.snarkvm_b200_msm_g2.argtypes = [vp, vp, sz, vp, sz]
    L.snarkvm_b200_msm_precompute_device.argtypes = [ctypes.POINTER(vp), vp, sz, sz, vp]
    L.snarkvm_b200_msm_precomputed_free.argtypes = [vp]
    L.snarkvm_b200_msm_precomputed_info.argtypes = [vp, ctypes.POINTER(sz), ctypes.POINTER(i32), ctypes.POINTER(i32), ctypes.POINTER(sz)]
    L.snarkvm_b200_msm_precomputed_device.argtypes = [vp, vp, vp, sz, vp]
    L.snarkvm_b200_kzg_commit_precomputed_device.argtypes = [vp, vp, vp, sz, vp]
    L.snarkvm_b200_kzg_commit_hiding_device.argtypes = [vp, vp, sz, vp, sz, vp, vp, sz, vp]
    L.snarkvm_b200_kzg_commit_batch_device.argtypes = [vp, vp, sz, vp, vp, sz, vp]
    L.snarkvm_b200_g1_ntt_device.argtypes = [vp, sz, vp, sz, u32, i32, vp]
    L.snarkvm_b200_fr_batch_inversion_and_mul_device.argtypes = [vp, sz, vp, vp]
    L.snarkvm_b200_poly_divide_by_vanishing_device.argtypes = [vp, vp, vp, sz, sz, vp]
    L.snarkvm_b200_poly_evaluate_device.argtypes = [vp, vp, sz, vp, vp]
    L.snarkvm_b200_poly_divide_by_linear_device.argtypes = [vp, vp, sz, vp, vp]
    L.snarkvm_b200_sparse_matvec_device.argtypes = [vp, vp, vp, vp, sz, vp, sz, vp]
    L.snarkvm_b200_fr_vec_op_device.argtypes = [vp, vp, vp, sz, i32, vp]
    L.snarkvm_b200_fr_vec_scalar_op_device.argtypes = [vp, vp, vp, sz, i32, vp]
    L.snarkvm_b200_domain_elements_device.argtypes = [vp, u32, vp]
    L.snarkvm_b200_index_arithmetize_device.argtypes = [i32, vp, vp, vp, vp, vp, sz, sz, sz, vp, vp, vp]
    L.snarkvm_b200_msm_batch_device.argtypes = [vp, vp, sz, vp, vp, sz, vp]
    L.snarkvm_b200_msm_window_sums_plan_device.argtypes = [vp, vp, sz, vp, sz, vp, sz, vp]
    L.snarkvm_b200_kzg_commit_batch_hiding_device.argtypes = [vp, vp, sz, vp, vp, vp, vp, vp, sz, vp]
    L.snarkvm_b200_kzg_commit_batch_precomputed_device.argtypes = [vp, vp, vp, vp, sz, vp]
    L.snarkvm_b200_sonic_commit_batch_device.argtypes = [vp, sz, vp, vp, vp, vp, vp, vp, sz, vp]
    L.snarkvm_b200_generator_mul_device.argtypes = [vp, sz, vp, sz, vp]
    L.snarkvm_b200_msm_scratch_stats.argtypes = [ctypes.POINTER(sz), ctypes.POINTER(sz), ctypes.POINTER(sz)]
    L.snarkvm_b200_msm_set_scratch_limit.argtypes = [sz]
    L.snarkvm_b200_selftest_coop.argtypes = [u32, u64, ctypes.POINTER(u32), vp]
    L.snarkvm_b200_selftest_host_copy.argtypes = [sz, u64, ctypes.POINTER(u32)]
    L.snarkvm_b200_msm_window_sums_host.argtypes = [vp, vp, sz, vp, sz, vp, sz, vp]
    for s in SYMBOLS[5:]:
        getattr(L, s).restype = i32
    L.snarkvm_b200_launch_count.restype = u64
    L.snarkvm_b200_msm_g2.restype = _RustError
    _libc = ctypes.CDLL(None)
    _libc.free.argtypes = [ctypes.c_void_p]
    _lib = L
    return L


def check_rust_error(err: _RustError) -> None:
    """`if err.code != 0 { return Err(err) }` (lib.rs:93-96); frees the malloc'd message."""
    if err.code != 0:
        msg = ""
        if err.message:
            msg = ctypes.string_at(err.message).decode(errors="replace")
            _libc.free(err.message)
        raise CudaError(err.code, msg)


def check(code: int) -> None:
    if code != 0:
        raise CudaError(code, "see cudaError_t")


def launch_count() -> int:
    return int(lib().snarkvm_b200_launch_count())


PROF_MSM_SORT, PROF_MSM_ACCUMULATE, PROF_MSM_REDUCE, PROF_NTT_PASS = 0, 1, 2, 3


def profile_enable(on: bool) -> None:
    check(lib().snarkvm_b200_profile_enable(1 if on else 0))


def profile_collect(kind: int):
    """(total_ms, launches) of the recorded kernels of `kind` since the last collect."""
    ms, cnt = ctypes.c_double(), ctypes.c_uint64()
    check(lib().snarkvm_b200_profile_collect(kind, ctypes.byref(ms), ctypes.byref(cnt)))
    return ms.value, cnt.value
