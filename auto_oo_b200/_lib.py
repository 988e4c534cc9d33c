"""ctypes binding of ``liboo_b200.so`` (C ABI in ``include/oo_b200.h``).

There is deliberately no fallback: if the library is missing it is built with
nvcc, and if that is impossible importing a compute entry point raises.  Nothing
here routes to a CPU implementation.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

_c_double_p = C.c_void_p      # device pointers are passed as integers
_i32 = C.c_int
_i64 = C.c_int64
_f64 = C.c_double
_ptr = C.c_void_p
_size = C.c_size_t
_u32 = C.c_uint

OO_WS_ROTATION, OO_WS_INT2E, OO_WS_HESSIAN, OO_WS_INT1E, OO_WS_YMATRIX = 1, 2, 3, 4, 5
OO_WS_CLASS_TRANSFORM, OO_WS_CLASS_BUFFER, OO_WS_CLASS_HESSIAN, OO_WS_CLASS_TRANSFORM_SYM = 6, 7, 8, 9
OO_WS_CLASS_HESSIAN_VECTOR, OO_WS_HESSIAN_VECTOR, OO_WS_HESSIAN_DIAGONAL, OO_WS_KRYLOV = 10, 11, 12, 13
OO_WS_ROTATION_VJP = 14
# per-call variant switches (include/oo_b200.h)
OO_FLAG_HESSIAN_DENSE, OO_FLAG_HESSIAN_ASSEMBLE_PER_ELEMENT, OO_FLAG_HESSIAN_ASSEMBLE_TILED = 1, 2, 4
OO_FLAG_CLASS_UNFUSED_PACK, OO_FLAG_HESSIAN_GROUP_UNSTREAMED, OO_FLAG_HESSIAN_ASSEMBLE_UNSTREAMED = 8, 16, 32
OO_FLAG_CLASS_Q2_RECTANGULAR, OO_FLAG_CLASS_ERI_8FOLD, OO_FLAG_HESSIAN_REUSE_OPERANDS = 64, 128, 256
OO_FLAG_CLASS_DIRECT_STORES, OO_FLAG_HESSIAN_SPMM_UNPAIRED, OO_FLAG_CLASS_Q1_UNPAIRED = 512, 1024, 2048


def OO_FLAG_CLASS_STAGE(k):
    """Run only GEMM stage k (0: quarter 1; 1-3: Coulomb class; 4-6: exchange class) of the symmetric class transform."""
    return 1 << (16 + k)

ABI_VERSION = 2

# name -> (restype, argtypes); mirrors include/oo_b200.h one to one
_SIGNATURES = {
    "oo_abi_version": (_i32, []),
    "oo_error_string": (C.c_char_p, [_i32]),
    "oo_last_cuda_error": (_i32, []),
    "oo_launch_count": (C.c_ulonglong, []),
    "oo_device_info": (_i32, [C.POINTER(_i32)] * 3),
    "oo_workspace_bytes": (_size, [_i32, _i32, _i32, _i32, _i32]),
    "oo_dgemm_tn_f64": (_i32, [_ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _i64, _i64, _i32,
                               _i64, _i64, _i64, _ptr]),
    "oo_dgemm_tn_swap02_f64": (_i32, [_ptr, _ptr, _ptr, _ptr, _i32, _i32, _i32, _i64, _i64, _i64, _i64, _i64,
                                      _ptr]),
    "oo_dgemm_small_f64": (_i32, [_i32, _i32, _i32, _i32, _i32, _f64, _ptr, _i32, _i64, _ptr, _i32,
                                  _i64, _f64, _ptr, _i32, _i64, _f64, _ptr, _i32, _i64, _i32, _ptr]),
    "oo_kappa_rotation_f64": (_i32, [_ptr, _ptr, _ptr, _i32, _i32, _i32, _i32, _i32, _ptr, _ptr,
                                     _size, _ptr]),
    "oo_kappa_rotation_vjp_f64": (_i32, [_ptr, _ptr, _ptr, _i32, _i32, _i32, _i32, _i32, _ptr, _ptr, _ptr,
                                         _size, _ptr]),
    "oo_expm_device_squarings_max_n": (_i32, []),
    "oo_expm_f64": (_i32, [_ptr, _f64, _i32, _i32, _i32, _i32, _ptr, _ptr, _size, _ptr]),
    "oo_mo_coeff_f64": (_i32, [_ptr, _i64, _ptr, _i64, _ptr, _i64, _i32, _i32, _i32, _ptr, _ptr, _size, _ptr]),
    "oo_int1e_transform_f64": (_i32, [_ptr, _i64, _ptr, _i64, _i32, _i32, _i32, _ptr, _ptr, _size, _ptr]),
    "oo_int2e_transform_f64": (_i32, [_ptr, _i64, _ptr, _ptr, _ptr, _ptr, _i64, _i32, _i32, _i32,
                                      _ptr, _ptr, _size, _ptr]),
    "oo_active_hamiltonian_f64": (_i32, [_ptr, _ptr, _i32, _i32, _i32, _i32, _i32, _f64, _ptr, _ptr, _ptr,
                                         _ptr, _ptr]),
    "oo_energy_f64": (_i32, [_ptr, _ptr, _ptr, _ptr, _i64, _ptr, _i64, _i32, _i32, _ptr, _ptr]),
    "oo_fock_gradient_f64": (_i32, [_ptr, _ptr, _ptr, _i64, _ptr, _i64, _i32, _i32, _i32, _i32, _i32,
                                    _ptr, _ptr, _i32, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr]),
    "oo_fock_gradient_vjp_f64": (_i32, [_ptr, _ptr, _ptr, _i32, _i32, _i32, _i32, _ptr, _ptr, _ptr]),
    "oo_hessian_f64": (_i32, [_ptr, _ptr, _ptr, _ptr, _ptr, _i32, _i32, _i32, _i32, _ptr, _ptr, _i32,
                              _ptr, _ptr, _size, _u32, _ptr]),
    "oo_transpose_f64": (_i32, [_ptr, _ptr, _i64, _i64, _ptr]),
    "oo_class_transform_f64": (_i32, [_ptr, _i64, _ptr, _i64, _i32, _i32, _i32, _i32, _ptr, _ptr, _size, _ptr]),
    "oo_eri_symmetry_defect_f64": (_i32, [_ptr, _i32, _ptr, _ptr]),
    "oo_pair_ld": (_i64, [_i32]),
    "oo_pack_eri_pairs_f64": (_i32, [_ptr, _ptr, _i32, _ptr]),
    "oo_pack_eri_8fold_f64": (_i32, [_ptr, _ptr, _i32, _ptr]),
    "oo_class_transform_sym_f64": (_i32, [_ptr, _i64, _ptr, _i64, _i32, _i32, _i32, _i32, _ptr, _ptr, _size, _u32,
                                          _ptr]),
    "oo_class_transform_sym_slab_f64": (_i32, [_ptr, _i64, _i64, _i64, _ptr, _i64, _i32, _i32, _i32, _i32, _ptr, _ptr,
                                               _size, _u32, _ptr]),
    "oo_class_active_hamiltonian_f64": (_i32, [_ptr, _i32, _i32, _i32, _i32, _i32, _i32, _f64, _ptr, _ptr, _ptr,
                                               _ptr, _ptr]),
    "oo_class_fock_gradient_f64": (_i32, [_ptr, _ptr, _i64, _ptr, _i64, _i32, _i32, _i32, _i32, _i32, _i32,
                                          _ptr, _ptr, _i32, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr]),
    "oo_class_fock_gradient_vjp_f64": (_i32, [_ptr, _ptr, _ptr, _i32, _i32, _i32, _i32, _i32, _ptr, _ptr, _ptr]),
    "oo_class_hessian_f64": (_i32, [_ptr, _ptr, _ptr, _i64, _ptr, _i64, _i32, _i32, _i32, _i32, _i32, _i32, _ptr,
                                    _ptr, _i32, _ptr, _ptr, _size, _u32, _ptr]),
    "oo_class_hessian_vector_f64": (_i32, [_ptr, _ptr, _ptr, _ptr, _i32, _i32, _i32, _i32, _i32, _ptr, _ptr, _i32,
                                           _ptr, _i32, _ptr, _ptr, _size, _ptr]),
    "oo_class_hessian_diagonal_f64": (_i32, [_ptr, _ptr, _ptr, _ptr, _i32, _i32, _i32, _i32, _i32, _ptr, _ptr, _i32,
                                             _ptr, _ptr, _size, _ptr]),
    "oo_hessian_vector_f64": (_i32, [_ptr, _ptr, _ptr, _ptr, _ptr, _i32, _i32, _i32, _i32, _ptr, _ptr, _i32, _ptr,
                                     _i32, _ptr, _ptr, _size, _ptr]),
    "oo_hessian_diagonal_f64": (_i32, [_ptr, _ptr, _ptr, _ptr, _ptr, _i32, _i32, _i32, _i32, _ptr, _ptr, _i32, _ptr,
                                       _ptr, _size, _ptr]),
    "oo_subspace_eigh_f64": (_i32, [_ptr, _i32, _i32, _i64, _i32, _ptr, _i64, _ptr, _i32, _i64, _ptr]),
    "oo_davidson_project_f64": (_i32, [_ptr, _i64, _i64, _i32, _ptr, _ptr, _i32, _ptr, _i32, _ptr]),
    "oo_davidson_expand_f64": (_i32, [_ptr, _ptr, _i64, _i64, _i32, _i32, _ptr, _i32, _ptr, _ptr, _f64, _ptr, _i32,
                                      _ptr, _ptr, _ptr, _ptr, _ptr, _size, _ptr]),
    "oo_pcg_step_f64": (_i32, [_i64, _ptr, _f64, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _i32, _ptr, _size,
                               _ptr]),
    "oo_pack_lower_f64": (_i32, [_ptr, _i32, _i32, _ptr, _ptr]),
    "oo_copy_f64": (_i32, [_ptr, _ptr, _i64, _ptr]),
    "oo_rdm_columns": (_i64, [_i32]),
    "oo_rdm_excitations_f64": (_i32, [_ptr, _i32, _i32, _i32, _i64, _i64, _i32, _ptr, _ptr, _i64, _ptr]),
    "oo_rdm_sector_flags_f64": (_i32, [_ptr, _i32, _i32, _i32, _ptr, _ptr]),
    "oo_rdm_sector_mask": (_i32, [_ptr, _i32, _i32, _ptr, _ptr]),
    "oo_rdm_accumulate_f64": (_i32, [_ptr, _i32, _i64, _ptr, _ptr]),
    "oo_rdm_assemble_f64": (_i32, [_ptr, _i32, _ptr, _ptr, _ptr]),
    "oo_rdm_operator_matrix_f64": (_i32, [_ptr, _ptr, _i32, _ptr, _ptr]),
    "oo_rdm_apply_gather_f64": (_i32, [_ptr, _ptr, _i32, _i32, _i64, _i64, _ptr, _ptr, _ptr, _ptr]),
    "oo_full_rdms_f64": (_i32, [_ptr, _ptr, _i32, _i32, _i32, _ptr, _ptr, _ptr]),
    "oo_y_matrix_f64": (_i32, [_ptr, _ptr, _i32, _i32, _ptr, _ptr, _size, _ptr]),
    "oo_pad_copy_f64": (_i32, [_ptr, _ptr, _i32, _i32, _i32, _i32, _i32, _ptr]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


class OOError(RuntimeError):
    pass


def library_path():
    return _build.LIB_PATH


def load():
    """Load (building first if necessary) and return the ctypes library handle."""
    global _lib
    if _lib is not None:
        return _lib
    # build_library() returns at once when the stamp next to the .so matches the digest of the sources in the
    # tree; an edited csrc/*.cu therefore never runs against a stale binary (raises if nvcc is unavailable)
    path = _build.build_library()
    lib = C.CDLL(path)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)                # AttributeError = symbol missing: fail loudly
        fn.restype = res
        fn.argtypes = args
    if lib.oo_abi_version() != ABI_VERSION:
        raise OOError(f"ABI mismatch: library {lib.oo_abi_version()} != binding {ABI_VERSION}")
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        lib = load()
        msg = lib.oo_error_string(rc).decode()
        extra = f" (cudaError {lib.oo_last_cuda_error()})" if rc == -4 else ""
        raise OOError(f"{what or 'liboo_b200'} failed: {msg}{extra}")
