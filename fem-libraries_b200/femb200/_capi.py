"""ctypes binding of libfemb200.so (the C ABI declared in include/femb200.h).

There is no CPU fallback: if the shared library is missing the import fails, and
every compute entry point needs a CUDA device (sm_100a).  Build the library with
`make -C fem-libraries_b200/csrc` (or `python -c "import __graft_entry__ as g; g.build()"`).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("FEMB200_LIB") or os.path.join(os.path.dirname(_HERE), "lib", "libfemb200.so")

P1, P2, Q2, Q1 = 0, 1, 2, 3
ROWMAJOR_INTERLEAVED, COLMAJOR_BYNODES = 0, 1
TANGENT_CLOSED, TANGENT_AD = 0, 1
OP_CSR, OP_PA = 0, 1
DIST_NCCL, DIST_P2P, DIST_BLOB_BYTES = 1, 2, 256
SC_FLAG, SC_ITERS, SC_FINAL, SC_RED_NOM, SC_RED_DEN, SC_RED_BETA, SC_COUNT = 4, 5, 6, 9, 10, 11, 16

vp, i32, i64, f64 = C.c_void_p, C.c_int, C.c_int64, C.c_double

# name -> argtypes; every function returns int (0 = ok) unless listed in _SPECIAL
SIGNATURES = {
    "femb200_device_info": [C.POINTER(C.c_int)] * 3,
    "femb200_fp64_probe": [i32, i32, vp, C.POINTER(i64), C.POINTER(f64), vp],
    "femb200_tabulate_tensor_batched": [i32, i64, vp, vp, i32, vp, vp, vp, f64, vp, vp, i32, i32, vp],
    "femb200_plan_create": [i32, i64, i64, vp, vp, vp, C.POINTER(vp)],
    "femb200_plan_sizes": [vp, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64), C.POINTER(i64), C.POINTER(C.c_int32),
                           C.POINTER(i64)],
    "femb200_plan_block_csr": [vp, C.POINTER(vp), C.POINTER(vp)],
    "femb200_plan_copy_block_csr": [vp, vp, vp, vp],
    "femb200_plan_scalar_csr": [vp, vp, vp, vp],
    "femb200_assemble_matrix": [vp, vp, i32, vp, f64, vp, vp, i32, vp, vp],
    "femb200_assemble_matrix_nobc": [vp, vp, i32, vp, f64, vp, vp, i32, vp, vp],
    "femb200_assemble_vector": [vp, vp, i32, vp, f64, vp, vp, vp, vp, vp],
    "femb200_apply_lifting": [vp, vp, vp, vp, f64, vp, vp, vp],
    "femb200_set_bc": [vp, vp, vp, f64, vp, vp],
    "femb200_axpy": [i64, f64, vp, vp, vp],
    "femb200_plan_set_dirichlet": [vp, vp, vp],
    "femb200_apply_dirichlet": [vp, vp, f64, vp],
    "femb200_matrix_norms": [vp, vp, vp, vp],
    "femb200_spmv": [vp, vp, vp, vp, vp],
    "femb200_spmv_dot": [vp, vp, vp, vp, vp, vp],
    "femb200_spmv_rows": [vp, vp, vp, vp, i64, i64, vp, i32, vp, vp],
    "femb200_extract_diagonal": [vp, vp, vp, vp],
    "femb200_jacobi_setup": [i64, vp, vp, vp],
    "femb200_pcg": [vp, i32, vp, vp, vp, vp, i64, f64, f64, i32, vp, i32, i32, vp, C.POINTER(C.c_int),
                    C.POINTER(C.c_double), C.POINTER(C.c_int), vp],
    "femb200_dot": [i64, vp, vp, vp, vp],
    "femb200_cg_set_tolerances": [vp, f64, f64, vp],
    "femb200_cg_init": [i64, vp, vp, vp, vp, vp, vp, vp],
    "femb200_cg_scalar_step": [vp, i32, vp],
    "femb200_cg_apply": [vp, i32, vp, vp, vp, vp, vp, vp],
    "femb200_cg_update_xr": [i64, vp, vp, vp, vp, vp, vp, vp],
    "femb200_cg_update_dir": [i64, vp, vp, vp, vp, vp],
    "femb200_pa_create": [i32, i64, i64, vp, vp, vp, i32, vp, f64, vp, C.POINTER(vp)],
    "femb200_pa_set_dirichlet": [vp, vp, f64, vp],
    "femb200_pa_apply": [vp, vp, vp, vp],
    "femb200_pa_diagonal": [vp, vp, vp],
    "femb200_gather": [i64, vp, vp, vp, vp],
    "femb200_scatter_rows": [i64, i32, vp, vp, vp, vp],
    "femb200_plan_set_option": [vp, C.c_char_p, i32],
    "femb200_plan_get_option": [vp, C.c_char_p, C.POINTER(C.c_int)],
    "femb200_dist_create": [vp, i32, i32, i64, i64, i32, vp, vp, vp, vp, vp, vp, C.POINTER(vp)],
    "femb200_dist_nccl_unique_id": [vp],
    "femb200_dist_nccl_comm_create": [vp, i32, i32, C.POINTER(vp)],
    "femb200_dist_nccl_comm_destroy": [vp],
    "femb200_dist_attach_nccl": [vp, vp],
    "femb200_dist_p2p_export": [vp, vp],
    "femb200_dist_p2p_attach": [vp, vp],
    "femb200_dist_set_transport": [vp, i32],
    "femb200_dist_allreduce_sum": [vp, vp, i32, vp],
    "femb200_dist_halo": [vp, vp, vp],
    "femb200_dist_mult": [vp, vp, vp, vp, vp],
    "femb200_dist_pcg": [vp, i32, vp, vp, vp, vp, f64, f64, i32, vp, i32, i32, i32, C.POINTER(C.c_int),
                         C.POINTER(C.c_double), C.POINTER(C.c_int), vp],
    "femb200_dist_vectors": [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)],
    "femb200_assemble_matrix_norms": [vp, vp, i32, vp, f64, vp, vp, i32, vp, vp, vp],
    "femb200_create_pattern": [i32, i64, i64, vp, vp, vp, C.POINTER(vp)],
    "femb200_element_grad_batched": [i32, i64, vp, vp, i32, vp, vp, vp, f64, vp, vp, i32, vp],
    "femb200_assemble_pa": [i32, i64, i64, vp, vp, vp, i32, vp, f64, vp, C.POINTER(vp)],
    "femb200_add_mult_pa": [vp, i64, vp, vp, vp, vp],
    "femb200_cg": [vp, i32, vp, vp, vp, vp, i64, f64, f64, i32, i32, C.POINTER(C.c_int), C.POINTER(C.c_double),
                   C.POINTER(C.c_int), vp],
    "femb200_smooth_damage": [vp, vp, vp, i32, f64, vp],
    "femb200_cell_strain_stress": [i32, i64, vp, vp, vp, i32, vp, f64, vp, vp, vp, vp, vp],
    "femb200_mg_create": [vp, i32, vp, vp, vp, i32, f64, vp, C.POINTER(vp)],
    "femb200_mg_create_op": [i32, vp, i32, vp, vp, i32, vp, i32, f64, vp, C.POINTER(vp)],
    "femb200_mg_sizes": [vp, C.POINTER(C.c_int), vp, vp, vp, C.POINTER(i64)],
    "femb200_mg_galerkin": [vp, vp, i32, vp],
    "femb200_mg_setup": [vp, vp, vp],
    "femb200_mg_level_values": [vp, i32, vp, vp],
    "femb200_mg_coarse_matrix": [vp, vp, vp],
    "femb200_mg_set_coarse_inverse": [vp, vp, vp],
    "femb200_mg_restrict": [vp, i32, vp, vp, vp, vp],
    "femb200_mg_prolong": [vp, i32, vp, vp, vp],
    "femb200_mg_vcycle": [vp, vp, vp, vp],
    "femb200_mg_vcycle_timed": [vp, vp, vp, vp, vp],
    "femb200_pcg_mg": [vp, vp, vp, f64, f64, i32, i32, vp, C.POINTER(C.c_int), C.POINTER(C.c_double),
                       C.POINTER(C.c_int), vp],
}
_SPECIAL = {
    "femb200_version": ([], C.c_int),
    "femb200_last_error": ([], C.c_char_p),
    "femb200_plan_destroy": ([vp], None),
    "femb200_tabulate_tensor_ufcx": ([C.POINTER(f64), C.POINTER(f64), C.POINTER(f64), C.POINTER(f64), C.POINTER(C.c_int),
                                      C.POINTER(C.c_uint8)], None),
    "femb200_dist_destroy": ([vp], None),
    "femb200_dist_transport": ([vp], C.c_int),
    "femb200_pa_destroy": ([vp], None),
    "femb200_mg_destroy": ([vp], None),
}
ALL_SYMBOLS = sorted(list(SIGNATURES) + list(_SPECIAL))

_lib = None


class Femb200Error(RuntimeError):
    pass


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} not found: build it with `make -C fem-libraries_b200/csrc` "
                              "(there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        for name, args in SIGNATURES.items():
            fn = getattr(L, name)
            fn.argtypes, fn.restype = args, C.c_int
        for name, (args, res) in _SPECIAL.items():
            fn = getattr(L, name)
            fn.argtypes, fn.restype = args, res
        _lib = L
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        raise Femb200Error(lib().femb200_last_error().decode(errors="replace"))


def call(name: str, *args) -> None:
    check(getattr(lib(), name)(*args))
