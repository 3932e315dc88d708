"""ctypes binding of libctl_b200.so (include/ctl_b200.h).

The CUDA library is the product: there is no CPU fallback.  Importing this module without
the built shared object raises; calling into it without a CUDA device fails with the
library's own error.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libctl_b200.so")

CTL_LAYOUT_BLOCK_MAJOR, CTL_LAYOUT_TIME_FASTEST = 0, 1
CTL_MAT_M, CTL_MAT_K, CTL_MAT_KT = 0, 1, 2
CTL_KSP_GMRES, CTL_KSP_FGMRES, CTL_KSP_MINRES = 0, 1, 2
CTL_PC_NONE, CTL_PC_BUILTIN, CTL_PC_CALLBACK = 0, 1, 2
CTL_PCMODE_TRIANGULAR, CTL_PCMODE_DIAGONAL = 0, 1
CTL_S0_JACOBI, CTL_S0_CHEBYSHEV, CTL_S0_AMG = 0, 1, 2
CTL_HISTORY_MAX = 1024


class ctl_config(C.Structure):
    _fields_ = [("n", C.c_int32), ("n_t", C.c_int32), ("CN", C.c_int32), ("device", C.c_int32),
                ("tau", C.c_double), ("beta", C.c_double), ("epsilon", C.c_double),
                ("stream", C.c_void_p), ("rank", C.c_int32), ("world", C.c_int32)]


class ctl_pc_options(C.Structure):
    _fields_ = [("mode", C.c_int32), ("solver_0", C.c_int32),
                ("cheb_emin", C.c_double), ("cheb_emax", C.c_double),
                ("cheb_steps", C.c_int32), ("amg_cycles", C.c_int32), ("amg_nu", C.c_int32),
                ("amg_nu_fine", C.c_int32),
                ("amg_max_levels", C.c_int32), ("amg_coarse_max", C.c_int32),
                ("amg_theta", C.c_double), ("amg_lo", C.c_double), ("amg_hi", C.c_double),
                ("amg_acc_lo", C.c_double), ("amg_acc_hi", C.c_double)]


class ctl_krylov_options(C.Structure):
    _fields_ = [("ksp_type", C.c_int32), ("restart", C.c_int32), ("max_it", C.c_int32),
                ("pc", C.c_int32), ("rtol", C.c_double), ("atol", C.c_double),
                ("divtol", C.c_double)]


class ctl_solve_result(C.Structure):
    _fields_ = [("its", C.c_int32), ("reason", C.c_int32), ("n_mult", C.c_int32),
                ("n_pc", C.c_int32), ("rnorm", C.c_double), ("ref_norm", C.c_double),
                ("n_history", C.c_int32), ("history", C.c_double * CTL_HISTORY_MAX),
                ("seconds_total", C.c_double), ("seconds_mult", C.c_double),
                ("seconds_pc", C.c_double)]


class ctl_stokes_pc_options(C.Structure):
    _fields_ = [("velocity", ctl_pc_options), ("inner_its", C.c_int32), ("mass_p", C.c_int32),
                ("mass_p_steps", C.c_int32), ("lambda_p_min", C.c_double), ("lambda_p_max", C.c_double),
                ("amg_p_nu", C.c_int32), ("amg_p_max_levels", C.c_int32),
                ("amg_p_coarse_max", C.c_int32), ("amg_p_cycles", C.c_int32),
                ("amg_p_theta", C.c_double), ("amg_p_lo", C.c_double), ("amg_p_hi", C.c_double)]


PC_CALLBACK = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_void_p)

_H = C.c_void_p
_I32P = C.POINTER(C.c_int32)
_F64P = C.c_void_p          # device or host pointers are passed as raw addresses

# name -> (restype, argtypes); mirrors include/ctl_b200.h one to one
SIGNATURES = {
    "ctl_create": (C.c_int, [C.POINTER(ctl_config), C.POINTER(_H)]),
    "ctl_destroy": (C.c_int, [_H]),
    "ctl_last_error": (C.c_char_p, [_H]),
    "ctl_version": (C.c_char_p, []),
    "ctl_set_pattern": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_int64]),
    "ctl_set_values": (C.c_int, [_H, C.c_int, C.c_int, C.c_void_p]),
    "ctl_set_bc": (C.c_int, [_H, C.c_void_p, C.c_int32]),
    "ctl_set_block_size": (C.c_int, [_H, C.c_int32]),
    "ctl_assemble": (C.c_int, [_H]),
    "ctl_n_blocks": (C.c_int32, [_H]),
    "ctl_ld": (C.c_int32, [_H]),
    "ctl_n_local": (C.c_int32, [_H]),
    "ctl_row_begin": (C.c_int32, [_H]),
    "ctl_vec_len": (C.c_int64, [_H, C.c_int]),
    "ctl_convert_layout": (C.c_int, [_H, _F64P, C.c_int, _F64P, C.c_int]),
    "ctl_kkt_apply": (C.c_int, [_H, _F64P, _F64P, C.c_int]),
    "ctl_pc_default_options": (C.c_int, [C.POINTER(ctl_pc_options)]),
    "ctl_pc_setup": (C.c_int, [_H, C.POINTER(ctl_pc_options)]),
    "ctl_pc_block_size": (C.c_int32, [_H]),
    "ctl_pc_apply": (C.c_int, [_H, _F64P, _F64P, C.c_int]),
    "ctl_pc_fn": (C.c_int, [_H, _F64P, _F64P, C.c_int]),
    "ctl_set_pc_callback": (C.c_int, [_H, PC_CALLBACK, C.c_void_p]),
    "ctl_krylov_default_options": (C.c_int, [C.POINTER(ctl_krylov_options)]),
    "ctl_solve": (C.c_int, [_H, _F64P, _F64P, C.c_int, C.POINTER(ctl_krylov_options),
                            C.POINTER(ctl_solve_result)]),
    "ctl_solve_host": (C.c_int, [_H, _F64P, _F64P, C.POINTER(ctl_krylov_options),
                                 C.POINTER(ctl_solve_result)]),
    "ctl_kkt_residual_norm": (C.c_int, [_H, _F64P, _F64P, C.c_int, C.POINTER(C.c_double)]),
    "ctl_nonlinear_residual": (C.c_int, [_H, _F64P, _F64P, _F64P, C.c_int, C.POINTER(C.c_double)]),
    "ctl_objective_host": (C.c_int, [_H, _F64P, _F64P, _F64P, C.POINTER(C.c_double)]),
    "ctl_objective": (C.c_int, [_H, _F64P, _F64P, _F64P, C.POINTER(C.c_double)]),
    "ctl_build_rhs": (C.c_int, [_H, _F64P, _F64P, _F64P, _F64P]),
    "ctl_lift_bc": (C.c_int, [_H, _F64P, _F64P, C.c_int]),
    "ctl_amg_num_hierarchies": (C.c_int32, [_H]),
    "ctl_amg_num_levels": (C.c_int32, [_H, C.c_int32]),
    "ctl_amg_level_size": (C.c_int, [_H, C.c_int32, C.c_int32, _I32P, C.POINTER(C.c_int64),
                                     C.POINTER(C.c_int64)]),
    "ctl_amg_get_csr": (C.c_int, [_H, C.c_int32, C.c_int32, C.c_int, C.c_void_p, C.c_void_p,
                                  C.c_void_p]),
    "ctl_amg_get_aggregates": (C.c_int, [_H, C.c_int32, C.c_int32, C.c_void_p]),
    "ctl_amg_solve": (C.c_int, [_H, C.c_int32, _F64P, _F64P]),
    "ctl_stokes_create": (C.c_int, [_H, _H, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(_H)]),
    "ctl_stokes_destroy": (C.c_int, [_H]),
    "ctl_stokes_vec_len": (C.c_int64, [_H]),
    "ctl_stokes_apply": (C.c_int, [_H, _F64P, _F64P]),
    "ctl_stokes_pc_default_options": (C.c_int, [C.POINTER(ctl_stokes_pc_options)]),
    "ctl_stokes_set_laplacian_p": (C.c_int, [_H, C.c_void_p]),
    "ctl_stokes_pc_setup": (C.c_int, [_H, C.POINTER(ctl_stokes_pc_options)]),
    "ctl_stokes_pc_apply": (C.c_int, [_H, _F64P, _F64P]),
    "ctl_stokes_pc_fn": (C.c_int, [_H, _F64P, _F64P]),
    "ctl_stokes_set_pc_callback": (C.c_int, [_H, PC_CALLBACK, C.c_void_p]),
    "ctl_stokes_solve": (C.c_int, [_H, _F64P, _F64P, C.POINTER(ctl_krylov_options),
                                   C.POINTER(ctl_solve_result)]),
    "ctl_stokes_lift_bc": (C.c_int, [_H, _F64P, _F64P]),
    "ctl_stokes_nonlinear_residual": (C.c_int, [_H, _F64P, _F64P, _F64P, C.POINTER(C.c_double)]),
    "ctl_stokes_time": (C.c_int, [_H, C.c_int, C.POINTER(C.c_double)]),
    "ctl_amg_setup_probe": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(ctl_pc_options),
                                      C.POINTER(C.c_int32), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ctl_comm_unique_id": (C.c_int, [C.c_void_p]),
    "ctl_comm_init": (C.c_int, [_H, C.c_void_p]),
    "ctl_kernel_launches": (C.c_int64, [_H]),
    "ctl_time_kkt_apply": (C.c_int, [_H, _F64P, _F64P, C.c_int, C.POINTER(C.c_float)]),
    "ctl_time_amg": (C.c_int, [_H, C.c_int32, C.c_int, C.c_int, C.POINTER(C.c_double)]),
}

_lib = None


def load():
    """Load the shared library (once) and attach the prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; "
            f"g.build()'` (or `make -C control_b200/csrc`).  control_b200 has no CPU fallback.")
    # torch's bundled NCCL must be the libnccl.so.2 the process resolves
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)        # AttributeError if the library lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class CtlError(RuntimeError):
    pass


def check(handle, rc):
    if rc != 0:
        msg = load().ctl_last_error(handle)
        raise CtlError(f"ctl_b200 error {rc}: {msg.decode() if msg else '?'}")
