"""ctypes binding of libfem_b200.so (include/fem_b200.h).  No CPU fallback: if the shared
library is missing or no CUDA device is visible, every compute entry point raises."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("FEM_B200_LIB") or os.path.join(_HERE, "libfem_b200.so")   # override: A/B builds of the kernels

STATUS = {0: "FEM_OK", 1: "FEM_ERR_INVALID_ARG", 2: "FEM_ERR_CUDA", 3: "FEM_ERR_NONFINITE_JACOBIAN",
          4: "FEM_ERR_PCG_BREAKDOWN", 5: "FEM_ERR_PCG_MAXIT", 6: "FEM_ERR_UNSUPPORTED", 7: "FEM_ERR_NO_DEVICE"}
FEM_ERR_PCG_MAXIT = 5


class FemError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"{STATUS.get(code, code)}: {msg}")
        self.code = code


class NonFiniteJacobian(FemError, ArithmeticError):
    pass


_vp, _i64, _i32, _dbl = C.c_void_p, C.c_int64, C.c_int, C.c_double

# name -> argtypes (restype is int unless listed in _RESTYPE)
SIGNATURES = {
    "fem_last_error_string": [],
    "fem_version": [],
    "fem_device_info": [C.POINTER(_i32), C.POINTER(_i32), C.POINTER(_i32), C.POINTER(_i64), C.POINTER(_i64)],
    "fem_plan_create": [_i64, _i64, _i32, _i32, _vp, _vp, C.POINTER(_dbl), C.POINTER(_dbl), C.POINTER(_dbl), _vp, C.POINTER(_vp)],
    "fem_plan_destroy": [_vp],
    "fem_plan_sizes": [_vp, C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_i32)],
    "fem_plan_pattern": [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_i64)],
    "fem_plan_blocks": [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_i64)],
    "fem_plan_geometry": [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp)],
    "fem_plan_stage_info": [_vp, C.POINTER(_i32), C.POINTER(_i32)],
    "fem_plan_bytes": [_vp],
    "fem_elastic_dmat": [_vp, _vp, _vp, _vp, _vp],
    "fem_assemble_elastic": [_vp, _vp, _vp, _vp, _vp],
    "fem_assemble_tangent": [_vp, _vp, _vp, _vp],
    "fem_assemble_tangent_ref": [_vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "fem_assemble_tangent_force": [_vp, _vp, _vp, _vp, _vp, _vp],
    "fem_strain": [_vp, _vp, _vp, _vp],
    "fem_internal_force": [_vp, _vp, _vp, _vp],
    "fem_dp_return_map": [_i64, _vp, C.POINTER(_dbl), _vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "fem_spmv": [_vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "fem_jacobi_setup": [_vp, _vp, _vp, _vp, _vp],
    "fem_pcg_init": [_i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "fem_pcg_spmv_dot": [_vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp],
    "fem_pcg_update_xr": [_i64, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp],
    "fem_pcg_update_p": [_i64, _vp, _vp, _vp, _vp, _i32, _vp],
    "fem_halo_push": [_vp, _i64, _i64, _vp, _i64, _i64, _vp, _vp],
    "fem_pcg_update_p_push": [_i64, _i64, _vp, _vp, _vp, _vp, _i32, _i64, _i64, _vp, _i64, _i64, _vp, _vp],
    "fem_ppcg_words": [],
    "fem_ppcg_begin": [_vp, _vp, _i32, _vp],
    "fem_ppcg_spmv_dot": [_vp, _vp, _vp, _vp, _vp, _vp, C.POINTER(_vp), _i32, _i32, _vp],
    "fem_ppcg_update_xr": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, C.POINTER(_vp), _i32, _i32, _vp],
    "fem_ppcg_update_p": [_vp, _i64, _i64, _vp, _vp, _vp, _i64, _i64, _vp, _i64, _i64, _vp, _vp, C.POINTER(_vp), _i32, _i32, _vp],
    "fem_pcg": [_vp, _vp, _vp, _vp, _dbl, _i32, _i32, _vp, _vp, C.POINTER(_i32), C.POINTER(_dbl), _vp],
    "fem_coarse_galerkin": [_vp, _vp, _vp, _vp, _vp, _dbl, _dbl, _dbl, _dbl, _i32, _i32, _vp, _vp],
    "fem_dense_gemv": [_i32, _vp, _vp, _vp, _vp, _vp],
    "fem_tl_init": [_i64, _vp, _vp, _vp, _vp, _vp, _dbl, _dbl, _dbl, _dbl, _i32, _i32, _vp, _vp, _vp, _vp],
    "fem_tl_update_xr": [_i64, _vp, _vp, _vp, _vp, _dbl, _dbl, _dbl, _dbl, _i32, _i32, _vp, _vp, _vp, _vp, _i32, _vp],
    "fem_tl_apply": [_i64, _i32, _vp, _vp, _vp, _vp, _dbl, _dbl, _dbl, _dbl, _i32, _i32, _vp, _vp, _vp, _i32, _i32, _vp],
    "fem_mg_sizeof": [_i32],
    "fem_mg_lattice": [_i64, _vp, _dbl, _dbl, _dbl, _dbl, _i32, _i32, _i32, _vp, _vp, _vp, _vp],
    "fem_mg_galerkin_fine": [_vp, _vp, _vp, _vp, _vp, _i32, _vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp],
    "fem_mg_galerkin_stencil": [_i32, _i32, _i32, _i32, _vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp],
    "fem_mg_block_jacobi": [_vp, _vp, _vp, _vp, _vp],
    "fem_mg_level_finalize": [_i64, _vp, _dbl, _vp, _vp],
    "fem_mg_stencil_apply": [_i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp],
    "fem_mg_stencil_to_dense": [_i32, _i32, _vp, _vp, _vp],
    "fem_mg_vcycle": [_vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "fem_peer_allreduce": [_vp, _i32, _vp, C.POINTER(_vp), _i64, _i64, _i64, _i32, _i32, _vp],
    "fem_mg_fine_step": [_vp, _vp, _i32, _vp, _vp, _vp, _vp, _dbl, _dbl, _vp, _vp],
    "fem_mg_to_f32": [_i64, _vp, _vp, _vp],
    "fem_mg_lattice_check": [_vp, _vp, _i32, _vp, _vp],
    "fem_mg_to_f32_lattice": [_vp, _vp, _vp, _vp, _i64, _i32, _i32, _vp],
    "fem_mg_fine_step_lattice": [_vp, _vp, _i32, _vp, _vp, _vp, _dbl, _dbl, _vp, _vp],
    "fem_mg_exchange_run": [_vp, _vp, _vp, _vp],
    "fem_mg_pcg_init": [_i64, _vp, _vp, _vp, _vp, _vp, _vp],
    "fem_mg_pcg_update_xr": [_i64, _vp, _vp, _vp, _vp, _vp, _i32, _vp],
    "fem_mg_pcg_update_p": [_i64, _vp, _vp, _vp, _i32, _vp],
    "fem_energy_norms": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "fem_vec_axpby": [_i64, _dbl, _vp, _dbl, _vp, _vp, _vp],
    "fem_transform": [_vp, _vp, _vp, _vp],
    "fem_vector_volume": [_vp, _vp, C.POINTER(_dbl), _vp, _vp],
    "fem_segment_sum_ordered": [_i64, _vp, _vp, _vp, _vp],
    "fem_midpoints_p2_count": [_i64, _i64, _vp, C.POINTER(_vp), C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_i32), _vp],
    "fem_midpoints_p2_fill": [_vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "fem_midpoints_p2_destroy": [_vp, _vp],
    "fem_set_tuning": [C.c_char_p, _i32],
}
_RESTYPE = {"fem_last_error_string": C.c_char_p, "fem_plan_bytes": _i64}

_lib = None


def load():
    """Load (once) and return the ctypes library; raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise ImportError(f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, args in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here = header/library mismatch
        fn.argtypes = args
        fn.restype = _RESTYPE.get(name, C.c_int)
    _lib = lib
    for kv in filter(None, os.environ.get("FEM_B200_TUNING", "").split(",")):      # launch-shape / diagnostic knobs: "key=value,..."
        k, v = kv.split("=")
        if lib.fem_set_tuning(k.strip().encode(), int(v)) != 0:
            raise ValueError(f"FEM_B200_TUNING: {kv!r} rejected: {lib.fem_last_error_string().decode()}")
    return lib


def check(code):
    if code != 0:
        msg = load().fem_last_error_string().decode()
        if code == 3:
            raise NonFiniteJacobian(code, msg)
        raise FemError(code, msg)


def call(name, *args):
    check(getattr(load(), name)(*args))
