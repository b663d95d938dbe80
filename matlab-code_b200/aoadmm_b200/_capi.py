"""ctypes binding of include/aoadmm.h (the C ABI of libaoadmm_b200.so).

The structs below are field-for-field copies of the C structs.  The library is REQUIRED: importing this
module raises if the CUDA extension has not been built (there is no CPU fallback).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libaoadmm_b200.so')

if not os.path.exists(LIB_PATH):
    raise ImportError(
        'libaoadmm_b200.so is missing (%s): build it with `make` or `python -c "import __graft_entry__ as g; '
        'g.build()"`.  The B200 engine has no CPU fallback.' % LIB_PATH)

lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)

c_uint8_p = C.POINTER(C.c_uint8)
c_double_p = C.POINTER(C.c_double)
c_int32_p = C.POINTER(C.c_int32)
c_int64_p = C.POINTER(C.c_int64)

STATUS_NAMES = {0: 'OK', 1: 'INVALID_ARG', 2: 'UNSUPPORTED', 3: 'NOT_POSITIVE_DEFINITE', 4: 'NON_FINITE',
                5: 'CUDA', 6: 'NCCL', 7: 'OOM', 8: 'NO_DEVICE'}

MODEL_CP, MODEL_PAR2 = 0, 1

FIELD_FAC, FIELD_CONSTRAINT_FAC, FIELD_CONSTRAINT_DUAL, FIELD_COUPLING_FAC, FIELD_COUPLING_DUAL = 0, 1, 2, 3, 4
FIELD_PAR2_P, FIELD_PAR2_DELTAB, FIELD_PAR2_MU_DELTAB = 5, 6, 7

# Z.constraints{m}{1} -> aoadmm_constraint_kind (functions/constraints_to_prox.m:13-91)
CONSTRAINT_KINDS = {
    'non-negativity': 1, 'box': 2, 'simplex column-wise': 3, 'simplex row-wise': 4, 'non-decreasing': 5,
    'non-increasing': 6, 'unimodality': 7, 'l1-ball': 8, 'l2-ball': 9, 'non-negative l2-ball': 10,
    'non-negative l2-sphere': 11, 'orthonormal': 12, 'l1 regularization': 13, 'l0 regularization': 14,
    'l2 regularization': 15, 'ridge': 16, 'quadratic regularization': 17, 'GL smoothness': 18,
    'TV regularization': 19, 'tPARAFAC2': 20, 'custom': 21,
}


class Constraint(C.Structure):
    _fields_ = [('kind', C.c_int32), ('p0', C.c_double), ('p1', C.c_double), ('matrix', c_double_p),
                ('matrix_n', C.c_int64)]


class Object(C.Structure):
    _fields_ = [('model', C.c_int32), ('order', C.c_int32), ('modes', c_int32_p), ('weight', C.c_double),
                ('znorm_const', C.c_double), ('data', c_double_p), ('shard_offset', C.c_int64),
                ('shard_extent', C.c_int64), ('slices', C.POINTER(c_double_p)), ('n_slices', C.c_int32),
                ('miss', c_uint8_p), ('miss_slices', C.POINTER(c_uint8_p))]


class Problem(C.Structure):
    _fields_ = [('nb_modes', C.c_int32), ('mode_rows', c_int64_p), ('mode_rank', c_int32_p),
                ('slice_rows', C.POINTER(c_int64_p)), ('n_slices', c_int32_p), ('n_objects', C.c_int32),
                ('objects', C.POINTER(Object)), ('lin_coupled_modes', c_int32_p), ('n_couplings', C.c_int32),
                ('coupling_type', c_int32_p), ('trafo', C.POINTER(c_double_p)), ('trafo_rows', c_int64_p),
                ('trafo_cols', c_int64_p), ('trafo2', C.POINTER(c_double_p)), ('trafo2_rows', c_int64_p),
                ('trafo2_cols', c_int64_p), ('coupling_rows', c_int64_p), ('coupling_cols', c_int64_p),
                ('constrained_modes', c_int32_p), ('constraints', C.POINTER(Constraint)), ('ridge', c_double_p)]


class SparseObject(C.Structure):
    _fields_ = [('nnz', C.c_int64), ('subs', c_int64_p), ('vals', c_double_p)]


class Dist(C.Structure):
    _fields_ = [('rank', C.c_int32), ('world_size', C.c_int32), ('device', C.c_int32),
                ('nccl_unique_id', C.c_uint8 * 128)]


class Options(C.Structure):
    _fields_ = [('MaxOuterIters', C.c_int32), ('MaxInnerIters', C.c_int32), ('AbsFuncTol', C.c_double),
                ('OuterRelTol', C.c_double), ('innerRelPrTol_coupl', C.c_double), ('innerRelPrTol_constr', C.c_double),
                ('innerRelDualTol_coupl', C.c_double), ('innerRelDualTol_constr', C.c_double), ('bsum', C.c_int32),
                ('bsum_weight', C.c_double), ('iter_start_PAR2Bkconstraint', C.c_int32),
                ('has_increase_factor_rhoBk', C.c_int32), ('increase_factor_rhoBk', C.c_double),
                ('mttkrp_precision', C.c_int32), ('dimtree', C.c_int32), ('fuse_inner', C.c_int32), ('graph', C.c_int32)]


class Out(C.Structure):
    _fields_ = [('f_tensors', C.c_double), ('f_couplings', C.c_double), ('f_constraints', C.c_double),
                ('f_PAR2_couplings', C.c_double), ('OuterIterations', C.c_int32), ('exit_flag', C.c_int32),
                ('func_val_conv', c_double_p), ('func_coupl_conv', c_double_p), ('func_constr_conv', c_double_p),
                ('func_PAR2_coupl', c_double_p), ('time_at_it', c_double_p), ('inner_iters', c_int32_p),
                ('error_mode', C.c_int32), ('f_rel_missing', C.c_double), ('func_rel_missing', c_double_p),
                ('non_finite_mode', C.c_int32)]


HandleP = C.c_void_p

# every symbol declared in include/aoadmm.h (tests check that the library exports all of them)
EXPORTS = ['aoadmm_abi_version', 'aoadmm_device_count', 'aoadmm_nccl_unique_id', 'aoadmm_create', 'aoadmm_destroy',
           'aoadmm_last_error', 'aoadmm_set_state', 'aoadmm_get_state', 'aoadmm_run', 'aoadmm_mttkrp', 'aoadmm_prox',
           'aoadmm_chol_solve', 'aoadmm_gram', 'aoadmm_generate_cp_data', 'aoadmm_time_mttkrp', 'aoadmm_launch_count',
           'aoadmm_phase_ms', 'aoadmm_last_run_ms', 'aoadmm_get_object_data', 'aoadmm_last_loop_ms', 'aoadmm_object_mttkrp', 'aoadmm_nvecs',
           'aoadmm_create_multi', 'aoadmm_gpu_count', 'aoadmm_comm_release', 'aoadmm_create_sparse',
           'aoadmm_create_sparse_masked', 'aoadmm_model_at', 'aoadmm_set_heldout', 'aoadmm_heldout_history',
           'aoadmm_sparse_shard_bounds', 'aoadmm_create_sparse_multi', 'aoadmm_set_heldout_stopping',
           'aoadmm_heldout_best', 'aoadmm_nvecs_sparse']

lib.aoadmm_abi_version.restype = C.c_int
lib.aoadmm_device_count.argtypes = [C.POINTER(C.c_int)]
lib.aoadmm_nccl_unique_id.argtypes = [C.POINTER(C.c_uint8)]
lib.aoadmm_create.argtypes = [C.POINTER(Problem), C.POINTER(Dist), C.POINTER(HandleP)]
lib.aoadmm_create_sparse.argtypes = [C.POINTER(Problem), C.POINTER(C.POINTER(SparseObject)), C.POINTER(Dist),
                                     C.POINTER(HandleP)]
lib.aoadmm_create_sparse_masked.argtypes = [C.POINTER(Problem), C.POINTER(C.POINTER(SparseObject)),
                                            C.POINTER(C.POINTER(SparseObject)), C.POINTER(Dist), C.POINTER(HandleP)]
lib.aoadmm_create_multi.argtypes = [C.POINTER(Problem), C.c_int32, c_int32_p, C.POINTER(HandleP)]
lib.aoadmm_sparse_shard_bounds.argtypes = [C.POINTER(SparseObject), C.c_int32, C.c_int64, C.c_int32, c_int64_p]
lib.aoadmm_create_sparse_multi.argtypes = [C.POINTER(Problem), C.POINTER(C.POINTER(SparseObject)),
                                           C.POINTER(C.POINTER(SparseObject)), C.c_int32, c_int32_p, C.POINTER(HandleP)]
lib.aoadmm_gpu_count.argtypes = [HandleP, c_int32_p]
lib.aoadmm_comm_release.argtypes = []
lib.aoadmm_destroy.argtypes = [HandleP]
lib.aoadmm_last_error.argtypes = [HandleP]
lib.aoadmm_last_error.restype = C.c_char_p
lib.aoadmm_set_state.argtypes = [HandleP, C.c_int32, C.c_int32, C.c_int32, c_double_p, C.c_int64, C.c_int64]
lib.aoadmm_get_state.argtypes = [HandleP, C.c_int32, C.c_int32, C.c_int32, c_double_p, C.c_int64, C.c_int64]
lib.aoadmm_run.argtypes = [HandleP, C.POINTER(Options), C.POINTER(Out)]
lib.aoadmm_mttkrp.argtypes = [c_double_p, C.c_int32, c_int64_p, C.POINTER(c_double_p), C.c_int32, C.c_int32,
                              c_double_p, C.c_int32]
lib.aoadmm_prox.argtypes = [C.POINTER(Constraint), c_double_p, C.c_int64, C.c_int64, C.c_double, c_double_p, C.c_int32]
lib.aoadmm_chol_solve.argtypes = [c_double_p, C.c_int32, c_double_p, C.c_int64, c_double_p, C.c_int32]
lib.aoadmm_gram.argtypes = [c_double_p, C.c_int64, C.c_int32, c_double_p, C.c_int32]
lib.aoadmm_generate_cp_data.argtypes = [HandleP, C.c_int32, C.POINTER(c_double_p), C.c_double, C.c_uint64]
lib.aoadmm_time_mttkrp.argtypes = [HandleP, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_float)]
lib.aoadmm_object_mttkrp.argtypes = [HandleP, C.c_int32, C.c_int32, C.c_int32, c_double_p]
lib.aoadmm_nvecs.argtypes = [HandleP, C.c_int32, C.c_int32, C.c_int32, c_double_p, C.c_int64, c_double_p]
lib.aoadmm_nvecs_sparse.argtypes = [HandleP, C.c_int32, C.c_int32, c_double_p, C.c_int64, c_double_p]
lib.aoadmm_launch_count.argtypes = [HandleP, C.POINTER(C.c_int64)]
lib.aoadmm_phase_ms.argtypes = [HandleP, c_double_p]
lib.aoadmm_last_run_ms.argtypes = [HandleP, c_double_p]
lib.aoadmm_last_loop_ms.argtypes = [HandleP, c_double_p]
lib.aoadmm_get_object_data.argtypes = [HandleP, C.c_int32, c_double_p, C.c_int64]
lib.aoadmm_model_at.argtypes = [HandleP, C.c_int32, C.POINTER(SparseObject), c_double_p]
lib.aoadmm_set_heldout.argtypes = [HandleP, C.c_int32, C.POINTER(SparseObject)]
lib.aoadmm_heldout_history.argtypes = [HandleP, C.c_int32, c_double_p, C.c_int64, c_int64_p]
lib.aoadmm_set_heldout_stopping.argtypes = [HandleP, C.c_int32]
lib.aoadmm_heldout_best.argtypes = [HandleP, c_int32_p, c_double_p]


class AoadmmError(RuntimeError):
    """Raised for a non-zero aoadmm_status (the C-ABI replacement of MATLAB error())."""

    def __init__(self, status, message):
        self.status = status
        self.status_name = STATUS_NAMES.get(status, str(status))
        super().__init__('aoadmm:%s: %s' % (self.status_name, message))


def check(status, handle=None):
    if status != 0:
        msg = lib.aoadmm_last_error(handle)
        raise AoadmmError(status, msg.decode('utf-8', 'replace') if msg else '')
