"""ctypes binding of liblurk_b200.so (C ABI: include/lurk_b200.h).  No CPU fallback: if the CUDA library is
missing or no GPU is present, calls raise."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liblurk_b200.so")

FIELD_BN254_FR, FIELD_BN254_FQ, FIELD_PALLAS_FQ, FIELD_PALLAS_FP = 0, 1, 2, 3
CURVE_BN254_G1, CURVE_GRUMPKIN, CURVE_PALLAS, CURVE_VESTA = 0, 1, 2, 3
FMT_CANONICAL, FMT_MONTGOMERY = 0, 1
OK, ERR_ARG, ERR_CUDA, ERR_OOM, ERR_RANGE, ERR_NOGPU, ERR_ORDER = 0, -1, -2, -3, -4, -5, -6


class LurkError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"liblurk_b200 error {code}: {msg}")
        self.code = code


class DagNode(C.Structure):
    _fields_ = [("kind", C.c_uint8), ("reserved", C.c_uint8), ("tag", C.c_uint16 * 4), ("child", C.c_uint32 * 4)]


class DagPlan(C.Structure):
    _fields_ = [("nodes", C.c_uint64), ("levels", C.c_uint64), ("max_width", C.c_uint64), ("est_gpu_us", C.c_uint64),
                ("est_cpu_core_us", C.c_uint64), ("use_gpu", C.c_int)]


class FoldConfig(C.Structure):
    _fields_ = [("curve_id", C.c_int), ("depth", C.c_int), ("n_w", C.c_uint64), ("n_x", C.c_uint64), ("n_rows", C.c_uint64),
                ("row_ptr", C.c_void_p * 3), ("col", C.c_void_p * 3), ("val", C.c_void_p * 3), ("fmt", C.c_int),
                ("world", C.c_int), ("rank", C.c_int), ("latency_sms", C.c_int)]


class FoldSpan(C.Structure):
    _fields_ = [("first", C.c_uint64), ("row_elems", C.c_uint64), ("stride", C.c_uint64), ("rows", C.c_uint64)]


class FoldResult(C.Structure):
    _fields_ = [("comm_W", C.c_uint8 * 96), ("comm_T", C.c_uint8 * 96), ("r", C.c_uint8 * 32), ("running_comm_W", C.c_uint8 * 96),
                ("running_comm_E", C.c_uint8 * 96), ("ro_hash", C.c_uint8 * 32), ("status", C.c_int), ("seq", C.c_uint64)]


FOLD_BUF_GLUE, FOLD_BUF_X2, FOLD_BUF_RO, FOLD_BUF_W2, FOLD_BUF_T, FOLD_BUF_Z1, FOLD_BUF_E1 = -1, -2, -3, -4, -5, -6, -7
FOLD_INPUTS_RESIDENT = 1
FOLD_RO_CONST, FOLD_RO_W_X, FOLD_RO_W_Y, FOLD_RO_W_INF, FOLD_RO_T_X, FOLD_RO_T_Y, FOLD_RO_T_INF = range(7)

_vp, _sz, _i = C.c_void_p, C.c_size_t, C.c_int
# lurk_challenge_fn: int (*)(void *user, int round, const uint8_t *message, size_t message_len, uint8_t challenge_out[32])
CHALLENGE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_uint8), C.c_size_t, C.POINTER(C.c_uint8))
SUMCHECK_QUAD, SUMCHECK_CUBIC = 0, 1
# every symbol declared in include/lurk_b200.h: name -> (restype, argtypes)
PROTOTYPES = {
    "lurk_last_error": (C.c_char_p, []),
    "lurk_version": (_i, []),
    "lurk_device_count": (_i, []),
    "lurk_field_modulus": (_i, [_i, _vp]),
    "lurk_poseidon_hash_batch": (_i, [_i, _i, _vp, _sz, _vp]),
    "lurk_poseidon_hash_batch_mont": (_i, [_i, _i, _vp, _sz, _vp]),
    "lurk_poseidon_hash_batch_dev": (_i, [_i, _i, _vp, _sz, _vp, _i, _vp]),
    "lurk_poseidon_constants": (_i, [_i, _i, C.POINTER(_i), C.POINTER(_i), _vp, _vp]),
    "lurk_poseidon_witness_block": (_sz, [_i, _i]),
    "lurk_poseidon_witness_batch": (_i, [_i, _i, _vp, _sz, _vp, _i]),
    "lurk_poseidon_witness_batch_dev": (_i, [_i, _i, _vp, _sz, _vp, _i, _vp]),
    "lurk_poseidon_witness_scatter_dev": (_i, [_i, _i, _vp, _sz, _vp, _vp, _i, _vp]),
    "lurk_bitdecomp_witness_scatter_dev": (_i, [_i, _vp, _sz, _vp, _vp, _i, _vp]),
    "lurk_bitdecomp_witness_block": (_sz, [_i]),
    "lurk_bitdecomp_witness_batch": (_i, [_i, _vp, _sz, _vp, _i]),
    "lurk_bitdecomp_witness_batch_dev": (_i, [_i, _vp, _sz, _vp, _i, _vp]),
    "lurk_dag_hash": (_i, [_i, _vp, _sz, _vp, _sz, _vp]),
    "lurk_dag_hash_plan": (_i, [_vp, _sz, _sz, C.POINTER(DagPlan)]),
    "lurk_msm_ctx_create": (_i, [_i, _vp, _sz, _i, C.POINTER(_vp)]),
    "lurk_msm_ctx_create_dev": (_i, [_i, _vp, _sz, C.POINTER(_vp)]),
    "lurk_msm_ctx_destroy": (None, [_vp]),
    "lurk_msm_ctx_run": (_i, [_vp, _vp, _sz, _i, _vp]),
    "lurk_msm_ctx_run_dev": (_i, [_vp, _vp, _sz, _i, _vp, _vp]),
    "lurk_msm": (_i, [_i, _vp, _vp, _sz, _i, _vp]),
    "lurk_msm_ctx_launch_dev": (_i, [_vp, _vp, _sz, _i, _vp]),
    "lurk_msm_ctx_finish": (_i, [_vp, _vp]),
    "lurk_msm_ctx_clone": (_i, [_vp, C.POINTER(_vp)]),
    "lurk_msm_ctx_precompute": (_i, [_vp]),
    "lurk_msm_ctx_set_profiling": (_i, [_vp, _i]),
    "lurk_msm_ctx_last_profile": (_i, [_vp, C.POINTER(C.c_float), C.POINTER(C.c_uint)]),
    "lurk_point_sum": (_i, [_i, _vp, _sz, _i, _vp]),
    "lurk_synthetic_bases": (_i, [_i, C.c_uint64, _sz, _i, _vp]),
    "lurk_ck_size": (_sz, [_sz, _sz, _sz]),
    "lurk_ck_generate": (_i, [_i, _vp, _sz, _sz, _i, _vp]),
    "lurk_ck_generate_dev": (_i, [_i, _vp, _sz, _sz, _vp, _vp]),
    "lurk_ck_generate_range_dev": (_i, [_i, _vp, _sz, _sz, _sz, _vp, _vp]),
    "lurk_hash_to_curve_batch": (_i, [_i, C.c_char_p, _vp, _sz, _sz, _i, _vp]),
    "lurk_hash_to_curve_batch_dev": (_i, [_i, C.c_char_p, _vp, _sz, _sz, _vp, _i, _vp]),
    "lurk_shake256": (_i, [_vp, _sz, _vp, _sz]),
    "lurk_sumcheck_prove_dev": (_i, [_i, _i, C.POINTER(_vp), _i, _vp, CHALLENGE_FN, _vp, _vp, _vp, _vp, _i, _vp]),
    "lurk_sumcheck_prove_batch_dev": (_i, [_i, _i, _i, C.POINTER(_vp), C.POINTER(_i), _vp, _vp, CHALLENGE_FN, _vp, _vp, _vp, _vp, _i, _vp]),
    "lurk_eq_evals_dev": (_i, [_i, _vp, _i, _vp, _i, _vp]),
    "lurk_inner_product_dev": (_i, [_i, _vp, _vp, _sz, _vp, _i, _vp]),
    "lurk_poly_combine_dev": (_i, [_i, _i, C.POINTER(_vp), C.POINTER(_sz), _vp, _vp, _sz, _i, _vp]),
    "lurk_ipa_fold_scalars_dev": (_i, [_i, _vp, _sz, _vp, _vp, _i, _vp]),
    "lurk_ipa_fold_bases_dev": (_i, [_i, _vp, _sz, _vp, _vp, _i, _vp]),
    "lurk_ipa_prove_dev": (_i, [_i, _vp, _vp, _vp, _vp, _i, CHALLENGE_FN, _vp, _vp, _vp, _vp, _vp, _i, _vp]),
    "lurk_msm_ctx_info": (_i, [_vp, C.POINTER(_i), C.POINTER(_sz)]),
    "lurk_ck_powers_dev": (_i, [_i, _vp, _vp, _sz, _vp, _i, _vp]),
    "lurk_hyperkzg_prove_dev": (_i, [_i, _vp, _vp, _vp, _i, CHALLENGE_FN, _vp, _vp, _vp, _vp, _i, _vp]),
    "lurk_axpy_dev": (_i, [_i, _vp, _vp, _vp, _sz, _vp, _vp]),
    "lurk_spmv_csr_dev": (_i, [_i, _vp, _vp, _vp, _sz, _vp, _vp, _vp]),
    "lurk_cross_term_dev": (_i, [_i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _vp]),
    "lurk_convert_dev": (_i, [_i, _vp, _sz, _i, _vp, _vp]),
    "lurk_ntt_dev": (_i, [_i, _vp, _i, _i, _vp]),
    "lurk_fold_ctx_create": (_i, [C.POINTER(FoldConfig), _vp, _vp, C.POINTER(_vp)]),
    "lurk_fold_ctx_destroy": (None, [_vp]),
    "lurk_fold_ctx_add_slot_batch": (_i, [_vp, _i, _sz, _vp]),
    "lurk_fold_ctx_set_spans": (_i, [_vp, _i, C.POINTER(FoldSpan)]),
    "lurk_fold_ctx_set_ro": (_i, [_vp, _i, C.POINTER(_i), _i]),
    "lurk_fold_ctx_host_buffer": (_i, [_vp, _i, _i, C.POINTER(_vp), C.POINTER(_sz)]),
    "lurk_fold_ctx_device_buffer": (_i, [_vp, _i, _i, C.POINTER(_vp), C.POINTER(_sz)]),
    "lurk_fold_ctx_exchange_handle": (_i, [_vp, _vp]),
    "lurk_fold_ctx_set_peers": (_i, [_vp, _vp]),
    "lurk_fold_ctx_set_running": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i]),
    "lurk_fold_ctx_get_running": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i]),
    "lurk_fold_ctx_stage_a": (_i, [_vp, _i, _i, _i]),
    "lurk_fold_ctx_init_running": (_i, [_vp, _i]),
    "lurk_fold_ctx_stage_b_launch": (_i, [_vp, _i]),
    "lurk_fold_ctx_collect": (_i, [_vp, _i, C.POINTER(FoldResult), _i]),
    "lurk_fold_ctx_check_running": (_i, [_vp, C.POINTER(C.c_uint64), C.POINTER(_i), C.POINTER(_i)]),
    "lurk_fold_ctx_stats": (_i, [_vp, C.POINTER(C.c_uint), C.POINTER(C.c_uint), C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "lurk_fold_ctx_sync": (_i, [_vp]),
}

_lib = None


def lib():
    """Loads the CUDA library; raises if it has not been built (python -c 'import __graft_entry__ as g; g.build()')."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise LurkError(ERR_NOGPU, f"{LIB_PATH} not built -- run __graft_entry__.build(); there is no CPU fallback")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(rc):
    if rc != OK:
        raise LurkError(rc, lib().lurk_last_error().decode())
    return rc


def np_ptr(a):
    return a.ctypes.data_as(C.c_void_p)
