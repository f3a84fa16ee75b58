"""ctypes binding of libbnmpc.so (C-ABI in include/bnmpc.h).  There is no CPU path: if the library is missing or no
CUDA device is present, the calls raise."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('BNMPC_LIB') or os.path.join(_HERE, 'lib', 'libbnmpc.so')      # BNMPC_LIB: another build of the same library (A/B timing)

MODEL_FORCE, MODEL_JERK, MODEL_FORCE_DENSE, MODEL_THRUST, MODEL_ATT = 0, 1, 2, 3, 4
MODELS = {'force': MODEL_FORCE, 'jerk': MODEL_JERK, 'force_dense': MODEL_FORCE_DENSE, 'thrust': MODEL_THRUST, 'att': MODEL_ATT}
FP64, FP32 = 0, 1
# acados return values (reference src/Readme.md:14-20)
SUCCESS, FAILURE, MAXITER, MINSTEP, QP_FAILURE = 0, 1, 2, 3, 4
FIELDS = {'x': 0, 'u': 1, 'yref': 2, 'lbx': 3, 'ubx': 4, 'p': 5, 'pi': 6, 'lam': 7, 'lbu': 8, 'ubu': 9}
STATS = {'status': 0, 'sqp_iter': 1, 'qp_iter': 2}


class Config(C.Structure):
    """struct bnmpc_config"""
    _fields_ = [('model', C.c_int32), ('horizon', C.c_int32), ('precision', C.c_int32), ('erk_stages', C.c_int32),
                ('sqp_max_iter', C.c_int32), ('qp_max_iter', C.c_int32), ('rti', C.c_int32), ('threads_per_block', C.c_int32),
                ('dt', C.c_double), ('W', C.c_double * 16), ('W_e', C.c_double * 12),
                ('lbx', C.c_double * 12), ('ubx', C.c_double * 12), ('lbu', C.c_double * 4), ('ubu', C.c_double * 4),
                ('tol', C.c_double * 4), ('qp_tol', C.c_double * 4),
                ('mu0', C.c_double), ('thr0', C.c_double), ('alpha_min', C.c_double), ('lam_min', C.c_double), ('t_min', C.c_double),
                ('sim_erk_stages', C.c_int32), ('sim_substeps', C.c_int32), ('sim_dt', C.c_double)]


class ClosedLoopArgs(C.Structure):
    """struct bnmpc_closed_loop_args"""
    _fields_ = [('n_steps', C.c_int32), ('first_step', C.c_int32), ('ref_rows', C.c_int32), ('ref_shared', C.c_int32),
                ('log_stride', C.c_int32), ('steps_per_launch', C.c_int32),
                ('ref', C.c_void_p), ('noise', C.c_void_p), ('Xsim', C.c_void_p), ('U_plant', C.c_void_p), ('U_ctrl', C.c_void_p),
                ('a_log', C.c_void_p), ('status', C.c_void_p), ('qp_iter', C.c_void_p),
                ('noise_philox', C.c_int32), ('reserved', C.c_int32), ('noise_seed', C.c_uint64), ('noise_std', C.c_double),
                ('first_instance', C.c_int64)]


class BnmpcError(RuntimeError):
    pass


_lib = None


def lib():
    """Load libbnmpc.so.  Raises if it has not been built (python -c 'import __graft_entry__ as g; g.build()')."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BnmpcError(f'{LIB_PATH} not found: build the CUDA library first (make -C drone_attitude_control_b200/csrc); '
                         'there is no CPU fallback')
    L = C.CDLL(LIB_PATH)
    vp, i32p, dp = C.c_void_p, C.POINTER(C.c_int32), C.c_void_p
    sig = {
        'bnmpc_version': (C.c_int, []),
        'bnmpc_last_error': (C.c_char_p, []),
        'bnmpc_config_default': (C.c_int, [C.c_int, C.POINTER(Config)]),
        'bnmpc_create': (C.c_int, [C.POINTER(Config), C.c_int, C.c_int, C.POINTER(vp)]),
        'bnmpc_destroy': (C.c_int, [vp]),
        'bnmpc_set_stream': (C.c_int, [vp, vp]),
        'bnmpc_synchronize': (C.c_int, [vp]),
        'bnmpc_dims': (C.c_int, [vp, i32p]),
        'bnmpc_workspace_bytes': (C.c_int64, [vp]),
        'bnmpc_set': (C.c_int, [vp, C.c_int, C.c_int, dp, C.c_int]),
        'bnmpc_get': (C.c_int, [vp, C.c_int, C.c_int, dp, C.c_int]),
        'bnmpc_set_yref_all': (C.c_int, [vp, dp, C.c_int]),
        'bnmpc_set_ref_table': (C.c_int, [vp, dp, C.c_int, C.c_int, C.c_int, C.c_int]),
        'bnmpc_set_yref_row': (C.c_int, [vp, C.c_int]),
        'bnmpc_reset': (C.c_int, [vp]),
        'bnmpc_solve': (C.c_int, [vp]),
        'bnmpc_get_stats': (C.c_int, [vp, C.c_int, vp, C.c_int]),
        'bnmpc_solve_for_x0': (C.c_int, [vp, dp, dp, vp, C.c_int]),
        'bnmpc_sim_step': (C.c_int, [vp, C.c_int, dp, dp, dp, dp, dp, C.c_int]),
        'bnmpc_step_for_x0': (C.c_int, [vp, dp, dp, dp, dp, dp, vp, dp, C.c_int]),
        'bnmpc_eval_sens_x0': (C.c_int, [vp, C.c_int, dp, dp, C.c_int]),
        'bnmpc_eval_adjoint_sens': (C.c_int, [vp, dp, dp, dp, dp, C.c_int]),
        'bnmpc_closed_loop_init': (C.c_int, [vp, dp, dp, dp]),
        'bnmpc_closed_loop_run': (C.c_int, [vp, C.POINTER(ClosedLoopArgs)]),
        'bnmpc_closed_loop_state': (C.c_int, [vp, dp, dp, dp, dp]),
        'bnmpc_closed_loop_failures': (C.c_int, [vp, vp, C.c_int]),
        'bnmpc_philox_noise': (C.c_int, [vp, C.c_uint64, C.c_double, C.c_int64, C.c_int, C.c_int, dp]),
        'bnmpc_gen_circle_table': (C.c_int, [vp, dp, C.c_int, dp]),
        'bnmpc_launch_count': (C.c_int64, [vp]),
        'bnmpc_debug_profile': (C.c_int, [vp, vp, C.c_int]),
        'bnmpc_measure_fma_peak': (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_double)]),
        'bnmpc_selftest_rcp': (C.c_int, [C.c_int, C.c_int64, C.c_int, C.POINTER(C.c_int64)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = res, args
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise BnmpcError(f'libbnmpc error {rc}: {lib().bnmpc_last_error().decode()}')


def default_config(model, **kw):
    cfg = Config()
    check(lib().bnmpc_config_default(MODELS[model] if isinstance(model, str) else int(model), C.byref(cfg)))
    for k, v in kw.items():
        cur = getattr(cfg, k)
        if hasattr(cur, '__len__'):
            vals = list(v) if hasattr(v, '__len__') else [v] * len(cur)
            for i, x in enumerate(vals):
                cur[i] = x
        else:
            setattr(cfg, k, v)
    return cfg
