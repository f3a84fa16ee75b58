"""ctypes binding of tests/hostsim_sens_p/sens_p.cpp (TEST HARNESS ONLY): the product's parameter-sensitivity templates
compiled for the host, so that the CPU-only test run can check them against the numpy restatement
(tests/sens_oracle_p.py).  Not part of the product."""
import ctypes as C
import os
import subprocess

import numpy as np

import hostsim

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, '_build', 'libhostsim_sens_p.so')
_SRC = [os.path.join(_HERE, 'sens_p.cpp')] + [
    os.path.join(_HERE, '..', '..', 'drone_attitude_control_b200', 'csrc', f)
    for f in ('bnmpc_core.cuh', 'bnmpc_loop.cuh', 'generated/models_gen.cuh')]

MODEL_FORCE, MODEL_JERK, MODEL_FORCE_DENSE = 0, 1, 2
FP64, FP32 = 0, 1


def build(force=False):
    newest = max(os.path.getmtime(f) for f in _SRC)
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < newest:
        os.makedirs(os.path.dirname(_SO), exist_ok=True)
        subprocess.check_call(['g++', '-O1', '-std=c++17', '-fPIC', '-shared', '-mfma', '-o', _SO, _SRC[0]])
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        assert _lib.hss_sizeof_opts() == C.sizeof(hostsim.Opts)
    return _lib


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double)) if a is not None else None


def _ip(a):
    return a.ctypes.data_as(C.POINTER(C.c_int)) if a is not None else None


def sens_p(model, prec, o, p, x, u, lam, pi, status=None, have_mult=None, bnd=None, stages=None, seed_x=None, seed_u=None,
           with_grad_p=True):
    """Parameter sensitivities (p = (mass, g)) of the product templates at a given stored solution: the arguments of sens()
    plus pi [B, N, nx], the multipliers of the dynamics.  Without seeds: forward (api_sens_p), returns
    (sens_x [B, stages, nx, 2], sens_u [B, min(stages, N), nu, 2]); with seed_x and / or seed_u: adjoint (api_sens_adj),
    returns (grad_x0 [B, nx], grad_yref [B, N*ny + nx], grad_p [B, 2]), all from one evaluation (with_grad_p = False:
    grad_p is NULL, the adjoint of bnmpc_eval_adjoint_sens, and the third result is None)."""
    x = np.ascontiguousarray(x, float); u = np.ascontiguousarray(u, float); lam = np.ascontiguousarray(lam, float)
    pi = np.ascontiguousarray(pi, float)
    B, N, nx, nu = x.shape[0], o.N, x.shape[2], u.shape[2]
    assert pi.shape == (B, N, nx), pi.shape
    p = np.ascontiguousarray(p, float)
    st = np.zeros(B, np.int32) if status is None else np.ascontiguousarray(status, np.int32)
    hm = np.ones(B, np.int32) if have_mult is None else np.ascontiguousarray(have_mult, np.int32)
    bnd = None if bnd is None else np.ascontiguousarray(bnd, float)
    if seed_x is None and seed_u is None:
        stages = N + 1 if stages is None else int(stages)
        sx = np.zeros((B, stages, nx, 2)); su = np.zeros((B, min(stages, N), nu, 2))
        rc = lib().hss_sens_p(model, prec, C.byref(o), 2, B, _dp(p), _dp(x), _dp(u), _dp(lam), _dp(pi), _ip(st), _ip(hm),
                              _dp(bnd), stages, _dp(sx), _dp(su), None, None, None, None, None)
        assert rc == 0, rc
        return sx, su
    sdx = None if seed_x is None else np.ascontiguousarray(seed_x, float)
    sdu = None if seed_u is None else np.ascontiguousarray(seed_u, float)
    gx = np.zeros((B, nx)); gy = np.zeros((B, N * (nx + nu) + nx)); gp = np.zeros((B, 2)) if with_grad_p else None
    rc = lib().hss_sens_p(model, prec, C.byref(o), 1, B, _dp(p), _dp(x), _dp(u), _dp(lam), _dp(pi), _ip(st), _ip(hm),
                          _dp(bnd), 0, None, None, _dp(sdx), _dp(sdu), _dp(gx), _dp(gy), _dp(gp))
    assert rc == 0, rc
    return gx, gy, gp
