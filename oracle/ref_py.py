"""ctypes loader for oracle/_ref/libedm_ref.so — the UNMODIFIED reference (EventDrivenMap.cu,
NewtonSolver.cpp, Stability.cpp) compiled for sm_100a by oracle/ref_build/Makefile.
TEST INFRASTRUCTURE ONLY: tests/ and tools/make_ref_golden.py use it to pin the CPU oracle and the
product's FP32 compatibility mode against the real reference.  Needs a GPU (the reference has no
CPU path); the product never imports this module."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
REF_SO = os.path.join(_HERE, "_ref", "libedm_ref.so")
REF_DRIVER = os.path.join(_HERE, "_ref", "Driver_ref")
_LIB = None
M = 3  # noSpikes, parameters.hpp:12 (compile-time in the reference)


def build():
    """Compile the reference where it lies: the checkout of the reference project that the environment
    variable B200_REFERENCE_DIR names (the reference is not part of this repository; without it, nothing)."""
    ref_dir = os.environ.get("B200_REFERENCE_DIR")
    if ref_dir and os.path.isdir(ref_dir):
        subprocess.check_call(["make", "-C", os.path.join(_HERE, "ref_build"), "REF=" + os.path.abspath(ref_dir)],
                              stdout=subprocess.DEVNULL)
    return os.path.exists(REF_SO)


def available():
    return os.path.exists(REF_SO)


def lib():
    global _LIB
    if _LIB is None:
        _LIB = C.CDLL(REF_SO)
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def run(z, beta, R, N=1024, T=5.0, sigma=0.0, seed=42, want_fields=True):
    """One reference ComputeF + staged replay.  Returns (F[3] float64, dict of raw reference buffers)."""
    z = np.ascontiguousarray(z, np.float64)
    f = np.empty(M)
    out = dict(coupling=np.empty(N, np.float32), init_index=np.empty(M, np.uint16),
               lift_v=np.empty((R, N), np.float32), lift_s=np.empty((R, N), np.float32),
               last_index=np.empty((M, R), np.uint16), last_time=np.empty((M, R), np.float32),
               crossed_index=np.empty((M, R), np.uint16), crossed_time=np.empty((M, R), np.float32),
               accept=np.empty(R, np.uint32), position=np.empty((M, R), np.float32),
               mean=np.empty(M, np.float32), beta=np.empty((R, N), np.float32),
               position_cf=np.empty((M, R), np.float32), mean_replay=np.empty(M, np.float32))
    fn = lib().edm_ref_run
    fn.restype = C.c_int
    fn.argtypes = [C.c_double, C.c_uint, C.c_int, C.c_float, C.c_float, C.c_ulonglong] + [C.c_void_p] * 16
    order = ["coupling", "init_index", "lift_v", "lift_s", "last_index", "last_time", "crossed_index",
             "crossed_time", "accept", "position", "mean", "beta", "position_cf", "mean_replay"]
    rc = fn(beta, R, N, T, sigma, seed, _p(z), _p(f), *[_p(out[k]) for k in order])
    if rc not in (0, 3):
        raise RuntimeError(f"edm_ref_run rc={rc}")
    out["replay_equal"] = (rc == 0)
    return f, out


def newton(z0, beta, R, N=1024, T=5.0, sigma=0.0, seed=42, tol=1e-4, maxit=10, eps=1e-2, damping=1.0):
    z0 = np.ascontiguousarray(z0, np.float64)
    z = np.empty(M); hist = np.empty(maxit + 1); jac = np.empty((M, M), order="F")
    fn = lib().edm_ref_newton
    fn.restype = C.c_int
    fn.argtypes = [C.c_double, C.c_uint, C.c_int, C.c_float, C.c_float, C.c_ulonglong, C.c_void_p,
                   C.c_double, C.c_int, C.c_double, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]
    flag = fn(beta, R, N, T, sigma, seed, _p(z0), tol, maxit, eps, damping, _p(z), _p(hist), _p(jac))
    return flag, z, hist, jac


def unstable(z, beta, R, N=1024, T=5.0, sigma=0.0, seed=42, eps=1e-2):
    z = np.ascontiguousarray(z, np.float64)
    fn = lib().edm_ref_unstable
    fn.restype = C.c_int
    fn.argtypes = [C.c_double, C.c_uint, C.c_int, C.c_float, C.c_float, C.c_ulonglong, C.c_void_p, C.c_double]
    return fn(beta, R, N, T, sigma, seed, _p(z), eps)


def time_compute_f(z, beta, R, N=1024, T=5.0, sigma=0.0, seed=42, warm=3, reps=10):
    """ms per call of the reference's own ComputeF on this GPU (host clock around its blocking calls)."""
    z = np.ascontiguousarray(z, np.float64)
    fn = lib().edm_ref_time_compute_f
    fn.restype = C.c_double
    fn.argtypes = [C.c_double, C.c_uint, C.c_int, C.c_float, C.c_float, C.c_ulonglong, C.c_void_p, C.c_int, C.c_int]
    return fn(beta, R, N, T, sigma, seed, _p(z), warm, reps)
