"""TEST INFRASTRUCTURE: ctypes binding of the dual-number instances of the step kernels compiled for the host
(tests/cpp/stepw_dual_host.cpp, tests/cpp/rigid_dual_host.cpp): the Jacobian-vector and vector-Jacobian products behind
tds_b200_step_{jvp,vjp}_device and tds_b200_rigid_{jvp,vjp}_device, executed on the CPU.  The dense Jacobians they are checked
against come from tests/emu.py.  The package never loads these libraries."""
import ctypes
import os
import subprocess

import numpy as np

from emu import _dp

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(ROOT, "tiny-differentiable-simulator_b200", "csrc")
_lib_w = None
_lib_r = None


def _build(src, so, kernel):
    deps = [src] + [os.path.join(CSRC, f) for f in (kernel, "tds_wcommon.cuh", "tds_math.cuh", "tds_dual.cuh", "tds_model.h", "tds_types.h")]
    if not (os.path.exists(so) and all(os.path.getmtime(d) <= os.path.getmtime(so) for d in deps)):
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-shared", "-fPIC", "-w", "-I" + CSRC, "-I" + os.path.join(ROOT, "include"),
                               "-I/usr/local/cuda/include", src, "-o", so + ".tmp"])
        os.replace(so + ".tmp", so)
    return ctypes.CDLL(so)


def lib_stepw():
    global _lib_w
    if _lib_w is None:
        L = _build(os.path.join(HERE, "cpp", "stepw_dual_host.cpp"), os.path.join(HERE, "cpp", "_stepw_dual_host.so"), "tds_stepw.cu")
        dp = ctypes.POINTER(ctypes.c_double)
        L.tdsemu_stepw_dual.restype = ctypes.c_int
        L.tdsemu_stepw_dual.argtypes = [dp, ctypes.c_int, dp, dp, ctypes.c_int, ctypes.c_int, ctypes.c_int] + [dp] * 11
        _lib_w = L
    return _lib_w


def lib_rigid():
    global _lib_r
    if _lib_r is None:
        L = _build(os.path.join(HERE, "cpp", "rigid_dual_host.cpp"), os.path.join(HERE, "cpp", "_rigid_dual_host.so"), "tds_rigid.cu")
        dp = ctypes.POINTER(ctypes.c_double)
        L.tdsemu_rigid_dual.restype = ctypes.c_int
        L.tdsemu_rigid_dual.argtypes = [dp, ctypes.c_int, dp, ctypes.c_int, dp, dp, ctypes.c_int] + [dp] * 6
        _lib_r = L
    return _lib_r


def _params(dt, gravity, friction, restitution, erp, cfm, pgs_iterations, keep_all_points, contact_model, spring_k, damper_d, exponent_n,
            v_transition, hard_contact_condition):
    return np.array([dt, *gravity, friction, restitution, erp, cfm, pgs_iterations, int(keep_all_points), contact_model, spring_k,
                     damper_d, exponent_n, v_transition, int(hard_contact_condition)], dtype=np.float64)


def _c(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.float64)


def step_dual(model, mode, q, qd, tau=None, use_pd=False, env=None, tangents=None, cotangent=None, want=(True, True, True), dt=1e-3,
              gravity=(0.0, 0.0, -9.81), friction=0.5, restitution=0.0, erp=0.2, cfm=1e-5, pgs_iterations=1, keep_all_points=False,
              contact_model=0, spring_k=50000.0, damper_d=5000.0, exponent_n=1.5, v_transition=0.01, hard_contact_condition=True):
    """JVP and / or VJP of one step through the host-compiled dual instance, launched like tds_b200_step_{jvp,vjp}_device.
    tangents: (t_q, t_qd, t_tau), each [n][dim] or None; cotangent [n][rows]; want: which gradient blocks (q, qd, tau) to request.
    Returns dict(jvp=[n][rows] or None, vjp=(g_q, g_qd, g_tau) with None for the blocks not requested, or None)."""
    m = np.ascontiguousarray(model, dtype=np.float64)
    q, qd = _c(q), _c(qd)
    n, n_q, n_qd = q.shape[0], int(m[3]), int(m[4])
    e = _c(env)
    n_in = int(e[0]) if use_pd else n_qd - (6 if int(m[2]) else 0)
    rows = n_qd if mode == 0 else n_q + n_qd
    params = _params(dt, gravity, friction, restitution, erp, cfm, pgs_iterations, keep_all_points, contact_model, spring_k, damper_d,
                     exponent_n, v_transition, hard_contact_condition)
    t = [None] * 3 if tangents is None else [_c(x) for x in tangents]
    t_out = np.zeros((n, rows)) if tangents is not None else None
    g_out = _c(cotangent)
    g = [np.zeros((n, d)) if (g_out is not None and w) else None for d, w in zip((n_q, n_qd, n_in), want)]
    rc = lib_stepw().tdsemu_stepw_dual(_dp(m), m.size, _dp(params), _dp(e), mode, int(use_pd), n, _dp(q), _dp(qd), _dp(_c(tau)),
                                           _dp(t[0]), _dp(t[1]), _dp(t[2]), _dp(t_out), _dp(g_out), _dp(g[0]), _dp(g[1]), _dp(g[2]))
    if rc < 0:
        raise RuntimeError(f"tdsemu_stepw_dual rc={rc}")
    return dict(jvp=t_out, vjp=tuple(g) if g_out is not None else None)


def rigid_dual(desc, state, force=None, steps=1, tangents=None, cotangent=None, want=(True, True), dt=1.0 / 60.0, gravity=(0.0, 0.0, -9.81),
               friction=0.5, restitution=0.0, erp=0.1, num_solver_iterations=1):
    """JVP and / or VJP of `steps` World::step calls through the host-compiled rigid dual instance, launched like
    tds_b200_rigid_{jvp,vjp}_device.  state [n][n_bodies][13], force / tangent of the force [n][n_bodies][3]; tangents (t_state, t_force);
    cotangent [n][n_bodies][13]; want: which gradient blocks (state, force).  Returns dict(jvp, vjp=(g_state, g_force)) like step_dual."""
    L = lib_rigid()
    d = np.ascontiguousarray(desc, dtype=np.float64)
    s = _c(state)
    n, nb = s.shape[0], d.shape[0]
    params = np.array([dt, *gravity, friction, restitution, erp, num_solver_iterations], dtype=np.float64)
    t = [None, None] if tangents is None else [_c(x) for x in tangents]
    t_out = np.zeros((n, nb, 13)) if tangents is not None else None
    g_out = _c(cotangent)
    g = [np.zeros((n, nb, k)) if (g_out is not None and w) else None for k, w in zip((13, 3), want)]
    rc = L.tdsemu_rigid_dual(_dp(d), nb, _dp(params), n, _dp(s), _dp(_c(force)), steps, _dp(t[0]), _dp(t[1]), _dp(t_out), _dp(g_out),
                             _dp(g[0]), _dp(g[1]))
    if rc:
        raise RuntimeError(f"tdsemu_rigid_dual rc={rc}")
    return dict(jvp=t_out, vjp=tuple(g) if g_out is not None else None)
