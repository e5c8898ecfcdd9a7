"""Batched worlds of rigid bodies on the GPU: the RigidBody path of the reference's World::step (src/world.hpp:293-363,
src/rigid_body.hpp, src/rb_constraint_solver.hpp; python/examples/billiard_optimization.py steps exactly this loop).
Host side of csrc/tds_rigid.cu / the tds_b200_rigid_* C-ABI (include/tds_b200.h)."""
import ctypes

import numpy as np

from . import _lib

SPHERE, PLANE, CAPSULE, BOX = 0, 1, 2, 4     # tds::GeometryTypes (src/geometry.hpp:30-38)


def sphere(mass, radius):
    return [mass, SPHERE, radius, 0.0, 0.0, 0.0]


def capsule(mass, radius, length):
    return [mass, CAPSULE, radius, length, 0.0, 0.0]


def box(mass, extents):
    return [mass, BOX, extents[0], extents[1], extents[2], 0.0]


def plane(normal=(0.0, 0.0, 1.0), constant=0.0):
    return [0.0, PLANE, normal[0], normal[1], normal[2], constant]


def _stream_arg(stream):
    """None: the world's own stream.  A torch stream: that stream; torch's default stream (handle 0) is passed as
    cudaStreamLegacy (1), since a null handle means the world's own stream to the tds_b200_rigid_*_device calls."""
    return None if stream is None else ctypes.c_void_p(stream.cuda_stream or 1)


def identity_state(n_worlds, n_bodies):
    """[n_worlds][n_bodies][13]: everything zero, orientations the identity quaternion (x, y, z, w) = (0, 0, 0, 1)."""
    s = np.zeros((n_worlds, n_bodies, 13))
    s[:, :, 6] = 1.0
    return s


class RigidWorld:
    """n_worlds independent worlds of the same bodies.  bodies: list of sphere() / capsule() / box() / plane() records, in the
    order the reference's World would hold them (contacts are enumerated over pairs i < j in that order)."""

    def __init__(self, bodies, n_worlds, device=0, **params):
        self._L = _lib.lib()
        self.desc = np.ascontiguousarray(bodies, dtype=np.float64).reshape(-1, 6)
        self.n_bodies, self.n_worlds, self.device = self.desc.shape[0], int(n_worlds), device
        self._h = self._L.tds_b200_rigid_create(ctypes.c_void_p(self.desc.ctypes.data), self.n_bodies, self.n_worlds, device)
        if not self._h:
            raise RuntimeError("tds_b200_rigid_create: " + _lib.last_error())
        self.set_params(**params)

    def close(self):
        if getattr(self, "_h", None):
            self._L.tds_b200_rigid_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc:
            raise RuntimeError(f"{what}: rc={rc} {_lib.last_error()}")

    def set_params(self, dt=1.0 / 60.0, gravity=(0.0, 0.0, -9.81), friction=0.5, restitution=0.0, erp=0.1, num_solver_iterations=1):
        g = np.asarray(gravity, dtype=np.float64)
        self._check(self._L.tds_b200_rigid_set_params(self._h, dt, ctypes.c_void_p(g.ctypes.data), friction, restitution, erp,
                                                      int(num_solver_iterations)), "rigid_set_params")

    def _args(self, state, force):
        s = np.ascontiguousarray(state, dtype=np.float64)
        assert s.shape == (self.n_worlds, self.n_bodies, 13), s.shape
        f = None
        if force is not None:
            f = np.ascontiguousarray(force, dtype=np.float64)
            assert f.shape == (self.n_worlds, self.n_bodies, 3), f.shape
        return s, f

    def step(self, state, force=None, steps=1):
        """`steps` calls of World::step(dt); force = apply_central_force before the first one.  Returns the new state."""
        s, f = self._args(state, force)
        out = np.zeros_like(s)
        self._check(self._L.tds_b200_rigid_step_host(self._h, ctypes.c_void_p(s.ctypes.data), ctypes.c_void_p(f.ctypes.data) if f is not None else None,
                                                     int(steps), ctypes.c_void_p(out.ctypes.data)), "rigid_step_host")
        return out

    def step_jacobian(self, state, force=None, steps=1):
        """(state_out, J): J [n_worlds][13 n_bodies][16 n_bodies] = d state_out / d (state | force), forward-mode on the GPU."""
        s, f = self._args(state, force)
        out = np.zeros_like(s)
        jac = np.zeros((self.n_worlds, 13 * self.n_bodies, 16 * self.n_bodies))
        self._check(self._L.tds_b200_rigid_jacobian_host(self._h, ctypes.c_void_p(s.ctypes.data), ctypes.c_void_p(f.ctypes.data) if f is not None else None,
                                                         int(steps), ctypes.c_void_p(out.ctypes.data), ctypes.c_void_p(jac.ctypes.data)), "rigid_jacobian_host")
        return out, jac

    def step_device(self, state_in, state_out, force=None, steps=1, stream=None):
        """CUDA tensors, fp64: state [13 * n_bodies][n_stride], force [3 * n_bodies][n_stride] or None; in place allowed.
        stream: a torch stream (torch's default stream included), or None for the world's own stream."""
        p = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
        self._check(self._L.tds_b200_rigid_step_device(self._h, p(state_in), p(state_out), p(force), int(steps), _stream_arg(stream)),
                    "rigid_step_device")

    def jvp_device(self, state, force, steps, t_state, t_force, t_out, stream=None):
        """Jacobian-vector product of `steps` steps with respect to (state | force), CUDA tensors fp64 in the layouts of step_device:
        tangents t_state [13 * n_bodies][n_stride], t_force [3 * n_bodies][n_stride] or None (zero) -> t_out like state."""
        p = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
        self._check(self._L.tds_b200_rigid_jvp_device(self._h, p(state), p(force), int(steps), p(t_state), p(t_force), p(t_out),
                                                      _stream_arg(stream)), "rigid_jvp_device")

    def vjp_device(self, state, force, steps, g_out, g_state=None, g_force=None, stream=None):
        """Vector-Jacobian product of `steps` steps: g_out (cotangent of the new state) -> g_state, g_force (None: not computed)."""
        p = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
        self._check(self._L.tds_b200_rigid_vjp_device(self._h, p(state), p(force), int(steps), p(g_out), p(g_state), p(g_force),
                                                      _stream_arg(stream)), "rigid_vjp_device")

    @property
    def n_stride(self):
        return (self.n_worlds + 31) & ~31
