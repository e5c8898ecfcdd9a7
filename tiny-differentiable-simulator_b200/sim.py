"""BatchSim: N independent copies of World{plane, MultiBody} resident on one GPU.

Python-side mirror of the fine-grained pytinydiffsim surface for the hot path
(forward_dynamics / integrate_euler_qdd / TinyWorld.step / integrate_euler,
python/pytinydiffsim.inl:659-663,857-876), batched: one call = one step of all environments.
torch is used for device memory and streams only.
"""
import ctypes

import numpy as np

from . import _lib
from .model import model_dims

MODE_FD, MODE_NOCONTACT, MODE_FULL = 0, 1, 2
MODE_WORLD = 3   # World::step(dt) alone (src/world.hpp:293-363): contacts + constraint solve on (q, qd) -> qd; world-frame kernel
PREC_MIXED, PREC_F64, PREC_F32, PREC_AUTO = 0, 1, 2, -1


def _dp(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_double)) if a is not None else None


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


class BatchSim:
    def __init__(self, model, n_envs, device=0, dt=1e-3, gravity=(0.0, 0.0, -9.81), friction=0.5,
                 restitution=0.0, erp=0.2, cfm=1e-5, pgs_iterations=1, keep_all_points=False,
                 precision=PREC_AUTO):
        self._L = _lib.lib()
        self.model = np.ascontiguousarray(model, dtype=np.float64)
        self.info = model_dims(self.model)
        self._h = self._L.tds_b200_create(_dp(self.model), self.model.size, int(n_envs), int(device))
        if not self._h:
            raise RuntimeError("tds_b200_create failed: " + _lib.last_error())
        dims = (ctypes.c_int * 8)()
        self._L.tds_b200_get_dims(self._h, dims)
        (self.n_envs, self.n_stride, self.n_q, self.n_qd, self.n_tau, self.n_links,
         self.n_contact_points, self.n_act) = list(dims)
        self.device = device
        self.auto_reset = False
        self.set_params(dt, gravity, friction, restitution, erp, cfm, pgs_iterations, keep_all_points)
        self.set_precision(precision)

    def close(self):
        if getattr(self, "_h", None):
            self._L.tds_b200_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc:
            raise RuntimeError(f"{what} failed (rc={rc}): {_lib.last_error()}")

    def set_params(self, dt=1e-3, gravity=(0.0, 0.0, -9.81), friction=0.5, restitution=0.0, erp=0.2, cfm=1e-5,
                   pgs_iterations=1, keep_all_points=False):
        g = np.asarray(gravity, dtype=np.float64)
        self.dt = dt
        self._check(self._L.tds_b200_set_params(self._h, dt, _dp(g), friction, restitution, erp, cfm,
                                                pgs_iterations, int(keep_all_points)), "set_params")

    def set_contact_model(self, contact_model=1, spring_k=50000.0, damper_d=5000.0, exponent_n=1.5, v_transition=0.01,
                          hard_contact_condition=True):
        """0: LCP / PGS (reference solver); 1: spring-damper law (parity unpinned, see include/tds_b200.h)."""
        self._check(self._L.tds_b200_set_contact_model(self._h, int(contact_model), spring_k, damper_d, exponent_n, v_transition,
                                                       int(hard_contact_condition)), "set_contact_model")

    def set_env(self, initial_poses, start_link=0, kp=0.0, kd=0.0, max_force=0.0, action_limit=0.4,
                reward_kind=0):
        ip = np.ascontiguousarray(initial_poses, dtype=np.float64)
        self._check(self._L.tds_b200_set_env(self._h, ip.size, _dp(ip), start_link, kp, kd, max_force,
                                             action_limit, reward_kind), "set_env")
        self.n_act = ip.size

    def set_auto_reset(self, enable, reset_q=None):
        rq = None if reset_q is None else np.ascontiguousarray(reset_q, dtype=np.float64)
        if rq is not None:
            assert rq.size == self.n_q
        self._check(self._L.tds_b200_set_auto_reset(self._h, int(enable), _dp(rq)), "set_auto_reset")
        self.auto_reset = bool(enable)

    def kernel_name(self):
        """Step kernel launched by the last step call (after the library's selection / fallbacks)."""
        return self._L.tds_b200_kernel_name(self._h).decode()

    def set_precision(self, precision):
        self._check(self._L.tds_b200_set_precision(self._h, precision), "set_precision")

    @property
    def precision(self):
        """The arithmetic selector that runs (PREC_AUTO resolved: mixed for a compiled model, else fp64)."""
        return self._L.tds_b200_get_precision(self._h)

    # ---- device-resident fast path (torch CUDA tensors, SoA [dim, n_stride] float32) ----
    def alloc(self, dim):
        import torch
        return torch.zeros((max(dim, 1), self.n_stride), dtype=torch.float32, device=f"cuda:{self.device}")

    def step_device(self, mode, q, qd, tau_or_action=None, q_out=None, qd_out=None, qdd_out=None, reward=None,
                    done=None, contact_dist=None, link_xf=None, use_pd=False, stream=None):
        import torch
        q_out = q if q_out is None else q_out
        qd_out = qd if qd_out is None else qd_out
        st = ctypes.c_void_p(stream.cuda_stream if stream is not None else torch.cuda.current_stream().cuda_stream)
        rc = self._L.tds_b200_step_device(self._h, mode, int(use_pd), _ptr(q), _ptr(qd), _ptr(tau_or_action),
                                          _ptr(q_out), _ptr(qd_out), _ptr(qdd_out), _ptr(reward), _ptr(done),
                                          _ptr(contact_dist), _ptr(link_xf), st)
        self._check(rc, "step_device")

    # ---- host-buffer path: numpy [n_envs, dim] float64 in / out ----
    def step_host(self, mode, q, qd, tau_or_action=None, use_pd=False, want_contacts=False):
        q = np.ascontiguousarray(q, dtype=np.float64)
        qd = np.ascontiguousarray(qd, dtype=np.float64)
        n = self.n_envs
        assert q.shape == (n, self.n_q) and qd.shape == (n, self.n_qd)
        t = None
        if tau_or_action is not None:
            t = np.ascontiguousarray(tau_or_action, dtype=np.float64)
            assert t.shape == (n, self.n_act if use_pd else self.n_tau), t.shape
        out = dict(q=np.zeros_like(q), qd=np.zeros_like(qd))
        qdd = np.zeros_like(qd) if mode == MODE_FD else None
        cd = np.zeros((n, max(self.n_contact_points, 1))) if want_contacts else None
        rc = self._L.tds_b200_step_host(self._h, mode, int(use_pd), _dp(q), _dp(qd), _dp(t), _dp(out["q"]),
                                        _dp(out["qd"]), _dp(qdd), _dp(cd))
        self._check(rc, "step_host")
        if qdd is not None:
            out["qdd"] = qdd
        if cd is not None:
            out["contact_dist"] = cd[:, :self.n_contact_points]
            # the contact-pair index list the constraint solver keeps in this step (computed on the device)
            cnt = np.zeros(n, dtype=np.int32)
            links = np.full((n, max(self.n_contact_points, 1), 2), -9, dtype=np.int32)
            self._check(self._L.tds_b200_contact_list_host(self._h, ctypes.c_void_p(cnt.ctypes.data),
                                                           ctypes.c_void_p(links.ctypes.data)), "contact_list_host")
            out["contact_count"] = cnt
            out["contact_links"] = links[:, :self.n_contact_points]
            # ... and which candidates (rows of contact_pairs()) they are: needed to tell the multibodies of a world apart
            cand = np.full((n, max(self.n_contact_points, 1)), -9, dtype=np.int32)
            self._check(self._L.tds_b200_contact_list_candidates_host(self._h, ctypes.c_void_p(cnt.ctypes.data),
                                                                      ctypes.c_void_p(cand.ctypes.data)), "contact_list_candidates_host")
            out["contact_candidates"] = cand[:, :self.n_contact_points]
        return out

    def step_jacobian_host(self, mode, q, qd, tau_or_action=None, use_pd=False):
        """Dense Jacobian of one step per environment (forward-mode dual numbers on the GPU): [n, rows, cols] float64,
        rows = q' | qd' (qdd for MODE_FD), cols = q | qd | tau, or q | qd | action | kp, kd, max_force with use_pd."""
        q = np.ascontiguousarray(q, dtype=np.float64)
        qd = np.ascontiguousarray(qd, dtype=np.float64)
        t = None if tau_or_action is None else np.ascontiguousarray(tau_or_action, dtype=np.float64)
        dims = (ctypes.c_int * 2)()
        self._check(self._L.tds_b200_jacobian_dims(self._h, mode, int(use_pd), dims), "jacobian_dims")
        jac = np.zeros((self.n_envs, dims[0], dims[1]))
        self._check(self._L.tds_b200_step_jacobian_host(self._h, mode, int(use_pd), _dp(q), _dp(qd), _dp(t), _dp(jac)), "step_jacobian_host")
        return jac

    def step_jvp_device(self, mode, q, qd, tau_or_action, t_q, t_qd, t_tau, t_out, use_pd=False, stream=None):
        """Jacobian-vector product of one step on the device, without the dense Jacobian: q, qd, tau_or_action as for step_device
        (float32 [dim, n_stride]); tangents t_q, t_qd, t_tau float64 [dim, n_stride] or None (zero); t_out float64
        [rows, n_stride] receives the tangent of q' | qd' (of qdd for MODE_FD).  Columns e >= n_envs are not written."""
        import torch
        st = ctypes.c_void_p(stream.cuda_stream if stream is not None else torch.cuda.current_stream().cuda_stream)
        self._check(self._L.tds_b200_step_jvp_device(self._h, mode, int(use_pd), _ptr(q), _ptr(qd), _ptr(tau_or_action), _ptr(t_q),
                                                     _ptr(t_qd), _ptr(t_tau), _ptr(t_out), st), "step_jvp_device")

    def step_vjp_device(self, mode, q, qd, tau_or_action, g_out, g_q=None, g_qd=None, g_tau=None, use_pd=False, stream=None):
        """Vector-Jacobian product of one step on the device: g_out float64 [rows, n_stride] is the cotangent of q' | qd' (of qdd
        for MODE_FD); g_q, g_qd, g_tau float64 [dim, n_stride] receive the gradient of each input block, or None: that block is
        not computed (its dual lanes are not launched)."""
        import torch
        st = ctypes.c_void_p(stream.cuda_stream if stream is not None else torch.cuda.current_stream().cuda_stream)
        self._check(self._L.tds_b200_step_vjp_device(self._h, mode, int(use_pd), _ptr(q), _ptr(qd), _ptr(tau_or_action), _ptr(g_out),
                                                     _ptr(g_q), _ptr(g_qd), _ptr(g_tau), st), "step_vjp_device")

    def integrate_host(self, q, qd, qdd, update_q=True):
        """integrate_euler (update_q) / integrate_euler_qdd of one state vector per environment, on the device
        (tds_b200_integrate_euler{,_qdd}_device); host arrays [n_q], [n_qd] for a one-environment simulator or [n, dim]."""
        import torch
        dev = f"cuda:{self.device}"
        def up(a, dim):
            t = torch.zeros((max(dim, 1), self.n_stride), dtype=torch.float32, device=dev)
            a = np.asarray(a, dtype=np.float64).reshape(-1, dim) if dim else np.zeros((self.n_envs, 0))
            if dim:
                t[:dim, :self.n_envs] = torch.tensor(np.ascontiguousarray(a.T), dtype=torch.float32)
            return t
        tq, tqd, tqdd = up(q, self.n_q), up(qd, self.n_qd), up(qdd, self.n_qd)
        st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        if update_q:
            self._check(self._L.tds_b200_integrate_euler_device(self._h, _ptr(tq), _ptr(tqd), _ptr(tqdd), st), "integrate_euler")
        else:
            self._check(self._L.tds_b200_integrate_euler_qdd_device(self._h, _ptr(tqd), _ptr(tqdd), st), "integrate_euler_qdd")
        torch.cuda.synchronize()
        qo = tq[:self.n_q, :self.n_envs].T.cpu().numpy().astype(np.float64)
        qdo = tqd[:self.n_qd, :self.n_envs].T.cpu().numpy().astype(np.float64)
        single = np.asarray(q).ndim == 1
        return (qo[0], qdo[0]) if single else (qo, qdo)

    def contact_pairs(self):
        """(body_a, link_a, body_b, link_b) of every candidate contact point, reference enumeration order
        (World::compute_contacts_multi_body_internal, src/world.hpp:212-281): what World::mb_contacts_ lists each step."""
        t = np.zeros((max(self.n_contact_points, 1), 4), dtype=np.int32)
        k = self._L.tds_b200_contact_pairs(self._h, ctypes.c_void_p(t.ctypes.data), t.shape[0])
        return t[:k]

    def contact_tuples(self):
        """(mb_a, link_a, geom_a, mb_b, link_b, geom_b) of every candidate contact point (geom: index among the link's collision
        shapes): the loop indices of World::compute_contacts_multi_body_internal at which the point is emitted."""
        t = np.zeros((max(self.n_contact_points, 1), 6), dtype=np.int32)
        k = self._L.tds_b200_contact_tuples(self._h, ctypes.c_void_p(t.ctypes.data), t.shape[0])
        return t[:k]

    # ---- resident environment state ----
    def env_set_state(self, q, qd):
        q = np.ascontiguousarray(q, dtype=np.float64)
        qd = np.ascontiguousarray(qd, dtype=np.float64)
        assert q.shape == (self.n_envs, self.n_q) and qd.shape == (self.n_envs, self.n_qd)
        self._check(self._L.tds_b200_env_set_state_host(self._h, _dp(q), _dp(qd)), "env_set_state")

    def env_get_state(self):
        q = np.zeros((self.n_envs, self.n_q))
        qd = np.zeros((self.n_envs, self.n_qd))
        self._check(self._L.tds_b200_env_get_state_host(self._h, _dp(q), _dp(qd)), "env_get_state")
        return q, qd

    def env_step_host(self, actions, obs, rewards, dones):
        """actions/obs/rewards/dones: float32 host arrays (numpy or pinned torch tensors)."""
        def hp(a):
            if a is None:
                return None
            return ctypes.c_void_p(a.data_ptr() if hasattr(a, "data_ptr") else a.ctypes.data)
        self._check(self._L.tds_b200_env_step_host(self._h, hp(actions), hp(obs), hp(rewards), hp(dones)),
                    "env_step_host")

    def num_visuals(self):
        return self._L.tds_b200_num_visuals(self._h)

    def env_step_visual_device(self, actions, positions, orientations, reward=None, done=None, stream=None):
        """Env step that also streams the visual transforms in the instancing renderer's layout:
        positions / orientations are float32 CUDA tensors [n_envs * n_visuals, 4] (xyz1 / quaternion xyzw)."""
        import torch
        st = ctypes.c_void_p(stream.cuda_stream if stream is not None else torch.cuda.current_stream().cuda_stream)
        self._check(self._L.tds_b200_env_step_visual_device(self._h, _ptr(actions), _ptr(reward), _ptr(done), _ptr(positions),
                                                            _ptr(orientations), st), "env_step_visual_device")

    # ---- environment layer on the device (reset with noise + settle steps, policy rollouts) ----
    def env_reset_device(self, mask=None, noise=None, noise_amp=0.05, seed=0, settle_steps=10, stream=None):
        """mask: float32 CUDA tensor [n] (None = all); noise: float32 CUDA tensor [n_act][n_stride] (None = generated).
        stream None = the simulator's own stream (the one the host-buffer calls use)."""
        st = ctypes.c_void_p(stream.cuda_stream) if stream is not None else None
        self._check(self._L.tds_b200_env_reset_device(self._h, _ptr(mask), _ptr(noise), float(noise_amp), int(seed),
                                                      int(settle_steps), st), "env_reset_device")

    def env_rollout_device(self, policy, rollout_length, shift, total_rewards, steps, stream=None):
        """policy: float32 CUDA tensor [n_params][n_stride]; total_rewards float32 [n], steps int32 [n] CUDA tensors.
        stream None = the simulator's own stream."""
        st = ctypes.c_void_p(stream.cuda_stream) if stream is not None else None
        self._check(self._L.tds_b200_env_rollout_device(self._h, _ptr(policy), int(policy.shape[0]), int(rollout_length),
                                                        float(shift), _ptr(total_rewards), _ptr(steps), st), "env_rollout_device")

    def ars_train_step(self, w, deltas, rollout_length, delta_std=0.025, step_size=0.02, shift=0.0, seed=0, settle_steps=10,
                       obs_stats=None):
        """One ARS iteration without leaving the GPU (ARSLearner::train_step, examples/ars/ars_learner.h:162-190): for the
        directions deltas [n_params][n_stride] (one per environment) a positive and a negative rollout of the linear policy
        w +- delta_std * delta from the same reset (noise keyed by `seed`), then w += step_size * g_hat.  w: float32 CUDA
        tensor [n_params], updated in place.  Returns (r_pos, r_neg) CUDA tensors."""
        import torch
        dev = w.device
        n_params = int(w.numel())
        # everything runs on the simulator's own stream (a NULL stream argument of the env-layer calls means exactly that
        # stream, which is non-blocking: work on torch's default stream would not be ordered against it)
        torch.cuda.current_stream().synchronize()          # w, deltas, obs_stats were produced on the caller's stream
        own = torch.cuda.ExternalStream(self._L.tds_b200_stream(self._h), device=dev)
        sp = ctypes.c_void_p(own.cuda_stream)
        with torch.cuda.stream(own):
            params = torch.empty((n_params, self.n_stride), dtype=torch.float32, device=dev)
            r = [torch.zeros(self.n_stride, dtype=torch.float32, device=dev) for _ in range(2)]
            steps = torch.zeros(self.n_stride, dtype=torch.int32, device=dev)
        self._check(self._L.tds_b200_env_set_obs_stats(self._h, _ptr(obs_stats)), "env_set_obs_stats")
        for k, sign in enumerate((1.0, -1.0)):
            self._check(self._L.tds_b200_ars_perturb_device(self._h, _ptr(w), _ptr(deltas), sign * delta_std, _ptr(params), n_params, sp),
                        "ars_perturb")
            self.env_reset_device(seed=seed, settle_steps=settle_steps, stream=own)
            self.env_rollout_device(params, rollout_length, shift, r[k], steps, stream=own)
        self._check(self._L.tds_b200_ars_update_device(self._h, _ptr(w), _ptr(deltas), _ptr(r[0]), _ptr(r[1]), delta_std, step_size,
                                                       n_params, sp), "ars_update")
        self._check(self._L.tds_b200_env_set_obs_stats(self._h, None), "env_set_obs_stats")
        own.synchronize()
        return r[0], r[1]

    def env_rollout_host(self, policy, rollout_length, shift=0.0, noise=None, noise_amp=0.05, seed=0, settle_steps=10):
        """Reset (noise [n][n_act] or generated) + rollout of per-environment linear policies [n][n_params] (host arrays).
        Returns (total_rewards float64 [n], steps int32 [n])."""
        pol = np.ascontiguousarray(policy, dtype=np.float64)
        assert pol.shape[0] == self.n_envs
        nz = None if noise is None else np.ascontiguousarray(noise, dtype=np.float64)
        tot = np.zeros(self.n_envs)
        steps = np.zeros(self.n_envs, dtype=np.int32)
        self._check(self._L.tds_b200_env_rollout_host(self._h, _dp(pol), int(pol.shape[1]), int(rollout_length), float(shift), _dp(nz),
                                                      float(noise_amp), int(seed), int(settle_steps), _dp(tot),
                                                      ctypes.c_void_p(steps.ctypes.data)), "env_rollout_host")
        return tot, steps

    def bind_env_step_host(self, actions, obs, rewards, dones):
        """Bind the four host buffers once and return a zero-argument callable that performs the env step on them (the
        per-call pointer marshalling of env_step_host is a measurable part of a 40 us step)."""
        def hp(a):
            return None if a is None else ctypes.c_void_p(a.data_ptr() if hasattr(a, "data_ptr") else a.ctypes.data)
        fn, h, args = self._L.tds_b200_env_step_host, self._h, (hp(actions), hp(obs), hp(rewards), hp(dones))
        keep = (actions, obs, rewards, dones)   # the buffers must outlive the callable

        def step():
            rc = fn(h, *args)
            if rc:
                self._check(rc, "env_step_host")
            return keep[1]
        return step

    def env_step_device(self, actions, reward=None, done=None, stream=None):
        import torch
        st = ctypes.c_void_p(stream.cuda_stream if stream is not None else torch.cuda.current_stream().cuda_stream)
        self._check(self._L.tds_b200_env_step_device(self._h, _ptr(actions), _ptr(reward), _ptr(done), st),
                    "env_step_device")
