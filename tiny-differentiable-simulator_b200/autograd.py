"""torch.autograd through batched steps: `loss.backward()`, `torch.autograd.forward_ad` and `torch.func.jvp` over rollouts of
BatchSim and RigidWorld.

    q1, qd1 = tds_b200.autograd.step(sim, q0, qd0, tau)          # tau.requires_grad -> tau.grad after loss.backward()
    state = tds_b200.autograd.rigid_step(world, state0, force, steps=50)

The forward value is the production step (BatchSim.step_device / RigidWorld.step_device: whichever kernel the simulator
selects).  Derivatives never need the dense Jacobian: backward is one vector-Jacobian product and forward mode one
Jacobian-vector product, both by forward-mode dual numbers (fp64) through the world-frame kernel (csrc/tds_stepw.cu,
csrc/tds_rigid.cu).  A backward launches one dual lane per environment and input direction of the blocks that need a gradient,
each writing one double; a JVP launches one lane per environment.  Only the inputs are saved for backward.

Semantics:
  * the derivative is that of the fp64 world-frame step at the fp32 inputs the forward pass stepped from, whichever kernel
    computed the forward value (the specialised / decomposed kernels agree with it to their precision, not bit for bit);
  * derivatives are taken with respect to the raw components of quaternion coordinates (floating base, spherical joints), as
    the dense Jacobian does: the tangent of a unit quaternion is not projected onto the sphere;
  * at a kink (contact activation, friction cone, PD clamps) the derivative is that of the branch taken;
  * PD gains are constants here (their derivatives: BatchSim.step_jacobian_host); backward is not differentiable again.
"""
import torch
from torch.autograd.function import once_differentiable

from .sim import MODE_FD, MODE_FULL, MODE_WORLD


def _device(obj):
    return torch.device("cuda", obj.device)


def _check(x, name, shape, dtypes, device):
    if not isinstance(x, torch.Tensor):
        raise TypeError(f"{name}: expected a tensor, got {type(x).__name__}")
    if tuple(x.shape) != tuple(shape):
        raise ValueError(f"{name}: expected shape {tuple(shape)}, got {tuple(x.shape)}")
    if x.dtype not in dtypes:
        raise TypeError(f"{name}: expected dtype {' or '.join(str(d) for d in dtypes)}, got {x.dtype}")
    if x.device != device:
        raise ValueError(f"{name}: expected a tensor on {device}, got {x.device}")


def _plain(t):
    """The tensor under torch.func's wrappers (the kernels read raw device memory; the rules below run with torch.func's
    dispatch disabled and hand back plain tensors, which torch.func wraps again)."""
    while t is not None and torch._C._functorch.is_functorch_wrapped_tensor(t):
        t = torch._C._functorch.get_unwrapped(t)
    return t


def _soa(x, ns, dtype):
    """[n, ...] -> [dim, ns] (environment index fastest), zero padding columns."""
    x = x.detach().reshape(x.shape[0], -1)
    t = torch.zeros((max(x.shape[1], 1), ns), dtype=dtype, device=x.device)
    t[:x.shape[1], :x.shape[0]] = x.T
    return t


def _aos(t, dim, n, like):
    """[dim, ns] -> [n, dim] in the dtype of `like`."""
    return t[:dim, :n].T.to(like.dtype).contiguous()


class _Step(torch.autograd.Function):
    @staticmethod
    def forward(sim, mode, use_pd, q, qd, tau):
        n, ns = sim.n_envs, sim.n_stride
        q_s, qd_s, tau_s = _soa(q, ns, torch.float32), _soa(qd, ns, torch.float32), _soa(tau, ns, torch.float32)
        q_o, qd_o = sim.alloc(sim.n_q), sim.alloc(sim.n_qd)
        qdd_o = sim.alloc(sim.n_qd) if mode == MODE_FD else None
        sim.step_device(mode, q_s, qd_s, tau_s, q_out=q_o, qd_out=qd_o, qdd_out=qdd_o, use_pd=use_pd)
        if mode == MODE_FD:
            return _aos(qdd_o, sim.n_qd, n, q)
        return _aos(q_o, sim.n_q, n, q), _aos(qd_o, sim.n_qd, n, q)

    @staticmethod
    def setup_context(ctx, inputs, output):
        sim, mode, use_pd, q, qd, tau = inputs
        ctx.sim, ctx.mode, ctx.use_pd = sim, mode, use_pd
        ctx.save_for_backward(q, qd, tau)
        ctx.save_for_forward(q, qd, tau)

    @staticmethod
    def _inputs(ctx):
        q, qd, tau = (_plain(t) for t in ctx.saved_tensors)
        ns = ctx.sim.n_stride
        return q, (_soa(q, ns, torch.float32), _soa(qd, ns, torch.float32), _soa(tau, ns, torch.float32))

    @staticmethod
    @once_differentiable
    def backward(ctx, *grads):
        with torch._C._DisableFuncTorch():
            return _Step._backward(ctx, *(_plain(g) for g in grads))

    @staticmethod
    def _backward(ctx, *grads):
        sim, mode = ctx.sim, ctx.mode
        q, ins = _Step._inputs(ctx)
        n, ns = sim.n_envs, sim.n_stride
        if mode == MODE_FD:
            rows = [(grads[0], sim.n_qd)]
        else:
            rows = [(grads[0], sim.n_q), (grads[1], sim.n_qd)]
        g_out = torch.cat([_soa(g, ns, torch.float64)[:d] if g is not None else torch.zeros((d, ns), dtype=torch.float64, device=q.device)
                           for g, d in rows])
        dims = (sim.n_q, sim.n_qd, sim.n_act if ctx.use_pd else sim.n_tau)
        need = ctx.needs_input_grad[3:6]
        g_in = [torch.zeros((max(d, 1), ns), dtype=torch.float64, device=q.device) if w else None for d, w in zip(dims, need)]
        sim.step_vjp_device(mode, *ins, g_out, *g_in, use_pd=ctx.use_pd)
        return (None, None, None) + tuple(None if g is None else _aos(g, d, n, q) for g, d in zip(g_in, dims))

    @staticmethod
    def jvp(ctx, _sim, _mode, _use_pd, t_q, t_qd, t_tau):
        with torch._C._DisableFuncTorch():
            return _Step._jvp(ctx, _plain(t_q), _plain(t_qd), _plain(t_tau))

    @staticmethod
    def _jvp(ctx, t_q, t_qd, t_tau):
        sim, mode = ctx.sim, ctx.mode
        q, ins = _Step._inputs(ctx)
        n, ns = sim.n_envs, sim.n_stride
        rows = sim.n_qd if mode == MODE_FD else sim.n_q + sim.n_qd
        t_out = torch.zeros((rows, ns), dtype=torch.float64, device=q.device)
        tan = [None if t is None else _soa(t, ns, torch.float64) for t in (t_q, t_qd, t_tau)]
        sim.step_jvp_device(mode, *ins, *tan, t_out, use_pd=ctx.use_pd)
        if mode == MODE_FD:
            return _aos(t_out, sim.n_qd, n, q)
        return _aos(t_out, sim.n_q, n, q), _aos(t_out[sim.n_q:], sim.n_qd, n, q)


class _RigidStep(torch.autograd.Function):
    @staticmethod
    def forward(world, steps, state, force):
        ns = world.n_stride
        s, f = _soa(state, ns, torch.float64), _soa(force, ns, torch.float64)
        out = torch.empty_like(s)
        world.step_device(s, out, f, steps, stream=torch.cuda.current_stream(state.device))
        return _aos(out, 13 * world.n_bodies, world.n_worlds, state).reshape(state.shape)

    @staticmethod
    def setup_context(ctx, inputs, output):
        world, steps, state, force = inputs
        ctx.world, ctx.steps = world, steps
        ctx.save_for_backward(state, force)
        ctx.save_for_forward(state, force)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        with torch._C._DisableFuncTorch():
            return _RigidStep._backward(ctx, _plain(g))

    @staticmethod
    def _backward(ctx, g):
        world = ctx.world
        state, force = (_plain(t) for t in ctx.saved_tensors)
        ns, nb, nw = world.n_stride, world.n_bodies, world.n_worlds
        need = ctx.needs_input_grad[2:4]
        g_s = torch.zeros((13 * nb, ns), dtype=torch.float64, device=state.device) if need[0] else None
        g_f = torch.zeros((3 * nb, ns), dtype=torch.float64, device=state.device) if need[1] else None
        world.vjp_device(_soa(state, ns, torch.float64), _soa(force, ns, torch.float64), ctx.steps, _soa(g, ns, torch.float64), g_s, g_f,
                         stream=torch.cuda.current_stream(state.device))
        return (None, None, None if g_s is None else _aos(g_s, 13 * nb, nw, state).reshape(state.shape),
                None if g_f is None else _aos(g_f, 3 * nb, nw, force).reshape(force.shape))

    @staticmethod
    def jvp(ctx, _world, _steps, t_state, t_force):
        with torch._C._DisableFuncTorch():
            return _RigidStep._jvp(ctx, _plain(t_state), _plain(t_force))

    @staticmethod
    def _jvp(ctx, t_state, t_force):
        world = ctx.world
        state, force = (_plain(t) for t in ctx.saved_tensors)
        ns = world.n_stride
        t_out = torch.zeros((13 * world.n_bodies, ns), dtype=torch.float64, device=state.device)
        world.jvp_device(_soa(state, ns, torch.float64), _soa(force, ns, torch.float64), ctx.steps,
                         None if t_state is None else _soa(t_state, ns, torch.float64),
                         None if t_force is None else _soa(t_force, ns, torch.float64), t_out,
                         stream=torch.cuda.current_stream(state.device))
        return _aos(t_out, 13 * world.n_bodies, world.n_worlds, state).reshape(state.shape)


def step(sim, q, qd, tau=None, mode=MODE_FULL, use_pd=False):
    """One differentiable step of every environment of `sim` (a BatchSim).

    q [n_envs, n_q], qd [n_envs, n_qd], tau [n_envs, n_tau] (or the actions [n_envs, n_act] with use_pd; None = zero): tensors on
    the simulator's device, all float32 or all float64.  The step runs on their fp32 values (the state precision of the product);
    returns (q_next, qd_next), or qdd for MODE_FD, in the inputs' dtype.  float64 inputs keep the gradients of a long rollout in
    fp64; the values are the same.  Gradients / tangents flow to q, qd and tau (see the module docstring for what they are)."""
    if mode == MODE_WORLD or mode not in (0, 1, 2):
        raise ValueError("autograd.step: modes MODE_FD, MODE_NOCONTACT, MODE_FULL (MODE_WORLD is not differentiable here)")
    if getattr(sim, "auto_reset", False):
        raise ValueError("autograd.step: the simulator resets environments on done, which a gradient cannot follow; "
                         "call sim.set_auto_reset(False) first")
    n_in = sim.n_act if use_pd else sim.n_tau
    if use_pd and sim.n_act == 0:
        raise ValueError("autograd.step: use_pd needs BatchSim.set_env")
    dev, dtypes = _device(sim), (torch.float32, torch.float64)
    _check(q, "q", (sim.n_envs, sim.n_q), dtypes, dev)
    _check(qd, "qd", (sim.n_envs, sim.n_qd), (q.dtype,), dev)
    if tau is None:
        tau = torch.zeros((sim.n_envs, n_in), dtype=q.dtype, device=dev)
    _check(tau, "action" if use_pd else "tau", (sim.n_envs, n_in), (q.dtype,), dev)
    return _Step.apply(sim, int(mode), bool(use_pd), q, qd, tau)


def rigid_step(world, state, force=None, steps=1):
    """`steps` differentiable World::step calls of every world of `world` (a RigidWorld): state [n_worlds, n_bodies, 13] and force
    [n_worlds, n_bodies, 3] (None = zero; applied before the first step) float64 tensors on the world's device.  Returns the new
    state (float64).  One dual lane carries the derivative through all `steps`, so memory does not grow with `steps`."""
    if int(steps) < 0:
        raise ValueError("rigid_step: steps >= 0")
    dev = _device(world)
    _check(state, "state", (world.n_worlds, world.n_bodies, 13), (torch.float64,), dev)
    if force is None:
        force = torch.zeros((world.n_worlds, world.n_bodies, 3), dtype=torch.float64, device=dev)
    _check(force, "force", (world.n_worlds, world.n_bodies, 3), (torch.float64,), dev)
    return _RigidStep.apply(world, int(steps), state, force)
