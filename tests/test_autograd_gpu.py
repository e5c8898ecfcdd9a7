"""torch.autograd through the batched steps on the GPU (tds_b200.autograd, tds_b200_step_{jvp,vjp}_device,
tds_b200_rigid_{jvp,vjp}_device): the device products against the dense Jacobians of the same instance, gradients of one step
against central differences of the C oracle, rollouts chained through autograd against chained Jacobians, and the billiard
optimisation of the reference's python/examples through rigid_step."""
import numpy as np
import pytest

import tds_b200
import tds_b200.workloads as wl
from tds_b200.model import fixture_path, load_model
from oracle import port

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
ag = tds_b200.autograd


def rel_err(a, ref):
    return float(np.max(np.abs(a - ref) / np.maximum(1.0, np.abs(ref)))) if ref.size else 0.0


def soa(a, ns, dtype=torch.float64):
    a = np.asarray(a).reshape(a.shape[0], -1)
    t = torch.zeros((max(a.shape[1], 1), ns), dtype=dtype, device="cuda:0")
    t[:a.shape[1], :a.shape[0]] = torch.tensor(a.T, dtype=dtype)
    return t


def aos(t, dim, n):
    return t[:dim, :n].T.cpu().numpy().astype(np.float64)


def check_device_products(sim, mode, q, qd, tau, use_pd=False):
    n, ns = sim.n_envs, sim.n_stride
    n_in = sim.n_act if use_pd else sim.n_tau
    J = sim.step_jacobian_host(mode, q, qd, tau, use_pd=use_pd)[:, :, :sim.n_q + sim.n_qd + n_in]
    rows = J.shape[1]
    r = np.random.default_rng(11)
    dims = (sim.n_q, sim.n_qd, n_in)
    tan = [r.normal(size=(n, d)) for d in dims]
    cot = r.normal(size=(n, rows))
    ins = (soa(q, ns, torch.float32), soa(qd, ns, torch.float32), soa(tau if tau is not None else np.zeros((n, n_in)), ns, torch.float32))
    t_out = torch.full((rows, ns), 7.0, dtype=torch.float64, device="cuda:0")
    sim.step_jvp_device(mode, *ins, *[soa(t, ns) for t in tan], t_out, use_pd=use_pd)
    g = [torch.full((max(d, 1), ns), 7.0, dtype=torch.float64, device="cuda:0") for d in dims]
    sim.step_vjp_device(mode, *ins, soa(cot, ns), *g, use_pd=use_pd)
    torch.cuda.synchronize()
    assert rel_err(aos(t_out, rows, n), np.einsum("erc,ec->er", J, np.concatenate(tan, axis=1))) <= 1e-10
    assert rel_err(np.concatenate([aos(x, d, n) for x, d in zip(g, dims)], axis=1), np.einsum("erc,er->ec", J, cot)) <= 1e-10
    if ns > n:   # padding columns are not written
        assert torch.all(t_out[:, n:] == 7.0) and all(torch.all(x[:, n:] == 7.0) for x in g)
    # actions / tau only: the same numbers as that block of the full product
    g_tau = torch.zeros((max(n_in, 1), ns), dtype=torch.float64, device="cuda:0")
    sim.step_vjp_device(mode, *ins, soa(cot, ns), None, None, g_tau, use_pd=use_pd)
    torch.cuda.synchronize()
    assert torch.equal(g_tau[:n_in, :n], g[2][:n_in, :n])


@pytest.mark.parametrize("name,gen", [("pendulum5", wl.pendulum5), ("cartpole", wl.cartpole), ("sphere2", wl.sphere2), ("box", wl.box),
                                      ("humanoid", wl.humanoid)])
def test_device_products_equal_dense_jacobian_products(name, gen):
    n = 40   # ragged: a second warp with 8 live lanes
    w = gen(n, seed=2718)
    sim = tds_b200.BatchSim(load_model(fixture_path(name)), n, **w["params"])
    tau = w.get("tau")
    tau = None if tau is None or not sim.n_tau else tau[:, -sim.n_tau:]
    check_device_products(sim, w["mode"], w["q"], w["qd"], tau)


def test_device_products_laikago_pd_and_multibody_world():
    w = wl.laikago_perturbed(40, seed=3)
    check_device_products(tds_b200.laikago_sim(40), 2, w["q"], w["qd"], w["action"], use_pd=True)
    w = wl.multibody_world("capsule_sphere", 40, seed=4)
    check_device_products(tds_b200.BatchSim(w["model"], 40, **w["params"]), 2, w["q"], w["qd"], w["tau"])


def test_rigid_device_products_equal_dense_jacobian_products():
    n, steps = 40, 3
    w = wl.rigid_world("billiard", n, seed=5)
    world = tds_b200.RigidWorld(w["bodies"], n, **w["params"])
    _, J = world.step_jacobian(w["state"], w["force"], steps)
    ns, nb = world.n_stride, world.n_bodies
    r = np.random.default_rng(6)
    t_s, t_f, cot = r.normal(size=(n, nb * 13)), r.normal(size=(n, nb * 3)), r.normal(size=(n, nb * 13))
    s, f = soa(w["state"], ns), soa(w["force"], ns)
    t_out = torch.zeros((13 * nb, ns), dtype=torch.float64, device="cuda:0")
    st = torch.cuda.current_stream()
    world.jvp_device(s, f, steps, soa(t_s, ns), soa(t_f, ns), t_out, stream=st)
    g_s, g_f = torch.zeros_like(s), torch.zeros((3 * nb, ns), dtype=torch.float64, device="cuda:0")
    world.vjp_device(s, f, steps, soa(cot, ns), g_s, g_f, stream=st)
    torch.cuda.synchronize()
    assert rel_err(aos(t_out, 13 * nb, n), np.einsum("erc,ec->er", J, np.concatenate([t_s, t_f], axis=1))) <= 1e-10
    g = np.einsum("erc,er->ec", J, cot)
    assert rel_err(aos(g_s, 13 * nb, n), g[:, :13 * nb]) <= 1e-10 and rel_err(aos(g_f, 3 * nb, n), g[:, 13 * nb:]) <= 1e-10


@pytest.mark.parametrize("name,gen", [("pendulum5", wl.pendulum5), ("cartpole", wl.cartpole)])
def test_step_backward_vs_oracle_central_differences(name, gen):
    n = 16
    model = load_model(fixture_path(name))
    w = gen(n, seed=99)
    mode = w["mode"]
    sim = tds_b200.BatchSim(model, n, **w["params"])
    P = port.make_params(**w["params"])
    q, qd, tau = (torch.tensor(x, dtype=torch.float64, device="cuda:0", requires_grad=True) for x in (w["q"], w["qd"], w["tau"]))
    out = ag.step(sim, q, qd, tau, mode=mode)
    out = (out,) if mode == 0 else out
    r = np.random.default_rng(1)
    c = [r.normal(size=tuple(o.shape)) for o in out]
    sum((o * torch.tensor(ci, device="cuda:0")).sum() for o, ci in zip(out, c)).backward()
    grad = np.concatenate([x.grad.cpu().numpy() for x in (q, qd, tau)], axis=1)
    n_q, n_qd = sim.n_q, sim.n_qd
    cc = np.concatenate(c, axis=1)
    for e in range(n):
        def f(x):
            s = port.step(model, P, mode, x[:n_q], x[n_q:n_q + n_qd], x[n_q + n_qd:])
            return s["qdd"] if mode == 0 else np.concatenate([s["q"], s["qd"]])
        x0 = np.concatenate([w["q"][e], w["qd"][e], w["tau"][e]]).astype(np.float64)
        ref = np.zeros(x0.size)
        for j in range(x0.size):
            xp, xm = x0.copy(), x0.copy(); xp[j] += 1e-6; xm[j] -= 1e-6
            ref[j] = cc[e] @ (f(xp) - f(xm)) / 2e-6
        assert rel_err(grad[e], ref) <= 1e-4, (e, grad[e], ref)


def _rollout_case(name, n=8):
    if name == "laikago":
        w = wl.laikago_perturbed(n, seed=21)
        sim = tds_b200.laikago_sim(n, precision=tds_b200.PREC_F64)
        return sim, w["q"], w["qd"], [w["action"] * (0.5 + 0.1 * k) for k in range(10)], True
    w = (wl.pendulum5 if name == "pendulum5" else wl.cartpole)(n, seed=22)
    sim = tds_b200.BatchSim(load_model(fixture_path(name)), n, **w["params"])
    r = np.random.default_rng(23)
    return sim, w["q"], w["qd"], [w["tau"] + 0.1 * r.normal(size=w["tau"].shape) for _ in range(20)], False


@pytest.mark.parametrize("name", ["pendulum5", "cartpole", "laikago"])
def test_rollout_gradient_and_jvp_equal_chained_jacobians(name):
    sim, q0, qd0, taus, use_pd = _rollout_case(name)
    n, n_x = sim.n_envs, sim.n_q + sim.n_qd
    dev = "cuda:0"
    leaves = [torch.tensor(t, dtype=torch.float64, device=dev, requires_grad=True) for t in taus]
    q, qd = torch.tensor(q0, dtype=torch.float64, device=dev), torch.tensor(qd0, dtype=torch.float64, device=dev)
    states = []
    for t in leaves:
        states.append((q.detach().cpu().numpy(), qd.detach().cpu().numpy()))
        q, qd = ag.step(sim, q, qd, t, mode=tds_b200.MODE_FULL, use_pd=use_pd)
    c = np.random.default_rng(24).normal(size=(n, n_x))
    (torch.cat([q, qd], dim=1) * torch.tensor(c, device=dev)).sum().backward()
    # reference: per-step Jacobians at the states the forward pass produced, chained backwards / forwards
    Js = [sim.step_jacobian_host(tds_b200.MODE_FULL, sq, sqd, t, use_pd=use_pd) for (sq, sqd), t in zip(states, taus)]
    lam = c.copy()
    ref = [None] * len(Js)
    for k in range(len(Js) - 1, -1, -1):
        ref[k] = np.einsum("erc,er->ec", Js[k][:, :, n_x:n_x + taus[k].shape[1]], lam)
        lam = np.einsum("erc,er->ec", Js[k][:, :, :n_x], lam)
    for k, t in enumerate(leaves):
        assert rel_err(t.grad.cpu().numpy(), ref[k]) <= 1e-8, k
    r = np.random.default_rng(25)
    v = [r.normal(size=t.shape) for t in taus]

    def roll(*ts):
        a, b = torch.tensor(q0, dtype=torch.float64, device=dev), torch.tensor(qd0, dtype=torch.float64, device=dev)
        for t in ts:
            a, b = ag.step(sim, a, b, t, mode=tds_b200.MODE_FULL, use_pd=use_pd)
        return torch.cat([a, b], dim=1)
    _, tangent = torch.func.jvp(roll, tuple(t.detach() for t in leaves), tuple(torch.tensor(x, device=dev) for x in v))
    D = np.zeros((n, n_x))
    for k, J in enumerate(Js):
        D = np.einsum("erc,ec->er", J[:, :, :n_x], D) + np.einsum("erc,ec->er", J[:, :, n_x:n_x + v[k].shape[1]], v[k])
    assert rel_err(tangent.cpu().numpy(), D) <= 1e-8


def test_rigid_step_gradient_and_billiard_descent():
    w = wl.rigid_world("billiard", 8, seed=31)
    world = tds_b200.RigidWorld(w["bodies"], 8, **w["params"])
    state = torch.tensor(w["state"], device="cuda:0")
    force = torch.tensor(w["force"], device="cuda:0", requires_grad=True)
    out = ag.rigid_step(world, state, force, steps=50)
    g = np.random.default_rng(32).normal(size=tuple(out.shape))
    (out * torch.tensor(g, device="cuda:0")).sum().backward()
    ref_out, J = world.step_jacobian(w["state"], w["force"], steps=50)
    assert rel_err(out.detach().cpu().numpy(), ref_out) <= 1e-10
    nb = world.n_bodies
    assert rel_err(force.grad.cpu().numpy().reshape(8, -1), np.einsum("erc,er->ec", J, g.reshape(8, -1))[:, 13 * nb:]) <= 1e-10
    # the billiard optimisation: push the cue ball so that the ball it hits ends closer to a goal point
    import tds_b200.rigid as rg
    n = 4
    world = tds_b200.RigidWorld([rg.sphere(1.0, 0.5), rg.sphere(1.0, 0.5)], n, gravity=(0.0, 0.0, 0.0), num_solver_iterations=50)
    s = rg.identity_state(n, 2)
    s[:, 1, 0] = 1.6
    s[:, 1, 1] = np.linspace(0.1, 0.3, n)
    state = torch.tensor(s, device="cuda:0")
    f = np.zeros((n, 2, 3))
    f[:, 0, 0] = 150.0
    force = torch.tensor(f, device="cuda:0", requires_grad=True)
    goal = torch.tensor([3.0, 0.6, 0.0], dtype=torch.float64, device="cuda:0")
    dist = []
    for _ in range(5):
        d = ((ag.rigid_step(world, state, force, steps=50)[:, 1, 0:3] - goal) ** 2).sum(dim=1)
        dist.append(d.detach().sqrt().cpu().numpy())
        force.grad = None
        d.sum().backward()
        with torch.no_grad():
            force -= 2.0 * force.grad
    assert all(np.all(b < a) for a, b in zip(dist, dist[1:])), dist


def test_refusals():
    n = 4
    w = wl.pendulum5(n)
    sim = tds_b200.BatchSim(load_model(fixture_path("pendulum5")), n)
    q, qd, tau = (torch.tensor(x, dtype=torch.float32, device="cuda:0") for x in (w["q"], w["qd"], w["tau"]))
    with pytest.raises(ValueError, match="MODE_WORLD"):
        ag.step(sim, q, qd, tau, mode=tds_b200.MODE_WORLD)
    with pytest.raises(ValueError, match="shape"):
        ag.step(sim, q[:, :3], qd, tau)
    with pytest.raises(TypeError, match="dtype"):
        ag.step(sim, q, qd.double(), tau)
    with pytest.raises(TypeError, match="dtype"):
        ag.step(sim, q.half(), qd.half(), tau.half())
    with pytest.raises(ValueError, match="cuda:0"):
        ag.step(sim, q.cpu(), qd.cpu(), tau.cpu())
    with pytest.raises(ValueError, match="set_env"):
        ag.step(sim, q, qd, None, use_pd=True)
    lk = tds_b200.laikago_sim(n, auto_reset=True)
    wl_ = wl.laikago(n)
    with pytest.raises(ValueError, match="reset"):
        ag.step(lk, *(torch.tensor(x, device="cuda:0") for x in (wl_["q"], wl_["qd"], wl_["action"])), use_pd=True)
    # the C-ABI refusals behind the low-level wrappers
    ns = sim.n_stride
    ins = (soa(w["q"], ns, torch.float32), soa(w["qd"], ns, torch.float32), soa(w["tau"], ns, torch.float32))
    g_out = torch.zeros((10, ns), dtype=torch.float64, device="cuda:0")
    with pytest.raises(RuntimeError, match="rc=-2"):
        sim.step_vjp_device(tds_b200.MODE_WORLD, *ins, g_out, g_q=torch.zeros_like(g_out))
    with pytest.raises(RuntimeError, match="rc=-3"):
        sim.step_jvp_device(tds_b200.MODE_FULL, *ins, None, None, None, g_out, use_pd=True)
    with pytest.raises(RuntimeError, match="rc=-1"):
        sim.step_jvp_device(tds_b200.MODE_FULL, *ins, None, None, None, None)
    world = tds_b200.RigidWorld(wl.rigid_world("billiard", n)["bodies"], n)
    with pytest.raises(TypeError, match="dtype"):
        ag.rigid_step(world, torch.zeros((n, 7, 13), dtype=torch.float32, device="cuda:0"))
    with pytest.raises(ValueError, match="shape"):
        ag.rigid_step(world, torch.zeros((n, 6, 13), dtype=torch.float64, device="cuda:0"))
    with pytest.raises(RuntimeError, match="rc=-1"):
        world.vjp_device(None, None, 1, None)
