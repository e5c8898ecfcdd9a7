"""Jacobian-vector and vector-Jacobian products of the dual-number step kernels (the path behind tds_b200.autograd), executed on
the CPU by the host-compiled kernel sources (tests/cpp/stepw_dual_host.cpp, tests/cpp/rigid_dual_host.cpp): J v and g^T J must equal
the products with the dense Jacobian the same instance computes on the same inputs (tests/cpp/stepw_host.cpp, rigid_host.cpp).  The arithmetic of every lane is the same; only
the order of the final summation differs, hence the 1e-10 bar."""
import os

import numpy as np
import pytest

import tds_b200.workloads as wl
from tds_b200.envs import ANT_INITIAL_POSES, ANT_KD, ANT_KP, ANT_MAX_FORCE, LAIKAGO_INITIAL_POSES, LAIKAGO_KD, LAIKAGO_KP, LAIKAGO_MAX_FORCE
from tds_b200.model import fixture_path, load_model
import emu
import emu_dual

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CONFIGS = ["cartpole", "pendulum5", "sphere2", "laikago", "humanoid", "ant", "box", "cartpole_plane", "pendulum5spherical", "humanoid_spherical"]
TOL = 1e-10
LAIKAGO_ENV = [12, 6, LAIKAGO_KP, LAIKAGO_KD, LAIKAGO_MAX_FORCE, 0.4, *LAIKAGO_INITIAL_POSES]
ANT_ENV = [8, 6, ANT_KP, ANT_KD, ANT_MAX_FORCE, 0.4, *ANT_INITIAL_POSES]


def rel_err(a, ref):
    return float(np.max(np.abs(a - ref) / np.maximum(1.0, np.abs(ref)))) if ref.size else 0.0


def golden_inputs(name, n=8):
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    model = load_model(fixture_path(name))
    n_tau = int(model[4]) - (6 if int(model[2]) else 0)
    tau = g["tau"][:n, -n_tau:] if "tau" in g.files else np.zeros((n, n_tau))
    params = {}
    for k in g.files:
        if k.startswith("param_"):
            v = g[k]
            params[k[6:]] = tuple(v.tolist()) if v.ndim else (bool(v) if k == "param_keep_all_points" else float(v))
    return model, int(g["mode"]), g["q_in"][:n], g["qd_in"][:n], tau, params


def check_products(model, mode, q, qd, tau, use_pd=False, env=None, seed=0, **params):
    """JVP and VJP against the dense Jacobian (without its PD-gain columns) of the same instance on the same inputs."""
    n, n_q, n_qd = q.shape[0], int(model[3]), int(model[4])
    n_in = int(env[0]) if use_pd else n_qd - (6 if int(model[2]) else 0)
    J = emu.step(model, mode, q, qd, tau, use_pd=use_pd, env=env, jacobian=True, **params)["jac"][:, :, :n_q + n_qd + n_in]
    rows = J.shape[1]
    r = np.random.default_rng(seed)
    tangents = (r.normal(size=(n, n_q)), r.normal(size=(n, n_qd)), r.normal(size=(n, n_in)))
    cot = r.normal(size=(n, rows))
    out = emu_dual.step_dual(model, mode, q, qd, tau, use_pd=use_pd, env=env, tangents=tangents, cotangent=cot, **params)
    assert out["jvp"].shape == (n, rows)
    assert rel_err(out["jvp"], np.einsum("erc,ec->er", J, np.concatenate(tangents, axis=1))) <= TOL
    assert rel_err(np.concatenate(out["vjp"], axis=1), np.einsum("erc,er->ec", J, cot)) <= TOL
    return J, out


@pytest.mark.parametrize("name", CONFIGS)
def test_fixture_products_equal_dense_jacobian_products(name):
    model, mode, q, qd, tau, params = golden_inputs(name)
    check_products(model, mode, q, qd, tau, seed=1, **params)


@pytest.mark.parametrize("name,gen,env", [("laikago", wl.laikago_perturbed, LAIKAGO_ENV), ("ant", wl.ant_perturbed, ANT_ENV)])
def test_pd_products_equal_dense_jacobian_products(name, gen, env):
    w = gen(6, seed=31)
    check_products(load_model(fixture_path(name)), 2, w["q"], w["qd"], w["action"], use_pd=True, env=env, seed=2, **w["params"])


@pytest.mark.parametrize("kind", wl.MULTIBODY_WORLDS)
def test_multibody_world_products_equal_dense_jacobian_products(kind):
    w = wl.multibody_world(kind, 6, seed=41)
    check_products(w["model"], 2, w["q"], w["qd"], w["tau"], seed=3, **w["params"])


def test_spring_damper_products_equal_dense_jacobian_products():
    model, _, q, qd, tau, params = golden_inputs("sphere2")
    law = dict(contact_model=1, spring_k=40000.0, damper_d=3000.0, exponent_n=1.5, v_transition=0.02, hard_contact_condition=True)
    check_products(model, 2, q, qd, tau, seed=4, **law, **params)


@pytest.mark.parametrize("mode", [0, 2])
def test_ragged_batch(mode):
    """33 environments: a second warp with one live lane; every environment must still be right."""
    w = wl.cartpole(33, seed=5)
    check_products(load_model(fixture_path("cartpole")), mode, w["q"], w["qd"], w["tau"], seed=5, **w["params"])


@pytest.mark.parametrize("mode", [0, 2])
def test_partial_vjp_and_null_tangents(mode):
    """A VJP that asks for the actions only launches the action directions and returns the action block of the full VJP bit for
    bit; a null tangent block is a zero tangent."""
    w = wl.laikago_perturbed(4, seed=6)
    model = load_model(fixture_path("laikago"))
    rows = 18 if mode == 0 else 36
    r = np.random.default_rng(6)
    cot = r.normal(size=(4, rows))
    full = emu_dual.step_dual(model, mode, w["q"], w["qd"], w["action"], use_pd=True, env=LAIKAGO_ENV, cotangent=cot, **w["params"])["vjp"]
    part = emu_dual.step_dual(model, mode, w["q"], w["qd"], w["action"], use_pd=True, env=LAIKAGO_ENV, cotangent=cot,
                              want=(False, False, True), **w["params"])["vjp"]
    assert part[0] is None and part[1] is None
    assert np.array_equal(part[2], full[2])
    t_qd = r.normal(size=(4, 18))
    a = emu_dual.step_dual(model, mode, w["q"], w["qd"], w["action"], use_pd=True, env=LAIKAGO_ENV, tangents=(None, t_qd, None), **w["params"])
    b = emu_dual.step_dual(model, mode, w["q"], w["qd"], w["action"], use_pd=True, env=LAIKAGO_ENV,
                           tangents=(np.zeros((4, 18)), t_qd, np.zeros((4, 12))), **w["params"])
    assert np.array_equal(a["jvp"], b["jvp"])


@pytest.mark.parametrize("kind", wl.RIGID_WORLDS)
@pytest.mark.parametrize("steps", [1, 5])
def test_rigid_products_equal_dense_jacobian_products(kind, steps):
    n = 4
    w = wl.rigid_world(kind, n, seed=7)
    nb = w["bodies"].shape[0]
    _, J = emu.rigid_step(w["bodies"], w["state"], w["force"], steps, jacobian=True, **w["params"])
    r = np.random.default_rng(8)
    t_s, t_f, cot = r.normal(size=(n, nb, 13)), r.normal(size=(n, nb, 3)), r.normal(size=(n, nb, 13))
    out = emu_dual.rigid_dual(w["bodies"], w["state"], w["force"], steps, tangents=(t_s, t_f), cotangent=cot, **w["params"])
    v = np.concatenate([t_s.reshape(n, -1), t_f.reshape(n, -1)], axis=1)
    assert rel_err(out["jvp"].reshape(n, -1), np.einsum("erc,ec->er", J, v)) <= TOL
    g = np.einsum("erc,er->ec", J, cot.reshape(n, -1))
    assert rel_err(out["vjp"][0].reshape(n, -1), g[:, :13 * nb]) <= TOL
    assert rel_err(out["vjp"][1].reshape(n, -1), g[:, 13 * nb:]) <= TOL
    only_f = emu_dual.rigid_dual(w["bodies"], w["state"], w["force"], steps, cotangent=cot, want=(False, True), **w["params"])["vjp"]
    assert only_f[0] is None and np.array_equal(only_f[1], out["vjp"][1])


def test_rigid_null_force_is_zero_force():
    w = wl.rigid_world("stack", 3, seed=9)
    nb = w["bodies"].shape[0]
    r = np.random.default_rng(9)
    cot = r.normal(size=(3, nb, 13))
    a = emu_dual.rigid_dual(w["bodies"], w["state"], None, 2, tangents=(None, r.normal(size=(3, nb, 3))), cotangent=cot, **w["params"])
    b = emu_dual.rigid_dual(w["bodies"], w["state"], np.zeros((3, nb, 3)), 2, tangents=(None, None), cotangent=cot, **w["params"])
    _, J = emu.rigid_step(w["bodies"], w["state"], np.zeros((3, nb, 3)), 2, jacobian=True, **w["params"])
    assert rel_err(b["vjp"][1].reshape(3, -1), np.einsum("erc,er->ec", J, cot.reshape(3, -1))[:, 13 * nb:]) <= TOL
    assert np.array_equal(a["vjp"][1], b["vjp"][1])
    assert not np.any(b["jvp"])
