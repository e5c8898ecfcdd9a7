#!/usr/bin/env python
"""Cost of the derivative products behind tds_b200.autograd next to the forward step they differentiate.

    python scripts/bench_autograd.py [--n 4096] [--reps 20]

For pendulum5 (forward dynamics), Laikago with PD (full step) and the rigid billiard world (steps 1 and 50), all with --n
environments: the forward step (step_device: the production kernel), one JVP (one dual lane per environment), one VJP for every
input block, and one VJP for the torques / actions / forces only.  Every timed call is preceded by writing a 256 MB buffer,
which evicts the 126 MB L2, and is timed alone with CUDA events after three warm-up calls; the median and the spread of --reps
calls are printed.  The first lines give the device name and its power limit.
"""
import argparse
import json
import os
import subprocess
import sys

sys.dont_write_bytecode = True
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np
import torch

import tds_b200
import tds_b200.workloads as wl
from tds_b200.model import fixture_path, load_model


def soa(a, ns, dtype):
    a = np.asarray(a).reshape(a.shape[0], -1)
    t = torch.zeros((max(a.shape[1], 1), ns), dtype=dtype, device="cuda:0")
    t[:a.shape[1], :a.shape[0]] = torch.tensor(a.T, dtype=dtype)
    return t


def timed(fn, reps, flush):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    return dict(median_ms=round(float(np.median(ms)), 4), min_ms=round(float(np.min(ms)), 4), max_ms=round(float(np.max(ms)), 4))


def multibody(name, n, reps, flush):
    if name == "laikago_pd":
        w = wl.laikago_perturbed(n, seed=1)
        sim, mode, use_pd, tau = tds_b200.laikago_sim(n), tds_b200.MODE_FULL, True, w["action"]
    else:
        w = wl.pendulum5(n, seed=1)
        sim, mode, use_pd, tau = tds_b200.BatchSim(load_model(fixture_path("pendulum5")), n), w["mode"], False, w["tau"]
    ns = sim.n_stride
    n_in = sim.n_act if use_pd else sim.n_tau
    rows = sim.n_qd if mode == tds_b200.MODE_FD else sim.n_q + sim.n_qd
    q, qd, t = soa(w["q"], ns, torch.float32), soa(w["qd"], ns, torch.float32), soa(tau, ns, torch.float32)
    q_o, qd_o, qdd_o = sim.alloc(sim.n_q), sim.alloc(sim.n_qd), sim.alloc(sim.n_qd)
    r = np.random.default_rng(2)
    tan = [soa(r.normal(size=(n, d)), ns, torch.float64) for d in (sim.n_q, sim.n_qd, n_in)]
    t_out = torch.zeros((rows, ns), dtype=torch.float64, device="cuda:0")
    cot = soa(r.normal(size=(n, rows)), ns, torch.float64)
    g = [torch.zeros((max(d, 1), ns), dtype=torch.float64, device="cuda:0") for d in (sim.n_q, sim.n_qd, n_in)]
    res = dict(case=name, n=n, mode=mode, use_pd=use_pd, dual_lanes_per_env_vjp_all=sim.n_q + sim.n_qd + n_in, dual_lanes_per_env_vjp_tau=n_in)
    res["forward"] = timed(lambda: sim.step_device(mode, q, qd, t, q_out=q_o, qd_out=qd_o, qdd_out=qdd_o, use_pd=use_pd), reps, flush)
    res["forward_kernel"] = sim.kernel_name()
    res["jvp"] = timed(lambda: sim.step_jvp_device(mode, q, qd, t, *tan, t_out, use_pd=use_pd), reps, flush)
    res["vjp_all"] = timed(lambda: sim.step_vjp_device(mode, q, qd, t, cot, *g, use_pd=use_pd), reps, flush)
    res["vjp_tau_only"] = timed(lambda: sim.step_vjp_device(mode, q, qd, t, cot, None, None, g[2], use_pd=use_pd), reps, flush)
    return res


def rigid(n, steps, reps, flush):
    w = wl.rigid_world("billiard", n, seed=3)
    world = tds_b200.RigidWorld(w["bodies"], n, **w["params"])
    ns, nb = world.n_stride, world.n_bodies
    s, f = soa(w["state"], ns, torch.float64), soa(w["force"], ns, torch.float64)
    out = torch.zeros_like(s)
    r = np.random.default_rng(4)
    t_s, t_f = soa(r.normal(size=(n, 13 * nb)), ns, torch.float64), soa(r.normal(size=(n, 3 * nb)), ns, torch.float64)
    cot = soa(r.normal(size=(n, 13 * nb)), ns, torch.float64)
    g_s, g_f = torch.zeros_like(s), torch.zeros((3 * nb, ns), dtype=torch.float64, device="cuda:0")
    st = torch.cuda.current_stream()
    res = dict(case="rigid_billiard", n=n, steps=steps, dual_lanes_per_world_vjp_all=16 * nb, dual_lanes_per_world_vjp_force=3 * nb)
    res["forward"] = timed(lambda: world.step_device(s, out, f, steps, stream=st), reps, flush)
    res["jvp"] = timed(lambda: world.jvp_device(s, f, steps, t_s, t_f, out, stream=st), reps, flush)
    res["vjp_all"] = timed(lambda: world.vjp_device(s, f, steps, cot, g_s, g_f, stream=st), reps, flush)
    res["vjp_force_only"] = timed(lambda: world.vjp_device(s, f, steps, cot, None, g_f, stream=st), reps, flush)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    print(json.dumps(dict(device=torch.cuda.get_device_name(0), nvidia_smi=smi.stdout.strip().splitlines()[:1],
                          l2="flushed before every timed call (256 MB write)")), flush=True)
    flush = torch.empty(64 << 20, dtype=torch.float32, device="cuda:0")
    for name in ("pendulum5", "laikago_pd"):
        print(json.dumps(multibody(name, a.n, a.reps, flush)), flush=True)
    for steps in (1, 50):
        print(json.dumps(rigid(a.n, steps, a.reps, flush)), flush=True)


if __name__ == "__main__":
    main()
