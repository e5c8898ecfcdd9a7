"""bench.py contract checks: the reference arm (the reference's own CPU implementation of the path, oracle/_ref) prints
exactly ONE JSON line on stdout with the keys the driver reads; --dump-outputs writes what the last timed step returned,
the same arrays from run to run (GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.skipif(not ref.available(), reason="oracle/_ref/libtds_ref.so not built (needs /root/reference)")
def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "2",
                        "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout[:500]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 3   # both arms clamp the warm-up to >= 3 (timing rules)
    assert d["metric"].startswith("env-steps/sec") and d["unit"] == "env-steps/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"] and d["config"]["host"]["usable_cores"] >= d["cpu_baseline"]["cores"]
    assert d["cpu_baseline_codegen"]["value"] > 0 and set(d["config"]["threads_sweep_templated"]) >= {"1"}


@pytest.mark.skipif(not ref.available(), reason="oracle/_ref/libtds_ref.so not built (needs /root/reference)")
@pytest.mark.parametrize("config", ["cartpole64", "pendulum5_fd", "sphere2_16384", "humanoid4096"])
def test_reference_arm_of_every_config(config):
    """bench.py --impl reference --config <c>: one JSON line per BASELINE configuration, bounded sample, same keys."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", config, "--steps", "2",
                        "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["value"] > 0 and d["cpu_baseline"]["cores"] == 1 and d["e2e"]["value"] == d["value"]
    assert "BASELINE.json configs" in d["config"]["workload"]


def _bench(*args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--no-cpu-baseline", "--min-seconds", "0"]
                       + list(args), capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout[:500]
    return json.loads(lines[0])


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def _flagship_rollout(K, W, graph):
    """The env steps bench.py runs for the Laikago workload with --min-seconds 0, launched one by one: 10 settle steps, W
    warm-up steps, then with a CUDA graph one step outside the capture and four replays of the K captured steps (one after
    the capture, the 2 // 2 before the timed one, the timed one); without, the K timed steps.  Returns the state before
    and after the last step, and that step's reward and done."""
    import torch
    import tds_b200
    import tds_b200.workloads as wl
    n, ring = 4096, 768
    sim = tds_b200.laikago_sim(n, device=0, precision=0, auto_reset=True)
    w = wl.laikago(n, seed=wl.SEED)
    sim.env_set_state(w["q"], w["qd"])
    ns = sim.n_stride
    g = torch.Generator(device="cpu").manual_seed(1234)
    actions = (torch.rand((ring, 12, ns), generator=g) * 0.8 - 0.4).cuda()
    reward, done = torch.zeros(ns, device="cuda"), torch.zeros(ns, device="cuda")
    zero = torch.zeros((12, ns), device="cuda")
    for _ in range(10):
        sim.env_step_device(zero, reward, done)
    timed = list(range(W + 1, W + 1 + K))
    order = list(range(W)) + ([W] + timed * 3 if graph else timed)
    for i in order[:-1]:
        sim.env_step_device(actions[i % ring], reward, done)
    before = sim.env_get_state()
    sim.env_step_device(actions[order[-1] % ring], reward, done)
    q, qd = sim.env_get_state()
    out = {"q": q, "qd": qd, "reward": reward[:n].cpu().numpy(), "done": done[:n].cpu().numpy()}
    sim.close()
    return before, out


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [True, False])
def test_dump_outputs_are_the_last_timed_step(graph, tmp_path):
    """--dump-outputs writes what the env step returned in the last of exactly --steps timed steps: bit for bit the state,
    reward and done of the same steps launched one by one, and not the state one step earlier."""
    K, W = 3, 4
    d = _bench("--steps", str(K), "--warmup", str(W), "--dump-outputs", str(tmp_path), *([] if graph else ["--no-graph"]))
    assert d["steps"] == K and d["warmup"] == W
    out = _load(tmp_path)
    assert set(out) == {"q", "qd", "reward", "done"}
    assert out["q"].shape == (4096, 18) and out["qd"].shape == (4096, 18) and out["reward"].shape == (4096,)
    assert out["q"].dtype == np.float64 and out["reward"].dtype == np.float32 and out["done"].dtype == np.float32
    before, expect = _flagship_rollout(K, W, graph)
    for k, v in out.items():
        assert np.all(np.isfinite(v)), k
        assert np.array_equal(v, expect[k]), (k, np.abs(v - expect[k]).max())
    assert not np.array_equal(out["qd"], before[1])


@pytest.mark.gpu
@pytest.mark.parametrize("config,names", [("pendulum5_fd", {"qdd"}),
                                          ("sphere2_16384", {"q", "qd", "contact_dist", "contact_count", "contact_links"})])
def test_dump_outputs_of_a_config(config, names, tmp_path):
    d = _bench("--config", config, "--envs", "256", "--steps", "2", "--warmup", "1", "--dump-outputs", str(tmp_path))
    assert d["steps"] == 2
    out = _load(tmp_path)
    assert set(out) == names
    for k, v in out.items():
        assert v.shape[0] == 256 and v.dtype in (np.float32, np.float64) and np.all(np.isfinite(v)), k


def test_dump_outputs_needs_the_b200_arm(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert r.returncode == 2 and "--dump-outputs needs --impl b200" in r.stderr
