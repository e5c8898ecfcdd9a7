#!/usr/bin/env python
"""Headline benchmark: env-steps/sec of the batched Laikago-on-plane step (BASELINE.json configs[3]:
"laikago on plane, 4096 envs, full step + PD actuators") on N B200s of one node.

    python bench.py --gpus 1 --steps 200 --warmup 20
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference's own CPU path on the host cores
    python bench.py --gpus 1 --steps 200 --warmup 20 --dump-outputs DIR   # + what the last timed step computed

One "step" = one env-step of every environment (PD -> ABA -> integrate -> collide -> LCP/PGS ->
integrate).  Environments are sharded across ranks (4096 per GPU: weak scaling), there is no
data-path collective.  Rank 0 prints ONE JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

# the benchmark writes nothing into the tree it runs from, writable or not: without this, the first import of a module
# (tds_b200.parallel, oracle.ref, ...) leaves a __pycache__ directory beside its source
sys.dont_write_bytecode = True

# stdout carries exactly ONE JSON line: everything else that libraries print there (NCCL's version banner, the
# reference's "Loading URDF" chatter) is sent to stderr by pointing fd 1 at fd 2; the result goes to the saved fd.
_JSON_FD = os.dup(1)
os.dup2(2, 1)


def emit(line):
    os.write(_JSON_FD, (json.dumps(line) + "\n").encode())


ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ENVS_PER_GPU = 4096
ALGO_BYTES_PER_ENV_STEP = 344       # SURVEY.md section 8d: q18+qd18+action12 read, q18+qd18+reward+done written (fp32)
FLOPS_PER_ENV_STEP = 27e3           # op count of the reference's CppAD tape (SURVEY.md section 8d)
METRIC = "env-steps/sec (N parallel sims)"
DUMP_LIMIT_BYTES = 64_000_000


def dump_outputs(dirname, arrays):
    """--dump-outputs: writes each array (one row per environment) as <dirname>/<name>.npy, float32 or float64 (integer
    outputs as float64), so that two builds run with the same arguments can be compared output for output.  Above
    DUMP_LIMIT_BYTES in all, the same fixed, seeded sample of environments is kept from every array; env_index.npy then
    lists which."""
    arrays = {k: np.asarray(v) for k, v in arrays.items()}
    arrays = {k: v if v.dtype in (np.float32, np.float64) else v.astype(np.float64) for k, v in arrays.items()}
    n = next(iter(arrays.values())).shape[0]
    row_bytes = sum(v.nbytes for v in arrays.values()) // n
    budget = DUMP_LIMIT_BYTES - 4096 * (len(arrays) + 1)   # room for the .npy headers
    if n * row_bytes > budget:
        keep = budget // (row_bytes + 8)
        idx = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        arrays = {k: v[idx] for k, v in arrays.items()}
        arrays["env_index"] = idx.astype(np.float64)
    os.makedirs(dirname, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(dirname, k + ".npy"), np.ascontiguousarray(v))


def _measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json, burst copy bandwidth)"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons during the timed region: through NVML (sub-millisecond per sample, so that a
    15 ms timed region still yields a handful of samples), falling back to polling nvidia-smi."""

    _NVML_REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        self.source = "nvidia-smi"
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._handle = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._handle, pynvml.NVML_CLOCK_SM))
            pynvml.nvmlDeviceGetClockInfo(self._handle, pynvml.NVML_CLOCK_SM)
            self._nvml = pynvml
            self.source = "nvml"
        except Exception:
            self._nvml = None

    def _sample_nvml(self):
        n = self._nvml
        self.samples.append(float(n.nvmlDeviceGetClockInfo(self._handle, n.NVML_CLOCK_SM)))
        try:
            get = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
            mask = int(get(self._handle))
            for bit, nm in self._NVML_REASONS.items():
                if mask & bit:
                    self.reasons.add(nm)
        except Exception:
            pass

    def _sample_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={q}",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
        f = [x.strip() for x in out.strip().split(",")]
        self.samples.append(float(f[0]))
        self.max_mhz = float(f[1])
        for nm, v in zip(names, f[2:6]):
            if v.lower().startswith("active"):
                self.reasons.add(nm)

    def run(self):
        while not self._halt.is_set():
            try:
                if self._nvml is not None:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                if self._nvml is not None:   # NVML stopped answering: fall back for the rest of the run
                    self._nvml = None
                    self.source = "nvidia-smi"
            self._halt.wait(0.001 if self._nvml is not None else 0.1)

    def stop(self):
        self._halt.set()
        self.join(timeout=5)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s), "source": self.source}


WORKLOAD = "laikago on plane, 4096 envs/GPU, full step + PD actuators (BASELINE.json configs[3])"


def host_cores():
    """Cores this process may actually use: min(affinity mask, cgroup CPU quota).  os.cpu_count() reports the
    machine, not the lease (round 1: 128 'cores' printed, CFS-throttled to far fewer)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:        # cgroup v2: "<quota|max> <period>"
            q, p = f.read().split()[:2]
            if q != "max":
                quota = float(q) / float(p)
    except Exception:
        try:                                             # cgroup v1
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:
                q = float(f.read())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                p = float(f.read())
            if q > 0:
                quota = q / p
        except Exception:
            pass
    if quota is not None:
        n = max(1, min(n, int(quota + 0.5)))
    return n


def _laikago_inputs(envs, seed=12345):
    import tds_b200.workloads as wl
    w = wl.laikago(envs, seed=seed)
    x = np.zeros((envs, 51))
    x[:, :18], x[:, 18:36], x[:, 36:48], x[:, 48:] = w["q"], w["qd"], w["action"], [100.0, 2.0, 50.0]
    return x


def cpu_reference_rate(seconds=3.0, envs=ENVS_PER_GPU, impl=0, threads=1, x0=None):
    """env-steps/s of the reference's own CPU implementation (oracle/_ref, compiled in place from
    /root/reference by oracle/build_ref.sh): LocomotionContactSimulation::step_forward_original
    (impl 0, one instance per thread) or its codegen kernel (impl 1), on `threads` host threads."""
    from oracle import ref
    L = ref.LaikagoRef(threads)
    x = (_laikago_inputs(envs) if x0 is None else x0).copy()
    out = np.zeros((envs, L.output_dim))
    L.step(x, impl, out)  # warm-up
    n_batches, t0 = 0, time.perf_counter()
    best = 0.0
    while True:
        t1 = time.perf_counter()
        L.step(x, impl, out)
        best = max(best, envs / (time.perf_counter() - t1))
        x[:, :36] = out[:, :36]
        n_batches += 1
        el = time.perf_counter() - t0
        if el >= seconds and n_batches >= 2:
            break
    L.close()
    return envs * n_batches / el, best, f"{n_batches} batches of {envs} env-steps in {el:.1f} s on {threads} threads"


def cpu_reference_sweep(impl, budget_s, envs=ENVS_PER_GPU):
    """The reference's CPU path at {1, 1/4, 1/2, all} of the usable cores; returns (best mean rate, threads, sample, table).
    Oversubscribed OpenMP teams are CFS-throttled and contend in malloc (the templated path heap-allocates per
    temporary), so 'all cores' is not always the fastest: the best figure is the honest baseline."""
    cores = host_cores()
    cands = sorted({1, max(1, cores // 4), max(1, cores // 2), cores})
    x0 = _laikago_inputs(envs)
    table, best = {}, (0.0, 1, "")
    for t in cands:
        e = envs if t > 1 else min(envs, 512)
        v, _, sample = cpu_reference_rate(seconds=budget_s / len(cands), envs=e, impl=impl, threads=t, x0=x0[:e])
        table[str(t)] = v
        if v > best[0]:
            best = (v, t, sample)
    return best[0], best[1], best[2], table


def run_reference_arm(args, rank, world):
    """--impl reference: the reference's CPU path for the same metric/config, rank 0 only."""
    if rank != 0:
        return
    envs = args.envs
    from oracle import ref
    K, W = args.steps, max(args.warmup, 3)
    # thread count: the best of the sweep for the templated World::step path (the baseline BASELINE.json names)
    v_t, threads, sample_t, table_t = cpu_reference_sweep(0, 8.0, envs)
    v_c, threads_c, sample_c, table_c = cpu_reference_sweep(1, 4.0, envs)
    # a step of this arm = one batch of `sample` env-steps, sized so that K + W steps end within ~2 minutes
    sample = int(min(envs, max(64, v_t * 120.0 / (K + W))))
    L = ref.LaikagoRef(threads)
    x = _laikago_inputs(envs)
    out = np.zeros((envs, L.output_dim))
    for _ in range(W):
        L.step(x[:sample], 0, out[:sample])
        x[:sample, :36] = out[:sample, :36]
    t0 = time.perf_counter()
    for _ in range(K):
        L.step(x[:sample], 0, out[:sample])
        x[:sample, :36] = out[:sample, :36]
    el = time.perf_counter() - t0
    val = sample * K / el
    line = {"metric": METRIC, "value": val, "unit": "env-steps/s", "impl": "reference", "n_gpus": args.gpus,
            "steps": K, "warmup": W, "ms_per_step": 1e3 * el / K, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "envs_per_gpu": envs,
                       "envs_per_step": sample, "path": "LocomotionContactSimulation::step_forward_original (templated CPU path, "
                       "World::step), one instance per OpenMP thread",
                       "threads_sweep_templated": table_t, "threads_sweep_codegen": table_c,
                       "host": {"usable_cores": host_cores(), "os_cpu_count": os.cpu_count()}},
            "cpu_baseline": {"value": val, "unit": "env-steps/s", "cores": threads, "kind": "reference",
                             "sample": f"{K} steps x {sample} envs on {threads} threads (best of the thread sweep)"},
            "cpu_baseline_codegen": {"value": v_c, "unit": "env-steps/s", "cores": threads_c, "kind": "reference", "sample": sample_c,
                                     "path": "omp_model_laikago_forward_zero_kernel (the reference's fastest CPU path, "
                                             "examples/ars/ars_vectorized_environment.h:110-137)"},
            "e2e": {"value": val, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# ---- the other BASELINE.json configurations (the headline one, laikago4096, is main() below) --------------------------
# bytes = SURVEY.md section 8d, ALGORITHMIC bytes per env-step (fp32 state in, fp32 state out)
CONFIGS = {
    "laikago4096": dict(envs=4096, bytes=344, model="laikago", workload=WORKLOAD),
    "cartpole64": dict(envs=64, bytes=36, model="cartpole", gen="cartpole",
                       workload="cartpole.urdf, 64 parallel envs, no contacts: FD -> integrate_euler (BASELINE.json configs[0])"),
    "pendulum5_fd": dict(envs=4096, bytes=80, model="pendulum5", gen="pendulum5",
                         workload="pendulum5.urdf, 4096 envs, forward_dynamics only (BASELINE.json configs[1])"),
    "sphere2_16384": dict(envs=16384, bytes=124, model="sphere2", gen="sphere2",
                          workload="sphere2.urdf on plane_implicit, 16384 envs, contact LCP solve + contact record (BASELINE.json configs[2])"),
    "humanoid4096": dict(envs=4096, bytes=532, model="humanoid", gen="humanoid",
                         workload="humanoid.urdf on plane, 4096 envs/GPU (32768 on 8 GPUs), full step, LCP contacts (BASELINE.json configs[4])"),
    "humanoid4096_spring": dict(envs=4096, bytes=532, model="humanoid", gen="humanoid", spring=True,
                                workload="humanoid.urdf on plane, 4096 envs/GPU (32768 on 8 GPUs), full step, spring-damper contacts "
                                         "(BASELINE.json configs[4]; law of DESIGN.md, parity unpinned: no reference source)"),
}


def _config_reference_rate(name, w, model, seconds):
    """The reference's own CPU implementation of the same pipeline (oracle/_ref: forward_dynamics / World::step, templated
    path), one host thread, batches stepped inside one foreign call."""
    from oracle import ref
    sim = ref.RefSim.from_model(model)
    sim.set_params(**w["params"])
    n, mode = w["q"].shape[0], w["mode"]
    tau = w.get("tau")
    full = None
    if tau is not None:
        full = np.zeros((n, sim.n_tau)); full[:, -tau.shape[1]:] = tau
    b = min(n, 256)
    sim.step_batch(mode, w["q"][:b], w["qd"][:b], None if full is None else full[:b])
    k, t0 = 0, time.perf_counter()
    while True:
        sim.step_batch(mode, w["q"][:b], w["qd"][:b], None if full is None else full[:b])
        k += b
        if time.perf_counter() - t0 >= seconds:
            break
    el = time.perf_counter() - t0
    return k / el, f"{k} env-steps in {el:.1f} s on 1 thread"


def run_config(args, rank, world, local_rank):
    """cartpole64 / pendulum5_fd / sphere2_16384 / humanoid4096: same metric, same JSON contract, through the generic
    device entry point tds_b200_step_device (value) and the host-buffer entry point tds_b200_step_host (e2e)."""
    C = CONFIGS[args.config]
    import tds_b200
    import tds_b200.workloads as wl
    from tds_b200.model import fixture_path, load_model
    n, K, W = args.envs, args.steps, max(args.warmup, 3)
    model = load_model(fixture_path(C["model"]))
    w = getattr(wl, C["gen"])(n, seed=wl.SEED + rank)
    mode = w["mode"]
    if args.impl == "reference":
        if rank != 0:
            return
        if C.get("spring"):
            emit({"impl": "reference", "unavailable": "the reference snapshot has no spring-damper solver source (MultiBodyConstraintSolverSpring absent); "
                                                      "compare with --config humanoid4096 (LCP)"})
            return
        sample_s = 4.0
        v, sample = _config_reference_rate(args.config, w, model, sample_s)
        per = max(16, int(v * 60.0 / (K + W)))          # a step of this arm = a bounded sample of the batch
        per = min(per, n)
        from oracle import ref
        sim = ref.RefSim.from_model(model); sim.set_params(**w["params"])
        tau = w.get("tau"); full = None
        if tau is not None:
            full = np.zeros((n, sim.n_tau)); full[:, -tau.shape[1]:] = tau
        def batch():
            sim.step_batch(mode, w["q"][:per], w["qd"][:per], None if full is None else full[:per])
        for _ in range(W):
            batch()
        t0 = time.perf_counter()
        for _ in range(K):
            batch()
        el = time.perf_counter() - t0
        val = per * K / el
        emit({"metric": METRIC, "value": val, "unit": "env-steps/s", "impl": "reference", "n_gpus": args.gpus, "steps": K, "warmup": W,
              "ms_per_step": 1e3 * el / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
              "data": "synthetic", "config": {"workload": C["workload"], "envs_per_gpu": n, "envs_per_step": per,
                                              "path": "forward_dynamics / World::step (templated CPU path), one thread"},
              "cpu_baseline": {"value": val, "unit": "env-steps/s", "cores": 1, "kind": "reference", "sample": f"{K} steps x {per} envs"},
              "e2e": {"value": val, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
        return
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the b200 arm has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    prec = {0: tds_b200.PREC_AUTO, 1: tds_b200.PREC_F64, 2: tds_b200.PREC_F32, 3: tds_b200.PREC_MIXED}[args.precision]
    sim = tds_b200.BatchSim(model, n, device=local_rank, precision=prec, **w["params"])
    if C.get("spring"):
        sim.set_contact_model(1)
    ns = sim.n_stride
    def soa(a, dim):
        t = torch.zeros((max(dim, 1), ns), device=dev)
        if a is not None and dim:
            t[:dim, :n] = torch.tensor(np.ascontiguousarray(a.T), dtype=torch.float32)
        return t
    q, qd = soa(w["q"], sim.n_q), soa(w["qd"], sim.n_qd)
    tau = w.get("tau")
    ring = 16
    g = torch.Generator(device="cpu").manual_seed(99 + rank)
    taus = None
    if tau is not None and sim.n_tau:
        base = soa(tau[:, -sim.n_tau:], sim.n_tau)
        taus = [base * float(s) for s in (0.5 + torch.rand(ring, generator=g))]
    qdd = sim.alloc(sim.n_qd) if mode == 0 else None
    cdist = sim.alloc(sim.n_contact_points) if (mode == 2 and sim.n_contact_points) else None
    ccount = torch.zeros(ns, dtype=torch.int32, device=dev) if cdist is not None else None
    clinks = torch.zeros((2 * max(sim.n_contact_points, 1), ns), dtype=torch.int32, device=dev) if cdist is not None else None
    L, st = sim._L, torch.cuda.current_stream().cuda_stream
    import ctypes

    # every timed step processes the same synthetic batch: outputs go to a second pair of buffers (an unactuated humanoid
    # left to fall for hundreds of steps ends up in states no configuration of BASELINE.json describes)
    q2, qd2 = torch.zeros_like(q), torch.zeros_like(qd)

    def one_step(i):
        sim.step_device(mode, q, qd, None if taus is None else taus[i % ring], q_out=q2, qd_out=qd2, qdd_out=qdd, contact_dist=cdist)
        if cdist is not None:   # the contact record of SURVEY 8d: count + (link_a, link_b) list of the step, on the device
            L.tds_b200_contact_list_device(sim._h, ctypes.c_void_p(cdist.data_ptr()), ctypes.c_void_p(ccount.data_ptr()),
                                           ctypes.c_void_p(clinks.data_ptr()), ctypes.c_void_p(st))
    flush = torch.empty(192 * 1024 * 1024 // 4, device=dev)   # 192 MiB > the 126 MB L2
    for i in range(W):
        one_step(i)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start(); time.sleep(0.25)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    for i in range(K):
        flush.zero_()                       # L2 flush between timed iterations (outside the event pair)
        ev[i][0].record()
        one_step(W + i)
        ev[i][1].record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    clocks = sampler.stop() if sampler else None
    dev_ms = float(sum(a.elapsed_time(b) for a, b in ev))
    t = torch.tensor([dev_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    if not bool(torch.isfinite(q2).all()) or not bool(torch.isfinite(qd2).all()):
        raise SystemExit("bench.py: non-finite state after the timed region")
    if args.dump_outputs and rank == 0:   # what step_device / the contact record of the last timed step returned
        def rows(t, dim):
            return t[:dim, :n].T.cpu().numpy()
        out = {"qdd": rows(qdd, sim.n_qd)} if mode == 0 else {"q": rows(q2, sim.n_q), "qd": rows(qd2, sim.n_qd)}
        if cdist is not None:
            out.update(contact_dist=rows(cdist, sim.n_contact_points), contact_count=ccount[:n].cpu().numpy(),
                       contact_links=rows(clinks, 2 * sim.n_contact_points))
        dump_outputs(args.dump_outputs, out)
    # end to end through tds_b200_step_host: fp64 AoS host buffers in and out (the MultiBody-style arrays a
    # VectorizedEnvironment caller holds), copies + layout conversion + step inside the timed region
    hq, hqd = w["q"].copy(), w["qd"].copy()
    htau = None if tau is None or not sim.n_tau else np.ascontiguousarray(tau[:, -sim.n_tau:])
    Ke = min(K, 100)
    for _ in range(3):
        sim.step_host(mode, hq, hqd, htau)
    t0 = time.perf_counter()
    for _ in range(Ke):
        sim.step_host(mode, hq, hqd, htau)
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    value = n * world * K / (total_ms * 1e-3)
    peaks, peak_src = _measured_peaks()
    achieved = C["bytes"] * n / ((total_ms * 1e-3) / K) / 1e9
    in_b = 8 * n * (sim.n_q + sim.n_qd + (sim.n_tau if htau is not None else 0))
    out_b = 8 * n * (sim.n_qd if mode == 0 else sim.n_q + sim.n_qd)
    line = {"metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": ["f32 + f64 (mixed)", "f64", "f32"][sim.precision], "data": "synthetic",
            "config": {"workload": C["workload"], "envs_per_gpu": n, "global_envs": n * world, "mode": int(mode),
                       "parallelism": f"env-sharded x{world}, no data-path collective",
                       "timing": "CUDA events around each of the K steps (individual launches), summed, max over ranks",
                       "l2": "flushed between timed steps (192 MiB written outside the event pairs)"},
            "gpu_launches": K * (2 if cdist is not None else 1),
            "e2e": {"value": n * world * Ke / float(te.item()), "unit": "env-steps/s", "h2d_bytes_per_step": in_b, "d2h_bytes_per_step": out_b,
                    "steps": Ke, "api": "tds_b200_step_host (fp64 AoS host arrays in / out, pageable)"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
                         "traffic": None, "peak_source": peak_src, "kernel": sim.kernel_name(),
                         "algorithmic_bytes_per_env_step": C["bytes"]},
            "clocks": clocks}
    if not args.no_cpu_baseline and world == 1:
        try:
            v, sample = _config_reference_rate(args.config, w, model, 5.0)
            line["cpu_baseline"] = {"value": v, "unit": "env-steps/s", "cores": 1, "kind": "reference", "sample": sample}
        except Exception as ex:
            line["cpu_baseline"] = {"value": None, "unit": "env-steps/s", "cores": 0, "kind": "reference", "sample": f"unavailable: {ex}"}
    emit(line)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=100)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs", type=int, default=None, help="environments per GPU (default: the size the config names)")
    ap.add_argument("--config", default="laikago4096", choices=sorted(CONFIGS),
                    help="BASELINE.json configuration; the default is the one the metric is quoted on (configs[3])")
    ap.add_argument("--precision", type=int, default=0, help="0 mixed (fp32 ABA + fp64 contact), 1 fp64, 2 fp32")
    ap.add_argument("--no-graph", action="store_true", help="launch the timed steps one by one instead of replaying a CUDA graph")
    ap.add_argument("--small-ring", action="store_true", help="16 action buffers (L2-resident) instead of 768 (> L2)")
    ap.add_argument("--min-seconds", type=float, default=1.0, help="keep the GPU busy this long for clock sampling")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--gather-reward", action="store_true",
                    help="all-gather {reward, done} per step (only needed by a single centralized policy): the step kernel "
                         "writes into the NCCL send buffer, the collective is captured in the same CUDA graph")
    ap.add_argument("--gather-overlap", action="store_true", help="with --gather-reward: the gather of step k runs on a side stream under step k+1")
    ap.add_argument("--strong", action="store_true", help="strong scaling: the config's environments are divided over the ranks")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned (rank 0's environments) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        # the reference arms size their batch from a measured rate, so their outputs differ from run to run
        ap.error("--dump-outputs needs --impl b200")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.envs is None:
        args.envs = CONFIGS[args.config]["envs"]
    if args.config != "laikago4096":
        run_config(args, rank, world, local_rank)
        return
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import tds_b200
    import tds_b200.workloads as wl

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the b200 arm has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")   # keep NCCL's version banner off stdout (one JSON line only)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    n = args.envs
    if args.strong:   # strong scaling: the 4096 environments of the config are divided over the ranks
        from tds_b200.parallel import shard_range
        lo, hi = shard_range(args.envs, rank, world)
        n = hi - lo
    K, W = args.steps, max(args.warmup, 3)

    sim = tds_b200.laikago_sim(n, device=local_rank, precision=args.precision, auto_reset=True)
    w = wl.laikago(n, seed=wl.SEED + rank)
    sim.env_set_state(w["q"], w["qd"])
    ns = sim.n_stride
    # Resident synthetic policy outputs: a ring of action tensors LARGER THAN L2 (768 x 12 x ns fp32 = 151 MB
    # > 126 MB), so every timed step reads its actions from HBM; q/qd (0.6 MB) are the kernel's own previous
    # output and stay wherever the hardware leaves them, as in any rollout.
    ring = 768 if not args.small_ring else 16
    g = torch.Generator(device="cpu").manual_seed(1234 + rank)
    actions = (torch.rand((ring, 12, ns), generator=g) * 0.8 - 0.4).to(dev)
    gathered = None
    if args.gather_reward and world > 1:
        from tds_b200.parallel import RewardDoneExchange
        gathered = RewardDoneExchange(ns, world, dev, depth=2 if args.gather_overlap else 1)
    reward = torch.zeros(ns, device=dev) if gathered is None else gathered.reward(0)
    done = torch.zeros(ns, device=dev) if gathered is None else gathered.done(0)

    zero = torch.zeros((12, ns), device=dev)
    for _ in range(10):  # settle like LaikagoContactSimulation::reset (laikago_environment2.h:96-104)
        sim.env_step_device(zero, reward, done)

    def one_step(i):
        if gathered is None:
            sim.env_step_device(actions[i % ring], reward, done)
        else:   # the kernel's reward / done stores fill the send buffer; the collective follows in stream order
            gathered.before_step(i)
            sim.env_step_device(actions[i % ring], gathered.reward(i), gathered.done(i))
            gathered.gather(i)

    for i in range(W):
        one_step(i)
    torch.cuda.synchronize()
    graph = None
    if not args.no_graph:
        # the K timed steps are captured once into a CUDA graph (K kernel nodes) and replayed: launch-bound
        # inner loops belong in graphs; the work per step is unchanged
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            one_step(W)          # first launch on the capture stream outside capture
        torch.cuda.synchronize()
        if gathered is not None:   # nothing recorded outside the capture may be waited on inside it
            with torch.cuda.stream(side):
                gathered.join()
            torch.cuda.synchronize()
            gathered.reset()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            for i in range(K):
                one_step(W + 1 + i)
            if gathered is not None:
                gathered.join()
        torch.cuda.synchronize()
        graph.replay()            # one untimed replay: the timed one is not the first launch of a fresh graph
        torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.25)

    def last_outputs():
        """What the env step returned in the last timed step (one_step(W + K)): the resident state the observations are
        read from, reward and done.  Called after the closing event, so it is not timed."""
        if not args.dump_outputs or rank != 0:
            return None
        torch.cuda.synchronize()
        q_o, qd_o = sim.env_get_state()
        r, d = (reward, done) if gathered is None else (gathered.reward(W + K), gathered.done(W + K))
        return {"q": q_o, "qd": qd_o, "reward": r[:n].cpu().numpy(), "done": d[:n].cpu().numpy()}

    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.perf_counter()
    reps = 1
    if graph is not None:
        # The K-step graph is replayed for about min_seconds so that the clocks can be sampled around the timed region
        # and so that a short run (K = 20 is 0.3 ms) is not timed while the GPU is still ramping up from its idle clocks:
        # half of the replays run before the timed one (extra warm-up, untimed), half after; exactly ONE replay = exactly K
        # steps lies between the two events.
        reps = max(2, int(args.min_seconds / max(1e-6, K * 60e-6)))
        for _ in range(reps // 2):
            graph.replay()
        ev0.record()
        graph.replay()
        ev1.record()
        outputs = last_outputs()
        for _ in range(reps - reps // 2 - 1):
            graph.replay()
        torch.cuda.synchronize()
    else:
        ev0.record()
        for i in range(K):
            one_step(W + 1 + i)
        if gathered is not None:
            gathered.join()
        ev1.record()
        outputs = last_outputs()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t_wall = time.perf_counter() - t_wall0
    clocks = sampler.stop() if sampler else None
    dev_ms = float(ev0.elapsed_time(ev1))                         # device time of exactly K steps
    t = torch.tensor([dev_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    q_chk, _ = sim.env_get_state()
    if not np.all(np.isfinite(q_chk)):
        raise SystemExit("bench.py: non-finite state after the timed region")
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)

    # ---- end-to-end through the public host API: pinned host actions in, obs/reward/done out, every step
    act_h = torch.rand((n, 12)).mul_(0.8).sub_(0.4).pin_memory()
    # one pinned block, obs | reward | done adjacent: the library then returns all three with a single copy
    out_h = torch.zeros(n * 38).pin_memory()
    obs_h, rew_h, done_h = out_h[:n * 36].view(n, 36), out_h[n * 36:n * 37], out_h[n * 37:]
    Ke = min(K, 200)
    step_host = sim.bind_env_step_host(act_h, obs_h, rew_h, done_h)   # same C entry point, buffers bound once
    for _ in range(5):
        step_host()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(Ke):
        step_host()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_val = n * world * Ke / float(te.item())

    if rank != 0:
        if world > 1:
            if gathered is not None:   # collectives captured in a CUDA graph: leave without the process-group teardown
                torch.cuda.synchronize()
                dist.barrier()
                os._exit(0)
            dist.destroy_process_group()
        return
    value = n * world * K / (total_ms * 1e-3)
    peaks, peak_src = _measured_peaks()
    kernel_s = (total_ms * 1e-3) / K
    achieved = ALGO_BYTES_PER_ENV_STEP * n / kernel_s / 1e9
    traffic = None
    for prof in ("r02_step_kernel_ncu.json", "r01_step_kernel_ncu.json"):   # one `ncu --set full` capture of the step kernel
        prof = os.path.join(ROOT, "profiles", prof)
        if os.path.exists(prof):
            try:
                with open(prof) as f:
                    traffic = json.load(f).get("dram_bytes_per_launch")
                break
            except Exception:
                pass
    line = {
        "metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "strong" if args.strong else "weak", "vs_baseline": None,
        "dtype": ["f32 (ABA, factorisation, PGS) + f64 (kinematics, inertias, CRBA, Jacobians, LCP rhs)", "f64", "f32"][args.precision], "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "envs_per_gpu": n, "global_envs": n * world, "dt": 1e-3, "parallelism": f"env-sharded x{world}, no data-path collective"
                   + ((" + all-gather(reward,done) in the graph, step kernel writes the send buffer" + (", overlapped with the next step" if args.gather_overlap else "")) if gathered is not None else ""),
                   "state": "SoA fp32 resident in HBM",
                   "timing": "CUDA events around exactly K steps (" + (f"one CUDA-graph replay of K kernel nodes, preceded and followed by untimed replays of the same graph for the clock sampler: {reps} replays in all" if graph is not None else "K individual launches") + "), max over ranks",
                   "l2": (f"inputs larger than L2: ring of {ring} action tensors = {ring * 12 * ns * 4 / 2**20:.0f} MiB, one per step"
                          if ring >= 700 else f"ring of {ring} action tensors (L2-resident)"),
                   "wall_s_all_replays": t_wall},
        "gpu_launches": K, "e2e": {"value": e2e_val, "unit": "env-steps/s", "h2d_bytes_per_step": n * 12 * 4,
                                    "d2h_bytes_per_step": n * 36 * 4 + n * 4 + n * 4, "steps": Ke, "gpu_launches_per_step": 1, "path": "zero-copy: the step kernel reads the pinned host actions and writes obs / reward / done to pinned host memory itself (PCIe traffic inside the timed kernel)",
                                    "api": "tds_b200_env_step_host (actions host->device, obs/reward/done device->host, pinned)"},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                     "frac": achieved / peaks["hbm_gbs"], "traffic": traffic, "peak_source": peak_src,
                     "kernel": sim.kernel_name(), "algorithmic_bytes_per_env_step": ALGO_BYTES_PER_ENV_STEP,
                     "note": "the step is not bandwidth bound: ~27 kFLOP and 344 B per env-step, one wave of 128 CTAs whose critical path "
                             "is one warp's instruction stream (instruction fetch + dependent-issue latency, see DESIGN.md and "
                             "profiles/); fp32-equivalent GFLOP/s reported beside the HBM figure",
                     "gflops": FLOPS_PER_ENV_STEP * n / kernel_s / 1e9},
        "clocks": clocks,
    }
    if not args.no_cpu_baseline and world == 1:
        try:
            v, cores, sample, table = cpu_reference_sweep(0, 12.0)
            line["cpu_baseline"] = {"value": v, "unit": "env-steps/s", "cores": cores, "kind": "reference", "sample": sample,
                                    "path": "step_forward_original (templated World::step path), one instance per thread",
                                    "threads_sweep": table, "usable_cores": host_cores(), "os_cpu_count": os.cpu_count()}
            v2, cores2, sample2, table2 = cpu_reference_sweep(1, 4.0)
            line["cpu_baseline_codegen"] = {"value": v2, "unit": "env-steps/s", "cores": cores2, "kind": "reference",
                                            "sample": sample2, "threads_sweep": table2,
                                            "path": "omp_model_laikago_forward_zero_kernel (reference's codegen CPU path)"}
        except Exception as ex:  # the oracle library did not travel: report it, do not fake it
            line["cpu_baseline"] = {"value": None, "unit": "env-steps/s", "cores": 0, "kind": "reference", "sample": f"unavailable: {ex}"}
    emit(line)
    if world > 1:
        if gathered is not None:       # (round 2: the teardown hung for the full timeout after the line was printed)
            torch.cuda.synchronize()
            dist.barrier()
            os._exit(0)
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
