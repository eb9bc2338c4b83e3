#!/usr/bin/env python
"""Benchmark of the MSACL fused rollout hot path (BASELINE.json metric: fused env-steps/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--env NAME] [--envs-per-gpu M] [--dump-outputs DIR]

Headline workload (config 5 of BASELINE.json, per-GPU share): QuadTracking, 2^21 env instances per GPU
(16 Mi envs on 8 GPUs), default-init StochaPolicy actor (seed 0), Philox resets, one "step" =
one fused rollout launch of `--inner` (16) env steps over all instances, transitions
materialised in HBM.  Weak scaling: per-GPU work is fixed, env ids are sharded by rank.

The JSON line also carries a `configs` block: the other BASELINE configs (2: Pendulum / DuctedFan 65 536 envs,
3: TwoLink 2^20 envs + MSACL targets over 2^20 windows + learner iteration times, 4: SingleTrackCar 2^22 envs sharded
over the ranks, 1: VanderPol training loop with the reference's default arguments) and the FP32 engine, each with its
own value and roofline fraction.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "fused rollout env-steps/sec"
UNIT = "env-steps/s"


def actor_flops(d, a):      # SURVEY.md 8d: 2*(D*256 + 256*256 + 256*2A)
    return 2 * (d * 256 + 256 * 256 + 256 * 2 * a)


DYN_FLOPS = {"VanderPol": 70, "Pendulum": 70, "DuctedFan": 200, "TwoLink": 270, "SingleTrackCar": 430, "QuadTracking": 950}


def transition_bytes(d, a):  # obs, act, rew, cost, obs2, logp (f32) + done, emit (u8) per env-step
    return 4 * (2 * d + a + 3) + 2


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 4), ("hw_thermal_slowdown", 5), ("sw_thermal_slowdown", 6), ("sw_power_cap", 7)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------
# CPU arms.  (a) the oracle port of the same fused step (actor + sample + env + reward/cost + autoreset), vectorised
# NumPy, one process per host core; (b) the reference AS SHIPPED (unmodified `RL` package installed into baseline/_ref
# by __graft_entry__.build(), imported through the gymnasium stub): its own NstepOffSampler.sample() at the reference's
# default env_num = 4, one sampler per host core.
# ------------------------------------------------------------------------------------------
def cpu_rollout(env_name, n_envs, steps, seed=0):
    from oracle import actor as oactor, envs as oenv, rollout as oroll
    spec = oenv.SPECS[env_name]
    w = oactor.init_policy_weights(spec.obs_dim, spec.act_dim, seed=0)
    ids = np.arange(n_envs, dtype=np.uint64)
    venv = oroll.VectorEnv(env_name, oroll.philox_reset(env_name, seed, ids, np.zeros(n_envs, np.int64)), seed=seed, env_ids=ids)
    rng = np.random.default_rng(seed)
    t0 = time.perf_counter()
    for _ in range(steps):
        eps = rng.standard_normal((n_envs, spec.act_dim)).astype(np.float32)
        oroll.sampler_step(venv, w, eps)
    return time.perf_counter() - t0


def _cpu_worker(job):
    env_name, n_envs, steps, seed = job
    try:
        from threadpoolctl import threadpool_limits
        with threadpool_limits(limits=1):                 # one BLAS thread per process: the processes cover the cores
            return cpu_rollout(env_name, n_envs, steps, seed)
    except ImportError:
        return cpu_rollout(env_name, n_envs, steps, seed)


def cpu_rollout_all_cores(env_name, n_per_proc, steps, procs):
    """P independent processes (no IPC on the step path), each stepping its own n_per_proc env instances with the
    NumPy port -- the embarrassingly-parallel best case of BASELINE.md section 3.  Returns env-steps/s over the
    slowest process."""
    import multiprocessing as mp
    ctx = mp.get_context("fork")
    with ctx.Pool(procs) as pool:
        times = pool.map(_cpu_worker, [(env_name, n_per_proc, steps, 1000 + p) for p in range(procs)])
    return procs * n_per_proc * steps / max(times)


def cpu_baseline(env_name, budget_s=10.0):
    n, procs = 4096, os.cpu_count() or 1
    t1 = cpu_rollout(env_name, n, 1)                      # includes first-call overheads
    t2 = cpu_rollout(env_name, n, 2)
    per = max((t2 - t1), 1e-3) * 1.5                      # processes slow each other down a little
    steps = int(min(max(budget_s / per, 2), 200))
    val = cpu_rollout_all_cores(env_name, n, steps, procs)
    return {"value": val, "unit": UNIT, "cores": procs, "kind": "port",
            "sample": f"{env_name}: {procs} processes x {n} envs x {steps} fused steps (NumPy oracle port, one process per host core)"}


REF_DIR = os.path.join(ROOT, "baseline", "_ref")
GYM_STUB = os.path.join(ROOT, "tests", "golden", "_gym_stub")


def reference_available():
    return os.path.isdir(os.path.join(REF_DIR, "RL")) and os.path.isdir(GYM_STUB)


def _reference_args(env_name, env_num, horizon):
    """Keyword set of example/msacl_train.py (reference defaults) that RL.create_pkg.create_sampler consumes."""
    return dict(
        env_name=env_name, algorithm="msacl", enable_cuda=False, use_gpu=False, env_num=env_num, env_seed=1, capture_video=False,
        target_value=0.0, reward_scale=100.0, cost_scale=100.0, value_func_name="ActionValue", value_func_type="MLP",
        value_hidden_sizes=[256, 256], value_hidden_activation="relu", value_output_activation="linear",
        lyapunov_func_name="LyapunovValue", lyapunov_func_type="MLP", lyapunov_hidden_sizes=[256, 256],
        lyapunov_hidden_activation="tanh", lyapunov_output_dim=256, lyapunov_output_activation="linear",
        lyapunov_single_input_dim=False, policy_func_name="StochaPolicy", policy_func_type="MLP",
        policy_act_distribution="TanhGaussDistribution", policy_hidden_sizes=[256, 256], policy_hidden_activation="relu",
        policy_min_log_std=-20, policy_max_log_std=1, q_learning_rate=1e-3, lyapunov_learning_rate=1e-3, policy_learning_rate=3e-4,
        alpha_learning_rate=1e-3, lya_diff_scale=10.0, lya_zero_scale=1.0, lya_positive_scale=1.0, tau=0.005, disable_auto_alpha=False,
        alpha=1.0, set_alpha_bound=False, alpha_bound=2.0, policy_frequency=2, target_network_frequency=1, anneal_lr=False, alpha1=1,
        alpha2=2, lya_eta=0.15, clip_coef=0.1, trainer="nstep_off_serial_trainer", max_iteration=1000000, buffer_name="nstep_replay_buffer",
        buffer_warm_size=5000, buffer_max_size=1000000, replay_batch_size=256,
        n_step=20, gamma=0.99, retrace_lambda=0.95, sampler_name="nstep_off_sampler",
        sample_batch_size=horizon, noise_params=None, action_type="continu", batch_size_per_sampler=horizon, seed=0)


_REF_SAMPLER = None


def _reference_init(env_name, env_num, horizon):
    """Pool initializer: one process = one unmodified reference sampler
    (RL.trainer.sampler.nstep_off_sampler.NstepOffSampler built by RL.create_pkg.create_sampler)."""
    global _REF_SAMPLER
    for p in (GYM_STUB, REF_DIR):
        if p not in sys.path:
            sys.path.insert(0, p)
    if not hasattr(np, "float_"):
        np.float_ = np.float64               # RL/utils/common_utils.py:50 uses the removed NumPy 1.x name
    import io
    import random
    from contextlib import redirect_stdout
    import torch
    torch.set_num_threads(1)                 # the processes cover the cores
    seed = os.getpid()
    random.seed(seed); np.random.seed(seed % (2 ** 31)); torch.manual_seed(seed)
    with redirect_stdout(io.StringIO()):
        import gymnasium as gym
        from RL.create_pkg.create_sampler import create_sampler
        from RL.env.make_env import make_env
        probe = gym.vector.SyncVectorEnv([make_env(env_name, 1, 0, False, "bench")])
        sa, so = probe.single_action_space, probe.single_observation_space
        args = _reference_args(env_name, env_num, horizon)
        args.update(obs_dim=so.shape[0], act_dim=sa.shape[0], action_high_limit=sa.high.astype("float32"),
                    action_low_limit=sa.low.astype("float32"))
        _REF_SAMPLER = create_sampler(**args)
        _REF_SAMPLER.sample()                # first-call overheads


def _reference_calls(calls):
    import io
    from contextlib import redirect_stdout
    with redirect_stdout(io.StringIO()):
        t0 = time.perf_counter()
        for _ in range(calls):
            _REF_SAMPLER.sample()
        return time.perf_counter() - t0


class ReferencePool:
    """The unmodified reference sampler path on all host cores: one reference sampler per core, each with the reference's
    default env_num = 4 and sample_batch_size = 20 (example/msacl_train.py)."""

    def __init__(self, env_name, env_num=4, horizon=20):
        import multiprocessing as mp
        self.env_name, self.env_num, self.horizon = env_name, env_num, horizon
        self.procs = os.cpu_count() or 1
        self.pool = mp.get_context("fork").Pool(self.procs, initializer=_reference_init, initargs=(env_name, env_num, horizon))
        self.step(1)                         # every worker is up and has built its sampler

    def step(self, calls):
        """Every worker runs `calls` sample() calls; env-steps/s over the slowest worker."""
        times = self.pool.map(_reference_calls, [calls] * self.procs, chunksize=1)
        return self.procs * self.env_num * self.horizon * calls / max(times)

    def describe(self, calls):
        return (f"{self.env_name}: {self.procs} processes x the unmodified reference NstepOffSampler.sample() (env_num {self.env_num}, "
                f"sample_batch_size {self.horizon}) x {calls} calls per step; RL package from baseline/_ref, gymnasium 0.28.1 stub")

    def close(self):
        self.pool.close()
        self.pool.join()


def reference_as_shipped(env_name, calls=2, steps=3):
    pool = ReferencePool(env_name)
    try:
        val = float(np.mean([pool.step(calls) for _ in range(steps)]))
        return {"value": val, "unit": UNIT, "cores": pool.procs, "kind": "reference", "sample": pool.describe(calls)}
    finally:
        pool.close()


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    procs = os.cpu_count() or 1
    workload = f"{args.env} fused rollout (actor+sample+env+reward/cost+autoreset), bounded CPU sample of config 5"
    port = None
    if reference_available():
        pool = ReferencePool(args.env)
        calls = 2
        try:
            for _ in range(args.warmup):
                pool.step(calls)
            t0 = time.perf_counter()
            vals = [pool.step(calls) for _ in range(args.steps)]
            el = time.perf_counter() - t0
        finally:
            pool.close()
        val = float(np.mean(vals))
        cpu = {"value": val, "unit": UNIT, "cores": procs, "kind": "reference", "sample": pool.describe(calls)}
        port = cpu_rollout_all_cores(args.env, 4096, 2, procs)
    else:
        n, steps_per = 4096, 4
        for _ in range(args.warmup):
            cpu_rollout(args.env, n, 1)
        t0 = time.perf_counter()
        vals = [cpu_rollout_all_cores(args.env, n, steps_per, procs) for _ in range(args.steps)]
        el = time.perf_counter() - t0
        val = float(np.mean(vals))
        cpu = {"value": val, "unit": UNIT, "cores": procs, "kind": "port",
               "sample": f"{args.env}: each step = {procs} processes x {n} envs x {steps_per} fused env steps on the NumPy oracle port "
                         "(baseline/_ref not present on this box)"}
    out = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": el / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": {"workload": workload},
        "cpu_baseline": cpu,
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if port is not None:
        out["cpu_baseline_port"] = {"value": port, "unit": UNIT, "cores": procs, "kind": "port",
                                    "sample": f"{args.env}: {procs} processes x 4096 envs x 2 fused steps, vectorised NumPy oracle port "
                                              "(~100x faster than the reference's per-env Python loop; reported for context)"}
    print(json.dumps(out))


# ------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------
class Ctx:
    pass


def make_policy(torch, D, A):
    torch.manual_seed(0)
    return torch.nn.Sequential(torch.nn.Linear(D, 256), torch.nn.ReLU(), torch.nn.Linear(256, 256), torch.nn.ReLU(),
                               torch.nn.Linear(256, 2 * A))


def time_rollout(cx, env, n, K, engine, steps, warmup, keep=False, clocks=False, settle_s=0.0):
    """Device-resident throughput of the fused rollout: `steps` launches of K env steps over n envs per rank.
    Returns dict(value, total_ms, kern_ms [, ro, actor])."""
    torch, dist = cx.torch, cx.dist
    from msacl_b200.sampler import ActorWeights, FusedRollout
    from msacl_b200.specs import get_spec
    spec = get_spec(env)
    pol = make_policy(torch, spec.obs_dim, spec.act_dim)
    lin = [m for m in pol if isinstance(m, torch.nn.Linear)]
    actor = ActorWeights([(l.weight, l.bias) for l in lin], device=cx.dev)
    ro = FusedRollout(env, n, K, n_step=20, seed=0, env_base=cx.rank * n, device=cx.dev, engine=engine,
                      history_chunks=None if keep else 1)
    ro.state.reset()
    for _ in range(warmup):
        ro.run(actor)
    burst = None
    if settle_s > 0:
        # (1) burst figure: the K launches right after the W warm-up launches, as round 1 measured it
        cx.barrier()
        b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        b0.record(cx.stream)
        for _ in range(steps):
            ro.run(actor)
        b1.record(cx.stream)
        cx.barrier()
        burst = n * K * steps * cx.world / (cx.max_over_ranks(b0.elapsed_time(b1)) * 1e-3)
        # (2) untimed settling launches: the part runs at its 1 kW power cap (sw_power_cap) and the SM clock of a cool GPU
        # sags by 3-5 % over the first second of back-to-back launches.  `value` and `e2e` are both taken after the clocks
        # have settled, so that they are comparable with each other (a burst `value` next to a settled `e2e` made the e2e
        # path look 4 % slower than it is) and with the SUSTAINED tensor peak.
        t_s = time.perf_counter()
        while time.perf_counter() - t_s < settle_s:
            for _ in range(4):
                ro.run(actor)
            torch.cuda.synchronize()
    cx.barrier()
    cs = None
    if clocks:
        cs = ClockSampler(cx.local)
        cs.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record(cx.stream)
    for i in range(steps):
        ro.run(actor, timing=ev[i])
    t1.record(cx.stream)
    cx.barrier()
    clk = cs.stop() if cs else None
    total_ms = cx.max_over_ranks(t0.elapsed_time(t1))
    kern_ms = float(np.mean([a.elapsed_time(b) for a, b in ev]))
    out = {"value": n * K * steps * cx.world / (total_ms * 1e-3), "total_ms": total_ms, "kern_ms": kern_ms, "clocks": clk,
           "value_burst": burst}
    if keep:
        out.update(ro=ro, actor=actor, host_w=[p.detach().clone().pin_memory() for p in pol.parameters()])
    else:
        del ro, actor
        torch.cuda.empty_cache()
    return out


def last_launch_outputs(ro, env_base, seed=0, budget=48 << 20):
    """What the last launch of `ro` handed its caller: the K new transition slices ([K, m, .] per field, float32), for
    all n env instances or, beyond `budget` bytes, a fixed seeded sample of m of them; `env_index` holds the global
    env ids of the m columns."""
    import torch
    tr = ro.tr
    fields = {k: v[tr.H:] for k, v in tr.fields().items()}
    per_env = 4 * sum(v[:, 0].numel() for v in fields.values())
    m = min(tr.n, max(1, budget // per_env))
    idx = np.arange(tr.n) if m == tr.n else np.sort(np.random.default_rng(seed).choice(tr.n, m, replace=False))
    cols = torch.as_tensor(idx, device=fields["obs"].device)
    out = {k: v.index_select(1, cols).float().cpu().numpy() for k, v in fields.items()}
    out["env_index"] = (idx + env_base).astype(np.float64)
    return out


def time_general_rollout(cx, env="TwoLink", n=1 << 18, K=16, hidden=(64, 64), steps=3, warmup=2):
    """The general rollout engine (a policy the fused kernels are not specialised for: per-layer tcgen05 GEMMs +
    msacl_rollout_step, launches per env step instead of one per K steps)."""
    torch = cx.torch
    from msacl_b200.sampler import FusedRollout, GeneralActor
    from msacl_b200.specs import get_spec
    spec = get_spec(env)
    torch.manual_seed(0)
    sizes = [spec.obs_dim, *hidden, 2 * spec.act_dim]
    lin = [torch.nn.Linear(a, b) for a, b in zip(sizes[:-1], sizes[1:])]
    actor = GeneralActor([(l.weight, l.bias) for l in lin], [torch.nn.Tanh() for _ in hidden] + [torch.nn.Identity()], device=cx.dev)
    ro = FusedRollout(env, n, K, n_step=20, seed=0, env_base=cx.rank * n, device=cx.dev, history_chunks=1)
    ro.state.reset()
    for _ in range(warmup):
        ro.run(actor)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0.record(cx.stream)
    for _ in range(steps):
        ro.run(actor)
    t1.record(cx.stream)
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1) / steps
    del ro, actor
    torch.cuda.empty_cache()
    return {"env": env, "envs_per_gpu": n, "inner_steps": K, "engine": "general", "policy_hidden_sizes": list(hidden),
            "policy_hidden_activation": "tanh", "value": n * K / (ms * 1e-3), "unit": UNIT, "ms_per_launch_of_K_steps": ms,
            "gpu_launches_per_env_step": len(hidden) + 2}


def rollout_roofline(cx, env, n, K, engine, kern_ms, ffma_peak):
    from msacl_b200.specs import get_spec
    spec = get_spec(env)
    D, A = spec.obs_dim, spec.act_dim
    flops = actor_flops(D, A) + DYN_FLOPS[env]
    achieved = flops * n * K / (kern_ms * 1e-3) / 1e12
    bytes_per_step = transition_bytes(D, A)
    state_bytes = 2 * (4 * spec.sf_rows + 8 * spec.sd_rows + 20)      # read + write once per launch
    hbm_gbs = (bytes_per_step * n * K + state_bytes * n) / (kern_ms * 1e-3) / 1e9
    hbm = {"achieved_gbs": hbm_gbs, "peak_gbs": cx.hbm_peak, "frac": hbm_gbs / cx.hbm_peak,
           "algorithmic_bytes_per_env_step": bytes_per_step + state_bytes / K}
    kernel = ("rollout_tc_kernel" if engine == "tc" else "rollout_fused_kernel") + f"<{env}>"
    # DRAM traffic: ncu dram__bytes_read.sum + dram__bytes_write.sum of this kernel from the committed capture
    # (profiles/ncu_traffic.json, written by tools/ncu_traffic.py from the ncu --set full raw CSV), scaled per env-step
    traffic, tsrc = None, None
    rec = cx.ncu_traffic.get(kernel)
    if rec:
        traffic = rec["dram_bytes_per_launch"] / rec["env_steps_per_launch"] * n * K
        tsrc = rec["source"]
    if engine == "ffma":
        return {"bound": "fp32_ffma", "achieved": achieved, "peak": ffma_peak, "unit": "TFLOP/s", "frac": achieved / ffma_peak,
                "traffic": traffic, "traffic_source": tsrc,
                "peak_source": "measured in this run: msacl_ffma_probe (8 independent FFMA chains/thread, 2x256 threads/SM); "
                               "MEASURED_PEAKS.json has no FP32 figure (theoretical 148*128*2*1.965 GHz = 74.4)",
                "kernel": kernel, "kernel_ms": kern_ms, "algorithmic_flops_per_env_step": flops, "hbm": hbm}
    # tensor path: algorithmic FLOPs (one FP32-equivalent pass) against the measured dense bf16 peak; the
    # split-bf16 scheme issues 3 UMMAs per algorithmic product, so tensor-pipe utilisation is ~3x `frac`.
    return {"bound": "tensor", "achieved": achieved, "peak": cx.tensor_peak, "unit": "TFLOP/s", "frac": achieved / cx.tensor_peak,
            "traffic": traffic, "traffic_source": tsrc,
            "peak_source": ("MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)" if cx.peaks
                            else "fallback 1.4 PFLOP/s sustained"),
            "peak_burst": cx.tensor_burst, "tensor_issue_factor": 3,
            "tensor_pipe_frac_incl_split": 3 * achieved * (1 - 2 * 256 * 2 * A / flops) / cx.tensor_peak,
            "fp32_ffma_peak_tflops": ffma_peak, "kernel": kernel, "kernel_ms": kern_ms,
            "algorithmic_flops_per_env_step": flops, "hbm": hbm}


def ffma_probe(cx, mode=0, iters=20000):
    torch = cx.torch
    from msacl_b200 import _lib
    lib = _lib.load()
    sink = torch.rand(128, device=cx.dev)
    fl = C.c_double(0.0)
    for _ in range(2):
        _lib.check(lib.msacl_ffma_probe(mode, iters, sink.data_ptr(), C.byref(fl), _lib.current_stream()))
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record(cx.stream)
    _lib.check(lib.msacl_ffma_probe(mode, iters, sink.data_ptr(), C.byref(fl), _lib.current_stream()))
    p1.record(cx.stream)
    torch.cuda.synchronize()
    return fl.value / (p0.elapsed_time(p1) * 1e-3) / 1e12


def time_targets(cx, B=1 << 20, n=20, D=4):
    """BASELINE config 3: the MSACL target kernels over B TwoLink windows (C-ABI calls on preallocated outputs)."""
    torch = cx.torch
    from msacl_b200 import _lib, targets as tg
    lib, st, dev = _lib.load(), _lib.current_stream(), cx.dev
    g = torch.Generator(device=dev).manual_seed(0)
    r = lambda *s: torch.randn(*s, device=dev, generator=g)
    obs, obs2 = r(B, n, D) * 0.5, r(B, n, D) * 0.5
    lpn, lpo, v1, v2 = r(B, n), r(B, n), r(B, n).abs(), r(B, n).abs()
    rew, done, q1, q2 = r(B, n), (torch.rand(B, n, device=dev, generator=g) < 0.1).float(), r(B, n), r(B, n)
    coef = tg.Coefficients(n, device=dev)

    def timeit(fn, reps=10):
        for _ in range(3):
            fn()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); a.record()
        for _ in range(reps):
            fn()
        b.record(); torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    def line(ms, nbytes):
        gbs = nbytes / (ms * 1e-3) / 1e9
        return {"ms": ms, "windows_per_s": B / (ms * 1e-3), "achieved_gbs": gbs, "frac_of_hbm": gbs / cx.hbm_peak, "bound": "hbm"}

    out = {}
    parts = torch.empty(3, dtype=torch.float64, device=dev)
    g1, g2 = torch.empty_like(v1), torch.empty_like(v2)
    ms = timeit(lambda: _lib.check(lib.msacl_lyapunov_risk(
        B, n, D, obs.data_ptr(), obs2.data_ptr(), lpn.data_ptr(), lpo.data_ptr(), v1.data_ptr(), v2.data_ptr(),
        coef.son.data_ptr(), coef.diff.data_ptr(), coef.sl.data_ptr(), coef.alpha1, coef.alpha2, 10.0, 1.0,
        parts.data_ptr(), g1.data_ptr(), g2.data_ptr(), None, None, st)))
    out["lyapunov_risk_fwd_bwd"] = line(ms, B * n * 4 * (2 * D + 4 + 2))
    bk = torch.empty_like(rew)
    ms = timeit(lambda: _lib.check(lib.msacl_q_backup(B * n, rew.data_ptr(), done.data_ptr(), q1.data_ptr(), q2.data_ptr(),
                                                      lpn.data_ptr(), 0.99, 0.2, bk.data_ptr(), st)))
    out["q_backup"] = line(ms, B * n * 4 * 6)
    v0 = v1[:, 0].contiguous()
    raw, adv, mom = torch.empty_like(v0), torch.empty_like(v0), torch.empty(2, dtype=torch.float64, device=dev)

    def _adv():
        _lib.check(lib.msacl_stability_advantage(B, n, v0.data_ptr(), v2.data_ptr(), coef.diff.data_ptr(), coef.sl.data_ptr(),
                                                 raw.data_ptr(), mom.data_ptr(), st))
        _lib.check(lib.msacl_advantage_normalize(B, raw.data_ptr(), mom.data_ptr(), adv.data_ptr(), st))

    out["stability_advantage_normalize"] = line(timeit(_adv), B * 4 * (n + 1 + 3))
    del obs, obs2, lpn, lpo, v1, v2, rew, done, q1, q2, bk, g1, g2
    torch.cuda.empty_cache()
    return out


def time_learner(cx, env="TwoLink", batches=(256, (1 << 20) // 20), iters=6):
    """model_update wall time per iteration (CUDA events over `iters` iterations incl. the policy updates every second one)."""
    torch = cx.torch
    import msacl_b200
    from msacl_b200.specs import get_spec
    spec = get_spec(env)
    D, A, n = spec.obs_dim, spec.act_dim, 20
    out = {}
    for B in batches:
        alg = msacl_b200.create_alg(algorithm="msacl", env_name=env, obs_dim=D, act_dim=A, n_step=n, action_low_limit=spec.act_low,
                                    action_high_limit=spec.act_high, q_learning_rate=1e-3, lyapunov_learning_rate=1e-3,
                                    policy_learning_rate=3e-4, alpha_learning_rate=1e-3, lya_diff_scale=10.0, device=cx.dev)
        g = torch.Generator(device=cx.dev).manual_seed(1)
        r = lambda *s: torch.randn(*s, device=cx.dev, generator=g)
        lo, hi = (torch.as_tensor(x, device=cx.dev) for x in (spec.act_low, spec.act_high))
        data = dict(obs=r(B, n, D) * 0.4, act=(lo + (hi - lo) * torch.rand(B, n, A, device=cx.dev, generator=g)) * 0.98,
                    rew=-torch.rand(B, n, device=cx.dev, generator=g) * 50, cost=torch.rand(B, n, device=cx.dev, generator=g),
                    done=(torch.rand(B, n, device=cx.dev, generator=g) < 0.1).float(), logp=r(B, n) - 1.0)
        data["obs2"] = data["obs"] + 0.05 * r(B, n, D)
        for it in range(2, 6):
            alg.model_update(data, it)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); a.record()
        for it in range(6, 6 + iters):
            alg.model_update(data, it)
        b.record(); torch.cuda.synchronize()
        out[f"B{B}"] = {"ms_per_iter": a.elapsed_time(b) / iters, "replay_batch": B, "rows": B * n,
                        "engine": getattr(alg, "engine_name", "torch")}
        del alg, data
        torch.cuda.empty_cache()
    out["reference_cpu_ms_per_iter_B256"] = 440.0      # SURVEY.md section 6 probe (8 vCPU container), for context
    return out


def time_training_loop(cx, env="VanderPol", iters=60):
    """BASELINE config 1: the reference's default training configuration (example/msacl_train.py: env_num 4, n_step 20,
    sample_batch_size 20, replay_batch_size 256) through sampler.sample -> buffer.add_batch -> sample_batch ->
    model_update; wall-clock ms per iteration, host included (this config is latency-bound by design)."""
    torch = cx.torch
    import msacl_b200
    from msacl_b200.specs import get_spec
    spec = get_spec(env)
    kw = dict(env_name=env, obs_dim=spec.obs_dim, act_dim=spec.act_dim, n_step=20, action_low_limit=spec.act_low,
              action_high_limit=spec.act_high, q_learning_rate=1e-3, lyapunov_learning_rate=1e-3, policy_learning_rate=3e-4,
              alpha_learning_rate=1e-3, lya_diff_scale=10.0, env_num=4, env_seed=1, sample_batch_size=20, action_type="continu",
              reward_scale=100.0, cost_scale=100.0, noise_params=None, target_value=0.0, buffer_max_size=100000, device=cx.dev)
    alg = msacl_b200.create_alg(algorithm="msacl", **kw)
    sampler = msacl_b200.create_sampler(**kw)
    buffer = msacl_b200.create_buffer(**kw)
    sampler.networks = alg.networks
    for _ in range(30):                               # fill: 30 x 80 transitions
        buffer.add_batch(sampler.sample()[0])
    for it in range(2, 8):
        buffer.add_batch(sampler.sample()[0])
        alg.model_update(buffer.sample_batch(256), it)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for it in range(8, 8 + iters):
        buffer.add_batch(sampler.sample()[0])
        alg.model_update(buffer.sample_batch(256), it)
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3 / iters
    return {"workload": f"{env} MSACL training, reference default args (env_num 4, n_step 20, sample_batch_size 20, replay 256)",
            "wall_ms_per_iteration": ms, "env_steps_per_iteration": 80, "learner_engine": getattr(alg, "engine_name", "torch")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10,
                    help="timed launches of the headline rollout, of the e2e region and of every rollout in `configs`; the "
                         "target-kernel, learner and training-loop configs time fixed repetition counts of their own")
    ap.add_argument("--warmup", type=int, default=3, help="untimed launches before each timed region (at least 3 for b200)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--env", default="QuadTracking")
    ap.add_argument("--envs-per-gpu", type=int, default=1 << 21)
    ap.add_argument("--inner", type=int, default=16, help="env steps per fused launch")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the `configs` block (other BASELINE configs)")
    ap.add_argument("--replay-batch", type=int, default=256)
    ap.add_argument("--e2e-full-d2h", action="store_true",
                    help="also time a variant that copies EVERY transition of the chunk to pinned host memory")
    ap.add_argument("--engine", default="tc", choices=["tc", "ffma"],
                    help="actor engine: tcgen05 split-bf16 tensor cores (default) or FP32 FFMA")
    ap.add_argument("--settle", type=float, default=0.0,
                    help="seconds of untimed back-to-back launches before the timed `value` region (sustained-clock figure; the burst "
                         "figure is then reported as value_burst)")
    ap.add_argument("--cooldown", type=float, default=2.0,
                    help="idle seconds before the e2e region, so that it starts from the same thermal state as the `value` region")
    ap.add_argument("--exchange", default="side", choices=["side", "main", "none"],
                    help="N>1 e2e diagnosis: all-gather on a side stream (default), on the main stream, or skipped")
    ap.add_argument("--reserve-sms", type=int, default=0, help="N>1 e2e: SMs left free for the side-stream NCCL all-gather")
    ap.add_argument("--replay", default="indexed", choices=["indexed", "ring"],
                    help="e2e replay store: index-based windows over the transition store (default) or the reference-layout ring")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the transitions of the last timed launch (rank 0; a fixed seeded sample of about 48 MB of env "
                         "instances when all of them are more) as DIR/<field>.npy, to compare two builds on identical inputs")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs records the b200 rollout")
    if args.dump_outputs and args.settle > 0:
        ap.error("--dump-outputs needs --settle 0: the number of settling launches, and so the state the timed launches "
                 "start from, depends on timing")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    if args.impl == "reference":
        return run_reference_arm(args)

    import torch
    import torch.distributed as dist

    import msacl_b200  # noqa: F401
    from msacl_b200 import _lib
    from msacl_b200.buffer import B200IndexedReplayBuffer, B200NstepReplayBuffer
    from msacl_b200.sampler import ActorWeights
    from msacl_b200.specs import get_spec
    from msacl_b200 import distributed as mdist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    cx = Ctx()
    cx.torch, cx.dist = torch, dist
    cx.rank = int(os.environ.get("RANK", "0"))
    cx.world = int(os.environ.get("WORLD_SIZE", "1"))
    cx.local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(cx.local)
    if cx.world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", cx.local))
    cx.dev = torch.device("cuda", cx.local)
    cx.stream = torch.cuda.current_stream()
    rank, world, dev, stream = cx.rank, cx.world, cx.dev, cx.stream

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            tt = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return float(tt.item())
        return float(ms)

    cx.barrier, cx.max_over_ranks = barrier, max_over_ranks
    cx.peaks = {}
    try:
        cx.peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    cx.hbm_peak = float(cx.peaks.get("hbm_gbs", 6650.0))
    cx.tensor_peak = float(cx.peaks.get("bf16_tflops_sustained", 1400.0))
    cx.tensor_burst = float(cx.peaks.get("bf16_tflops", 1590.0))
    cx.ncu_traffic = {}
    try:
        cx.ncu_traffic = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
    except Exception:
        pass

    spec = get_spec(args.env)
    n, K, n_step = args.envs_per_gpu, args.inner, 20
    D, A = spec.obs_dim, spec.act_dim

    # ---------------- device-resident throughput (`value`) + dominant-kernel timing
    main_run = time_rollout(cx, args.env, n, K, args.engine, args.steps, args.warmup, keep=True, clocks=True, settle_s=args.settle)
    ro, host_w = main_run["ro"], main_run["host_w"]
    value, total_ms, kern_ms, clk = main_run["value"], main_run["total_ms"], main_run["kern_ms"], main_run["clocks"]
    main_run_burst = main_run["value_burst"]
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in last_launch_outputs(ro, rank * n).items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
    steps_total = n * K * args.steps * world
    h2d_bytes = sum(p.numel() * 4 for p in host_w)

    def upload_actor():
        dw = [p.to(dev, non_blocking=True) for p in host_w]
        return ActorWeights([(dw[0], dw[1]), (dw[2], dw[3]), (dw[4], dw[5])], device=dev)

    # ---------------- end to end through the public API with host buffers
    if args.replay == "indexed":
        # every emitted window stays sampleable for as long as its slices are in the sampler's transition store
        cap = (ro.tr.M - 2) * K * n
        buf = B200IndexedReplayBuffer(obs_dim=D, act_dim=A, buffer_max_size=cap, n_step=n_step, device=dev)
    else:
        cap = 1_000_000
        buf = B200NstepReplayBuffer(obs_dim=D, act_dim=A, buffer_max_size=cap, n_step=n_step, device=dev)
    Bq = args.replay_batch // world if world > 1 else args.replay_batch
    fields = {"obs": (D,), "act": (A,), "rew": (), "cost": (), "obs2": (D,), "done": (), "logp": ()}
    # One packed buffer per rank carries the 7 batch fields + the statistics: the gather kernel writes the sampled windows
    # straight into it, N>1 all-gathers it on a side stream (consumed one step later), and ONE contiguous D2H copy brings
    # the [G, P] result into pinned host memory, where the learner-facing {field: [B, n, .]} dict is a set of views.
    exch = mdist.BatchExchange(fields, Bq, n_step, dev, depth=2 if world > 1 else 1)   # 2: a rank's step never waits for a straggler's
    if args.exchange == "main":
        exch.side = None
    host_packed = [torch.empty(world, exch.P, dtype=torch.float32).pin_memory() for _ in range(2)]
    host_ready = [None, None]
    d2h_bytes = host_packed[0].numel() * 4
    step_no = [0]
    consumed = [0.0]
    e2e_kernel_events = []
    copy_stream = torch.cuda.Stream(dev)

    def e2e_step():
        cur = step_no[0] & 1
        a = upload_actor()                               # H2D: the learner's current policy (pinned host memory)
        kev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
        e2e_kernel_events.append(kev)
        batch = ro.run(a, timing=kev)                    # fused K-step rollout
        buf.add_batch(batch)                             # n-step windows -> device replay store
        sub = buf.sample_batch(Bq, out=exch.views())     # replay batch for the learner, gathered into the packed buffer
        if args.exchange == "none" and world > 1:
            exch.send[0][exch.stats_off:].view(torch.float64).copy_(ro.stats[:8])
            packed = exch.send[0][None].expand(world, -1)
        else:
            packed = exch.exchange(sub, ro.stats[:8], unpack=False)   # N>1: NCCL all-gather on a side stream, previous result back
        # D2H of the replay batch + episode statistics on a copy stream: a copy engine moves it while the next rollout launch
        # already runs (at N = 8 the gathered buffer is 5.2 MB = 0.2 ms of PCIe time that used to sit between two launches)
        ready = torch.cuda.Event()
        ready.record(stream)
        copy_stream.wait_event(ready)
        with torch.cuda.stream(copy_stream):
            host_packed[cur].copy_(packed, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        exch.guard_reuse(ev)
        host_ready[cur] = ev
        # the host (learner side) consumes the batch of the PREVIOUS step while this step's launches are in flight: the
        # learner's data is one iteration stale by design, so the per-step host wait never drains the GPU queue
        prev = host_ready[1 - cur]
        if prev is not None:
            prev.synchronize()
            hb, hs = exch.host_views(host_packed[1 - cur])
            consumed[0] += float(hs[0]) + float(hb["rew"][0, 0])       # touch the data like a consumer would
        step_no[0] += 1

    # Same thermal state for both timed regions: the part runs at its 1 kW power cap and the SM clock of a cool GPU sags by
    # 3-5 % over the first second of back-to-back launches, so an e2e region measured right after the `value` region looked
    # 4 % slower than it is (round 1: e2e/value 0.96 at N = 8; skipping the NCCL exchange entirely changed nothing).
    barrier()
    time.sleep(args.cooldown)
    if world > 1 and args.engine == "tc":
        # the side-stream all-gather needs an SM while the persistent rollout kernel runs: reserve NCCL's CTAs instead of
        # letting them displace rollout CTAs (which stretched every launch by the collective's cross-rank wait: 0.6 ms)
        ro.reserve_sms(args.reserve_sms)
    for _ in range(args.warmup):
        e2e_step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        e2e_step()
    host_ready[(step_no[0] - 1) & 1].synchronize()       # the last step's batch has reached the host inside the timed region
    e1.record(stream)
    barrier()
    ro.reserve_sms(0)
    e2e_ms = max_over_ranks(e0.elapsed_time(e1))
    e2e_kernel_ms = float(np.mean([a_.elapsed_time(b_) for a_, b_ in e2e_kernel_events[-args.steps:]]))
    e2e_value = steps_total / (e2e_ms * 1e-3)
    windows_kept = int(buf.size)

    # ---------------- optional: the same step but with every transition of the chunk copied to the host
    e2e_full = None
    if args.e2e_full_d2h:
        tr = ro.tr
        dev_fields = {k: v[tr.H:] for k, v in tr.fields().items()}
        host_fields = {k: torch.empty(v.shape, dtype=v.dtype).pin_memory() for k, v in dev_fields.items()}
        full_bytes = sum(v.numel() * v.element_size() for v in host_fields.values())

        def full_step():
            a = upload_actor()
            ro.run(a)
            cur = tr.fields()                            # views of the chunk this launch wrote
            for k in host_fields:
                host_fields[k].copy_(cur[k][tr.H:], non_blocking=True)
            stream.synchronize()

        for _ in range(2):
            full_step()
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record(stream)
        for _ in range(args.steps):
            full_step()
        f1.record(stream)
        barrier()
        full_ms = f0.elapsed_time(f1)
        e2e_full = {"value": steps_total / (full_ms * 1e-3), "unit": UNIT, "ms_per_step": full_ms / args.steps,
                    "d2h_bytes_per_step": full_bytes, "what": "rollout + D2H of all K x n transition records (pinned host memory)"}
    del ro, buf, main_run
    torch.cuda.empty_cache()

    # ---------------- roofline of the dominant kernel
    ffma_peak = ffma_probe(cx, 0)
    roofline = rollout_roofline(cx, args.env, n, K, args.engine, kern_ms, ffma_peak)
    if args.engine == "ffma":
        roofline["register_tiled_sgemm_ceiling_tflops"] = ffma_probe(cx, 1)
        roofline["register_tiled_ffma2_ceiling_tflops"] = ffma_probe(cx, 2)

    # ---------------- the other BASELINE configs
    configs = None
    if not args.no_configs:
        configs = {}
        S, W = args.steps, args.warmup

        def rollout_cfg(env, n_c, K_c, engine="tc"):
            r = time_rollout(cx, env, n_c, K_c, engine, S, W)
            rf = rollout_roofline(cx, env, n_c, K_c, engine, r["kern_ms"], ffma_peak)
            return {"env": env, "envs_per_gpu": n_c, "inner_steps": K_c, "engine": engine, "value": r["value"], "unit": UNIT,
                    "ms_per_launch": r["total_ms"] / S, "kernel_ms": r["kern_ms"],
                    "roofline": {k: rf[k] for k in ("bound", "achieved", "peak", "unit", "frac")}, "hbm_frac": rf["hbm"]["frac"]}

        car_n = (1 << 22) // world
        configs["4_singletrackcar_4M_envs_sharded"] = rollout_cfg("SingleTrackCar", car_n, 16)
        configs["4_singletrackcar_4M_envs_sharded"]["total_envs"] = car_n * world
        if world == 1:
            configs["2_pendulum_65536_envs"] = rollout_cfg("Pendulum", 65536, 256)
            configs["2_ductedfan_65536_envs"] = rollout_cfg("DuctedFan", 65536, 256)
            c3 = rollout_cfg("TwoLink", 1 << 20, 16)
            c3["msacl_targets_2^20_windows_n20"] = time_targets(cx)
            try:
                c3["learner_model_update"] = time_learner(cx)
            except Exception as e:      # never lose the headline line to an auxiliary measurement
                c3["learner_model_update"] = {"error": repr(e)}
            configs["3_twolink_1M_envs_msacl_targets"] = c3
            configs["5_quadtracking_fp32_ffma_engine"] = rollout_cfg(args.env, n, K, "ffma" if args.engine == "tc" else "tc")
            try:
                configs["general_engine_twolink_hidden_64x64_tanh"] = time_general_rollout(cx, steps=S, warmup=W)
            except Exception as e:
                configs["general_engine_twolink_hidden_64x64_tanh"] = {"error": repr(e)}
            try:
                configs["1_vanderpol_training_reference_defaults"] = time_training_loop(cx)
            except Exception as e:
                configs["1_vanderpol_training_reference_defaults"] = {"error": repr(e)}

    if rank == 0:
        cpu, cpu_ref = None, None
        if not args.no_cpu_baseline and world == 1:
            cpu = cpu_baseline(args.env)
            if reference_available():
                try:
                    cpu_ref = reference_as_shipped(args.env, calls=2, steps=5)
                except Exception as e:
                    cpu_ref = {"error": repr(e), "kind": "reference"}
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if args.engine == "ffma" else "bf16x3 (split-bf16 tensor-core products, f32 accumulate; f32/f64 dynamics)",
            "data": "synthetic",
            "config": {"workload": f"{args.env} fused rollout (actor MLP + TanhGauss sample + env ODE step + reward/cost + autoreset), "
                                   f"{n} envs/GPU (BASELINE config 5 per-GPU share), {K} env steps per launch, transitions written to HBM",
                       "engine": args.engine, "envs_per_gpu": n, "inner_steps": K, "n_step": n_step, "l2": "inputs larger than L2 (state + transitions per launch >> 126 MB)",
                       "settle_s": args.settle, "cooldown_before_e2e_s": args.cooldown,
                       "parallelism": f"env-sharded x{world}, no step-path collective"},
            "value_burst": main_run_burst, "clocks": clk, "gpu_launches": args.steps,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                    "ms_per_step": e2e_ms / args.steps, "rollout_kernel_ms_inside_e2e": e2e_kernel_ms, "gpu_launches_per_step": 6, "replay": args.replay,
                    "replay_capacity_windows": cap, "replay_windows_resident_after_run": windows_kept,
                    "what": "per step: H2D actor weights (pinned) -> sampler rollout -> buffer.add_batch (device window index scatter) -> "
                            "buffer.sample_batch (n-step gather) -> [one packed NCCL all-gather of the sub-batches + statistics on a side "
                            "stream, consumed one step later, if N>1] -> D2H replay batch + episode stats (pinned, double-buffered: the host reads step t-1's "
                            "batch while step t runs)"},
            "roofline": roofline,
        }
        if configs is not None:
            out["configs"] = configs
        if cpu is not None:
            out["cpu_baseline"] = cpu_ref if (cpu_ref and "value" in cpu_ref) else cpu
            out["cpu_baseline_port"] = cpu
        if e2e_full is not None:
            out["e2e_full_transition_d2h"] = e2e_full
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
