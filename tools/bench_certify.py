#!/usr/bin/env python
"""Throughput of the Lyapunov-certificate verifier (state-steps/s) and the split of its time into the greedy rollout, the V
GEMMs and the check kernels, measured with CUDA events; the check kernels' share of HBM bandwidth is their algorithmic bytes
(4 D + 4 + 1 per state-step, plus the per-state records) over their time, against a device-to-device copy measured in the
same run.  One JSON line per configuration, preceded by the card's name and power limit.

    python tools/bench_certify.py [--out FILE] [--repeats 3]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

import msacl_b200  # noqa: E402
from msacl_b200.algorithm import ApproxContainer  # noqa: E402
from msacl_b200.specs import get_spec  # noqa: E402

CONFIGS = [("QuadTracking", 1 << 21, 20), ("VanderPol", 1 << 22, 20)]
RECORD_BYTES = 4 + 8 + 1 + 4 + 4 + 4 + 8        # v0, s0, flags, first_violation, first_decrease, end_step, worst_ratio


class EventTimer:
    def __init__(self):
        self.pairs = {}

    def __call__(self, name):
        timer = self

        class _Section:
            def __enter__(self):
                self.a, self.b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                self.a.record()

            def __exit__(self, *exc):
                self.b.record()
                timer.pairs.setdefault(name, []).append((self.a, self.b))
        return _Section()

    def ms(self):
        torch.cuda.synchronize()
        return {k: sum(a.elapsed_time(b) for a, b in v) for k, v in self.pairs.items()}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def copy_peak_gbs(nbytes=4 << 30, reps=10):
    src = torch.empty(nbytes // 4, dtype=torch.float32, device="cuda").fill_(1.0)
    dst = torch.empty_like(src)
    dst.copy_(src)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        dst.copy_(src)
    b.record()
    torch.cuda.synchronize()
    return 2 * nbytes * reps / (a.elapsed_time(b) * 1e-3) / 1e9


def networks(env_name):
    spec = get_spec(env_name)
    torch.manual_seed(0)
    return ApproxContainer(obs_dim=spec.obs_dim, act_dim=spec.act_dim, action_low_limit=spec.act_low, action_high_limit=spec.act_high,
                           lyapunov_output_dim=256, q_learning_rate=1e-3, lyapunov_learning_rate=1e-3, policy_learning_rate=3e-4,
                           alpha_learning_rate=1e-3).cuda()


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--out")
    p.add_argument("--repeats", type=int, default=3)
    a = p.parse_args()
    lines = [{"card": card(), "copy_peak_GBps": round(copy_peak_gbs(), 1)}]
    print(json.dumps(lines[0]), flush=True)
    peak = lines[0]["copy_peak_GBps"]
    for name, N, T in CONFIGS:
        nets = networks(name)
        D = get_spec(name).obs_dim
        msacl_b200.create_certifier(networks=nets, env_name=name, num_states=N, horizon=T).run()        # warm-up: every shape
        for rep in range(a.repeats):
            timer = EventTimer()
            ver = msacl_b200.create_certifier(networks=nets, env_name=name, num_states=N, horizon=T, timer=timer)
            start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            start.record()
            report = ver.run()
            end.record()
            ms = timer.ms()
            total = start.elapsed_time(end)
            visited = int(ver.records["end_step"].long().sum())          # state-steps actually checked (k = 1..e)
            check_bytes = visited * (4 * D + 4 + 1) + N * (4 * D + 4) + 2 * N * RECORD_BYTES * (-(-T // ver.chunk))
            rec = {"env": name, "states": N, "horizon": T, "chunk_steps": ver.chunk, "repeat": rep,
                   "state_steps_per_s": N * T / (total * 1e-3), "total_ms": round(total, 2),
                   "rollout_ms": round(ms.get("rollout", 0.0), 2), "lyapunov_ms": round(ms.get("lyapunov", 0.0), 2),
                   "check_ms": round(ms.get("check", 0.0), 3),
                   "check_GBps": round(check_bytes / (ms["check"] * 1e-3) / 1e9, 1),
                   "check_fraction_of_copy_peak": round(check_bytes / (ms["check"] * 1e-3) / 1e9 / peak, 3),
                   "certified": report.certified, "escaped": report.escaped, "decrease": report.decrease}
            lines.append(rec)
            print(json.dumps(rec), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write("\n".join(json.dumps(r) for r in lines) + "\n")


if __name__ == "__main__":
    main()
