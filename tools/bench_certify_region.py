#!/usr/bin/env python
"""Throughput of the region verifier's interval kernel (cells/s) at default network shapes, and its FFMA rate: algorithmic
FMAs (4 per weight of the 256x256 layers per cell: the V net's two layers at C and at F^m(C), the policy's layer m times)
over CUDA-event kernel time, against msacl_ffma_probe mode 1 (register-tiled FFMA outer product) and mode 8 (the same with
FFMA.RM / FFMA.RP) measured in the same run.  Writes one JSON line per configuration, preceded by the card's name and
power limit, to --out (default profiles/r4_certify_region_bench.jsonl) and stdout.

With --robust every env is also timed under bounded disturbances (all three sets nonzero: sensor noise, an actuator bias,
process noise), alternating robust and nominal launches on the same cells in the same process, and each robust line gives
its cells/s over the nominal one (default --out profiles/r5_certify_region_robust_bench.jsonl).

    python tools/bench_certify_region.py [--out FILE] [--cells 1048576] [--repeats 5] [--robust]
"""
import argparse
import ctypes as C
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

import msacl_b200  # noqa: E402
from msacl_b200 import _lib  # noqa: E402
from msacl_b200.algorithm import ApproxContainer  # noqa: E402
from msacl_b200.specs import get_spec  # noqa: E402

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from bench_certify import card  # noqa: E402

HID = 256


def probe_fma_rate(mode, iters=20000):
    """FMAs/s of msacl_ffma_probe `mode` (FLOPs / 2)."""
    lib = _lib.load()
    sink = torch.ones(128, dtype=torch.float32, device="cuda")
    fl = C.c_double(0)
    _lib.check(lib.msacl_ffma_probe(mode, iters, sink.data_ptr(), C.byref(fl), _lib.current_stream()))
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    _lib.check(lib.msacl_ffma_probe(mode, iters, sink.data_ptr(), C.byref(fl), _lib.current_stream()))
    b.record()
    torch.cuda.synchronize()
    return fl.value / 2 / (a.elapsed_time(b) * 1e-3)


def setup(name, n, steps, robust=False):
    """Nominal verifier (and, with robust, one under disturbances) of default networks, the packed image and n cells of width
    2e-3 of the box."""
    s = get_spec(name)
    torch.manual_seed(0)
    nets = ApproxContainer(obs_dim=s.obs_dim, act_dim=s.act_dim, action_low_limit=s.act_low, action_high_limit=s.act_high,
                           q_learning_rate=1e-3, lyapunov_learning_rate=1e-3, policy_learning_rate=3e-4,
                           alpha_learning_rate=1e-3).cuda()
    lo0, hi0 = s.obs_low * 0.25, s.obs_high * 0.25
    kw = dict(networks=nets, env_name=name, box=(lo0, hi0), steps=steps)
    vers = [msacl_b200.create_region_certifier(**kw)]
    if robust:
        ar = s.act_high - s.act_low
        vers.append(msacl_b200.create_region_certifier(**kw, disturbance=dict(obs=1e-3 * (hi0 - lo0), act=(0.01 * ar, 0.02 * ar),
                                                                               state=1e-3 * (hi0 - lo0))))
    g = torch.Generator(device="cuda").manual_seed(0)
    lo0t, span = torch.as_tensor(lo0, device="cuda"), torch.as_tensor(hi0 - lo0, device="cuda")
    c = lo0t + span * torch.rand(n, s.obs_dim, device="cuda", generator=g)
    w = span * 1e-3
    lo, hi = (c - w).contiguous(), (c + w).contiguous()
    image = vers[0].pack()
    for v in vers:
        v.evaluate(lo, hi, image)                     # warm-up (module load, smem attribute)
    return vers, lo, hi, image


def time_eval(ver, lo, hi, image):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    ver.evaluate(lo, hi, image)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e-3


def bench(name, n, steps, repeats, robust=False):
    """One record per verifier (nominal first); with robust, the two are timed alternately."""
    vers, lo, hi, image = setup(name, n, steps, robust)
    times = [[] for _ in vers]
    for _ in range(repeats):
        for v, t in zip(vers, times):
            t.append(time_eval(v, lo, hi, image))
    fmas = 4.0 * HID * HID * (4 + steps) * n
    out = []
    for v, t in zip(vers, times):
        r = dict(env=name, cells=n, steps=steps, seconds=min(t), seconds_all=t, cells_per_s=n / min(t), fma_per_s=fmas / min(t))
        if v.disturbance is not None:
            r["disturbance"] = {k: [lo_.tolist(), hi_.tolist()] for k, (lo_, hi_) in v.disturbance.items()}
            r["over_nominal"] = r["cells_per_s"] / out[0]["cells_per_s"]
        out.append(r)
    return out


def main(argv=None):
    p = argparse.ArgumentParser()
    p.add_argument("--out")
    p.add_argument("--cells", type=int, default=1 << 20)
    p.add_argument("--repeats", type=int, default=5)
    p.add_argument("--robust", action="store_true", help="also time the verifier under disturbances against the nominal one")
    a = p.parse_args(argv)
    a.out = a.out or os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                  "r5_certify_region_robust_bench.jsonl" if a.robust else "r4_certify_region_bench.jsonl")
    lines = [{"card": card()}]
    ffma, rmrp = probe_fma_rate(1), probe_fma_rate(8)
    lines.append({"ffma_probe_mode1_fma_per_s": ffma, "ffma_probe_mode8_rm_rp_fma_per_s": rmrp, "mode8_over_mode1": rmrp / ffma})
    for name in ("VanderPol", "TwoLink"):
        for r in bench(name, a.cells, 1, a.repeats, a.robust):
            r["of_ffma_probe"] = r["fma_per_s"] / ffma
            r["of_rm_rp_probe"] = r["fma_per_s"] / rmrp
            lines.append(r)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        for ln in lines:
            fh.write(json.dumps(ln) + "\n")
            print(json.dumps(ln), flush=True)


if __name__ == "__main__":
    main()
