"""Lyapunov-certificate verifier: closed-loop checks of boundedness and exponential decrease over many initial states.

MSACL trains a controller together with a Lyapunov certificate V(o) = sum_j z_j(o)^2 (`networks.lyapunov`).  This module
answers, for a trained ApproxContainer, the two questions a user asks of such a certificate:

  1. does alpha1 |o|^2 <= V(o) <= alpha2 |o|^2 hold on the states of interest, and
  2. does V decay at least like (1 - eta)^k along the greedy closed loop, and from which sublevel set {V < c*} does it hold?

It is a SAMPLING-BASED EMPIRICAL CHECK over the sampled initial states and the horizon T, not a formal proof: a state that
passes was only observed to satisfy the conditions along its own T-step trajectory.

For every initial state the greedy closed loop (mode() actions, as the evaluator) runs for up to T steps on the fused rollout
kernels; a trajectory stops at its first `done` (the env's time limit is set above T, so `done` means the state left the
env's domain) and that final observation is checked too.  V is evaluated on every visited observation with the split-bf16
tcgen05 GEMMs (`FusedMLP(..., sumsq_head=True)`), and csrc/certify.cu checks, per state and visited step k, with
s_k = sum_j o_k[j]^2 and c_k = (1 - eta)^k in float64:

  NONFINITE       some component of o_k or V_k is NaN / Inf
  BOUND_LO        V_k < alpha1 s_k - v_atol             BOUND_HI  V_k > alpha2 s_k + v_atol
  DECREASE        k >= 1 and V_k > c_k V_0 + v_atol      ESCAPED   a `done` occurred at some step <= T
  NOT_EXP_STABLE  k >= 1 and s_k > (alpha2 / alpha1) c_k s_0  (model-free: the squared exponential-stability label)

A state is certified when it has none of the first five flags.  The report (`CertificateReport`) counts every flag, the
certified states and the states where DECREASE and NOT_EXP_STABLE disagree (does V's decay predict the true decay?), gives a
histogram of the step of the first DECREASE, c* = min V_0 over the uncertified states and roa_count = #{i : V_0,i < c*}.
With init=("box", lo, hi) roa_fraction = roa_count / N estimates the fraction of the box covered by the sampled sublevel set
{V < c*}.

With torch.distributed initialised the N states are sharded over the ranks (global state ids key the resets and the box
draws, so the result does not depend on the number of GPUs) and the reports are combined (`distributed.combine_certificate`).
The actor is packed from the policy's CURRENT parameters on every `run()`.
"""
import contextlib
import ctypes as C
import json
import math
import warnings
from dataclasses import asdict, dataclass

import numpy as np
import torch
import torch.distributed as dist

from . import _lib
from . import distributed as mdist
from .sampler import FusedRollout, actor_from_policy
from .specs import get_spec

FLAG_NAMES = ("nonfinite", "bound_lo", "bound_hi", "decrease", "escaped", "not_exp_stable")
FLAG_BITS = {name: 1 << b for b, name in enumerate(FLAG_NAMES)}
SUM_HIST = 11                    # MSACL_CERT_SUM_HIST: summary = [11 counters / keys] + [horizon] histogram
MAX_HORIZON = 8192               # MSACL_CERT_MAX_HORIZON


@dataclass
class CertificateReport:
    """Summary of one verifier run (all N states, every rank combined)."""
    env_name: str
    num_states: int
    horizon: int
    init: str
    lya_eta: float
    alpha1: float
    alpha2: float
    v_atol: float
    nonfinite: int
    bound_lo: int
    bound_hi: int
    decrease: int
    escaped: int
    not_exp_stable: int
    certified: int
    inconsistent: int                 # states where DECREASE and NOT_EXP_STABLE disagree
    first_decrease_hist: list         # [horizon]: entry k - 1 = states whose first DECREASE is at step k
    c_star: float                     # min V_0 over uncertified states (+inf if every state is certified)
    roa_count: int                    # #{i : V_0,i < c_star}
    roa_fraction: float

    def to_json(self):
        d = asdict(self)
        d["c_star"] = d["c_star"] if math.isfinite(d["c_star"]) else str(d["c_star"])
        return json.dumps(d)


def decay_table(horizon, lya_eta):
    """c_0 = 1, c_k = c_{k-1} (1 - eta) in float64, by repeated multiplication (bit-identical wherever it is restated)."""
    c = [1.0]
    base = 1.0 - float(lya_eta)
    for _ in range(horizon):
        c.append(c[-1] * base)
    return c


class TrajectoryChecker:
    """Per-state records and the check kernels of csrc/certify.cu for n states (one shard): `begin` with the initial
    observations and V_0, `steps` once per chunk of visited observations (transition-store layout), `finish` for the
    summary.  Works on any trajectories, not only the verifier's own rollouts."""

    def __init__(self, n, obs_dim, horizon, lya_eta=0.15, alpha1=1.0, alpha2=2.0, v_atol=0.0, device="cuda"):
        self.n, self.D, self.T = int(n), int(obs_dim), int(horizon)
        self.device = torch.device(device)
        e = lambda dt: torch.empty(self.n, dtype=dt, device=self.device)
        self.rec = dict(v0=e(torch.float32), s0=e(torch.float64), flags=e(torch.uint8), first_violation=e(torch.int32),
                        first_decrease=e(torch.int32), end_step=e(torch.int32), worst_ratio=e(torch.float64))
        self.rdesc = _lib.CertRecords(**{k: v.data_ptr() for k, v in self.rec.items()})
        self.decay = torch.tensor(decay_table(self.T, lya_eta), dtype=torch.float64, device=self.device)
        self.params = _lib.CertParams(horizon=self.T, alpha1=float(alpha1), alpha2=float(alpha2), v_atol=float(v_atol),
                                      decay=self.decay.data_ptr())
        self.lib = _lib.load()

    def begin(self, obs0, v0):
        """obs0 [n, D], v0 [n] float32 CUDA (contiguous)."""
        _lib.check(self.lib.msacl_certify_begin(self.n, self.D, _lib.ptr(obs0), _lib.ptr(v0), C.byref(self.params),
                                                C.byref(self.rdesc), _lib.current_stream()))

    def steps(self, k0, obs2, V, done):
        """Visited steps k0 .. k0 + K - 1: obs2 [K, n, D], V [K, n] float32, done [K, n] uint8 (steps beyond the horizon
        are ignored)."""
        _lib.check(self.lib.msacl_certify_steps(self.n, self.D, int(obs2.shape[0]), int(k0), _lib.ptr(obs2), _lib.ptr(V),
                                                _lib.ptr(done), C.byref(self.params), C.byref(self.rdesc), _lib.current_stream()))

    def finish(self, summary=None):
        """int64 [SUM_HIST + horizon] summary of this shard (layout MSACL_CERT_SUM_* of include/msacl_b200.h)."""
        if summary is None:
            summary = torch.zeros(SUM_HIST + self.T, dtype=torch.int64, device=self.device)
        _lib.check(self.lib.msacl_certify_finish(self.n, self.T, C.byref(self.rdesc), summary.data_ptr(), _lib.current_stream()))
        return summary

    def count_below(self, c_star, summary):
        """#{i : V_0,i < c_star} of this shard (written to summary[MSACL_CERT_SUM_ROA] and returned)."""
        _lib.check(self.lib.msacl_certify_roa(self.n, self.rec["v0"].data_ptr(), float(c_star), summary.data_ptr(),
                                              _lib.current_stream()))
        return int(summary[mdist.CERT_ROA].item())

    def records(self):
        """The per-state records (device tensors); worst_ratio as float32."""
        return {**self.rec, "worst_ratio": self.rec["worst_ratio"].float()}


class B200CertificateVerifier:
    """B200CertificateVerifier(networks=..., env_name=..., num_states=N, horizon=T, ...).run() -> CertificateReport.

    kwargs: networks (ApproxContainer: `.policy` and `.lyapunov` are used), env_name, num_states, horizon (default n_step or
    20), lya_eta (0.15), alpha1 (1), alpha2 (2), v_atol (0), seed (0), init ("reset" or ("box", lo, hi): uniform per
    observation dimension, box envs only, inside the observation bounds), rollout_engine ("tc"; a policy the fused kernels
    do not hold runs on the general engine), chunk_steps (rollout steps per launch, default min(T, 10)), precision (6: bf16x6
    GEMMs for V), workspace_bytes (cap of the V GEMM activations, default 2 GiB), distributed (True), device ("cuda"),
    trace (optional callable(k0, obs [K, n, D], V [K, n], done [K, n] or None) called with device views of every visited
    chunk, k0 = 0 for the initial states; for tests and inspection), timer (optional callable(name) -> context manager
    around the "rollout", "lyapunov" and "check" phases, e.g. CUDA event pairs; for benchmarks).

    After run(), `records` holds this rank's per-state records (device tensors: v0, s0, flags, first_violation,
    first_decrease, end_step, worst_ratio)."""

    def __init__(self, **kwargs):
        self.networks = kwargs["networks"]
        self.env_name = kwargs["env_name"]
        self.spec = get_spec(self.env_name)
        self.num_states = int(kwargs["num_states"])
        horizon = kwargs.get("horizon", kwargs.get("n_step"))
        self.horizon = 20 if horizon is None else int(horizon)
        self.lya_eta = float(kwargs.get("lya_eta", 0.15))
        self.alpha1, self.alpha2 = float(kwargs.get("alpha1", 1.0)), float(kwargs.get("alpha2", 2.0))
        self.v_atol = float(kwargs.get("v_atol", 0.0))
        self.seed = int(kwargs.get("seed") or 0)
        self.engine = kwargs.get("rollout_engine", "tc")
        self.chunk = int(kwargs.get("chunk_steps") or min(self.horizon, 10))
        self.precision = int(kwargs.get("precision", 6))
        self.workspace_bytes = int(kwargs.get("workspace_bytes", 2 << 30))
        self.distributed = bool(kwargs.get("distributed", True))
        self.device = torch.device(kwargs.get("device", "cuda"))
        self.trace = kwargs.get("trace")
        self.timer = kwargs.get("timer") or (lambda name: contextlib.nullcontext())
        self.records = None
        if self.num_states < 1:
            raise ValueError("num_states must be >= 1")
        if not 1 <= self.horizon <= MAX_HORIZON:
            raise ValueError(f"horizon must be in [1, {MAX_HORIZON}]")
        if self.chunk < 1:
            raise ValueError("chunk_steps must be >= 1")
        if not 0.0 <= self.lya_eta < 1.0:
            raise ValueError("lya_eta must be in [0, 1)")
        if not (self.alpha1 > 0 and self.alpha2 > 0 and math.isfinite(self.alpha1) and math.isfinite(self.alpha2)):
            raise ValueError("alpha1 and alpha2 must be positive and finite")
        if not (self.v_atol >= 0 and math.isfinite(self.v_atol)):
            raise ValueError("v_atol must be >= 0 and finite")
        self.box = self._parse_init(kwargs.get("init", "reset"))

    def _parse_init(self, init):
        if isinstance(init, str) and init == "reset":
            return None
        if not (isinstance(init, (tuple, list)) and len(init) == 3 and init[0] == "box"):
            raise ValueError('init must be "reset" or ("box", lo, hi)')
        if self.env_name == "QuadTracking":
            raise ValueError("init=('box', ...) needs an env whose state is its observation; QuadTracking's is not")
        D = self.spec.obs_dim
        lo = np.broadcast_to(np.asarray(init[1], np.float32), (D,)).copy()
        hi = np.broadcast_to(np.asarray(init[2], np.float32), (D,)).copy()
        if not (np.all(np.isfinite(lo)) and np.all(np.isfinite(hi)) and np.all(lo <= hi)):
            raise ValueError("box: need finite lo <= hi")
        if np.any(lo < self.spec.obs_low) or np.any(hi > self.spec.obs_high):
            raise ValueError(f"box [{lo.tolist()}, {hi.tolist()}] is not inside the observation bounds of {self.env_name} "
                             f"[{self.spec.obs_low.tolist()}, {self.spec.obs_high.tolist()}]")
        return lo, hi

    # ---- V = networks.lyapunov on [rows, D] row blocks
    def _lyapunov_fn(self, max_rows):
        lya = self.networks.lyapunov
        dev = self.device
        try:
            from .learner import FusedMLP
            mlp = FusedMLP(lya.lya, dev, precision=self.precision, sumsq_head=True)
        except ValueError as e:
            warnings.warn(f"certificate verifier: the fused GEMMs do not take this Lyapunov network ({e}); evaluating "
                          "networks.lyapunov with PyTorch")
            rb = max(1, min(max_rows, self.workspace_bytes // (4 * 3 * 256)))

            def torch_fn(x, out):
                with torch.no_grad():
                    for r0 in range(0, x.shape[0], rb):
                        out[r0:r0 + rb].copy_(lya(x[r0:r0 + rb]))
            return torch_fn
        per_row = 4 * (mlp.h1 + mlp.h2 + mlp.dout)
        rb = min(max_rows, max(128, self.workspace_bytes // per_row // 128 * 128))
        ws = mlp.workspace("certify", rb, sumsq=True)
        pad = []

        def fused_fn(x, out):
            rows = x.shape[0]
            for r0 in range(0, rows, rb):
                r1 = min(rows, r0 + rb)
                xs = x[r0:r1]
                if r1 - r0 < rb:            # one workspace for every call: a short block is padded to rb rows
                    if not pad:
                        pad.append(torch.zeros(rb, mlp.din, dtype=torch.float32, device=dev))
                    pad[0][:r1 - r0].copy_(xs)
                    xs = pad[0]
                mlp.forward(xs, ws)
                out[r0:r1].copy_(ws.v[:r1 - r0])
        return fused_fn

    def _run_shard(self, lo, n, summary):
        lib, dev, spec = _lib.load(), self.device, self.spec
        D, T, K = spec.obs_dim, self.horizon, min(self.chunk, self.horizon)
        actor = actor_from_policy(self.networks.policy, device=dev)       # packed from the current parameters, every run
        ro = FusedRollout(self.env_name, n, K, n_step=1, seed=self.seed, env_base=lo, device=dev, max_step=T + 1,
                          engine=self.engine, history_chunks=1)
        ro.state.reset()
        if self.box is not None:
            blo, bhi = self.box
            _lib.check(lib.msacl_certify_box_init(C.byref(ro.state.desc), blo.ctypes.data_as(_lib.c_f32p),
                                                  bhi.ctypes.data_as(_lib.c_f32p), _lib.current_stream()))
        chk = TrajectoryChecker(n, D, T, self.lya_eta, self.alpha1, self.alpha2, self.v_atol, dev)
        lya = self._lyapunov_fn(K * n)
        obs0, v0 = ro.state.obs, chk.rec["v0"]
        with self.timer("lyapunov"):
            lya(obs0, v0)
        if self.trace is not None:
            self.trace(0, obs0[None], v0[None], None)
        with self.timer("check"):
            chk.begin(obs0, v0)
        V = torch.empty(K, n, dtype=torch.float32, device=dev)
        for k0 in range(1, T + 1, K):
            with self.timer("rollout"):
                ro.run(actor, deterministic=True)
            tr = ro.tr
            kv = min(K, T - k0 + 1)
            obs2, done = tr.obs2[tr.H:tr.H + kv], tr.done[tr.H:tr.H + kv]
            with self.timer("lyapunov"):
                lya(obs2.reshape(kv * n, D), V[:kv].view(-1))
            if self.trace is not None:
                self.trace(k0, obs2, V[:kv], done)
            with self.timer("check"):
                chk.steps(k0, obs2, V[:kv], done)
        with self.timer("check"):
            chk.finish(summary)
        return chk

    def run(self) -> CertificateReport:
        N, T, dev = self.num_states, self.horizon, self.device
        lo, hi = 0, N
        if self.distributed and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            lo, hi = mdist.shard_env_range(N, dist.get_rank(), dist.get_world_size())
        n = hi - lo
        summary = torch.zeros(SUM_HIST + T, dtype=torch.int64, device=dev)
        chk = None
        if n > 0:
            chk = self._run_shard(lo, n, summary)
        else:                              # a rank without states still takes part in the collectives
            summary[mdist.CERT_CSTAR_KEY] = mdist.float_order_key(math.inf)
        total, c_star = mdist.combine_certificate(summary, lambda c: chk.count_below(c, summary) if chk is not None else 0)
        self.records = chk.records() if chk is not None else None
        s = total.cpu().tolist()
        init = "reset" if self.box is None else f"box({self.box[0].tolist()}, {self.box[1].tolist()})"
        return CertificateReport(env_name=self.env_name, num_states=N, horizon=T, init=init, lya_eta=self.lya_eta,
                                 alpha1=self.alpha1, alpha2=self.alpha2, v_atol=self.v_atol,
                                 **{name: int(s[1 + b]) for b, name in enumerate(FLAG_NAMES)},
                                 certified=int(s[7]), inconsistent=int(s[8]), first_decrease_hist=[int(x) for x in s[SUM_HIST:]],
                                 c_star=float(c_star), roa_count=int(s[mdist.CERT_ROA]), roa_fraction=s[mdist.CERT_ROA] / N)
