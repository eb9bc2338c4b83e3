"""Sound region verifier of the Lyapunov certificate: interval branch-and-bound over state boxes on the GPU.

The empirical verifier (`certify.py`) checks sampled states.  This module answers the question sampling cannot: does the
certificate condition hold for EVERY state of a region, and which sublevel set is then provably a region of attraction?

For an env, a box X0 inside the observation bounds, an inner box B (around the origin), eta, alpha1, alpha2 and m >= 1
closed-loop steps, the verifier partitions X0 \\ B into cells and proves, per cell C, with outward-rounded interval
arithmetic (csrc/certify_region.cu):

  DECREASE ok   sup V(F^m(C)) <= (1 - eta)^m inf V(C)
  ESCAPED ok    F^j(C) lies strictly inside the env's observation bounds for j = 1..m, so the env cannot terminate
  BOUND ok      alpha1 sup |x|^2 <= inf V(C) and sup V(C) <= alpha2 inf |x|^2 over C (sufficient for alpha1 |x|^2 <= V <= alpha2 |x|^2)
  NONFINITE     some bound overflowed or is NaN; the cell is then never "verified"

A cell is verified when DECREASE and ESCAPED are proven and it is not NONFINITE.  F is one greedy closed-loop step: the
policy mean mu, a = half tanh(mu) + mid, the clip to the action box, then the env's CONTROL_STEP explicit-Euler sub-steps.

THE VERIFIED OBJECT IS THE REAL-ARITHMETIC CLOSED LOOP.  The networks are exact real functions of their stored float32
parameters, sin / cos / tanh are exact, and the Euler map is evaluated in exact arithmetic with the env's constants (the
float32 values of env_dynamics.cuh, float64 in TwoLink's solve) read as exact reals.  The verifier does not model the rounding
of any particular implementation, such as the split-bf16 rollout GEMMs or the float32 env kernels.

Cells are dyadic: depth t bisects dimension t mod D (the widest one scaled by the box width); B is snapped outward to the
dyadic grid of 2^(max_depth // D) cells per dimension, and cells entirely inside the snapped B ("inner" cells) are checked for
c_in instead of DECREASE.  A failing cell's centre c is evaluated as the degenerate interval [c, c]: if inf V(F^m(c)) >
(1 - eta)^m sup V(c), or some F^j(c) provably leaves the observation box, c is a proven counterexample and the cell is
"refuted" (not split).  Other failing cells are split up to max_depth ("undecided" there).

From the cells the report derives one sound statement.  c_sound is the least inf V(C) over cells outside B that are not
verified, or whose image F^m(C) is not proven to stay inside X0 (the sublevel set must be a subset of X0; the BOUND condition
does not count).  If every inner cell maps into X0 without leaving the observation box and c_in = sup V(F^m(inner cells)) <
c_sound, then S = {x in X0 : V(x) < c_sound} is forward invariant under F^m, and the F^m-trajectories from S reach
{V <= max(c_in, sup V(inner cells))} in finitely many steps (eta > 0).  Otherwise c_sound is reported as "none".

The frontier is a stack of at most max_cells cells, processed depth-first in chunks.  The actor and V net are packed from
the CURRENT parameters on every `run()`.

BOUNDED DISTURBANCES (`disturbance=dict(obs=..., act=..., state=...)`).  One disturbed closed-loop step is

  F_d(x) = Phi(x, clip(half tanh(mu(x + n)) + mid) + u) + w,   n in N, u in U, w in W

with Phi the CONTROL_STEP Euler map: n is sensor noise that only the policy sees (V is evaluated at the true state), u an
actuator disturbance added after the clip (not re-clipped, held over the sub-steps), w a process disturbance added once after
the sub-steps.  N, U, W are boxes, possibly asymmetric and not containing 0 (a constant bias), and each of the m steps takes
its own (n, u, w).  Every condition -- DECREASE, ESCAPED, LEAVES, the inner-cell conditions, c_in -- then holds for EVERY
admissible disturbance sequence, and the invariance statement becomes robust invariance of S plus the ultimate bound
{V <= reach_level} (practical stability).  A counterexample is still the centre [c, c] with the sets as intervals: its
violation holds for every sequence, and its margin is the least violation over them.  With all sets {0} the verifier is the
nominal one, bit for bit.
"""
import ctypes as C
import json
import math
from dataclasses import asdict, dataclass, field
from fractions import Fraction

import numpy as np
import torch

from . import _lib
from .distributed import float_from_order_key, float_order_key
from .specs import get_spec

SUPPORTED = ("VanderPol", "Pendulum", "DuctedFan", "TwoLink")
HIDDEN = 256                 # MSACL_REGION_HIDDEN
MAX_DEPTH = 50               # MSACL_REGION_MAX_DEPTH
FLAG_NAMES = ("nonfinite", "decrease", "escaped", "bound", "leaves")
FLAGS = {"nonfinite": 1, "decrease": 2, "escaped": 4, "bound": 8, "leaves": 16, "refute_decrease": 32, "refute_escaped": 64}
STATUS = ("split", "verified", "refuted", "undecided", "inner")
ST = dict(verified=0, refuted=1, undecided=2, inner=3, split=4, evaluated=5, probed=6, flags=7, volume=12, c_sound=16, c_in=17,
          v_inner=18, inner_fail=19, count=20)          # MSACL_REGION_ST_* of include/msacl_b200.h
VOLUME_UNIT = 2.0 ** -MAX_DEPTH


def decay_bounds(lya_eta, steps):
    """(1 - eta)^m rounded down and up to float64 (exact rational arithmetic)."""
    exact = (1 - Fraction(float(lya_eta))) ** int(steps)
    f = float(exact)
    lo = f if Fraction(f) <= exact else math.nextafter(f, -math.inf)
    hi = f if Fraction(f) >= exact else math.nextafter(f, math.inf)
    return lo, hi


def _round_out(x, down):
    f = float(x)
    if down and Fraction(f) > x:
        return math.nextafter(f, -math.inf)
    if not down and Fraction(f) < x:
        return math.nextafter(f, math.inf)
    return f


def snap_inner(x0_lo, x0_hi, b_lo, b_hi, level):
    """B snapped outward to the grid of 2^level cells per dimension of X0: integer grid bounds and the box (rounded out)."""
    glo, ghi, blo, bhi = [], [], [], []
    for xl, xh, l, h in zip(x0_lo, x0_hi, b_lo, b_hi):
        xl, w = Fraction(float(xl)), Fraction(float(xh)) - Fraction(float(xl))
        i0 = math.floor((Fraction(float(l)) - xl) / w * 2 ** level)
        i1 = math.ceil((Fraction(float(h)) - xl) / w * 2 ** level)
        i0, i1 = max(0, i0), min(2 ** level, i1)
        glo.append(i0); ghi.append(i1)
        blo.append(_round_out(xl + w * i0 / 2 ** level, True))
        bhi.append(_round_out(xl + w * i1 / 2 ** level, False))
    return glo, ghi, blo, bhi


@dataclass
class RegionReport:
    """Result of one region verification (fractions are of the volume of X0)."""
    env_name: str
    box: list
    inner: list                   # B snapped outward to the cell grid
    steps: int
    lya_eta: float
    alpha1: float
    alpha2: float
    max_depth: int
    verified: int
    refuted: int
    undecided: int
    inner_cells: int
    verified_fraction: float
    refuted_fraction: float
    undecided_fraction: float
    inner_fraction: float
    verified_fraction_outside: float     # of X0 \ (inner cells)
    failed: dict                  # leaf cells outside B with each condition not proven (nonfinite, decrease, escaped, bound, leaves)
    c_sound: object               # float, or "none" when the invariance statement was not proven
    c_sound_candidate: float      # least inf V over cells outside B that are not verified or may leave X0 (+inf if none)
    c_in: float                   # sup V(F^m(C)) over inner cells (-inf if none)
    v_inner: float                # sup V(C) over inner cells
    inner_failed: int             # inner cells that may leave X0 or the observation box, or are nonfinite
    invariant: bool               # {x in X0 : V(x) < c_sound} is forward invariant under F^m
    reach_level: object           # max(c_in, v_inner): trajectories from the invariant set reach {V <= reach_level}
    counterexamples: list = field(default_factory=list)   # {"x", "kind": "decrease" | "escaped", "margin"}
    rounds: int = 0
    evaluated: int = 0

    def to_json(self):
        d = asdict(self)
        for k, v in d.items():
            if isinstance(v, float) and not math.isfinite(v):
                d[k] = str(v)
        return json.dumps(d)

    @classmethod
    def from_stats(cls, stats, examples, **meta):
        """Derive the report from the MSACL_REGION_ST_* statistics (a sequence of ints) and the counterexample rows."""
        s = [int(v) for v in stats]
        vol = [s[ST["volume"] + j] * VOLUME_UNIT for j in range(4)]
        c_cand = float_from_order_key(s[ST["c_sound"]])
        c_in = float_from_order_key(s[ST["c_in"]])
        v_inner = float_from_order_key(s[ST["v_inner"]])
        inner = s[ST["inner"]]
        eta = float(meta["lya_eta"])
        invariant = s[ST["inner_fail"]] == 0 and c_in < c_cand and c_cand > 0 and eta > 0 and inner > 0
        outside = 1.0 - vol[3]
        return cls(**meta, verified=s[ST["verified"]], refuted=s[ST["refuted"]], undecided=s[ST["undecided"]], inner_cells=inner,
                   verified_fraction=vol[0], refuted_fraction=vol[1], undecided_fraction=vol[2], inner_fraction=vol[3],
                   verified_fraction_outside=vol[0] / outside if outside > 0 else 1.0,
                   failed={n: s[ST["flags"] + b] for b, n in enumerate(FLAG_NAMES)},
                   c_sound=c_cand if invariant else "none", c_sound_candidate=c_cand, c_in=c_in, v_inner=v_inner,
                   inner_failed=s[ST["inner_fail"]], invariant=invariant,
                   reach_level=max(c_in, v_inner) if invariant else None, counterexamples=examples)


@dataclass
class RobustRegionReport(RegionReport):
    """RegionReport of a run under bounded disturbances: every statement holds for every admissible disturbance sequence."""
    disturbance: dict = field(default_factory=dict)     # {"obs" | "act" | "state": [lo list, hi list]}: the proven boxes


@dataclass
class RobustnessMargin:
    """Result of B200RegionVerifier.robustness_margin (every scale is that of a full run)."""
    s_proven: object              # largest tested scale whose run proved invariance with c_sound >= level; None if s = 0 failed
    s_failed: object              # smallest tested scale whose run did not; None if s_max passed
    runs: int
    report: RobustRegionReport    # the run at s_proven (at s = 0 when the nominal loop is not proven)
    nominal_proven: bool


DIST_KEYS = ("obs", "act", "state")


def _f32_out(x, down):
    """float32 array of x rounded outward (down for lower bounds), so the proven box contains the requested one."""
    x = np.asarray(x, np.float64)
    f = x.astype(np.float32)
    bad = f.astype(np.float64) > x if down else f.astype(np.float64) < x
    return np.where(bad, np.nextafter(f, np.float32(-np.inf if down else np.inf)), f).astype(np.float32)


def parse_disturbance(dist, obs_dim, act_dim):
    """{"obs" | "act" | "state": (lo, hi) float32 arrays} from the user's dict: each entry is a radius r >= 0 (scalar, or a list
    / array per dimension) meaning [-r, r], or a tuple (lo, hi) of scalars or per-dimension values; missing keys are {0}.
    Bounds are rounded outward to float32."""
    if not isinstance(dist, dict):
        raise ValueError(f"disturbance must be a dict with keys {DIST_KEYS}, got {type(dist).__name__}")
    unknown = set(dist) - set(DIST_KEYS)
    if unknown:
        raise ValueError(f"disturbance: unknown keys {sorted(unknown)}; allowed: {DIST_KEYS}")
    out = {}
    for key, n in zip(DIST_KEYS, (obs_dim, act_dim, obs_dim)):
        v = dist.get(key, 0.0)
        if isinstance(v, tuple):
            if len(v) != 2:
                raise ValueError(f"disturbance {key}: a (lo, hi) pair needs 2 entries, got {len(v)}")
            lo, hi = (np.asarray(b, np.float64) for b in v)
        else:
            r = np.asarray(v, np.float64)
            if np.any(r < 0):
                raise ValueError(f"disturbance {key}: a radius must be >= 0, got {r.tolist()}")
            lo, hi = -r, r
        vals = []
        for b in (lo, hi):
            if b.ndim > 1 or (b.ndim == 1 and b.shape[0] not in (1, n)):
                raise ValueError(f"disturbance {key}: need a scalar or {n} values per bound, got shape {list(b.shape)}")
            vals.append(np.broadcast_to(b, (n,)).astype(np.float64))
        lo, hi = vals
        if not (np.all(np.isfinite(lo)) and np.all(np.isfinite(hi))):
            raise ValueError(f"disturbance {key}: bounds must be finite, got [{lo.tolist()}, {hi.tolist()}]")
        if not np.all(lo <= hi):
            raise ValueError(f"disturbance {key}: need lo <= hi, got [{lo.tolist()}, {hi.tolist()}]")
        out[key] = (_f32_out(lo, True), _f32_out(hi, False))
    return out


def _layers(seq, what):
    lin = [m for m in seq if isinstance(m, torch.nn.Linear)]
    other = [m for m in seq if not isinstance(m, torch.nn.Linear)]
    shape = [tuple(m.weight.shape) for m in lin] + [type(m).__name__ for m in other]
    if len(lin) != 3 or len(other) != 3 or not isinstance(other[2], torch.nn.Identity) or type(other[0]) is not type(other[1]):
        raise ValueError(f"{what}: need two hidden layers with one activation and a linear output, got {shape}")
    if lin[0].out_features > HIDDEN or lin[1].out_features > HIDDEN or lin[2].out_features > HIDDEN:
        raise ValueError(f"{what}: layer widths must be <= {HIDDEN}, got {shape}")
    return lin, other[0]


class B200RegionVerifier:
    """B200RegionVerifier(networks=..., env_name=..., box=(lo, hi), inner=(lo, hi) or radius, ...).run() -> RegionReport.

    kwargs: networks (ApproxContainer: `.policy` and `.lyapunov`), env_name (VanderPol, Pendulum, DuctedFan, TwoLink), box
    (X0, inside the observation bounds; scalars broadcast), inner (B inside X0: a (lo, hi) pair or a radius r for
    [-r, r]^D; default 0.05 of the box width around the origin), lya_eta (0.15, in (0, 1)), alpha1 (1), alpha2 (2), steps
    (m, 1), max_depth (30, <= 50), max_cells (2^22: frontier capacity), max_examples (16), chunk (cells per round, default
    max_cells // (2 (max_depth + 1))), device ("cuda"), trace (optional callable(lo, hi, status) with device views of every
    round's cell boxes and their status, for tests and inspection), disturbance (optional dict with keys obs / act / state:
    the boxes N, U, W of the module docstring, each a radius r >= 0 -- scalar, or a list / array per dimension -- for
    [-r, r], or a tuple (lo, hi); missing keys are {0}; run() then returns a RobustRegionReport)."""

    def __init__(self, **kw):
        self.networks = kw["networks"]
        self.env_name = kw["env_name"]
        if self.env_name not in SUPPORTED:
            why = ("its kinematic / dynamic model switch needs interval case splits" if self.env_name == "SingleTrackCar" else
                   "its state is not its observation" if self.env_name == "QuadTracking" else "unknown env")
            get_spec(self.env_name)
            raise ValueError(f"region verifier: {self.env_name} is not supported ({why}); supported: {', '.join(SUPPORTED)}")
        self.spec = spec = get_spec(self.env_name)
        D = spec.obs_dim
        self.steps = int(kw.get("steps", 1))
        self.lya_eta = float(kw.get("lya_eta", 0.15))
        self.alpha1, self.alpha2 = float(kw.get("alpha1", 1.0)), float(kw.get("alpha2", 2.0))
        self.max_depth = int(kw.get("max_depth", 30))
        self.max_cells = int(kw.get("max_cells", 1 << 22))
        self.max_examples = int(kw.get("max_examples", 16))
        self.device = torch.device(kw.get("device", "cuda"))
        self.trace = kw.get("trace")
        if self.steps < 1:
            raise ValueError("steps must be >= 1")
        if not 0.0 < self.lya_eta < 1.0:
            raise ValueError("lya_eta must be in (0, 1)")
        if not (self.alpha1 > 0 and self.alpha2 > 0 and math.isfinite(self.alpha1) and math.isfinite(self.alpha2)):
            raise ValueError("alpha1 and alpha2 must be positive and finite")
        if not 1 <= self.max_depth <= MAX_DEPTH:
            raise ValueError(f"max_depth must be in [1, {MAX_DEPTH}]")
        if self.max_cells < 2 * (self.max_depth + 2):
            raise ValueError(f"max_cells must be >= {2 * (self.max_depth + 2)}")
        if self.max_examples < 0:
            raise ValueError("max_examples must be >= 0")
        self.chunk = int(kw.get("chunk") or max(1, self.max_cells // (2 * (self.max_depth + 1))))
        box = kw["box"]
        lo = np.broadcast_to(np.asarray(box[0], np.float32), (D,)).copy()
        hi = np.broadcast_to(np.asarray(box[1], np.float32), (D,)).copy()
        if not (np.all(np.isfinite(lo)) and np.all(np.isfinite(hi)) and np.all(lo < hi)):
            raise ValueError("box: need finite lo < hi")
        if np.any(lo < spec.obs_low) or np.any(hi > spec.obs_high):
            raise ValueError(f"box [{lo.tolist()}, {hi.tolist()}] is not inside the observation bounds of {self.env_name} "
                             f"[{spec.obs_low.tolist()}, {spec.obs_high.tolist()}]")
        self.box = (lo, hi)
        inner = kw.get("inner", 0.05 * float(np.min(hi - lo)) / 2)
        if np.ndim(inner) == 0:
            r = float(inner)
            if not r > 0:
                raise ValueError("inner radius must be > 0")
            ilo, ihi = np.full(D, -r, np.float32), np.full(D, r, np.float32)
        else:
            ilo = np.broadcast_to(np.asarray(inner[0], np.float32), (D,)).copy()
            ihi = np.broadcast_to(np.asarray(inner[1], np.float32), (D,)).copy()
        if not (np.all(ilo <= ihi) and np.all(ilo >= lo) and np.all(ihi <= hi)):
            raise ValueError(f"inner box [{ilo.tolist()}, {ihi.tolist()}] is not inside box [{lo.tolist()}, {hi.tolist()}]")
        self.inner_level = self.max_depth // D
        self.inner_grid = snap_inner(lo, hi, ilo, ihi, self.inner_level)
        self.p_lin, pact = _layers(self.networks.policy.policy, "policy")
        if not isinstance(pact, torch.nn.ReLU):
            raise ValueError(f"policy: the hidden activation must be ReLU, got {type(pact).__name__}")
        if self.p_lin[2].out_features != 2 * spec.act_dim or self.p_lin[0].in_features != D:
            raise ValueError(f"policy: shapes {[tuple(m.weight.shape) for m in self.p_lin]} do not match {self.env_name}")
        self.v_lin, vact = _layers(self.networks.lyapunov.lya, "lyapunov")
        if not isinstance(vact, (torch.nn.ReLU, torch.nn.Tanh)):
            raise ValueError(f"lyapunov: the hidden activation must be ReLU or Tanh, got {type(vact).__name__}")
        if self.v_lin[0].in_features != D:
            raise ValueError(f"lyapunov: input width {self.v_lin[0].in_features} != obs_dim {D}")
        self.v_tanh = isinstance(vact, torch.nn.Tanh)
        dist = kw.get("disturbance")
        self.disturbance = None if dist is None else parse_disturbance(dist, D, spec.act_dim)
        self._lib = None

    # ---- device plumbing
    def params(self):
        lo, hi = decay_bounds(self.lya_eta, self.steps)
        p = _lib.RegionParams(env_id=self.spec.env_id, steps=self.steps, v_tanh=int(self.v_tanh), decay_lo=lo, decay_hi=hi,
                              alpha1=self.alpha1, alpha2=self.alpha2)
        for d in range(self.spec.obs_dim):
            p.x0_lo[d], p.x0_hi[d] = float(self.box[0][d]), float(self.box[1][d])
        return p

    def _dist(self, dist):
        d = _lib.RegionDisturbance()
        for key, (lo, hi) in dist.items():
            for j in range(lo.shape[0]):
                getattr(d, key + "_lo")[j], getattr(d, key + "_hi")[j] = float(lo[j]), float(hi[j])
        return d

    def _scaled(self, s):
        """The disturbance boxes times s >= 0, rounded outward to float32."""
        return {k: (_f32_out(np.float64(s) * lo.astype(np.float64), True), _f32_out(np.float64(s) * hi.astype(np.float64), False))
                for k, (lo, hi) in self.disturbance.items()}

    def pack(self):
        """The network image from the current parameters (device float tensor)."""
        lib = self._lib = _lib.load()
        img = torch.empty(lib.msacl_region_image_bytes() // 4, dtype=torch.float32, device=self.device)
        t = [m.weight.detach().float().contiguous() for m in self.p_lin] + [m.bias.detach().float().contiguous() for m in self.p_lin]
        v = [m.weight.detach().float().contiguous() for m in self.v_lin] + [m.bias.detach().float().contiguous() for m in self.v_lin]
        self._keep = t + v
        nets = _lib.RegionNets(env_id=self.spec.env_id, obs_dim=self.spec.obs_dim, act_dim=self.spec.act_dim,
                               p_h1=self.p_lin[0].out_features, p_h2=self.p_lin[1].out_features,
                               p_w1=t[0].data_ptr(), p_b1=t[3].data_ptr(), p_w2=t[1].data_ptr(), p_b2=t[4].data_ptr(),
                               p_w3=t[2].data_ptr(), p_b3=t[5].data_ptr(),
                               v_h1=self.v_lin[0].out_features, v_h2=self.v_lin[1].out_features, v_out=self.v_lin[2].out_features,
                               v_w1=v[0].data_ptr(), v_b1=v[3].data_ptr(), v_w2=v[1].data_ptr(), v_b2=v[4].data_ptr(),
                               v_w3=v[2].data_ptr(), v_b3=v[5].data_ptr())
        _lib.check(lib.msacl_region_pack(C.byref(nets), img.data_ptr(), _lib.current_stream()))
        return img

    def _out(self, n, trace=False):
        D, A, dev = self.spec.obs_dim, self.spec.act_dim, self.device
        f = lambda *s: torch.empty(*s, dtype=torch.float32, device=dev)
        o = dict(v_lo=f(n), v_hi=f(n), vm_lo=f(n), vm_hi=f(n), img_lo=f(n, D), img_hi=f(n, D),
                 flags=torch.empty(n, dtype=torch.uint8, device=dev), margin=f(n))
        if trace:
            o["trace"] = f(n, self.steps, 4 * A + 2 * D)
        desc = _lib.RegionOut(**{k: v.data_ptr() for k, v in o.items()})
        return o, desc

    def evaluate(self, lo, hi, image=None, trace=False):
        """Enclosures for the boxes [lo, hi] ([n, D] float32 CUDA): dict of device tensors (v_lo, v_hi, vm_lo, vm_hi, img_lo,
        img_hi, flags, margin and, with trace, [n, m, 4A + 2D] = mu lo, mu hi, a lo, a hi, F^j lo, F^j hi)."""
        image = self.pack() if image is None else image
        self._lib = self._lib or _lib.load()
        lo, hi = lo.float().contiguous(), hi.float().contiguous()
        o, desc = self._out(lo.shape[0], trace)
        p = self.params()
        args = (C.byref(p), image.data_ptr(), lo.shape[0], None, lo.data_ptr(), hi.data_ptr(), C.byref(desc), _lib.current_stream())
        if self.disturbance is None:
            _lib.check(self._lib.msacl_region_eval(*args))
        else:
            _lib.check(self._lib.msacl_region_eval_robust(*args, C.byref(self._dist(self.disturbance))))
        return o

    def run(self) -> RegionReport:
        """Verify the region: a RegionReport, or a RobustRegionReport when the verifier has a disturbance."""
        return self._run(self.disturbance)

    def run_scaled(self, s) -> RobustRegionReport:
        """run() with every disturbance box scaled by s >= 0 (s = 0 is the nominal loop)."""
        if self.disturbance is None:
            raise ValueError("run_scaled needs a verifier created with a disturbance")
        return self._run(self._scaled(s))

    def robustness_margin(self, s_max, iters=8, level=0.0) -> RobustnessMargin:
        """Bisect the scale s in [0, s_max] of the disturbance shape for the largest s whose run proves `invariant` with
        c_sound >= level.  Runs s = 0 (the nominal loop) first: if that is not proven there is no margin (s_proven None).
        Then s_max, then `iters` bisection steps.  Every reported scale is that of a full run, and each such run is a sound
        statement at its own scale; whether the proof is monotone in s (a larger set can only lose) only decides how tight
        the bracket [s_proven, s_failed] is, not whether s_proven is sound."""
        s_max = float(s_max)
        if not (s_max > 0 and math.isfinite(s_max)):
            raise ValueError("s_max must be positive and finite")
        if int(iters) < 0:
            raise ValueError("iters must be >= 0")
        ok = lambda r: bool(r.invariant) and r.c_sound != "none" and r.c_sound >= level
        runs = 1
        rep = self.run_scaled(0.0)
        if not ok(rep):
            return RobustnessMargin(s_proven=None, s_failed=0.0, runs=runs, report=rep, nominal_proven=False)
        good, good_rep, bad = 0.0, rep, s_max
        rep = self.run_scaled(s_max)
        runs += 1
        if ok(rep):
            return RobustnessMargin(s_proven=s_max, s_failed=None, runs=runs, report=rep, nominal_proven=True)
        for _ in range(int(iters)):
            mid = 0.5 * (good + bad)
            rep = self.run_scaled(mid)
            runs += 1
            if ok(rep):
                good, good_rep = mid, rep
            else:
                bad = mid
        return RobustnessMargin(s_proven=good, s_failed=bad, runs=runs, report=good_rep, nominal_proven=True)

    def _run(self, dist):
        D, dev = self.spec.obs_dim, self.device
        W = 1 + D
        image = self.pack()
        p = self.params()
        glo, ghi, blo, bhi = self.inner_grid
        b = _lib.RegionBnb(max_depth=self.max_depth, inner_level=self.inner_level, max_examples=self.max_examples)
        for d in range(D):
            b.inner_lo[d], b.inner_hi[d], b.inner_box_lo[d], b.inner_box_hi[d] = glo[d], ghi[d], blo[d], bhi[d]
        stack = torch.zeros(self.max_cells, W, dtype=torch.int32, device=dev)     # uint32 words; cell 0 = X0
        stats = torch.zeros(ST["count"], dtype=torch.int64, device=dev)
        stats[ST["c_sound"]] = float_order_key(math.inf)
        stats[ST["c_in"]] = float_order_key(-math.inf)
        stats[ST["v_inner"]] = float_order_key(-math.inf)
        examples = torch.zeros(max(1, self.max_examples), D + 2, dtype=torch.float32, device=dev)
        children = torch.zeros(1, dtype=torch.int64, device=dev)
        K = min(self.chunk, self.max_cells)
        res, rdesc = self._out(K)
        pres, pdesc = self._out(K)
        nb = (K + 255) // 256
        wsb = dict(cells=torch.empty(K, W, dtype=torch.int32, device=dev), lo=torch.empty(K, D, device=dev),
                   hi=torch.empty(K, D, device=dev), plo=torch.empty(K, D, device=dev), phi=torch.empty(K, D, device=dev),
                   probe=torch.empty(K, dtype=torch.int32, device=dev), status=torch.empty(K, dtype=torch.uint8, device=dev),
                   scan=torch.zeros(3 * nb + 8, dtype=torch.int64, device=dev))
        ws = _lib.RegionWs(res=rdesc, pres=pdesc, **{k: v.data_ptr() for k, v in wsb.items()})
        top, rounds = 1, 0
        wd = None if dist is None else self._dist(dist)
        while top > 0:
            k = min(K, top, self.max_cells - top)
            if k < 1:
                raise RuntimeError(f"region verifier: the frontier exceeds max_cells = {self.max_cells}")
            args = (C.byref(p), C.byref(b), image.data_ptr(), stack.data_ptr(), top, k, C.byref(ws), stats.data_ptr(),
                    examples.data_ptr(), children.data_ptr(), _lib.current_stream())
            if wd is None:
                _lib.check(self._lib.msacl_region_round(*args))
            else:
                _lib.check(self._lib.msacl_region_round_robust(*args, C.byref(wd)))
            if self.trace is not None:
                self.trace(wsb["lo"][:k], wsb["hi"][:k], wsb["status"][:k])
            rounds += 1
            top = top - k + int(children.item())
        s = stats.cpu().tolist()
        ex = examples[:min(self.max_examples, s[ST["refuted"]])].cpu().numpy()
        exs = [{"x": r[:D].tolist(), "kind": "decrease" if r[D + 1] == 1.0 else "escaped", "margin": float(r[D])} for r in ex]
        meta = dict(env_name=self.env_name, box=[self.box[0].tolist(), self.box[1].tolist()], inner=[blo, bhi], steps=self.steps,
                    lya_eta=self.lya_eta, alpha1=self.alpha1, alpha2=self.alpha2, max_depth=self.max_depth)
        if dist is None:
            rep = RegionReport.from_stats(s, exs, **meta)
        else:
            rep = RobustRegionReport.from_stats(s, exs, **meta,
                                                disturbance={k: [lo.tolist(), hi.tolist()] for k, (lo, hi) in dist.items()})
        rep.rounds, rep.evaluated = rounds, s[ST["evaluated"]]
        return rep
