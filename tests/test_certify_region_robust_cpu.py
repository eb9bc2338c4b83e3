"""Region verifier under bounded disturbances, without a GPU: argument refusals and broadcasting of the disturbance boxes, the
nominal report unchanged, robustness_margin's bracketing against a stubbed run, and the disturbed float64 closed loop that
the GPU tests compare against."""
import math

import numpy as np
import pytest

from oracle import envs as oenv
from oracle import region as oreg
from test_certify_region_cpu import BASE, _cells_to_stats, _make


def closed_loop_disturbed(name, policy_layers, x, steps, dist=None, xp=np):
    """[(mu, a, F^j(x)) for j = 1..steps] of the disturbed greedy closed loop
    F_d(x) = Phi(x, clip(half tanh(mu(x + n)) + mid) + u) + w, built from the float64 oracle's unchanged pieces.  dist is
    None or one (n, u, w) per step ([N, D], [N, A], [N, D] arrays, any of them None for {0})."""
    A = oenv.SPECS[name].act_dim
    out = []
    for j in range(steps):
        n, u, w = dist[j] if dist is not None else (None, None, None)
        mu = oreg.policy_mean(policy_layers, x if n is None else x + n, A, xp)
        a = oreg.action(name, mu, xp)
        if u is not None:
            a = a + u
        x = oreg.env_step(name, x, a, xp)
        if w is not None:
            x = x + w
        out.append((mu, a, x))
    return out


@pytest.mark.parametrize("dist,msg", [
    (dict(obs=(0.1, -0.1)), "lo <= hi"),
    (dict(state=((0.0, 0.2), (0.1, 0.1))), "lo <= hi"),
    (dict(act=float("nan")), "finite"),
    (dict(state=(-math.inf, 0.0)), "finite"),
    (dict(obs=[0.1, 0.2, 0.3]), "2 values"),
    (dict(act=(np.zeros(2), np.zeros(2))), "1 values"),
    (dict(obs=-1e-3), "radius must be >= 0"),
    (dict(state=[1e-3, -1e-3]), "radius must be >= 0"),
    (dict(noise=0.1), "unknown keys"),
    (dict(obs=(0.0, 0.1, 0.2)), "2 entries"),
    (0.1, "must be a dict"),
])
def test_disturbance_refusals(dist, msg):
    with pytest.raises(ValueError, match=msg):
        _make(disturbance=dist)


def test_disturbance_broadcasting_and_outward_rounding():
    v = _make(env_name="DuctedFan", box=(-1.0, 1.0), disturbance=dict(obs=1e-3, act=(0.5, [1.0, 2.0]),
                                                                      state=[1e-4, 2e-4, 3e-4, 4e-4, 5e-4, 6e-4]))
    d = v.disturbance
    assert set(d) == {"obs", "act", "state"}
    assert all(lo.dtype == np.float32 and hi.dtype == np.float32 for lo, hi in d.values())
    assert d["obs"][0].shape == (6,) and d["act"][0].shape == (2,) and d["state"][1].shape == (6,)
    # 1e-3 is not a float32: the box is rounded outward, so it contains the requested one
    assert np.all(d["obs"][0].astype(np.float64) <= -1e-3) and np.all(d["obs"][1].astype(np.float64) >= 1e-3)
    assert np.all(d["obs"][1] - np.float32(1e-3) <= np.spacing(np.float32(1e-3)))
    assert d["act"][0].tolist() == [0.5, 0.5] and d["act"][1].tolist() == [1.0, 2.0]
    assert np.all(d["state"][1].astype(np.float64) >= np.array([1e-4, 2e-4, 3e-4, 4e-4, 5e-4, 6e-4]))
    assert np.all(d["state"][0] == -d["state"][1])
    # missing keys are {0}; a per-dimension radius of length 1 broadcasts
    v = _make(disturbance=dict(state=[2e-3]))
    assert v.disturbance["obs"][0].tolist() == [0.0, 0.0] and v.disturbance["act"][1].tolist() == [0.0]
    assert v.disturbance["state"][0].shape == (2,)
    # scaling keeps the shape and rounds outward
    lo, hi = v._scaled(0.5)["state"]
    assert np.all(hi.astype(np.float64) >= 0.5 * v.disturbance["state"][1].astype(np.float64)) and np.all(lo == -hi)
    assert v._scaled(0.0)["state"][0].tolist() == [0.0, 0.0]


def test_nominal_report_unchanged_without_disturbance():
    from msacl_b200.certify_region import RegionReport, RobustRegionReport
    from dataclasses import fields
    v = _make()
    assert v.disturbance is None
    with pytest.raises(ValueError, match="disturbance"):
        v.run_scaled(1.0)
    with pytest.raises(ValueError, match="disturbance"):
        v.robustness_margin(1.0)
    meta = dict(env_name="VanderPol", box=[[-1, -1], [1, 1]], inner=[[-0.1], [0.1]], steps=1, lya_eta=0.15, alpha1=1.0,
                alpha2=2.0, max_depth=4)
    stats = _cells_to_stats(BASE)
    r = RegionReport.from_stats(stats, [], **meta)
    assert type(r) is RegionReport
    assert [f.name for f in fields(RegionReport)] == [
        "env_name", "box", "inner", "steps", "lya_eta", "alpha1", "alpha2", "max_depth", "verified", "refuted", "undecided",
        "inner_cells", "verified_fraction", "refuted_fraction", "undecided_fraction", "inner_fraction",
        "verified_fraction_outside", "failed", "c_sound", "c_sound_candidate", "c_in", "v_inner", "inner_failed", "invariant",
        "reach_level", "counterexamples", "rounds", "evaluated"]
    dist = {"obs": [[0.0, 0.0], [0.0, 0.0]], "act": [[-0.5], [0.5]], "state": [[0.0, 0.0], [0.0, 0.0]]}
    rr = RobustRegionReport.from_stats(stats, [], **meta, disturbance=dist)
    assert isinstance(rr, RegionReport)
    import json
    a, b = json.loads(r.to_json()), json.loads(rr.to_json())
    assert b.pop("disturbance") == dist and a == b
    assert r.to_json() == rr.to_json().replace(', "disturbance": ' + json.dumps(dist), "")


class _Rep:
    def __init__(self, s, invariant, c_sound):
        self.s, self.invariant, self.c_sound = s, invariant, c_sound


def _stubbed(proven, c_sound=lambda s: 1.0):
    """A verifier whose run_scaled(s) proves invariance iff proven(s); records every tested s."""
    v = _make(disturbance=dict(state=1e-3))
    calls = []

    def run_scaled(s):
        calls.append(float(s))
        ok = proven(s)
        return _Rep(s, ok, c_sound(s) if ok else "none")
    v.run_scaled = run_scaled
    return v, calls


def test_robustness_margin_brackets_a_threshold():
    v, calls = _stubbed(lambda s: s <= 0.3)
    r = v.robustness_margin(1.0, iters=8)
    assert r.nominal_proven and calls[:2] == [0.0, 1.0] and r.runs == len(calls) == 10
    assert r.s_proven in calls and r.s_failed in calls and r.report.s == r.s_proven
    assert r.s_proven <= 0.3 < r.s_failed and r.s_failed - r.s_proven == 2.0 ** -8
    assert r.s_proven == max(s for s in calls if s <= 0.3) and r.s_failed == min(s for s in calls if s > 0.3)


def test_robustness_margin_nominal_not_proven():
    v, calls = _stubbed(lambda s: False)
    r = v.robustness_margin(1.0, iters=8)
    assert calls == [0.0] and r.runs == 1 and r.s_proven is None and not r.nominal_proven and r.s_failed == 0.0
    assert r.report.s == 0.0


def test_robustness_margin_s_max_proven():
    v, calls = _stubbed(lambda s: True)
    r = v.robustness_margin(2.5, iters=8)
    assert calls == [0.0, 2.5] and r.s_proven == 2.5 and r.s_failed is None and r.runs == 2


def test_robustness_margin_level():
    # invariant everywhere, but c_sound falls with s: the level decides
    v, calls = _stubbed(lambda s: True, c_sound=lambda s: 1.0 - s)
    r = v.robustness_margin(1.0, iters=10, level=0.6)
    assert r.s_proven <= 0.4 < r.s_failed and r.report.c_sound >= 0.6
    assert r.s_proven in calls and r.s_failed in calls
    v, calls = _stubbed(lambda s: True, c_sound=lambda s: 0.5)
    r = v.robustness_margin(1.0, level=0.6)
    assert r.s_proven is None and calls == [0.0]
    v, calls = _stubbed(lambda s: True, c_sound=lambda s: math.inf)
    assert v.robustness_margin(1.0, level=1e30).s_proven == 1.0


def test_robustness_margin_non_monotone_reports_only_tested_scales():
    v, calls = _stubbed(lambda s: s < 0.1 or 0.5 <= s < 0.6)
    r = v.robustness_margin(1.0, iters=6)
    assert r.s_proven in calls and r.s_failed in calls and r.s_proven < r.s_failed
    assert r.s_proven < 0.1 or 0.5 <= r.s_proven < 0.6


@pytest.mark.parametrize("kw,msg", [(dict(s_max=0.0), "s_max"), (dict(s_max=math.inf), "s_max"),
                                    (dict(s_max=1.0, iters=-1), "iters")])
def test_robustness_margin_arguments(kw, msg):
    v, _ = _stubbed(lambda s: True)
    with pytest.raises(ValueError, match=msg):
        v.robustness_margin(**kw)


@pytest.mark.parametrize("name", ["VanderPol", "Pendulum", "DuctedFan", "TwoLink"])
def test_disturbed_loop_with_zero_disturbance_is_the_nominal_loop(name):
    from oracle import actor as oactor
    spec = oenv.SPECS[name]
    D, A = spec.obs_dim, spec.act_dim
    w = oactor.init_policy_weights(D, A, seed=1)
    layers = [(W.astype(np.float64), b.astype(np.float64)) for W, b in w]
    rng = np.random.default_rng(2)
    x = rng.uniform(spec.obs_low * 0.1, spec.obs_high * 0.1, (256, D))
    zero = [(np.zeros((256, D)), np.zeros((256, A)), np.zeros((256, D)))] * 3
    want = oreg.closed_loop(name, layers, x, 3)
    for dist in (None, zero):
        got = closed_loop_disturbed(name, layers, x, 3, dist)
        for (m0, a0, x0), (m1, a1, x1) in zip(want, got):
            assert np.array_equal(m0, m1) and np.array_equal(a0, a1) and np.array_equal(x0, x1)
    # a nonzero process disturbance shifts the state after the step, an actuator one the action, sensor noise the policy input
    n, u, wd = rng.normal(size=(256, D)) * 1e-3, rng.normal(size=(256, A)) * 1e-3, rng.normal(size=(256, D)) * 1e-3
    ((mu, a, x1),) = closed_loop_disturbed(name, layers, x, 1, [(n, u, wd)])
    assert np.array_equal(mu, oreg.policy_mean(layers, x + n, A))
    assert np.array_equal(a, oreg.action(name, mu) + u)
    assert np.array_equal(x1, oreg.env_step(name, x, a) + wd)
