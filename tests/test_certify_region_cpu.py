"""Region verifier without a GPU: argument validation, report bookkeeping from hand-built statistics, and the float64
real-arithmetic oracle (oracle/region.py) against the golden env steps."""
import math
import os

import numpy as np
import pytest

from oracle import envs as oenv
from oracle import region as oreg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _networks(name, **kw):
    from msacl_b200.algorithm import ApproxContainer
    spec = oenv.SPECS[name]
    return ApproxContainer(obs_dim=spec.obs_dim, act_dim=spec.act_dim, action_low_limit=spec.act_low, action_high_limit=spec.act_high,
                           q_learning_rate=1e-3, lyapunov_learning_rate=1e-3, policy_learning_rate=3e-4, alpha_learning_rate=1e-3,
                           **kw)


def _make(**kw):
    import msacl_b200
    args = dict(env_name="VanderPol", box=(-1.0, 1.0), inner=0.1, device="cpu")
    args.update(kw)
    if "networks" not in args:
        args["networks"] = _networks(args["env_name"])
    return msacl_b200.create_region_certifier(**args)


def test_valid_arguments_construct():
    v = _make(steps=3, max_depth=12)
    assert v.inner_level == 6 and v.steps == 3


@pytest.mark.parametrize("name", ["SingleTrackCar", "QuadTracking"])
def test_refused_envs(name):
    with pytest.raises(ValueError, match="not supported"):
        _make(env_name=name, box=(-0.5, 0.5), networks=_networks(name))


@pytest.mark.parametrize("kw,msg", [
    (dict(box=(-11.0, 1.0)), "not inside the observation bounds"),
    (dict(box=(-1.0, 1.0), inner=((-2.0, -0.1), (0.1, 0.1))), "not inside box"),
    (dict(steps=0), "steps"),
    (dict(lya_eta=0.0), "lya_eta"),
    (dict(max_depth=51), "max_depth"),
    (dict(box=(1.0, -1.0)), "lo < hi"),
])
def test_bad_arguments(kw, msg):
    with pytest.raises(ValueError, match=msg):
        _make(**kw)


@pytest.mark.parametrize("kw,msg", [
    (dict(policy_hidden_sizes=[300, 256]), "<= 256"),
    (dict(policy_hidden_sizes=[64, 64, 64]), "two hidden layers"),
    (dict(policy_hidden_activation="tanh"), "ReLU"),
    (dict(lyapunov_hidden_activation="elu"), "ReLU or Tanh"),
    (dict(lyapunov_output_dim=512), "<= 256"),
])
def test_unsupported_network_shapes(kw, msg):
    with pytest.raises(ValueError, match=msg):
        _make(networks=_networks("VanderPol", **kw))


def test_narrow_networks_accepted():
    _make(networks=_networks("TwoLink", policy_hidden_sizes=[64, 32], lyapunov_hidden_sizes=[48, 16], lyapunov_output_dim=8,
                             lyapunov_hidden_activation="relu"), env_name="TwoLink", box=(-0.5, 0.5))


def test_decay_bounds_bracket_the_exact_power():
    from fractions import Fraction
    from msacl_b200.certify_region import decay_bounds
    for eta, m in [(0.15, 1), (0.15, 3), (0.1, 7), (1e-3, 2)]:
        lo, hi = decay_bounds(eta, m)
        exact = (1 - Fraction(eta)) ** m
        assert Fraction(lo) <= exact <= Fraction(hi) and hi - lo <= 2 * math.ulp(hi)


def test_inner_box_snaps_outward():
    from msacl_b200.certify_region import snap_inner
    glo, ghi, blo, bhi = snap_inner([-1.0, -2.0], [1.0, 2.0], [-0.1, -0.3], [0.1, 0.25], 4)
    assert glo == [7, 6] and ghi == [9, 9]            # -0.1 -> grid 7.2 -> 7; 0.25 in [-2, 2] -> 9 exactly
    assert blo[0] <= -0.1 and bhi[0] >= 0.1 and blo[1] <= -0.3 and bhi[1] >= 0.25


def _cells_to_stats(cells):
    """Statistics as region_decide_kernel accumulates them, from a hand-built list of leaf cells."""
    from msacl_b200.certify_region import ST, FLAGS
    from msacl_b200.distributed import float_order_key
    s = [0] * ST["count"]
    c_sound, c_in, v_inner = math.inf, -math.inf, -math.inf
    for c in cells:
        vol = 1 << (50 - c["depth"])
        f = c.get("flags", 0)
        if c["status"] == "inner":
            s[ST["inner"]] += 1
            s[ST["volume"] + 3] += vol
            s[ST["inner_fail"]] += bool(f & (FLAGS["nonfinite"] | FLAGS["escaped"] | FLAGS["leaves"]))
            c_in, v_inner = max(c_in, c["vm_hi"]), max(v_inner, c["v_hi"])
            continue
        j = ("verified", "refuted", "undecided").index(c["status"])
        s[ST[c["status"]]] += 1
        s[ST["volume"] + j] += vol
        for b in range(5):
            s[ST["flags"] + b] += bool(f & (1 << b))
        if c["status"] != "verified" or f & FLAGS["leaves"]:
            c_sound = min(c_sound, -math.inf if math.isnan(c["v_lo"]) else c["v_lo"])   # a NaN bound counts as -inf
    s[ST["c_sound"]], s[ST["c_in"]], s[ST["v_inner"]] = map(float_order_key, (c_sound, c_in, v_inner))
    return s


def _report(cells, eta=0.15):
    from msacl_b200.certify_region import RegionReport
    return RegionReport.from_stats(_cells_to_stats(cells), [], env_name="VanderPol", box=[[-1, -1], [1, 1]], inner=[[-0.1], [0.1]],
                                   steps=1, lya_eta=eta, alpha1=1.0, alpha2=2.0, max_depth=4)


BASE = [dict(status="verified", depth=1, v_lo=0.5), dict(status="verified", depth=2, v_lo=0.2),
        dict(status="refuted", depth=3, v_lo=0.9, flags=2), dict(status="undecided", depth=4, v_lo=0.7, flags=2 | 8),
        dict(status="inner", depth=4, v_hi=0.05, vm_hi=0.04), dict(status="verified", depth=4, v_lo=0.3, flags=8),
        dict(status="verified", depth=4, v_lo=0.8, flags=16)]


def test_report_bookkeeping():
    r = _report(BASE)
    assert (r.verified, r.refuted, r.undecided, r.inner_cells) == (4, 1, 1, 1)
    assert r.verified_fraction == 0.5 + 0.25 + 2 / 16 and r.refuted_fraction == 1 / 8 and r.undecided_fraction == 1 / 16
    assert r.inner_fraction == 1 / 16 and r.verified_fraction_outside == pytest.approx((0.875) / (15 / 16))
    assert r.failed == {"nonfinite": 0, "decrease": 2, "escaped": 0, "bound": 2, "leaves": 1}
    assert r.c_sound_candidate == np.float32(0.7)      # least over not-verified (0.9, 0.7) and verified-but-leaving (0.8)
    assert r.invariant and r.c_sound == r.c_sound_candidate and r.reach_level == np.float32(0.05)
    assert '"c_sound": 0.7' in r.to_json().replace("0.699999988079071", "0.7")


@pytest.mark.parametrize("change,why", [
    (dict(vm_hi=0.75), "c_in >= c_sound"),
    (dict(flags=4), "inner cell may leave the box"),
    (dict(flags=1), "inner cell nonfinite"),
    (dict(status="verified", v_lo=0.01), "no inner cell"),
])
def test_invariance_needs_every_condition(change, why):
    cells = [dict(c) for c in BASE]
    cells[4].update(change)
    r = _report(cells)
    assert not r.invariant and r.c_sound == "none" and r.reach_level is None, why


def test_all_verified_gives_infinite_c_sound():
    r = _report([dict(status="verified", depth=1, v_lo=0.5), dict(status="inner", depth=1, v_hi=0.1, vm_hi=0.05)])
    assert r.c_sound == math.inf and r.invariant and r.verified_fraction_outside == 1.0
    assert '"c_sound": "inf"' in r.to_json()


def test_nan_lower_bound_blocks_invariance():
    r = _report([dict(status="undecided", depth=1, v_lo=float("nan")), dict(status="inner", depth=1, v_hi=0.1, vm_hi=0.05)])
    assert not r.invariant


@pytest.mark.parametrize("name", ["VanderPol", "Pendulum", "DuctedFan", "TwoLink"])
def test_oracle_real_step_matches_golden_to_float32_rounding(name):
    d = np.load(os.path.join(ROOT, "tests", "golden", f"env_step_{name}.npz"))
    x = d["obs_in"].astype(np.float64)
    a = d["act"].astype(np.float64)
    got = oreg.env_step(name, x, a)
    want = d["obs_out"].astype(np.float64)
    live = np.all(np.isfinite(want), -1) & np.all(np.abs(x) < 1e3, -1)
    scale = np.maximum(np.abs(want[live]), 1.0)
    assert np.max(np.abs(got[live] - want[live]) / scale) < 5e-6


def test_oracle_closed_loop_matches_oracle_actor():
    from oracle import actor as oactor
    spec = oenv.SPECS["TwoLink"]
    w = oactor.init_policy_weights(spec.obs_dim, spec.act_dim, seed=0)
    layers = [(W.astype(np.float64), b.astype(np.float64)) for W, b in w]
    x = np.random.default_rng(0).uniform(-0.5, 0.5, (64, 4))
    ((mu, a, x1),) = oreg.closed_loop("TwoLink", layers, x, 1)
    want = oenv.env_step("TwoLink", {"obs": x.astype(np.float32), "step": np.zeros(64, np.int32)}, a.astype(np.float32))[1]
    np.testing.assert_allclose(x1, want, rtol=1e-4, atol=1e-5)
    assert np.all(np.abs(a) <= 20.0)
