"""CPU checks of the Lyapunov-certificate verifier: the oracle's contract on hand-built trajectories, host-side argument
validation of the C ABI and of the Python front end, and the multi-rank combine under gloo (no GPU needed)."""
import ctypes as C
import math
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import msacl_b200
from msacl_b200 import _lib
from msacl_b200 import distributed as mdist
from oracle import certify as oc

NF, LO, HI, DEC, ESC, NES = oc.NONFINITE, oc.BOUND_LO, oc.BOUND_HI, oc.DECREASE, oc.ESCAPED, oc.NOT_EXP_STABLE


def _traj(T, N, D=2):
    return np.zeros((T + 1, N, D), np.float32), np.zeros((T + 1, N), np.float32), np.zeros((T + 1, N), bool)


def _geometric(o, V, i, T, r=0.5, x0=1.0, gain=1.5):
    """o_k = (x0 r^k, 0), V_k = gain |o_k|^2: inside the bounds for alpha1 <= gain <= alpha2, decreasing like r^2k."""
    for k in range(T + 1):
        o[k, i, 0] = x0 * r ** k
        V[k, i] = gain * float(o[k, i, 0]) ** 2


def test_oracle_flags_on_hand_built_trajectories():
    T, eta = 3, 0.5                            # c_k = 1, 0.5, 0.25, 0.125 exactly
    o, V, done = _traj(T, 9)
    _geometric(o, V, 0, T)                     # 0: certified
    _geometric(o, V, 1, T)
    o[2, 1, 0], V[2, 1] = np.nan, np.nan       # 1: NaN mid-trajectory (NaN compares false everywhere else)
    _geometric(o, V, 2, T)
    done[0, 2] = True                          # 2: done[0] is ignored ...
    done[1, 2] = True                          #    ... a done on the first step ends the trajectory at e = 1
    o[2:, 2] = 100.0                           #    and nothing after it is looked at
    V[2:, 2] = -1.0
    _geometric(o, V, 3, T)
    done[T, 3] = True                          # 3: done on the last step of the horizon
    # 4: V_0 = 0 at the origin and staying there: certified, 0 / 0 = 0
    # 5: V_0 = 0, then leaves the origin: DECREASE (x / 0 = inf) and NOT_EXP_STABLE agree
    o[1:, 5, 0], V[1:, 5] = 0.1, 1.5 * np.float32(0.1) ** 2
    _geometric(o, V, 6, T)
    V[0, 6] = 0.9                              # 6: BOUND_LO at k = 0 only (0.9 < |o_0|^2 = 1; V still decays fast enough)
    _geometric(o, V, 7, T)
    V[1, 7] = 2.5 * float(o[1, 7, 0]) ** 2     # 7: BOUND_HI at k = 1 (0.625 > 2 * 0.25; still below c_1 V_0 = 0.75)
    _geometric(o, V, 8, T, r=0.75)             # 8: V decays like 0.5625^k > 0.5^k: DECREASE from k = 1, s_k within 2 c_k s_0
    rec = oc.check(o, V, done, T, lya_eta=eta)
    flags = rec["flags"].tolist()
    assert flags == [0, NF, ESC, ESC, 0, DEC | NES, LO, HI, DEC]
    assert rec["first_violation"].tolist() == [-1, 2, 1, 3, -1, 1, 0, 1, 1]
    assert rec["first_decrease"].tolist() == [-1, -1, -1, -1, -1, 1, -1, -1, 1]
    assert rec["end_step"].tolist() == [3, 3, 1, 3, 3, 3, 3, 3, 3]
    wr = rec["worst_ratio"]
    assert wr[0] == np.float32(0.5) and wr[4] == 0 and math.isinf(wr[5])
    assert wr[2] == np.float32(0.5)            # only k = 1 is visited
    assert wr[8] == np.float32(1.125 ** 3)
    s = oc.summarize(rec, T)
    assert (s["nonfinite"], s["bound_lo"], s["bound_hi"], s["decrease"], s["escaped"], s["not_exp_stable"]) == (1, 1, 1, 2, 2, 1)
    assert s["certified"] == 2 and s["inconsistent"] == 1           # state 8: DECREASE without NOT_EXP_STABLE
    assert s["first_decrease_hist"].tolist() == [2, 0, 0]
    # c* = min V_0 over the uncertified states: state 5 (V_0 = 0) -> nothing lies strictly below it
    assert s["c_star"] == 0.0 and s["roa_count"] == 0


def test_oracle_v_atol_and_escape_after_horizon():
    T = 1
    o, V, done = _traj(T + 2, 2)
    for i in range(2):
        o[0, i, 0], V[0, i] = 1.0, 1.9
        o[1:, i, 0] = 0.85
        V[1:, i] = np.float32(0.75 * 1.9 + 1e-3)        # just above c_1 V_0 (eta = 0.25), inside the bounds
    done[T + 1, 1] = True                                 # beyond the horizon: not an escape
    without = oc.check(o, V, done, T, lya_eta=0.25)
    assert without["flags"].tolist() == [DEC, DEC] and without["end_step"].tolist() == [T, T]
    with_atol = oc.check(o, V, done, T, lya_eta=0.25, v_atol=1e-2)
    assert with_atol["flags"].tolist() == [0, 0]
    # v_atol also widens the bounds: alpha2 s + v_atol
    V2 = V.copy()
    V2[1] = np.float32(2.0 * np.float32(0.85) ** 2) + np.float32(5e-3)
    assert oc.check(o, V2, done, T, lya_eta=0.25)["flags"][0] & HI
    assert not oc.check(o, V2, done, T, lya_eta=0.25, v_atol=1e-2)["flags"][0] & HI


def test_oracle_long_horizon_decay_in_float64():
    """T = 400 at eta = 0.3: c_400 = 0.7^400 ~ 1e-62 underflows float32 to 0 but not float64."""
    T, eta = 400, 0.3
    c = oc.decay_table(T, eta)
    assert np.float32(c[T]) == 0 and c[T] > 0
    ref = 1.0
    for k in range(T):
        ref *= 0.7
    assert c[T] == ref                                   # repeated multiplication, not pow
    assert c.tolist() == msacl_b200_decay(T, eta)
    o, V, done = _traj(T, 2)
    o[0, :, 0], V[0] = 1.0, 1.5
    V[T, 0] = np.float32(1e-40)                          # a float32 subnormal, still far above c_400 V_0
    rec = oc.check(o, V, done, T, lya_eta=eta)
    assert rec["flags"].tolist() == [DEC | HI, 0]           # V_400 > 0 = alpha2 |o_400|^2 as well
    assert rec["first_decrease"].tolist() == [T, -1]
    assert np.isfinite(rec["worst_ratio"][0]) and rec["worst_ratio"][0] > 1e20      # float32: 1e-40 / 0 = inf
    assert rec["worst_ratio"][1] == 0


def msacl_b200_decay(T, eta):
    from msacl_b200.certify import decay_table
    return decay_table(T, eta)


def test_oracle_c_star_tie_and_nan():
    rec = dict(v0=np.array([1.0, 2.0, 2.0, 3.0, 0.5, np.nan, 2.0], np.float32),
               flags=np.array([0, DEC, ESC, LO, 0, NF, 0], np.uint8),
               first_decrease=np.array([-1, 2, -1, -1, -1, -1, -1], np.int32))
    s = oc.summarize(rec, 4)
    assert s["c_star"] == 2.0                            # NaN V_0 does not take part
    assert s["roa_count"] == 2                           # strict: the certified state at V_0 = c* is not counted
    assert s["first_decrease_hist"].tolist() == [0, 1, 0, 0]
    assert oc.summarize(dict(v0=rec["v0"][[0, 4]], flags=np.zeros(2, np.uint8), first_decrease=np.full(2, -1, np.int32)), 4)["c_star"] == math.inf


def test_float_order_key_round_trip_and_order():
    vals = [-math.inf, -3.5, -0.0, 0.0, 1e-45, 0.25, 2.0, 3e38, math.inf]
    keys = [mdist.float_order_key(v) for v in vals]
    assert keys == sorted(keys) and len(set(keys)) == len(keys)
    for v, k in zip(vals, keys):
        back = mdist.float_from_order_key(k)
        assert back == np.float32(v) and math.copysign(1, back) == math.copysign(1, v)
    assert mdist.float_order_key(math.inf) == 0xFF800000


def test_abi_argument_validation_without_gpu_work():
    lib = msacl_b200.load_library()
    err = lambda: lib.msacl_last_error()
    f = (C.c_float * 12)(*([0.0] * 12))
    g = (C.c_float * 12)(*([1.0] * 12))
    assert lib.msacl_certify_box_init(None, f, g, None) == -2 and b"certify_box_init" in err()
    st = _lib.EnvState(env_id=5, max_step=1000, n=4, stride=4, sf=0x1000)
    assert lib.msacl_certify_box_init(C.byref(st), f, g, None) == -2 and b"QuadTracking" in err()
    st.env_id = 0
    assert lib.msacl_certify_box_init(C.byref(st), g, f, None) == -2 and b"lo[j] <= hi[j]" in err()
    rec = _lib.CertRecords(**{k: 0x1000 for k, _ in _lib.CertRecords._fields_})
    good = _lib.CertParams(horizon=20, alpha1=1.0, alpha2=2.0, v_atol=0.0, decay=0x1000)
    for bad in (dict(horizon=0), dict(horizon=8193), dict(alpha1=0.0), dict(alpha2=float("nan")), dict(v_atol=-1.0), dict(decay=None)):
        kw = dict(horizon=20, alpha1=1.0, alpha2=2.0, v_atol=0.0, decay=0x1000)
        kw.update(bad)
        p = _lib.CertParams(**kw)
        assert lib.msacl_certify_begin(8, 2, 0x1000, 0x1000, C.byref(p), C.byref(rec), None) == -2
        assert b"bad parameters" in err()
    assert lib.msacl_certify_begin(8, 3, 0x1000, 0x1000, C.byref(good), C.byref(rec), None) == -2 and b"obs_dim 3" in err()
    assert lib.msacl_certify_begin(8, 4, 0x1008, 0x1000, C.byref(good), C.byref(rec), None) == -2 and b"aligned" in err()
    partial = _lib.CertRecords(v0=0x1000)
    assert lib.msacl_certify_begin(8, 2, 0x1000, 0x1000, C.byref(good), C.byref(partial), None) == -2 and b"record" in err()
    assert lib.msacl_certify_steps(8, 2, 0, 1, 0x1000, 0x1000, 0x1000, C.byref(good), C.byref(rec), None) == -2
    assert lib.msacl_certify_steps(8, 2, 4, 0, 0x1000, 0x1000, 0x1000, C.byref(good), C.byref(rec), None) == -2
    assert lib.msacl_certify_steps(8, 2, 4, 1, None, 0x1000, 0x1000, C.byref(good), C.byref(rec), None) == -2
    assert lib.msacl_certify_finish(0, 20, C.byref(rec), 0x1000, None) == -2
    assert lib.msacl_certify_finish(8, 9000, C.byref(rec), 0x1000, None) == -2 and b"horizon" in err()
    assert lib.msacl_certify_roa(0, 0x1000, 1.0, 0x1000, None) == -2 and b"certify_roa" in err()


def test_verifier_rejects_bad_arguments():
    from msacl_b200.certify import B200CertificateVerifier as V
    base = dict(networks=None, env_name="VanderPol", num_states=16)
    V(**base)                                            # constructing validates only; nothing runs
    V(**base, init=("box", [-10.0, -10.0], [10.0, 10.0]))
    for bad in (dict(num_states=0), dict(horizon=0), dict(horizon=9000), dict(lya_eta=1.0), dict(alpha1=0), dict(v_atol=-1),
                dict(init="uniform"), dict(init=("box", -11.0, 1.0)), dict(init=("box", 1.0, -1.0)),
                dict(init=("box", [-1.0, -1.0], [1.0, 10.5]))):
        with pytest.raises(ValueError):
            V(**{**base, **bad})
    with pytest.raises(ValueError, match="QuadTracking"):
        V(networks=None, env_name="QuadTracking", num_states=4, init=("box", -1.0, 1.0))
    with pytest.raises(ValueError, match="Unknown custom env"):
        V(networks=None, env_name="CartPole", num_states=4)


def _summary(rec, T):
    """int64 summary in the layout of include/msacl_b200.h (MSACL_CERT_SUM_*), from the oracle's summarize()."""
    s = oc.summarize(rec, T)
    out = np.zeros(11 + T, np.int64)
    out[0] = s["states"]
    for b, name in enumerate(oc.FLAG_NAMES):
        out[1 + b] = s[name]
    out[7], out[8] = s["certified"], s["inconsistent"]
    out[9] = mdist.float_order_key(s["c_star"])
    out[11:] = s["first_decrease_hist"]
    return torch.as_tensor(out)


def _random_records(N, T, seed=0):
    rng = np.random.default_rng(seed)
    v0 = rng.random(N).astype(np.float32) * 4
    v0[rng.choice(N, 5, replace=False)] = np.nan
    flags = np.where(v0 < 1.5, rng.integers(0, 64, N) & NES, rng.integers(0, 64, N)).astype(np.uint8)   # mostly certified below 1.5
    return dict(v0=v0, flags=flags, first_decrease=rng.integers(-1, T + 1, N).astype(np.int32))


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def _combine_worker(rank, world, port, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    N, T = 1001, 7
    rec = _random_records(N, T)
    lo, hi = mdist.shard_env_range(N, rank, world)
    mine = {k: v[lo:hi] for k, v in rec.items()}
    v0 = torch.as_tensor(mine["v0"])
    total, c_star = mdist.combine_certificate(_summary(mine, T), lambda c: int((v0 < c).sum()))
    q.put((rank, total.tolist(), c_star))
    dist.destroy_process_group()


def test_distributed_combine_gloo_world2_equals_single_process():
    N, T = 1001, 7
    rec = _random_records(N, T)
    v0 = torch.as_tensor(rec["v0"])
    single, c1 = mdist.combine_certificate(_summary(rec, T), lambda c: int((v0 < c).sum()))
    want = oc.summarize(rec, T)
    assert c1 == want["c_star"] and int(single[10]) == want["roa_count"] > 0
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_combine_worker, args=(r, 2, port, q)) for r in range(2)]
    [p.start() for p in procs]
    res = sorted(q.get(timeout=120) for _ in range(2))
    [p.join(60) for p in procs]
    for rank, total, c_star in res:
        assert total == single.tolist() and c_star == c1
