"""Lyapunov-certificate verifier on the GPU: the check kernels against oracle/certify.py (exact), the whole pipeline
(closed-loop rollout + V GEMMs + checks) against the oracle envs on an analytic case, V against torch on real network
shapes, fresh weights on every run, sharding invariance, and one full-size QuadTracking run with a subset replay."""
import numpy as np
import pytest
import torch

from oracle import certify as ocert
from oracle import envs as oenv
from oracle import philox as ophx
from oracle import rollout as oroll

pytestmark = pytest.mark.gpu

ETA, A1, A2 = 0.15, 1.0, 2.0


def _networks(name, **kw):
    from msacl_b200.algorithm import ApproxContainer
    spec = oenv.SPECS[name]
    return ApproxContainer(obs_dim=spec.obs_dim, act_dim=spec.act_dim, action_low_limit=spec.act_low, action_high_limit=spec.act_high,
                           q_learning_rate=1e-3, lyapunov_learning_rate=1e-3, policy_learning_rate=3e-4, alpha_learning_rate=1e-3,
                           **kw).cuda()


def _host_records(rec):
    return {k: v.cpu().numpy() for k, v in rec.items()}


def _summary_dict(summary, c_star):
    s = summary.cpu().numpy()
    out = {name: int(s[1 + b]) for b, name in enumerate(ocert.FLAG_NAMES)}
    out.update(states=int(s[0]), certified=int(s[7]), inconsistent=int(s[8]), roa_count=int(s[10]), c_star=c_star,
               first_decrease_hist=s[11:].tolist())
    return out


def _oracle_summary(rec, T):
    s = ocert.summarize(rec, T)
    s["first_decrease_hist"] = s["first_decrease_hist"].tolist()
    return s


def _assert_records_equal(got, want):
    for k in ("flags", "first_violation", "first_decrease", "end_step"):
        np.testing.assert_array_equal(got[k], want[k], err_msg=k)
    np.testing.assert_array_equal(got["v0"], want["v0"])
    g, w = got["worst_ratio"].astype(np.float64), want["worst_ratio"].astype(np.float64)
    assert np.array_equal(np.isinf(g), np.isinf(w))
    fin = np.isfinite(w)
    np.testing.assert_allclose(g[fin], w[fin], rtol=1e-6, atol=0)


@pytest.mark.parametrize("D,T,K,v_atol", [(2, 20, 7, 0.0), (12, 23, 5, 0.0), (7, 9, 4, 1e-3), (4, 3, 8, 0.0), (6, 1, 1, 0.0)])
def test_check_kernels_match_oracle_on_synthetic_trajectories(D, T, K, v_atol):
    """Random trajectories with NaN / Inf, done patterns, V near every threshold and T not a multiple of K: records,
    counters, histogram, c* and roa_count exact; worst_decrease_ratio to 1e-6 relative."""
    from msacl_b200 import distributed as mdist
    from msacl_b200.certify import TrajectoryChecker
    N = 40000 + D
    rng = np.random.default_rng(D * 100 + T)
    L = -(-T // K) * K + 1                              # the last chunk runs past the horizon
    o = np.zeros((L, N, D), np.float32)
    o[0] = rng.standard_normal((N, D)).astype(np.float32)
    decay = rng.uniform(0.6, 1.05, N).astype(np.float32)
    for k in range(1, L):
        o[k] = o[k - 1] * decay[:, None] + 0.05 * rng.standard_normal((N, D)).astype(np.float32)
    s = (o.astype(np.float64) ** 2).sum(-1)
    gain = rng.uniform(0.8, 2.2, (1, N))                # some states outside [alpha1, alpha2]
    V = (gain * s * rng.uniform(0.97, 1.03, (L, N))).astype(np.float32)
    V[1:, 64:128] = np.float32(1e-3)
    ties = rng.choice(np.arange(200, N), 500, replace=False)
    V[:, ties] = V[0, ties][None] * np.asarray(ocert.decay_table(L - 1, ETA), np.float32)[:, None]   # on the decrease threshold
    nan = rng.random((L, N)) < 2e-3
    o[nan, rng.integers(0, D, nan.sum())] = np.nan
    V[rng.random((L, N)) < 1e-3] = np.inf
    V[rng.random((L, N)) < 1e-3] = np.nan
    done = (rng.random((L, N)) < 0.03).astype(np.uint8)
    done[1, :500] = 1
    done[T, 500:1000] = 1
    o[:, :64], V[:, :64], done[:, :64] = 0.0, 0.0, 0        # at the origin: V_0 = 0, 0 / 0, certified below every c* > 0
    rec_o = ocert.check(o, V, done, T, lya_eta=ETA, alpha1=A1, alpha2=A2, v_atol=v_atol)

    dev = "cuda"
    chk = TrajectoryChecker(N, D, T, ETA, A1, A2, v_atol, dev)
    t = lambda a: torch.as_tensor(a).to(dev).contiguous()
    chk.begin(t(o[0]), t(V[0]))
    for k0 in range(1, L, K):
        chk.steps(k0, t(o[k0:k0 + K]), t(V[k0:k0 + K]), t(done[k0:k0 + K]))
    summary = chk.finish()
    total, c_star = mdist.combine_certificate(summary, lambda c: chk.count_below(c, summary))
    got = _host_records(chk.records())
    _assert_records_equal(got, rec_o)
    want = _oracle_summary(rec_o, T)
    assert _summary_dict(total, c_star) == want
    assert 0 < want["roa_count"] < N and want["decrease"] > 0 and want["nonfinite"] > 0 and want["escaped"] > 0


def _identity_lyapunov(nets, D):
    """W1 = [I; -I], W2 = I, W3 = [I, -I], zero biases, ReLU: z = relu(o) - relu(-o) = o, V = |o|^2 up to round-off."""
    lin = [m for m in nets.lyapunov.lya if isinstance(m, torch.nn.Linear)]
    eye = torch.eye(D, device="cuda")
    with torch.no_grad():
        lin[0].weight.copy_(torch.cat([eye, -eye], 0))
        lin[1].weight.copy_(torch.eye(2 * D, device="cuda"))
        lin[2].weight.copy_(torch.cat([eye, -eye], 1))
        for l in lin:
            l.bias.zero_()
    for p in nets.policy.parameters():
        with torch.no_grad():
            p.zero_()


def _margins_near(o, V, T, e, alpha1, alpha2, tol=1e-5):
    """States whose oracle margin to some threshold is within tol relative at a visited step (or whose obs is within tol of
    the VanderPol domain bound, where `done` decides)."""
    c = ocert.decay_table(T, ETA)
    s = (o.astype(np.float64) ** 2).sum(-1)
    Vd = V.astype(np.float64)
    near = np.zeros(o.shape[1], bool)
    rel = lambda a, b: np.abs(a - b) <= tol * np.maximum(np.abs(b), 1e-30)
    for k in range(T + 1):
        vis = k <= e
        m = rel(Vd[k], alpha1 * s[k]) | rel(Vd[k], alpha2 * s[k])
        if k >= 1:
            m |= rel(Vd[k], c[k] * Vd[0]) | rel(s[k], (alpha2 / alpha1) * c[k] * s[0])
        m |= (np.abs(np.abs(o[k]) - 10.0) <= 10.0 * tol).any(-1)
        near |= vis & m
    return near


def _oracle_closed_loop(name, o0, T):
    """Zero-action closed loop of the oracle env: o [T + 1, N, D], done [T + 1, N] (the state stops at its first done)."""
    N = o0.shape[0]
    st = {"obs": o0.copy(), "step": np.zeros(N, np.int32)}
    o = np.zeros((T + 1,) + o0.shape, np.float32)
    done = np.zeros((T + 1, N), bool)
    o[0] = o0
    ended = np.zeros(N, bool)
    for k in range(1, T + 1):
        with np.errstate(all="ignore"):               # states that already ended keep being stepped (and ignored)
            new, obs, _, term, _ = oenv.env_step(name, st, np.zeros((N, 1), np.float32))
        o[k] = np.where(ended[:, None], o[k - 1], obs)
        done[k] = term & ~ended
        ended |= term
        st = new
    return o, done


@pytest.mark.parametrize("init", ["reset", ("box", -10.0, 10.0)])
@pytest.mark.parametrize("engine", ["tc", "ffma"])
def test_vanderpol_analytic_case_matches_oracle(init, engine):
    import msacl_b200
    name, N, T, seed, alpha1 = "VanderPol", 20000, 20, 7, 0.5
    D = 2
    nets = _networks(name, lyapunov_hidden_activation="relu", lyapunov_hidden_sizes=[2 * D, 2 * D], lyapunov_output_dim=D)
    _identity_lyapunov(nets, D)
    seen = {}
    ver = msacl_b200.create_certifier(networks=nets, env_name=name, num_states=N, horizon=T, seed=seed, init=init, alpha1=alpha1,
                                      rollout_engine=engine, chunk_steps=6, trace=lambda k0, ob, v, d: seen.setdefault(k0, ob.cpu().numpy()[0]))
    rep = ver.run()
    ids = np.arange(N, dtype=np.uint64)
    if init == "reset":
        o0 = oroll.philox_reset(name, seed, ids, np.zeros(N, np.int64))["obs"]
    else:
        u = [ophx.u01(ophx.philox4x32_10(ids & ophx.MASK, ids >> np.uint64(32), np.uint64(j), np.uint64(0x63657274), seed, 0)[0])
             for j in range(D)]
        lo, hi = np.float32(-10.0), np.float32(10.0)
        o0 = np.stack([(lo + (hi - lo) * uj.astype(np.float32)).astype(np.float32) for uj in u], 1)
    np.testing.assert_array_equal(seen[0], o0)                     # the kernel's initial states, bit for bit
    o, done = _oracle_closed_loop(name, o0, T)
    V = (o.astype(np.float64) ** 2).sum(-1).astype(np.float32)
    want = ocert.check(o, V, done, T, lya_eta=ETA, alpha1=alpha1, alpha2=A2)
    got = _host_records(ver.records)
    near = _margins_near(o, V, T, np.minimum(want["end_step"], got["end_step"]), alpha1, A2)
    ok = ~near
    for k in ("flags", "end_step", "first_violation", "first_decrease"):
        np.testing.assert_array_equal(got[k][ok], want[k][ok], err_msg=k)
    assert near.sum() <= max(20, N // 1000), near.sum()
    ws = _oracle_summary(want, T)
    assert rep.num_states == N
    assert abs(rep.certified - ws["certified"]) <= near.sum() and abs(rep.escaped - ws["escaped"]) <= near.sum()
    if init != "reset":
        assert rep.escaped > 0 and rep.certified < N
    assert rep.bound_lo == 0 and rep.bound_hi == 0 and rep.nonfinite == 0      # V = |o|^2 sits well inside [0.5, 2] |o|^2
    print(name, init, engine, rep.to_json())


@pytest.mark.parametrize("hidden,out,act", [([256, 256], 256, "tanh"), ([64, 32], 16, "tanh"), ([48, 40], 8, "relu")])
def test_verifier_v_matches_torch_lyapunov(hidden, out, act):
    import msacl_b200
    name, N, T = "DuctedFan", 3000, 7
    torch.manual_seed(3)
    nets = _networks(name, lyapunov_hidden_sizes=hidden, lyapunov_output_dim=out, lyapunov_hidden_activation=act)
    chunks = []
    ver = msacl_b200.create_certifier(networks=nets, env_name=name, num_states=N, horizon=T, seed=1, chunk_steps=3,
                                      trace=lambda k0, ob, v, d: chunks.append((ob.clone(), v.clone(), None if d is None else d.clone())))
    ver.run()
    for ob, v, d in chunks:
        x = ob.reshape(-1, ob.shape[-1])
        with torch.no_grad():
            want = nets.lyapunov(x)
        got = v.reshape(-1)
        live = torch.isfinite(want)
        torch.testing.assert_close(got[live], want[live], rtol=2e-5, atol=1e-6 * float(want[live].abs().max()))
    np.testing.assert_array_equal(ver.records["v0"].cpu().numpy(), chunks[0][1][0].cpu().numpy())


def test_verifier_uses_fresh_policy_weights():
    """FusedAdam writes the policy through raw pointers (torch's _version is unchanged): a second run() of the same verifier
    must see the new weights, exactly as a freshly built verifier does."""
    import msacl_b200
    from msacl_b200.learner import FusedAdam
    name, N, T = "TwoLink", 8192, 12
    torch.manual_seed(0)
    nets = _networks(name)
    kw = dict(networks=nets, env_name=name, num_states=N, horizon=T, seed=5)
    ver = msacl_b200.create_certifier(**kw)
    first = ver.run()
    worst1 = ver.records["worst_ratio"].clone()
    params = list(nets.policy.parameters())
    versions = [p._version for p in params]
    nets.policy_optimizer.param_groups[0]["lr"] = 0.05
    adam = FusedAdam(nets.policy_optimizer, params)
    g = torch.Generator(device="cuda").manual_seed(1)
    adam.step([(torch.randn((1,) + tuple(p.shape), device="cuda", generator=g), 1) for p in params])
    torch.cuda.synchronize()
    assert [p._version for p in params] == versions
    second = ver.run()
    fresh_ver = msacl_b200.create_certifier(**kw)
    fresh = fresh_ver.run()
    assert second == fresh
    for k, v in ver.records.items():
        assert torch.equal(v, fresh_ver.records[k]), k
    assert not torch.equal(worst1, ver.records["worst_ratio"]) or first != second


@pytest.mark.parametrize("name,init", [("Pendulum", "reset"), ("SingleTrackCar", ("box", -0.5, 0.5)), ("QuadTracking", "reset")])
def test_sharding_invariance(name, init):
    """N states as one shard and as two shards (env_base): identical per-state records and combined counters."""
    import msacl_b200
    from msacl_b200 import distributed as mdist
    from msacl_b200.certify import SUM_HIST
    N, T, seed = 5000, 10, 3
    torch.manual_seed(4)
    nets = _networks(name)
    kw = dict(networks=nets, env_name=name, horizon=T, seed=seed, init=init, chunk_steps=4)
    whole = msacl_b200.create_certifier(num_states=N, **kw)
    rep = whole.run()
    parts, sums = [], []
    for lo, hi in [mdist.shard_env_range(N, r, 2) for r in range(2)]:
        v = msacl_b200.create_certifier(num_states=hi - lo, **kw)
        summary = torch.zeros(SUM_HIST + T, dtype=torch.int64, device="cuda")
        chk = v._run_shard(lo, hi - lo, summary)
        parts.append((chk, summary))
        sums.append(summary.clone())
    for k in whole.records:
        cat = torch.cat([chk.records()[k] for chk, _ in parts])
        assert torch.equal(cat, whole.records[k]), k
    total = sum(s for s in sums)
    key = min(int(s[mdist.CERT_CSTAR_KEY]) for s in sums)
    c_star = mdist.float_from_order_key(key)
    roa = sum(chk.count_below(c_star, s) for chk, s in parts)
    assert c_star == rep.c_star and roa == rep.roa_count
    assert total[1:9].tolist() == [rep.nonfinite, rep.bound_lo, rep.bound_hi, rep.decrease, rep.escaped, rep.not_exp_stable,
                                   rep.certified, rep.inconsistent]
    assert total[SUM_HIST:].tolist() == rep.first_decrease_hist


def test_quadtracking_full_size_subset_replay():
    """2^21 QuadTracking states x T = 20 on the tc engine: the report is consistent, and a random subset of >= 4096 states
    replayed through the oracle on the kernel's own observations and V (closed-loop round-off of the split-bf16 actor does
    not enter) has exactly the kernel's flags away from thresholds."""
    import msacl_b200
    name, N, T = "QuadTracking", 1 << 21, 20
    torch.manual_seed(0)
    nets = _networks(name)
    rng = np.random.default_rng(11)
    ids = np.unique(np.concatenate([np.arange(128), np.arange(N - 128, N), rng.choice(N, 4096, replace=False)]))
    idx = torch.as_tensor(ids, device="cuda")
    o = np.zeros((T + 1, len(ids), 12), np.float32)
    V = np.zeros((T + 1, len(ids)), np.float32)
    done = np.zeros((T + 1, len(ids)), np.uint8)

    def trace(k0, ob, v, d):
        kv = ob.shape[0]
        o[k0:k0 + kv] = ob[:, idx].cpu().numpy()
        V[k0:k0 + kv] = v[:, idx].cpu().numpy()
        if d is not None:
            done[k0:k0 + kv] = d[:, idx].cpu().numpy()

    ver = msacl_b200.create_certifier(networks=nets, env_name=name, num_states=N, horizon=T, seed=2, rollout_engine="tc", trace=trace)
    rep = ver.run()
    assert rep.num_states == N and 0 <= rep.certified <= N and rep.roa_count <= N and rep.nonfinite == 0
    assert rep.certified <= N - max(rep.bound_lo, rep.bound_hi, rep.decrease, rep.escaped)
    assert sum(rep.first_decrease_hist) == rep.decrease
    assert rep.roa_fraction == rep.roa_count / N
    # replay: after the first done the rollout autoresets, the checker ignores those steps -- and so does the oracle
    want = ocert.check(o, V, done, T, lya_eta=ETA, alpha1=A1, alpha2=A2)
    got = _host_records({k: v[idx] for k, v in ver.records.items()})
    _assert_records_equal(got, want)                      # same inputs, float64 comparisons: exact
    print(rep.to_json())
