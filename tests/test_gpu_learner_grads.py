"""The learner's parameter gradients BEFORE Adam vs the float64 oracle (oracle/learner.py, pinned to the reference by
tests/test_learner_reference_cpu.py).

Adam hides a gradient's scale: m_hat / (sqrt(v_hat) + eps) is the same for g and c g, and its first step is lr sign(g).
A kernel that halves a whole gradient, or weights one term of the policy loss wrongly, leaves the post-Adam parameters of
test_gpu_algorithm.py / test_gpu_learner.py nearly unchanged.  Here every update starts from the same state snapshot and
runs eagerly; for the fused engine the gradient each FusedAdam receives is captured (its `(partials, nsplit)` list cloned
and the splits summed in float64), for the torch engine `p.grad` is read after the update.  Each parameter tensor is then
compared with the oracle's gradient at that state, and so are the device statistics and log_alpha after the alpha step.

The data are built on the CPU from a seed so that every branch is taken (both hinges, both ESL labels, active decrease
terms under both labels, clip ratios on both sides of 1, done in {0, 1}, min-Q routed to each critic, the surrogate inside
the clip / outside and used / outside and zeroed, log_std clamped on some rows, log_alpha != 0) and no decision lies
within round-off of its threshold; |u| <= 3, so tanh is far from saturation (saturation is a kernel-level case in
tests/test_gpu_learner.py).

Tolerances, per update: relative Frobenius error of every tensor <= FRO, max |g - g_ref| <= MAX * max |g_ref| per tensor,
and the relative Frobenius error of the whole gradient vector <= ALL.  The test also asserts that 1 % of each single term of
the policy gradient (critic path, entropy, surrogate) exceeds ALL, i.e. that a 1 % error in any term would fail.
Measured on one NVIDIA B200 at a 1000 W power limit (worst over the four configurations and both engines):
  FRO   critic 3.8e-6, Lyapunov 8.1e-6, policy 4.2e-6   -> bound 5e-5
  MAX   critic 4.3e-6, Lyapunov 9.8e-6, policy 4.5e-6   -> bound 5e-5
  ALL   critic 2.9e-6, Lyapunov 6.6e-6, policy 3.3e-6   -> bound 5e-5
  statistics (losses, Q means, loss parts, entropy)     8.1e-6 relative -> bound 2.5e-5
  log_alpha after the alpha step                        1.3e-8 absolute -> bound 1e-6
The smallest single term is the critic path of the non-default shape, 4.6 % of the policy gradient, so a 1 % error in it
is a 4.6e-4 error of the whole vector.  The data also keep every ReLU of the policy at least 1e-5 of its input scale from
its kink: a unit within the GEMMs' round-off of the kink took the other branch on the GPU and moved whole rows of the
first-layer gradient (a 6e-4 error that is not a kernel error).
"""
import functools
import math

import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import learner as ol

pytestmark = pytest.mark.gpu

FRO, MAX, ALL, STAT = 5e-5, 5e-5, 5e-5, 2.5e-5

# (env, B, n, network sizes); TwoLink defaults, QuadTracking (D = 12, A = 4, target entropy -5), a non-default shape with
# M = 185 rows (not a multiple of 128), and n_step = 1 (every row is a surrogate row; lyapunov_risk takes its warp-per-window
# kernel)
CASES = {
    "twolink": ("TwoLink", 48, 20, {}),
    "quad": ("QuadTracking", 24, 20, {}),
    "shape": ("DuctedFan", 37, 5, dict(value_hidden_sizes=[128, 64], lyapunov_hidden_sizes=[64, 96], lyapunov_output_dim=32,
                                       policy_hidden_sizes=[96, 320])),
    "n1": ("TwoLink", 128, 1, {}),
}
LOG_CLIP = (math.log(0.9), math.log(1.1))


def _kwargs(name, max_log_std=1.0):
    from msacl_b200.specs import get_spec
    env, B, n, sizes = CASES[name]
    spec = get_spec(env)
    return dict(algorithm="msacl", env_name=env, obs_dim=spec.obs_dim, act_dim=spec.act_dim, n_step=n, action_low_limit=spec.act_low,
                action_high_limit=spec.act_high, q_learning_rate=1e-3, lyapunov_learning_rate=1e-3, policy_learning_rate=3e-4,
                alpha_learning_rate=1e-3, alpha=0.7, lya_diff_scale=10.0, policy_max_log_std=max_log_std, learner_graph=False, **sizes)


def _oracle_cfg(kw):
    return dict(gamma=0.99, lya_diff_scale=kw["lya_diff_scale"], max_log_std=kw["policy_max_log_std"])


def _decisions(sd, batch, eps_p, cfg, clip=0.1):
    """Every branch decision of the three updates at state `sd`, with its distance to the threshold."""
    _, _, lya = ol.lyapunov_update(sd, batch, cfg)
    _, _, pol = ol.policy_update(sd, batch, eps_p, cfg)
    v = lya["up"] + cfg.get("alpha2", 2.0) * (torch.as_tensor(batch["obs"]).double() ** 2).sum(-1)
    scale_v = torch.maximum(v.abs(), (lya["lo"] + v).abs()) + 1e-12
    q1, q2 = pol["q1"], pol["q2"]
    return dict(
        lya=lya, pol=pol,
        m_lo=(lya["lo"].abs() / scale_v), m_up=(lya["up"].abs() / scale_v),
        m_esl=lya["esl_arg"].abs(), m_inner=lya["inner"].abs() / (v.abs().max() + 1e-12),
        m_clip=torch.minimum((pol["log_ratio0"] - LOG_CLIP[0]).abs(), (pol["log_ratio0"] - LOG_CLIP[1]).abs()),
        m_q=(q1 - q2).abs() / torch.maximum(q1.abs().max(), q2.abs().max()),
        m_ls=(pol["log_std"] - cfg["max_log_std"]).abs(), m_kink=_policy_kinks(sd, batch["obs"]))


def _policy_kinks(sd, obs):
    """min over the policy's hidden units of |pre-activation| / sum |input| |weight| per row [B, n]: a unit closer to its ReLU
    kink than the GEMMs' round-off (1.5e-6 of that sum) may take the other branch on the GPU."""
    p = ol.params(sd, "policy.policy.", False)
    x, out = torch.as_tensor(obs).double(), []
    for i in (0, 2):
        w, b = p[f"policy.policy.{i}.weight"], p[f"policy.policy.{i}.bias"]
        pre = x @ w.T + b
        out.append((pre.abs() / (x.abs() @ w.abs().T + b.abs())).min(-1).values)
        x = torch.relu(pre)
    return torch.minimum(*out)


@functools.lru_cache(maxsize=None)
def _case(name):
    """-> (create_alg kwargs, float32 state dict, float32 batch, q eps, policy eps); CPU only, deterministic."""
    from msacl_b200.algorithm import ApproxContainer
    env, B, n, _ = CASES[name]
    kw = _kwargs(name)
    D, A = kw["obs_dim"], kw["act_dim"]
    torch.manual_seed(7)
    sd = {k: v.clone() for k, v in ApproxContainer(**kw).state_dict().items()}
    sd["log_alpha"] = torch.tensor(math.log(0.7), dtype=torch.float32)
    # V(0) = 0, as for a trained certificate, V four times as steep along obs[0] and its mean curvature at 0 set to 1.5 (between
    # alpha1 = 1 and alpha2 = 2): V / |o|^2 then depends strongly on the direction, so that both hinges occur and a state can grow in norm
    # while V falls (ESL -1 with an active decrease term)
    sd["lyapunov.lya.0.weight"][:, 0] *= 4.0
    z = lambda x: ol.mlp(ol.params(sd, "lyapunov.lya.", False), "lyapunov.lya.", x, "tanh")
    J = torch.autograd.functional.jacobian(lambda x: z(x[None])[0], torch.zeros(D, dtype=torch.float64))
    gain = math.sqrt(1.5 * D / float(torch.trace(J.T @ J)))
    sd["lyapunov.lya.4.weight"] *= gain
    sd["lyapunov.lya.4.bias"] *= gain
    sd["lyapunov.lya.4.bias"] -= z(torch.zeros(1, D, dtype=torch.float64))[0].float()
    g = torch.Generator().manual_seed(11)
    U = lambda lo, hi, *s: lo + (hi - lo) * torch.rand(*s, generator=g)
    lo_a, hi_a = sd["policy.act_low_lim"], sd["policy.act_high_lim"]

    def obs_pair(b):              # window scales from 0.05 to 3 (both hinges); obs2 shrinking or growing, turned at random
        sc = torch.exp(U(math.log(0.05), math.log(3.0), b, 1, 1))
        o = torch.randn(b, n, D, generator=g) * sc
        return o, o * U(0.3, 1.6, b, n, 1) + sc * torch.randn(b, n, D, generator=g)

    obs, obs2 = obs_pair(B)
    batch = dict(obs=obs, obs2=obs2, act=(lo_a + hi_a) / 2 + (hi_a - lo_a) / 2 * U(-0.95, 0.95, B, n, A),
                 rew=-U(0, 5, B, n), cost=U(0, 1, B, n), done=(torch.rand(B, n, generator=g) < 0.2).float(), logp=torch.zeros(B, n))
    eps_q = torch.randn(B, n, A, generator=g).clamp(-2.5, 2.5)
    eps_p = torch.randn(B, n, A, generator=g).clamp(-2.5, 2.5)
    # max_log_std in the widest gap between the 60th and 85th percentiles of the policy's log_std: some rows are clamped
    _, _, pol = ol.policy_update(sd, batch, eps_p, _oracle_cfg(kw))
    sd["q2.q.4.bias"] += float((pol["q1"] - pol["q2"]).median())      # Q2 below Q1 on about half of the rows
    ls = pol["log_std"].flatten().sort().values
    i0, i1 = int(0.6 * len(ls)), int(0.85 * len(ls))
    j = i0 + int(torch.argmax(ls[i0 + 1:i1] - ls[i0:i1 - 1]))
    kw = _kwargs(name, float(np.float32((ls[j] + ls[j + 1]) / 2)))
    cfg = _oracle_cfg(kw)
    # stored log-probs: the surrogate's step 0 inside the clip, above it or below it (one third each), other steps +-0.5
    cat = torch.arange(B) % 3
    lr0 = torch.where(cat == 0, U(-0.06, 0.06, B), torch.where(cat == 1, U(0.15, 0.5, B), U(-0.5, -0.15, B)))
    log_ratio = U(-0.5, 0.5, B, n)
    log_ratio[:, 0] = lr0
    for _ in range(20):                            # re-draw the windows / rows that put a decision near its threshold
        batch["logp"] = (ol.policy_log_prob(sd, batch, cfg) - log_ratio.double()).float()
        d = _decisions(sd, batch, eps_p, cfg)
        bad_w = ((d["m_lo"] < 1e-3) | (d["m_up"] < 1e-3) | (d["m_esl"] < 1e-3) | (d["m_inner"] < 1e-4)).any(1) | \
            (d["m_ls"] < 1e-4).flatten(1).any(1) | (d["m_kink"] < 1e-5).any(1)
        bad_r = d["m_q"] < 1e-3
        if not bad_w.any() and not bad_r.any():
            break
        nb = int(bad_w.sum())
        if nb:
            batch["obs"][bad_w], batch["obs2"][bad_w] = obs_pair(nb)
        eps_p[bad_r] = torch.randn(int(bad_r.sum()), A, generator=g).clamp(-2.5, 2.5)
    else:
        raise AssertionError(f"{name}: could not keep every decision away from its threshold")
    return kw, sd, batch, eps_q, eps_p


def _assert_branches(name, sd, batch, eps_p, cfg):
    d = _decisions(sd, batch, eps_p, cfg)
    lya, pol = d["lya"], d["pol"]
    B, n = batch["rew"].shape
    counts = dict(
        lo=int((lya["lo"] > 0).sum()), up=int((lya["up"] > 0).sum()), esl_p=int((lya["esl"] > 0).sum()), esl_m=int((lya["esl"] < 0).sum()),
        inner_p=int(((lya["inner"] > 0) & (lya["esl"] > 0)).sum()), inner_m=int(((lya["inner"] > 0) & (lya["esl"] < 0)).sum()),
        ratio_lt1=int((lya["log_ratio"] < 0).sum()), ratio_gt1=int((lya["log_ratio"] > 0).sum()),
        done0=int((batch["done"] == 0).sum()), done1=int((batch["done"] == 1).sum()),
        q1_min=int((pol["q1"] < pol["q2"]).sum()), q2_min=int((pol["q2"] < pol["q1"]).sum()),
        ls_clamped=int((pol["log_std"] > cfg["max_log_std"]).sum()), ls_free=int((pol["log_std"] < cfg["max_log_std"]).sum()))
    lr0, adv = pol["log_ratio0"], pol["adv"]
    inside = (lr0 > LOG_CLIP[0]) & (lr0 < LOG_CLIP[1])
    used = ((lr0 > LOG_CLIP[1]) & (adv < 0)) | ((lr0 < LOG_CLIP[0]) & (adv > 0))
    counts.update(sur_inside=int(inside.sum()), sur_used=int(used.sum()), sur_zeroed=int((~inside & ~used).sum()))
    assert min(counts.values()) >= 1, (name, counts)
    assert float(sd["log_alpha"]) != 0.0
    assert float(pol["u"].abs().max()) <= 3.0
    margins = {k: float(d[k].min()) for k in ("m_lo", "m_up", "m_esl", "m_inner", "m_clip", "m_q", "m_ls", "m_kink")}
    assert margins["m_lo"] >= 1e-3 and margins["m_up"] >= 1e-3 and margins["m_esl"] >= 1e-3 and margins["m_inner"] >= 1e-4, margins
    assert margins["m_clip"] >= 1e-2 and margins["m_q"] >= 1e-3 and margins["m_ls"] >= 1e-4 and margins["m_kink"] >= 1e-5, margins
    assert float(adv[~inside].abs().min()) > 1e-3
    return pol


def _compare(tag, got, ref):
    """Per-tensor relative Frobenius / max-abs errors and the whole-vector relative error; returns the errors."""
    errs = {}
    num = den = 0.0
    for k, r in ref.items():
        x = got[k].double().cpu().reshape(r.shape)
        e = x - r
        num, den = num + float((e ** 2).sum()), den + float((r ** 2).sum())
        errs[k] = (float(e.norm() / r.norm()), float(e.abs().max() / r.abs().max()))
    errs["all"] = math.sqrt(num / den)
    print(tag, {k: tuple(f"{v:.2e}" for v in e) if isinstance(e, tuple) else f"{e:.2e}" for k, e in errs.items()})
    for k, (fro, mx) in ((k, e) for k, e in errs.items() if k != "all"):
        assert fro <= FRO and mx <= MAX, (tag, k, fro, mx)
    assert errs["all"] <= ALL, (tag, errs["all"])
    return errs


def _rel(a, b):
    return abs(float(a) - float(b)) / max(abs(float(b)), 1e-12)


def _snapshot(alg):
    return {k: v.detach().cpu().clone() for k, v in alg.networks.state_dict().items()}


def _restore(alg, sd):
    alg.networks.load_state_dict({k: v for k, v in sd.items()})      # copies in place: kernel bindings stay valid


@pytest.mark.parametrize("engine", ["fused", "torch"])
@pytest.mark.parametrize("name", list(CASES))
def test_gradients_before_adam_match_float64_oracle(name, engine):
    import msacl_b200
    kw, sd, batch, eps_q, eps_p = _case(name)
    cfg = _oracle_cfg(kw)
    pol = _assert_branches(name, sd, batch, eps_p, cfg)
    alg = msacl_b200.create_alg(learner_engine=engine, **kw)
    assert alg.engine_name == engine and alg.n_step == CASES[name][2]
    if name == "quad":
        assert alg.target_entropy == -5 and kw["obs_dim"] == 12 and kw["act_dim"] == 4
    _restore(alg, sd)
    B, n = batch["rew"].shape
    M = B * n
    d = {k: v.cuda() for k, v in batch.items()}
    eq, ep = eps_q.cuda(), eps_p.cuda()
    net = alg.networks
    sd = _snapshot(alg)

    # oracle at the snapshot
    loss_q, g_q, info_q = ol.critic_update(sd, batch, eps_q, cfg)
    loss_l, g_l, info_l = ol.lyapunov_update(sd, batch, cfg)
    loss_p, g_p, info_p = ol.policy_update(sd, batch, eps_p, cfg, terms=True)

    got = {}
    if engine == "fused":
        fl = alg._fused_learner()
        rec = {}

        def recorder(tag, adam):
            orig = adam.step

            def step(grads):
                rec[tag] = [(t.clone(), s) for t, s in grads]
                return orig(grads)
            return step

        for tag, prefix in (("q1", "q1.q."), ("q2", "q2.q."), ("l", "lyapunov.lya."), ("p", "policy.policy.")):
            adam = getattr(fl, "adam_" + tag)
            adam.step = recorder(tag, adam)

        def grads_of(tag, module, prefix):
            names = [prefix + k for k, _ in module.named_parameters()]
            assert len(rec[tag]) == len(names)
            return {nm: t.double()[:s].sum(0) for nm, (t, s) in zip(names, rec[tag])}

        fl.q_update(d, eq)
        torch.cuda.synchronize()
        got["q"] = {**grads_of("q1", net.q1.q, "q1.q."), **grads_of("q2", net.q2.q, "q2.q.")}
        s = fl.stats[:4].tolist()
        stats_q = dict(loss=(s[0] + s[1]) / M, q1_mean=s[2] / M, q2_mean=s[3] / M)
        _restore(alg, sd)
        fl.lyapunov_update(d)
        torch.cuda.synchronize()
        got["l"] = grads_of("l", net.lyapunov.lya, "lyapunov.lya.")
        s = fl.stats[4:7].tolist()
        stats_l = dict(loss2=(s[0] + s[1]) / M * alg.lya_positive_scale, loss3=s[2] / B * alg.lya_diff_scale)
        _restore(alg, sd)
        fl.policy_update(d, ep)
        torch.cuda.synchronize()
        got["p"] = grads_of("p", net.policy.policy, "policy.policy.")
        s = fl.stats[8:11].tolist()
        stats_p = dict(q_term=s[0] / M, entropy=-s[1] / M, surrogate=s[2] / B)
        fl.alpha_update()
        torch.cuda.synchronize()
        stats_p["entropy_out"] = float(fl.entropy)
    else:
        grad_of = lambda module, prefix: {prefix + k: p.grad.detach().clone() for k, p in module.named_parameters()}
        lq, q1m, q2m = alg._q_update(d, eq)
        got["q"] = {**grad_of(net.q1.q, "q1.q."), **grad_of(net.q2.q, "q2.q.")}
        stats_q = dict(loss=float(lq), q1_mean=float(q1m), q2_mean=float(q2m))
        _restore(alg, sd)
        ll = alg._lyapunov_update(d)
        got["l"] = grad_of(net.lyapunov.lya, "lyapunov.lya.")
        stats_l = dict(loss=float(ll))
        _restore(alg, sd)
        lp, ent = alg._policy_update(d, ep)
        got["p"] = grad_of(net.policy.policy, "policy.policy.")
        stats_p = dict(loss=float(lp), entropy=float(ent))
        alg._alpha_update(ent)
        torch.cuda.synchronize()

    _compare(f"{name}/{engine} critic", got["q"], g_q)
    _compare(f"{name}/{engine} lyapunov", got["l"], g_l)
    _compare(f"{name}/{engine} policy", got["p"], g_p)

    # each term of the policy gradient is large enough that a 1 % error in it alone fails the whole-vector bound
    norm = lambda gs: math.sqrt(sum(float((v ** 2).sum()) for v in gs.values()))
    for term, gt in info_p["terms"].items():
        assert 0.01 * norm(gt) > ALL * norm(g_p), (name, term, norm(gt), norm(g_p))

    # device statistics
    want = dict(loss=float(loss_q), q1_mean=float(info_q["q1_mean"]), q2_mean=float(info_q["q2_mean"]))
    print(name, engine, "critic stats", {k: f"{_rel(v, want[k]):.1e}" for k, v in stats_q.items()})
    for k, v in stats_q.items():
        assert _rel(v, want[k]) <= STAT, (name, engine, k, v, want[k])
    want = dict(loss=float(loss_l), loss2=float(info_l["loss2"]), loss3=float(info_l["loss3"]))
    print(name, engine, "lyapunov stats", {k: f"{_rel(v, want[k]):.1e}" for k, v in stats_l.items()})
    for k, v in stats_l.items():
        assert _rel(v, want[k]) <= STAT, (name, engine, k, v, want[k])
    want = dict(loss=float(loss_p), q_term=float(info_p["q_term"]), surrogate=float(info_p["surrogate"]),
                entropy=float(info_p["entropy"]), entropy_out=float(info_p["entropy"]))
    print(name, engine, "policy stats", {k: f"{_rel(v, want[k]):.1e}" for k, v in stats_p.items()})
    for k, v in stats_p.items():
        assert _rel(v, want[k]) <= STAT, (name, engine, k, v, want[k])

    # log_alpha after one entropy-coefficient step (fresh Adam state) from the oracle's entropy
    ga = net.alpha_optimizer.param_groups[0]
    la, *_ = ol.alpha_update(float(sd["log_alpha"]), float(info_p["entropy"]), float(alg.target_entropy), ga["lr"], ga["betas"], ga["eps"])
    la_got = float(net.log_alpha.detach())
    print(name, engine, f"log_alpha error {abs(la_got - la):.1e}")
    assert abs(la_got - la) <= 1e-6, (la_got, la)
    assert la_got != float(sd["log_alpha"])


def test_fused_lyapunov_backward_chain_matches_reference_param_grads():
    """Reference -> CUDA directly: FusedMLP over [obs; obs2] with the recorded Lyapunov parameters, msacl_lyapunov_risk with
    the recorded logp_new, msacl_sumsq_bwd and the fused backward reproduce the reference's recorded parameter gradients
    (tolerance of the oracle's own test in test_oracle_golden.py)."""
    import msacl_b200
    from msacl_b200 import _lib
    from msacl_b200.algorithm import mlp
    from msacl_b200.learner import FusedMLP
    lib = msacl_b200.load_library()
    g = load_golden("msacl_targets_TwoLink.npz")
    B, n, D = g["obs"].shape
    M = B * n
    names = [str(k) for k in g["lya_param_names"]]
    seq = mlp([D, 256, 256, 256], torch.nn.Tanh).cuda()
    seq.load_state_dict({k[4:]: torch.as_tensor(g["lya_param_" + k]) for k in names})
    fm = FusedMLP(seq, "cuda", 6, sumsq_head=True)
    ws = fm.workspace("train", 2 * M, train=True, sumsq=True)
    cu = lambda k: torch.as_tensor(g[k]).cuda().contiguous()
    obs, obs2, logp_new, logp_old = cu("obs"), cu("obs2"), cu("logp_new"), cu("logp")
    xl = torch.cat([obs.reshape(M, D), obs2.reshape(M, D)]).contiguous()
    z = fm.forward(xl, ws)
    V = ws.v
    son, diff, sl = cu("coef_start_obs_norm"), cu("coef_lya_diff"), cu("coef_start_lya")
    parts = torch.zeros(3, dtype=torch.float64, device="cuda")
    dV = torch.empty(2 * M, device="cuda")
    st = _lib.current_stream()
    _lib.check(lib.msacl_lyapunov_risk(B, n, D, obs.data_ptr(), obs2.data_ptr(), logp_new.data_ptr(), logp_old.data_ptr(), V.data_ptr(),
                                       V[M:].data_ptr(), son.data_ptr(), diff.data_ptr(), sl.data_ptr(), 1.0, 2.0, 10.0, 1.0,
                                       parts.data_ptr(), dV.data_ptr(), dV[M:].data_ptr(), None, None, st))
    dz = torch.empty(2 * M, 256, device="cuda")
    _lib.check(lib.msacl_sumsq_bwd(2 * M, 256, z.data_ptr(), dV.data_ptr(), dz.data_ptr(), st))
    fm.backward(ws, dz)
    loss = float((parts[0] + parts[1]) / M + parts[2] / B * 10.0)
    np.testing.assert_allclose(loss, float(g["loss_lya"]), rtol=2e-5)
    for k, got in zip(names, fm.reduced_grads(ws)):
        ref = g["lya_grad_" + k]
        np.testing.assert_allclose(got.cpu().numpy(), ref, rtol=2e-4, atol=2e-6 * max(1.0, np.abs(ref).max()), err_msg=k)
