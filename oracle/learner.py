"""Oracle (test infrastructure): the four MSACL learner losses and their parameter gradients in float64.

torch on the CPU in float64 with autograd, restating RL/algorithm/msacl.py:227-438 from a state dict (the reference's
ApproxContainer keys: `q1.q.0.weight`, `lyapunov.lya.0.weight`, `policy.policy.0.weight`, `log_alpha`, ...):
  critic loss      :227-262   soft-TD backup with alpha = exp(log_alpha), mean squared error of both critics
  Lyapunov risk    :265-336   the formulas of oracle/targets.py written in torch so that autograd reaches the network;
                              V(obs) is evaluated twice, as the reference does (:289, :317)
  policy loss      :349-411   rsample on given N(0,1) draws, torch.minimum routing (half the gradient to each side on a
                              tie), entropy term, stability advantage (unbiased std + 1e-8), PPO-clipped surrogate on
                              step 0 of every window
  entropy coef.    :425-438   loss_alpha = exp(log_alpha) (entropy - target) and one Adam step on log_alpha
Every network is the reference's Linear-act-...-Linear stack (mlp.py:18-33); its activations are arguments.  Nothing
here launches a kernel: the oracle checks the CUDA learner and must not share code with it.
"""
import math

import torch

EPS = 1e-6                       # act_distribution_cls.py:7
f64 = torch.float64
ACT = {"relu": torch.relu, "tanh": torch.tanh}

DEFAULTS = dict(gamma=0.99, lya_eta=0.15, retrace_lambda=0.95, alpha1=1.0, alpha2=2.0, lya_diff_scale=1.0,
                lya_positive_scale=1.0, clip_coef=0.1, min_log_std=-20.0, max_log_std=1.0, value_act="relu",
                lyapunov_act="tanh", policy_act="relu")


def _cfg(cfg):
    out = dict(DEFAULTS)
    out.update(cfg or {})
    return out


def _t(x):
    return torch.as_tensor(x).detach().to(f64)


def params(sd, prefix, grad=True):
    """float64 leaf copies of the tensors of `sd` under `prefix` (e.g. "q1.q."), keyed by their full names."""
    return {k: _t(v).clone().requires_grad_(grad) for k, v in sd.items() if k.startswith(prefix)}


def mlp(p, prefix, x, act):
    """Linear-act-...-Linear (mlp.py:18-33) over the parameters `p[prefix + "<i>.weight"]`, in module-index order."""
    idx = sorted({int(k[len(prefix):].split(".")[0]) for k in p if k.startswith(prefix)})
    for j, i in enumerate(idx):
        x = x @ p[f"{prefix}{i}.weight"].T + p[f"{prefix}{i}.bias"]
        if j < len(idx) - 1:
            x = ACT[act](x)
    return x


def coefficients(n_step, lya_eta=0.15, retrace_lambda=0.95, alpha1=1.0, alpha2=2.0):
    """msacl.py:153-164 in float64 -> (start_obs_norm_coef, lya_diff_coef, start_lya_coef), [n]."""
    k = torch.arange(n_step, dtype=f64)
    son = ((1 - lya_eta) ** (k + 1) * (alpha2 / alpha1)) ** 0.5
    lam = retrace_lambda ** k
    return son, lam / lam.sum(), (1 - lya_eta) ** (k + 1)


# ---- TanhGaussDistribution (act_distribution_cls.py:30-95)
def _split_logits(logits, c):
    mean, log_std = torch.chunk(logits, 2, dim=-1)
    return mean, torch.clamp(log_std, c["min_log_std"], c["max_log_std"]).exp()          # mlp.py:134-135


def _normal_logp(u, mean, std):
    return (-((u - mean) ** 2) / (2 * std ** 2) - std.log() - math.log(math.sqrt(2 * math.pi))).sum(-1)


def rsample(mean, std, eps, low, high):
    """-> (action, log-prob, u) of the tanh-squashed Gaussian on explicit N(0,1) draws."""
    half, mid = (high - low) / 2, (high + low) / 2
    u = mean + std * eps
    th = torch.tanh(u)
    logp = _normal_logp(u, mean, std) - torch.log(1 + EPS - th ** 2).sum(-1) - torch.log(half).sum(-1)
    return half * th + mid, logp, u


def log_prob(mean, std, act, low, high):
    half, mid = (high - low) / 2, (high + low) / 2
    u = torch.atanh((1 - EPS) * (2 * act - 2 * mid) / (2 * half))
    return _normal_logp(u, mean, std) - torch.log(half * (1 + EPS - torch.tanh(u) ** 2)).sum(-1)


def _bounds(sd):
    return _t(sd["policy.act_low_lim"]), _t(sd["policy.act_high_lim"])


def _batch(batch):
    return {k: _t(v) for k, v in batch.items()}


# ---- losses over network outputs (the golden files record these directly)
def critic_loss_from_values(q1, q2, rew, done, next_q1, next_q2, next_logp, gamma, alpha):
    """msacl.py:249-257: backup = rew + (1 - done) gamma (min(Q1', Q2') - alpha logp'), loss = sum of the two MSEs."""
    backup = rew + (1 - done) * gamma * (torch.minimum(next_q1, next_q2) - alpha * next_logp)
    return ((q1 - backup) ** 2).mean() + ((q2 - backup) ** 2).mean()


def lyapunov_risk_from_values(obs, obs2, logp_new, logp_old, v_obs, v_obs2, v_obs_start, coefs, c):
    """msacl.py:280-329 -> dict(loss, loss2, loss3 and the decision quantities).  v_obs_start is the second evaluation of
    V(obs) (:317), whose step-0 column is the start value of the exponential-decrease term."""
    son, diff, sl = coefs
    ratio = torch.exp(logp_new - logp_old)
    isr = torch.cumprod(torch.clamp(ratio, 0, 1), dim=1)
    obs_pow2 = (obs ** 2).sum(-1)
    lo = c["alpha1"] * obs_pow2 - v_obs
    up = v_obs - c["alpha2"] * obs_pow2
    loss2 = (torch.relu(lo).mean() + torch.relu(up).mean()) * c["lya_positive_scale"]
    expanded = torch.sqrt((obs[:, 0, :] ** 2).sum(-1))[:, None] * son[None, :]
    obs2_norm = torch.sqrt((obs2 ** 2).sum(-1))
    esl_arg = expanded - obs2_norm
    esl = torch.where(esl_arg >= 0, 1.0, -1.0).to(f64)
    inner = esl * (v_obs2 - v_obs_start[:, 0:1] * sl[None, :])
    lya_diff = (diff[None, :] * isr * torch.relu(inner)).sum(1)
    loss3 = lya_diff.mean() * c["lya_diff_scale"]
    return dict(loss=loss2 + loss3, loss2=loss2, loss3=loss3, lo=lo, up=up, esl=esl, esl_arg=esl_arg, inner=inner,
                log_ratio=logp_new - logp_old)


def stability_advantage(v_obs0, v_obs2, coefs):
    """msacl.py:392-400 -> batch-normalised advantage [B] (unbiased std + 1e-8)."""
    _, diff, sl = coefs
    raw = (diff[None, :] * (v_obs0[:, None] * sl[None, :] - v_obs2)).sum(1)
    return (raw - raw.mean()) / (raw.std(unbiased=True) + 1e-8)


def clipped_surrogate(new_logp0, old_logp0, adv, clip_coef):
    """msacl.py:385-387,402-405: mean(min(ratio adv, clamp(ratio, 1 - c, 1 + c) adv))."""
    ratio = torch.exp(new_logp0 - old_logp0)
    return torch.min(ratio * adv, torch.clamp(ratio, 1 - clip_coef, 1 + clip_coef) * adv).mean()


# ---- the four updates from a state dict
def _grads(loss, p, keep=False):
    g = torch.autograd.grad(loss, list(p.values()), allow_unused=True, retain_graph=keep)
    return {k: (torch.zeros_like(v) if gi is None else gi) for (k, v), gi in zip(p.items(), g)}


def critic_update(sd, batch, eps, cfg=None):
    """_q_update (msacl.py:227-262).  eps: N(0,1) draws [B, n, A] of the next-action rsample.
    -> (loss_q, {q1.* / q2.* name: float64 gradient}, info with q1_mean, q2_mean and the backup)."""
    c, d = _cfg(cfg), _batch(batch)
    p = {**params(sd, "q1.q."), **params(sd, "q2.q.")}
    tp = {**params(sd, "q1_target.q.", False), **params(sd, "q2_target.q.", False), **params(sd, "policy.policy.", False)}
    low, high = _bounds(sd)
    alpha = math.exp(float(sd["log_alpha"]))
    xq = torch.cat([d["obs"], d["act"]], -1)
    q1, q2 = mlp(p, "q1.q.", xq, c["value_act"])[..., 0], mlp(p, "q2.q.", xq, c["value_act"])[..., 0]
    with torch.no_grad():
        mean, std = _split_logits(mlp(tp, "policy.policy.", d["obs2"], c["policy_act"]), c)
        next_act, next_logp, _ = rsample(mean, std, _t(eps), low, high)
        xq2 = torch.cat([d["obs2"], next_act], -1)
        nq1, nq2 = mlp(tp, "q1_target.q.", xq2, c["value_act"])[..., 0], mlp(tp, "q2_target.q.", xq2, c["value_act"])[..., 0]
    loss = critic_loss_from_values(q1, q2, d["rew"], d["done"], nq1, nq2, next_logp, c["gamma"], alpha)
    return loss.detach(), _grads(loss, p), dict(q1=q1.detach(), q2=q2.detach(), q1_mean=q1.detach().mean(), q2_mean=q2.detach().mean())


def policy_log_prob(sd, batch, cfg=None):
    """log pi(act | obs) of the stored actions under the policy of `sd` ([B, n], no gradient)."""
    c, d = _cfg(cfg), _batch(batch)
    p = params(sd, "policy.policy.", False)
    mean, std = _split_logits(mlp(p, "policy.policy.", d["obs"], c["policy_act"]), c)
    return log_prob(mean, std, d["act"], *_bounds(sd))


def lyapunov_update(sd, batch, cfg=None, logp_new=None):
    """_lyapunov_update (msacl.py:265-336).  logp_new: log pi(act | obs) [B, n]; computed from the policy of `sd` when
    None.  -> (loss_lya, {lyapunov.* name: float64 gradient}, info with loss2, loss3 and the decision quantities)."""
    c, d = _cfg(cfg), _batch(batch)
    n = d["obs"].shape[1]
    p = params(sd, "lyapunov.lya.")
    V = lambda x: (mlp(p, "lyapunov.lya.", x, c["lyapunov_act"]) ** 2).sum(-1)
    if logp_new is None:
        logp_new = policy_log_prob(sd, batch, cfg)
    coefs = coefficients(n, c["lya_eta"], c["retrace_lambda"], c["alpha1"], c["alpha2"])
    out = lyapunov_risk_from_values(d["obs"], d["obs2"], _t(logp_new), d["logp"], V(d["obs"]), V(d["obs2"]), V(d["obs"]), coefs, c)
    info = {k: v.detach() for k, v in out.items()}
    return out["loss"].detach(), _grads(out["loss"], p), info


def policy_update(sd, batch, eps, cfg=None, terms=False):
    """_policy_update (msacl.py:349-411).  eps: N(0,1) draws [B, n, A] of the new-action rsample.
    -> (loss_policy, {policy.* name: float64 gradient}, info).  info carries the loss parts (q_term = mean(min_q - alpha
    logp_new), surrogate), the entropy, the decision quantities and, with terms=True, the gradient of each of the three
    terms of the loss on its own: "critic" (-mean min_q), "entropy" (alpha mean logp_new) and "surrogate" (-L_lya)."""
    c, d = _cfg(cfg), _batch(batch)
    B, n = d["rew"].shape
    p = params(sd, "policy.policy.")
    qp = {**params(sd, "q1.q.", False), **params(sd, "q2.q.", False), **params(sd, "lyapunov.lya.", False)}
    low, high = _bounds(sd)
    alpha = math.exp(float(sd["log_alpha"]))
    logits = mlp(p, "policy.policy.", d["obs"], c["policy_act"])
    mean, std = _split_logits(logits, c)
    new_act, new_logp, u = rsample(mean, std, _t(eps), low, high)
    xq = torch.cat([d["obs"], new_act], -1)
    q1, q2 = mlp(qp, "q1.q.", xq, c["value_act"])[..., 0], mlp(qp, "q2.q.", xq, c["value_act"])[..., 0]
    min_q = torch.minimum(q1, q2)
    q_term = (min_q - alpha * new_logp).mean()
    new_logp_old_act = log_prob(mean, std, d["act"], low, high)
    coefs = coefficients(n, c["lya_eta"], c["retrace_lambda"], c["alpha1"], c["alpha2"])
    with torch.no_grad():
        V = lambda x: (mlp(qp, "lyapunov.lya.", x, c["lyapunov_act"]) ** 2).sum(-1)
        adv = stability_advantage(V(d["obs"][:, 0]), V(d["obs2"]), coefs)
    surrogate = clipped_surrogate(new_logp_old_act[:, 0], d["logp"][:, 0], adv, c["clip_coef"])
    loss = -q_term - surrogate
    grads = _grads(loss, p, keep=terms)
    log_std = torch.chunk(logits, 2, dim=-1)[1]
    info = dict(q_term=q_term.detach(), surrogate=surrogate.detach(), entropy=-new_logp.detach().mean(), q1=q1.detach(),
                q2=q2.detach(), u=u.detach(), log_std=log_std.detach(), adv=adv,
                log_ratio0=(new_logp_old_act[:, 0] - d["logp"][:, 0]).detach())
    if terms:
        info["terms"] = {"critic": _grads(-min_q.mean(), p, True), "entropy": _grads(alpha * new_logp.mean(), p, True),
                         "surrogate": _grads(-surrogate, p)}
    return loss.detach(), grads, info


def alpha_update(log_alpha, entropy, target_entropy, lr, betas=(0.9, 0.999), eps=1e-8, step=1, exp_avg=0.0, exp_avg_sq=0.0,
                 alpha_bound=None):
    """_alpha_update (msacl.py:425-438): gradient exp(log_alpha) (entropy - target) and one torch.optim.Adam step (step = the
    step number after this one) in float64, then the optional clamp to log(alpha_bound).
    -> (new log_alpha, exp_avg, exp_avg_sq, gradient)."""
    b1, b2 = betas
    g = math.exp(log_alpha) * (entropy - target_entropy)
    m = b1 * exp_avg + (1 - b1) * g
    v = b2 * exp_avg_sq + (1 - b2) * g * g
    la = log_alpha - lr / (1 - b1 ** step) * m / (math.sqrt(v) / math.sqrt(1 - b2 ** step) + eps)
    if alpha_bound is not None:
        la = min(la, math.log(alpha_bound))
    return la, m, v, g
