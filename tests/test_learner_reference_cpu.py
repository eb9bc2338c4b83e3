"""Pins the float64 learner oracle (oracle/learner.py) to the reference's recorded runs, so that the GPU gradient tests
(tests/test_gpu_learner_grads.py) compare the CUDA learner with something that is itself checked.  CPU only."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import learner as ol


def _lya_sd(g):
    return {"lyapunov." + str(n): g["lya_param_" + str(n)] for n in g["lya_param_names"]}


def test_lyapunov_parameter_gradients_match_reference():
    """Float64 autograd of the Lyapunov risk through the rebuilt net (V(obs) evaluated twice) vs the reference's recorded
    parameter gradients, at the tolerance of the NumPy oracle's own test; and the recorded loss."""
    g = load_golden("msacl_targets_TwoLink.npz")
    batch = {k: g[k] for k in ("obs", "obs2", "logp", "rew")}
    loss, grads, info = ol.lyapunov_update(_lya_sd(g), batch, dict(lya_diff_scale=10.0), logp_new=g["logp_new"])
    for n in g["lya_param_names"]:
        ref = g["lya_grad_" + str(n)]
        np.testing.assert_allclose(grads["lyapunov." + str(n)].numpy(), ref, rtol=2e-4, atol=2e-6 * max(1.0, np.abs(ref).max()),
                                   err_msg=str(n))
    np.testing.assert_allclose(float(loss), float(g["loss_lya"]), rtol=2e-6)
    # the recording takes both hinges, both ESL labels and active decrease terms under both labels
    assert (info["lo"] > 0).any() or (info["up"] > 0).any()
    assert (info["esl"] > 0).any() and (info["esl"] < 0).any()


def test_lyapunov_values_of_the_rebuilt_net_match_reference():
    g = load_golden("msacl_targets_TwoLink.npz")
    p = ol.params(_lya_sd(g), "lyapunov.lya.", False)
    v = (ol.mlp(p, "lyapunov.lya.", torch.as_tensor(g["obs"]).double(), "tanh") ** 2).sum(-1)
    np.testing.assert_allclose(v.numpy(), g["lya_obs"], rtol=2e-5, atol=1e-6)


def test_critic_loss_matches_reference():
    g = load_golden("msacl_targets_TwoLink.npz")
    t = lambda k: torch.as_tensor(g[k]).double()
    loss = ol.critic_loss_from_values(t("q1"), t("q2"), t("rew"), t("done"), t("next_q1"), t("next_q2"), t("next_logp"),
                                      float(g["gamma"]), float(g["alpha"]))
    np.testing.assert_allclose(float(loss), float(g["loss_q"]), rtol=3e-6)


def test_policy_surrogate_part_matches_reference():
    """loss_policy = -mean(min_q - alpha logp_new) - L_lya: the recorded first part plus the oracle's surrogate (stability
    advantage from the recorded V values, PPO clip on step 0) reproduce the recorded policy loss."""
    g = load_golden("msacl_targets_TwoLink.npz")
    t = lambda k: torch.as_tensor(g[k]).double()
    n = g["obs"].shape[1]
    coefs = ol.coefficients(n)
    for mine, ref in zip(coefs, ("coef_start_obs_norm", "coef_lya_diff", "coef_start_lya")):
        np.testing.assert_allclose(mine.numpy(), g[ref], rtol=2e-6)
    adv = ol.stability_advantage(t("pol_lya_obs0"), t("pol_lya_obs2"), coefs)
    surr = ol.clipped_surrogate(t("pol_new_logp0"), t("logp")[:, 0], adv, 0.1)
    np.testing.assert_allclose(float(-g["policy_q_term"] - surr), float(g["loss_policy"]), rtol=1e-6, atol=1e-6)
    assert abs(float(surr)) > 0.05 * abs(float(g["loss_policy"]))          # the surrogate is a visible part of the loss


def _update_golden():
    g = load_golden("msacl_update_TwoLink.npz")
    sd = {str(k): g["before_" + str(k)] for k in g["state_keys"]}
    batch = {k[5:]: g[k] for k in g if k.startswith("data_")}
    return g, sd, batch


def test_critic_update_matches_recorded_model_update():
    """The recorded model_update's critic loss and Q means, from the state before it and its first rsample draws."""
    g, sd, batch = _update_golden()
    loss, grads, info = ol.critic_update(sd, batch, g["eps_0"], dict(gamma=0.99))
    np.testing.assert_allclose(float(loss), float(g["tb_Loss_Critic_loss-RL_iter"]), rtol=2e-6)
    np.testing.assert_allclose(float(info["q1_mean"]), float(g["tb_MSACL_q1_mean-RL_iter"]), rtol=2e-5)
    np.testing.assert_allclose(float(info["q2_mean"]), float(g["tb_MSACL_q2_mean-RL_iter"]), rtol=2e-5)
    assert set(grads) == {k for k in sd if k.startswith(("q1.q.", "q2.q."))}


def test_lyapunov_update_matches_recorded_model_update():
    """The recorded Lyapunov loss: the critic step and the Polyak update before it do not touch the Lyapunov net or the
    policy, so it is the loss at the state before the update, with logp_new from that policy."""
    g, sd, batch = _update_golden()
    loss, grads, _ = ol.lyapunov_update(sd, batch, dict(lya_diff_scale=10.0))
    np.testing.assert_allclose(float(loss), float(g["tb_Loss_Lyapunov_loss-RL_iter"]), rtol=2e-6)
    assert set(grads) == {k for k in sd if k.startswith("lyapunov.")}


def test_oracle_gradients_match_finite_differences():
    """Float64 autograd of the policy and alpha losses vs central differences on a tiny net, so that the oracle's gradients
    are those of the losses it states (the routing, clamp and clip branches are kept away from their kinks)."""
    gen = torch.Generator().manual_seed(3)
    B, n, D, A, H = 6, 3, 3, 2, 5
    r = lambda *s: torch.randn(*s, generator=gen, dtype=torch.float64)
    sd = {}
    for net, din, dout in (("q1.q.", D + A, 1), ("q2.q.", D + A, 1), ("lyapunov.lya.", D, 4), ("policy.policy.", D, 2 * A)):
        for i, (a, b) in enumerate(((din, H), (H, H), (H, dout))):
            sd[f"{net}{2 * i}.weight"], sd[f"{net}{2 * i}.bias"] = r(b, a) * 0.5, r(b) * 0.1
    sd.update({"policy.act_low_lim": torch.tensor([-2.0, 0.0], dtype=torch.float64), "policy.act_high_lim": torch.tensor([2.0, 3.0], dtype=torch.float64),
               "log_alpha": torch.tensor(-0.3, dtype=torch.float64)})
    batch = dict(obs=r(B, n, D), obs2=r(B, n, D), act=torch.stack([torch.rand(B, n, generator=gen) * 3.6 - 1.8,
                                                                     torch.rand(B, n, generator=gen) * 2.8 + 0.1], -1).double(),
                 rew=r(B, n), done=(torch.rand(B, n, generator=gen) < 0.3).double(), logp=r(B, n))
    eps = r(B, n, A)
    cfg = dict(max_log_std=0.5)
    _, grads, _ = ol.policy_update(sd, batch, eps, cfg)
    for k in ("policy.policy.0.weight", "policy.policy.4.bias"):
        num = torch.zeros_like(sd[k])
        for i in range(sd[k].numel()):
            for s in (1, -1):
                sd2 = dict(sd)
                sd2[k] = sd[k].clone().view(-1)
                sd2[k][i] += s * 1e-6
                sd2[k] = sd2[k].view_as(sd[k])
                num.view(-1)[i] += s * float(ol.policy_update(sd2, batch, eps, cfg)[0]) / 2e-6
        np.testing.assert_allclose(grads[k].numpy(), num.numpy(), rtol=1e-5, atol=1e-8, err_msg=k)
    # one Adam step of log_alpha from a fresh optimizer is lr * sign(gradient)
    la, m, v, g = ol.alpha_update(-0.3, entropy=1.5, target_entropy=-2.0, lr=1e-3)
    assert g > 0 and abs(la - (-0.3 - 1e-3)) < 1e-9
