#!/usr/bin/env python
"""Generate golden vectors by RUNNING THE REFERENCE (read-only at /root/reference).

Run in the build container only:   python tests/golden/make_golden.py
Outputs tests/golden/*.npz (committed).  Nothing here is imported by the product package,
and nothing at test/bench run time reads /root/reference.

Shims (SURVEY.md section 8c): a gymnasium 0.28.1 stub (tests/golden/_gym_stub), np.float_ alias
(RL/utils/common_utils.py:50 uses the removed name), Tensor.cuda -> identity on this CPU-only
host (RL/algorithm/msacl.py:156-164 call .cuda() unconditionally).  The reference sources are
not modified; attribute overrides on *instances* (env.max_step, env.obs, ...) only set state.
"""
import json
import os
import random
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get("MSACL_REFERENCE", "/root/reference")
sys.path.insert(0, os.path.join(HERE, "_gym_stub"))
sys.path.insert(0, REF)
if not hasattr(np, "float_"):
    np.float_ = np.float64
torch.Tensor.cuda = lambda self, *a, **k: self
torch.nn.Module.cuda = lambda self, *a, **k: self

from RL.env.make_env import make_env  # noqa: E402

from golden_params import msacl_init_params, pack_parameters  # noqa: E402

f32 = np.float32
ENVS = ["VanderPol", "Pendulum", "DuctedFan", "TwoLink", "SingleTrackCar", "QuadTracking"]


def new_env(name):
    return make_env(name, 0, 0, False, "golden")().unwrapped


# ------------------------------------------------------------------ A. single env.step cases
def box_cases(name, rng, m=320):
    env = new_env(name)
    low, high = env.observation_space.low, env.observation_space.high
    alow, ahigh = env.action_space.low, env.action_space.high
    d, a = low.shape[0], alow.shape[0]
    obs_in = np.zeros((m, d), f32); step_in = np.zeros(m, np.int32); act = np.zeros((m, a), f32)
    for i in range(m):
        kind = i % 8
        if kind in (0, 1, 2):      # generic in-box state
            o = rng.uniform(low, high) * rng.uniform(0.05, 0.95)
        elif kind == 3:            # small reset-like state
            o = rng.uniform(-0.5, 0.5, size=d) * np.minimum(1.0, high)
        elif kind == 4:            # close to the boundary (termination on/off)
            o = rng.uniform(low, high) * 0.3
            j = rng.integers(d)
            o[j] = (high[j] if rng.random() < 0.5 else low[j]) * rng.uniform(0.9, 1.0)
        elif kind == 5:            # inside the origin box (bonus branch)
            o = rng.uniform(-0.004, 0.004, size=d)
        elif kind == 6:            # time-limit edge
            o = rng.uniform(low, high) * 0.2
        else:
            o = rng.uniform(low, high) * 0.6
        if name == "SingleTrackCar" and i % 16 == 7:
            o[3] = -1.0 + rng.uniform(-0.09, 0.09)     # |v| < 0.1 : kinematic branch
            o[3] = max(o[3], -0.9999)
        obs_in[i] = o.astype(f32)
        step_in[i] = 998 + (i // 8) % 2 if kind == 6 else rng.integers(0, 900)
        u = rng.uniform(alow, ahigh)
        if kind == 5:
            u = u * 0.001
        act[i] = u.astype(f32)
    obs_out = np.zeros_like(obs_in); rew = np.zeros(m, f32)
    term = np.zeros(m, bool); trunc = np.zeros(m, bool)
    for i in range(m):
        env.obs = obs_in[i].copy(); env.current_step = int(step_in[i])
        o, r, te, tr, _ = env.step(act[i].copy())
        assert o.dtype == np.float32 and np.asarray(r).dtype == np.float32, (o.dtype, np.asarray(r).dtype)
        obs_out[i], rew[i], term[i], trunc[i] = o, r, te, tr
    return dict(obs_in=obs_in, step_in=step_in, act=act, obs_out=obs_out, reward=rew, term=term, trunc=trunc)


def quad_hidden(env):
    return dict(x=env.x.copy(), v=env.v.copy(), R=env.R.copy(), Om=env.Omega.copy(),
                t=np.float64(env.current_time), t_last=np.float64(env.t_last[0]),
                Rd_last=np.asarray(env.Rd_last, dtype=np.float64).copy(), obs=env.obs.copy(),
                step=np.int32(env.current_step))


def quad_cases(rng, episodes=10, horizon=36):
    env = new_env("QuadTracking")
    hover = 4.34 * 9.8
    before, after, acts, rews, terms, truncs, resets = [], [], [], [], [], [], []
    for e in range(episodes):
        np.random.seed(1000 + e)            # reset draws the rotation from the global NumPy RNG
        env.reset(seed=500 + e)
        resets.append(quad_hidden(env))
        if e % 3 == 2:
            env.current_step = 1000 - horizon + 3   # reach the time limit inside the episode
        aggressive = e % 5 == 4
        for k in range(horizon):
            if aggressive:
                a = np.array([rng.uniform(0, 85.0), *rng.uniform(-10, 10, size=3)], dtype=f32)
            else:
                a = np.array([hover + rng.normal(0, 2.0), *rng.normal(0, 0.2, size=3)], dtype=f32)
            a = np.clip(a, env.action_space.low, env.action_space.high).astype(f32)
            before.append(quad_hidden(env))
            o, r, te, tr, _ = env.step(a.copy())
            assert np.asarray(r).dtype == np.float32
            after.append(quad_hidden(env)); acts.append(a); rews.append(r); terms.append(te); truncs.append(tr)
            if te or tr:
                break
    out = {}
    for tag, lst in (("in", before), ("out", after), ("reset", resets)):
        for k in lst[0]:
            out[f"{k}_{tag}"] = np.stack([h[k] for h in lst])
    out.update(act=np.stack(acts), reward=np.array(rews, f32), term=np.array(terms), trunc=np.array(truncs))
    return out


# ------------------------------------------------------------------ B. sampler pipeline
def base_args(name, env_num, n_step, buffer_max_size=1000):
    import gymnasium as gym
    probe = gym.vector.SyncVectorEnv([make_env(name, 1, 0, False, "g")])
    sa, so = probe.single_action_space, probe.single_observation_space
    return dict(
        env_name=name, algorithm="msacl", enable_cuda=False, use_gpu=False, env_num=env_num, env_seed=1,
        capture_video=False, target_value=0.0, reward_scale=100.0, cost_scale=100.0,
        value_func_name="ActionValue", value_func_type="MLP", value_hidden_sizes=[256, 256],
        value_hidden_activation="relu", value_output_activation="linear",
        lyapunov_func_name="LyapunovValue", lyapunov_func_type="MLP", lyapunov_hidden_sizes=[256, 256],
        lyapunov_hidden_activation="tanh", lyapunov_output_dim=256, lyapunov_output_activation="linear",
        lyapunov_single_input_dim=False,
        policy_func_name="StochaPolicy", policy_func_type="MLP", policy_act_distribution="TanhGaussDistribution",
        policy_hidden_sizes=[256, 256], policy_hidden_activation="relu", policy_min_log_std=-20, policy_max_log_std=1,
        q_learning_rate=1e-3, lyapunov_learning_rate=1e-3, policy_learning_rate=3e-4, alpha_learning_rate=1e-3,
        lya_diff_scale=10.0, lya_zero_scale=1.0, lya_positive_scale=1.0, gamma=0.99, retrace_lambda=0.95,
        tau=0.005, disable_auto_alpha=False, alpha=1.0, set_alpha_bound=False, alpha_bound=2.0, n_step=n_step,
        policy_frequency=2, target_network_frequency=1, anneal_lr=False, alpha1=1, alpha2=2, lya_eta=0.15,
        clip_coef=0.1, trainer="nstep_off_serial_trainer", max_iteration=1000000, sampler_name="nstep_off_sampler",
        sample_batch_size=20, noise_params=None, buffer_name="nstep_replay_buffer", buffer_warm_size=5000,
        buffer_max_size=buffer_max_size, replay_batch_size=256, obs_dim=so.shape[0], act_dim=sa.shape[0],
        action_type="continu", action_high_limit=sa.high.astype("float32"), action_low_limit=sa.low.astype("float32"),
        batch_size_per_sampler=20, seed=0,
    )


def policy_weights(policy):
    lin = [m for m in policy.policy if isinstance(m, torch.nn.Linear)]
    out = {}
    for i, l in enumerate(lin):
        out[f"W{i}"] = l.weight.detach().numpy().astype(f32).copy()
        out[f"b{i}"] = l.bias.detach().numpy().astype(f32).copy()
    return out


def env_full_state(name, e):
    u = e.unwrapped
    if name == "QuadTracking":
        return quad_hidden(u)
    return dict(obs=u.obs.copy(), step=np.int32(u.current_step))


def sampler_case(name, env_num=4, n_step=5, steps=40, max_step=13, ring=23, seed=7):
    from RL.create_pkg.create_sampler import create_sampler
    from RL.create_pkg.create_buffer import create_buffer
    random.seed(seed); np.random.seed(seed); torch.manual_seed(seed)
    args = base_args(name, env_num, n_step, buffer_max_size=ring)
    sampler = create_sampler(**args)
    buf = create_buffer(**args)
    for e in sampler.envs.envs:
        e.unwrapped.max_step = max_step        # instance attribute: shorter episodes -> truncations
    # make the policy less timid so the box envs also hit their bounds sometimes
    with torch.no_grad():
        last = [m for m in sampler.networks.policy.policy if isinstance(m, torch.nn.Linear)][-1]
        last.bias[: args["act_dim"]] += torch.linspace(-0.5, 0.5, args["act_dim"])
    out = policy_weights(sampler.networks.policy)
    st0 = [env_full_state(name, e) for e in sampler.envs.envs]
    for k in st0[0]:
        out[f"init_{k}"] = np.stack([s[k] for s in st0])
    rec = {k: [] for k in ("eps", "obs", "act", "rew", "cost", "obs2", "done", "logp", "next_obs", "emit")}
    post = {k: [] for k in st0[0]}
    win = {k: [] for k in ("obs", "act", "rew", "cost", "obs2", "done", "logp")}
    ptr_after, size_after = [], []
    a_dim = args["act_dim"]
    rec.update({k: [] for k in ("term", "trunc", "raw_reward", "valid")})
    captured = {}
    real_step = sampler.envs.step

    def spy_step(actions):
        ret = real_step(actions)
        captured["act"] = np.asarray(actions, f32).copy()
        captured["ret"] = ret
        return ret

    sampler.envs.step = spy_step
    for t in range(steps):
        rng_state = torch.get_rng_state()
        z = torch.empty(env_num, a_dim).normal_()        # what Normal.sample() will draw
        torch.set_rng_state(rng_state)
        obs_before = sampler.obs.copy()
        run_before = [len(d) for d in sampler.n_step_buffers]
        exps = sampler._n_step()
        next_obs, raw_rew, terms, truncs, infos = captured["ret"]
        dones = np.logical_or(terms, truncs)
        real_next = np.float32(next_obs).copy()
        for i in range(env_num):
            if dones[i]:
                real_next[i] = infos["final_observation"][i]
        rec["eps"].append(z.numpy().astype(f32)); rec["obs"].append(obs_before)
        rec["next_obs"].append(sampler.obs.copy())
        rec["act"].append(captured["act"]); rec["obs2"].append(real_next)
        rec["done"].append(dones.astype(f32)); rec["term"].append(np.asarray(terms)); rec["trunc"].append(np.asarray(truncs))
        rec["raw_reward"].append(np.float32(raw_rew))
        emit = np.array([run_before[i] + 1 >= n_step for i in range(env_num)])
        assert emit.sum() == len(exps)
        rec["emit"].append(emit)
        rew = np.full(env_num, np.nan, f32); cost = np.full(env_num, np.nan, f32); logp = np.full(env_num, np.nan, f32)
        valid = np.zeros(env_num, bool)
        j = 0
        for i in range(env_num):
            if emit[i]:
                w = exps[j]; j += 1
                rew[i], cost[i], logp[i] = w.n_step_rew[-1], w.n_step_cost[-1], w.n_step_log_prob[-1]
                valid[i] = True
                assert np.array_equal(w.n_step_act[-1], captured["act"][i]) and np.array_equal(w.n_step_obs2[-1], real_next[i])
                for k, src in (("obs", w.n_step_obs), ("act", w.n_step_act), ("rew", w.n_step_rew), ("cost", w.n_step_cost),
                               ("obs2", w.n_step_obs2), ("done", w.n_step_done), ("logp", w.n_step_log_prob)):
                    win[k].append(np.asarray(src, f32))
            elif len(sampler.n_step_buffers[i]):
                d = sampler.n_step_buffers[i][-1]
                rew[i], cost[i], logp[i] = d["rew"], d["cost"], d["log_prob"]
                valid[i] = True
        rec["rew"].append(rew); rec["cost"].append(cost); rec["logp"].append(logp); rec["valid"].append(valid)
        sts = [env_full_state(name, e) for e in sampler.envs.envs]
        for k in post:
            post[k].append(np.stack([s[k] for s in sts]))
        buf.add_batch(exps)
        ptr_after.append(buf.ptr); size_after.append(buf.size)
    for k, v in rec.items():
        out[f"step_{k}"] = np.stack(v)
    for k, v in post.items():
        out[f"post_{k}"] = np.stack(v)
    for k, v in win.items():
        out[f"win_{k}"] = np.stack(v) if v else np.zeros((0,), f32)
    for k, v in buf.n_step_buf.items():
        out[f"ring_{k}"] = v.copy()
    out.update(ptr_after=np.array(ptr_after), size_after=np.array(size_after), n_step=np.int32(n_step),
               max_step=np.int32(max_step), ring=np.int32(ring), act_low=args["action_low_limit"], act_high=args["action_high_limit"])
    return out


# ------------------------------------------------------------------ C. MSACL learner targets
def msacl_case(name="TwoLink", B=48, n_step=20, seed=11):
    from RL.create_pkg.create_alg import create_alg
    random.seed(seed); np.random.seed(seed); torch.manual_seed(seed)
    args = base_args(name, 4, n_step)
    args["replay_batch_size"] = B
    alg = create_alg(**args)
    net = alg.networks
    D, A = args["obs_dim"], args["act_dim"]
    g = torch.Generator().manual_seed(seed)
    lo = torch.as_tensor(args["action_low_limit"]); hi = torch.as_tensor(args["action_high_limit"])
    obs = torch.randn(B, n_step, D, generator=g) * 0.4
    obs2 = obs + 0.05 * torch.randn(B, n_step, D, generator=g)
    obs2[: B // 3] *= 0.6                     # some windows contract (ESL = +1)
    act = lo + (hi - lo) * torch.rand(B, n_step, A, generator=g)
    act = act.clamp(lo * 0.98, hi * 0.98)
    data = dict(obs=obs, act=act, rew=-torch.rand(B, n_step, generator=g) * 50, cost=torch.rand(B, n_step, generator=g),
                obs2=obs2, done=(torch.rand(B, n_step, generator=g) < 0.1).float(), logp=torch.randn(B, n_step, generator=g) - 1.0)
    out = {k: v.numpy().astype(f32) for k, v in data.items()}
    out.update(act_low=args["action_low_limit"], act_high=args["action_high_limit"])
    with torch.no_grad():
        # ---- lyapunov update inputs (network outputs BEFORE the update)
        logits = net.policy(obs); dist = net.create_action_distributions(logits)
        out["logp_new"] = dist.log_prob(act).numpy().astype(f32)
        out["pi_mean"], out["pi_std"] = (x.numpy().astype(f32) for x in torch.chunk(logits, 2, dim=-1))
        out["lya_obs"] = net.lyapunov(obs).numpy().astype(f32)
        out["lya_obs2"] = net.lyapunov(obs2).numpy().astype(f32)
    lya_state = {k: v.clone() for k, v in net.lyapunov.state_dict().items()}
    loss_lya = alg._lyapunov_update(data)
    out["loss_lya"] = f32(loss_lya.item())
    names = [n_ for n_, _ in net.lyapunov.named_parameters()]
    for n_, p in net.lyapunov.named_parameters():
        out["lya_grad_" + n_] = p.grad.numpy().astype(f32).copy()
        out["lya_param_" + n_] = lya_state[n_].numpy().astype(f32).copy()
    out["lya_param_names"] = np.array(names)
    net.lyapunov.load_state_dict(lya_state)     # undo the optimiser step for the next sections
    # ---- q update: replay the rsample noise
    alpha = alg._get_alpha()
    st = torch.get_rng_state()
    eps_q = torch.empty(B, n_step, A).normal_()
    torch.set_rng_state(st)
    with torch.no_grad():
        q1 = net.q1(obs, act); q2 = net.q2(obs, act)
        nl = net.policy(obs2); mean2, std2 = torch.chunk(nl, 2, dim=-1)
        u = mean2 + std2 * eps_q
        next_act = (hi - lo) / 2 * torch.tanh(u) + (hi + lo) / 2
        nd = net.create_action_distributions(nl)
        next_logp = (nd.gauss_distribution.log_prob(u) - torch.log(1 + 1e-6 - torch.tanh(u) ** 2).sum(-1)
                     - torch.log((hi - lo) / 2).sum(-1))
        out["next_q1"] = net.q1_target(obs2, next_act).numpy().astype(f32)
        out["next_q2"] = net.q2_target(obs2, next_act).numpy().astype(f32)
        out["next_logp"] = next_logp.numpy().astype(f32)
        out["q1"], out["q2"] = q1.numpy().astype(f32), q2.numpy().astype(f32)
    loss_q, _, _ = alg._q_update(data)
    out["loss_q"] = f32(loss_q.item()); out["alpha"] = f32(alpha); out["gamma"] = f32(alg.gamma)
    # ---- policy update: replay noise, record pieces
    st = torch.get_rng_state()
    eps_p = torch.empty(B, n_step, A).normal_()
    torch.set_rng_state(st)
    with torch.no_grad():
        nl = net.policy(obs); mean, std = torch.chunk(nl, 2, dim=-1)
        u = mean + std * eps_p
        new_act = (hi - lo) / 2 * torch.tanh(u) + (hi + lo) / 2
        nd = net.create_action_distributions(nl)
        new_act_logp = (nd.gauss_distribution.log_prob(u) - torch.log(1 + 1e-6 - torch.tanh(u) ** 2).sum(-1)
                        - torch.log((hi - lo) / 2).sum(-1))
        min_q = torch.min(net.q1(obs, new_act), net.q2(obs, new_act))
        out["policy_q_term"] = f32((min_q - alg._get_alpha() * new_act_logp).mean().item())
        out["pol_new_logp0"] = nd.log_prob(act)[:, 0].numpy().astype(f32)
        out["pol_lya_obs0"] = net.lyapunov(obs)[:, 0].numpy().astype(f32)
        out["pol_lya_obs2"] = net.lyapunov(obs2).numpy().astype(f32)
    loss_policy, entropy = alg._policy_update(data)
    out["loss_policy"] = f32(loss_policy.item()); out["entropy"] = f32(entropy.item())
    out["coef_start_obs_norm"] = alg.start_obs_norm_coef.numpy().astype(f32)[0]
    out["coef_lya_diff"] = alg.lya_diff_coef.numpy().astype(f32)[0]
    out["coef_start_lya"] = alg.start_lya_coef.numpy().astype(f32)[0]
    return out


# ------------------------------------------------------------------ D. one full MSACL.model_update
def msacl_update_case(name="TwoLink", B=32, n_step=20, seed=21):
    """State dict before, batch, the three rsample noise tensors (q update, two policy updates), the
    returned tb_info losses and the state dict after `MSACL.model_update(data, 2)`."""
    from RL.create_pkg.create_alg import create_alg
    random.seed(seed); np.random.seed(seed); torch.manual_seed(seed)
    args = base_args(name, 4, n_step)
    args["replay_batch_size"] = B
    alg = create_alg(**args)
    net = alg.networks
    D, A = args["obs_dim"], args["act_dim"]
    g = torch.Generator().manual_seed(seed)
    lo = torch.as_tensor(args["action_low_limit"]); hi = torch.as_tensor(args["action_high_limit"])
    obs = torch.randn(B, n_step, D, generator=g) * 0.4
    obs2 = obs + 0.05 * torch.randn(B, n_step, D, generator=g)
    obs2[: B // 3] *= 0.6
    act = (lo + (hi - lo) * torch.rand(B, n_step, A, generator=g)).clamp(lo * 0.98, hi * 0.98)
    data = dict(obs=obs, act=act, rew=-torch.rand(B, n_step, generator=g) * 50, cost=torch.rand(B, n_step, generator=g),
                obs2=obs2, done=(torch.rand(B, n_step, generator=g) < 0.1).float(), logp=torch.randn(B, n_step, generator=g) - 1.0)
    out = {"data_" + k: v.numpy().astype(f32) for k, v in data.items()}
    out.update(act_low=args["action_low_limit"], act_high=args["action_high_limit"])
    for k, v in net.state_dict().items():
        out["before_" + k] = v.detach().numpy().copy()
    st = torch.get_rng_state()
    for i in range(3):
        out[f"eps_{i}"] = torch.empty(B, n_step, A).normal_().numpy().astype(f32)
    torch.set_rng_state(st)
    tb = alg.model_update(data, 2)
    for k, v in tb.items():
        if "time" not in k.lower():
            out["tb_" + k.replace("/", "_").replace(" ", "_")] = f32(v)
    out["tb_keys"] = np.array([k for k in tb if "time" not in k.lower()])
    for k, v in net.state_dict().items():
        out["after_" + k] = v.detach().numpy().copy()
    out["state_keys"] = np.array(list(net.state_dict().keys()))
    return out


# ------------------------------------------------------------------ E. NormalizeOrientMatrix incl. the det < 0 branch
def quad_polar_case(seed=31, m=96):
    """Reference NormalizeOrientMatrix (QuadTracking.py:308-315) on (a) the inputs the dynamics produce (a rotation times
    I + h hat(w)) and (b) improper inputs (det < 0) with well separated singular values, which take the column-flip
    branch (:312-314)."""
    from RL.env.QuadTracking import NormalizeOrientMatrix
    from scipy.spatial.transform import Rotation
    rng = np.random.default_rng(seed)
    mats = []
    for i in range(m):
        Q = Rotation.from_rotvec(rng.normal(size=3) * rng.uniform(0.1, 3.0)).as_matrix()
        if i % 2 == 0:
            w = rng.normal(size=3) * rng.uniform(0.1, 12.0)
            hat = np.array([[0, -w[2], w[1]], [w[2], 0, -w[0]], [-w[1], w[0], 0]])
            M = Q @ (np.eye(3) + 0.01 * hat)
        else:
            Q2 = Rotation.from_rotvec(rng.normal(size=3)).as_matrix()
            sv = np.array([rng.uniform(1.2, 1.5), rng.uniform(0.9, 1.1), rng.uniform(0.5, 0.7)])
            M = Q @ np.diag(sv * np.array([1.0, 1.0, -1.0])) @ Q2          # det < 0
        mats.append(M.astype(f32))
    mats = np.stack(mats)
    out = np.stack([NormalizeOrientMatrix(M.copy()) for M in mats])
    assert out.dtype == np.float32
    return dict(mat_in=mats, mat_out=out, det_in=np.linalg.det(mats.astype(np.float64)))


# ------------------------------------------------------------------ F. Evaluator.run_parallel_episodes
def evaluator_case(name, episodes=12, max_step=60, seed=41, bias_shift=(-0.6, 0.9), spread=0.97):
    """Reference `Evaluator.run_parallel_episodes` (RL/trainer/evaluator.py:141-204) with recorded policy weights and
    recorded initial env states: the vector env's reset is called once by this script (states recorded), then
    `envs.reset` on the INSTANCE returns those observations, so the evaluation starts from known states."""
    from RL.trainer.evaluator import Evaluator
    random.seed(seed); np.random.seed(seed); torch.manual_seed(seed)
    args = base_args(name, episodes, 20)
    args.update(eval_env_seed=seed, num_eval_episode=episodes, is_render=False, save_folder="/tmp/msacl_golden_eval",
                is_parallel_eval=True)
    ev = Evaluator(**args)
    with torch.no_grad():      # a livelier policy: some episodes leave the box before the time limit
        last = [m for m in ev.networks.policy.policy if isinstance(m, torch.nn.Linear)][-1]
        last.bias[: args["act_dim"]] += torch.linspace(bias_shift[0], bias_shift[1], args["act_dim"])
    out = policy_weights(ev.networks.policy)
    for e in ev.envs.envs:
        e.unwrapped.max_step = max_step
    obs0, _ = ev.envs.reset(seed=seed)
    if name != "QuadTracking":     # spread the initial states over the box so that terminations happen
        rng = np.random.default_rng(seed)
        hi = ev.envs.single_observation_space.high
        for i, e in enumerate(ev.envs.envs):
            if i % 3 == 0:
                e.unwrapped.obs = (rng.uniform(-spread, spread, size=hi.shape) * hi).astype(f32)
        obs0 = np.stack([e.unwrapped.obs.copy() for e in ev.envs.envs])
    st0 = [env_full_state(name, e) for e in ev.envs.envs]
    for k in st0[0]:
        out[f"init_{k}"] = np.stack([s[k] for s in st0])
    ev.envs.reset = lambda seed=None, options=None: (obs0.copy(), {})
    ep_len = []
    real_step = ev.envs.step
    first_done = np.full(episodes, -1)
    counter = {"t": 0}

    def spy(actions):
        ret = real_step(actions)
        d = np.logical_or(ret[2], ret[3])
        for i in range(episodes):
            if d[i] and first_done[i] < 0:
                first_done[i] = counter["t"] + 1
        counter["t"] += 1
        return ret

    ev.envs.step = spy
    trm, trs, tcm, tcs = ev.run_parallel_episodes()
    out.update(trm=np.float64(trm), trs=np.float64(trs), tcm=np.float64(tcm), tcs=np.float64(tcs),
               first_episode_len=first_done.astype(np.int32), max_step=np.int32(max_step), episodes=np.int32(episodes),
               reward_scale=f32(args["reward_scale"]), cost_scale=f32(args["cost_scale"]))
    return out


def extra_cases():
    """Round-2 additions; separate seeds, so the round-1 files above reproduce bit for bit."""
    path = os.path.join(HERE, "quad_polar.npz")
    np.savez_compressed(path, **quad_polar_case())
    print("wrote", path)
    for name in ("VanderPol", "TwoLink", "QuadTracking"):
        path = os.path.join(HERE, f"evaluator_{name}.npz")
        kw = {"VanderPol": dict(max_step=60), "TwoLink": dict(max_step=60, bias_shift=(-0.2, 0.2), spread=0.45),
              "QuadTracking": dict(max_step=40, bias_shift=(0.0, 0.0))}[name]
        data = evaluator_case(name, **kw)
        np.savez_compressed(path, **data)
        print("wrote", path, {k: data[k] for k in ("trm", "trs", "tcm", "tcs")}, data["first_episode_len"])


def packed_targets_case(seed=11):
    out = msacl_case(seed=seed)
    names = [str(n) for n in out["lya_param_names"]]
    return pack_parameters(out, seed, out["obs"].shape[-1], out["act"].shape[-1], ["lya_param_" + n for n in names],
                           ["lyapunov." + n for n in names], [], [])


def packed_update_case(seed=21):
    out = msacl_update_case(seed=seed)
    D, A = out["data_obs"].shape[-1], out["data_act"].shape[-1]
    keys = [str(k) for k in out["state_keys"]]
    init = [k for k in keys if k in msacl_init_params(seed, D, A)]
    return pack_parameters(out, seed, D, A, ["before_" + k for k in init], init, ["after_" + k for k in keys],
                           ["before_" + k for k in keys])


def tb_tags_case():
    """The reference's TensorBoard tag table (RL/utils/tensorboard_setup.py:13-40): a naming contract with its CSV /
    plotting tools that msacl_b200.trainer.tb_tags keeps."""
    from RL.utils.tensorboard_setup import tb_tags
    path = os.path.join(HERE, "reference_tb_tags.json")
    with open(path, "w") as fh:
        json.dump(tb_tags, fh, indent=1)
        fh.write("\n")
    print("wrote", path)


def main():
    if "--only-extra" in sys.argv:
        return extra_cases()
    if "--only-tags" in sys.argv:
        return tb_tags_case()
    if "--only-update" in sys.argv:
        path = os.path.join(HERE, "msacl_update_TwoLink.npz")
        np.savez_compressed(path, **packed_update_case())
        print("wrote", path)
        return
    rng = np.random.default_rng(20261018)
    for name in ENVS:
        path = os.path.join(HERE, f"env_step_{name}.npz")
        data = quad_cases(rng) if name == "QuadTracking" else box_cases(name, rng)
        np.savez_compressed(path, **data)
        print("wrote", path, {k: v.shape for k, v in data.items() if hasattr(v, "shape")})
    for name in ENVS:
        path = os.path.join(HERE, f"sampler_{name}.npz")
        data = sampler_case(name)
        np.savez_compressed(path, **data)
        print("wrote", path, "windows:", len(data["win_rew"]), "dones:", int(data["step_done"].sum()))
    path = os.path.join(HERE, "msacl_targets_TwoLink.npz")
    np.savez_compressed(path, **packed_targets_case())
    print("wrote", path)
    path = os.path.join(HERE, "msacl_update_TwoLink.npz")
    np.savez_compressed(path, **packed_update_case())
    print("wrote", path)
    extra_cases()
    tb_tags_case()


if __name__ == "__main__":
    main()
