#!/usr/bin/env python
"""MSACL training loop entirely on one B200: fused rollout sampler -> device replay ring -> MSACL learner
(target kernels) -> greedy evaluator.  Mirrors `example/msacl_train.py` + `NstepOffSerialTrainer`
(RL/trainer/nstep_off_serial_trainer.py:22-162) with the reference's default hyper-parameters; only
`env_num` is raised (the GPU steps thousands of envs per launch) and logging is plain stdout.

    python examples/msacl_train_b200.py --env_name VanderPol --max_iteration 2000

With --certify_states N the trained controller's Lyapunov certificate is then checked on N initial states (msacl_b200.
create_certifier; an empirical check over the sampled states and n_step steps, not a proof) and the report printed as JSON.
"""
import argparse
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

import msacl_b200  # noqa: E402
from msacl_b200.evaluator import B200Evaluator  # noqa: E402
from msacl_b200.specs import get_spec  # noqa: E402


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--env_name", default="VanderPol")
    p.add_argument("--env_num", type=int, default=1024)
    p.add_argument("--sample_batch_size", type=int, default=20)
    p.add_argument("--n_step", type=int, default=20)
    p.add_argument("--replay_batch_size", type=int, default=256)
    p.add_argument("--buffer_warm_size", type=int, default=5000)
    p.add_argument("--buffer_max_size", type=int, default=1_000_000)
    p.add_argument("--max_iteration", type=int, default=2000)
    p.add_argument("--eval_interval", type=int, default=500)
    p.add_argument("--num_eval_episode", type=int, default=64)
    p.add_argument("--rollout_engine", default="tc")
    p.add_argument("--seed", type=int, default=0)
    p.add_argument("--certify_states", type=int, default=0, help="after training, check the Lyapunov certificate on this many "
                   "initial states (0: skip)")
    a = vars(p.parse_args())
    spec = get_spec(a["env_name"])
    torch.manual_seed(a["seed"])
    kw = dict(a, algorithm="msacl", obs_dim=spec.obs_dim, act_dim=spec.act_dim, action_type="continu",
              action_low_limit=spec.act_low, action_high_limit=spec.act_high, env_seed=a["seed"], reward_scale=100.0,
              cost_scale=100.0, noise_params=None, target_value=0.0, gamma=0.99, retrace_lambda=0.95, lya_eta=0.15, tau=0.005,
              alpha=1.0, policy_frequency=2, target_network_frequency=1, lya_diff_scale=10.0, lya_positive_scale=1.0,
              alpha1=1, alpha2=2, clip_coef=0.1, q_learning_rate=1e-3, lyapunov_learning_rate=1e-3, policy_learning_rate=3e-4,
              alpha_learning_rate=1e-3, lyapunov_output_dim=256, eval_env_seed=2)
    alg = msacl_b200.create_alg(**kw)
    sampler = msacl_b200.create_sampler(**kw)
    buffer = msacl_b200.create_buffer(**kw)
    evaluator = B200Evaluator(networks=alg.networks, **kw)
    sampler.networks = alg.networks                           # nstep_off_serial_trainer.py:33-35
    while buffer.size < a["buffer_warm_size"]:                # :61-63
        buffer.add_batch(sampler.sample()[0])
    t0 = time.time()
    for it in range(1, a["max_iteration"] + 1):               # :75-147
        samples, _ = sampler.sample()
        buffer.add_batch(samples)
        info = alg.model_update(buffer.sample_batch(a["replay_batch_size"]), it)
        if it % a["eval_interval"] == 0 or it == 1:
            trm, trs, tcm, tcs = evaluator.run_evaluation(it)
            env_steps = sampler.get_total_sample_number()
            print(f"iter {it:6d}  env-steps {env_steps:10d}  TRM {trm:10.3f} +- {trs:8.3f}  TCM {tcm:10.4f} +- {tcs:8.4f}  "
                  f"loss_q {info['Loss/Critic loss-RL iter'] if info else float('nan'):10.3f}  wall {time.time() - t0:6.1f}s", flush=True)
    if a["certify_states"] > 0:
        report = msacl_b200.create_certifier(networks=alg.networks, env_name=a["env_name"], num_states=a["certify_states"],
                                             horizon=a["n_step"], lya_eta=kw["lya_eta"], alpha1=kw["alpha1"], alpha2=kw["alpha2"],
                                             seed=a["seed"], rollout_engine=a["rollout_engine"]).run()
        print("certificate", report.to_json(), flush=True)


if __name__ == "__main__":
    main()
