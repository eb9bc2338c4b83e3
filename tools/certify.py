#!/usr/bin/env python
"""Check the Lyapunov certificate of a trained checkpoint on the GPU and print the report as one JSON line.

    python tools/certify.py --env_name VanderPol --checkpoint runs/apprfunc/apprfunc_2000.pkl --num_states 1048576

The checkpoint is the trainer's `apprfunc_{iteration}.pkl` (`networks.state_dict()`); it is loaded into an ApproxContainer
built with the network arguments of examples/msacl_train_b200.py (reference defaults, lyapunov_output_dim 256; override
with the flags below).  The result is an empirical check over the sampled initial states and the horizon, not a proof.

With --region LO HI the sound region verifier runs instead (interval branch-and-bound over the box [LO, HI]^obs_dim minus
the inner box --inner, for --steps closed-loop steps, cells down to --max_depth) and its RegionReport is printed:

    python tools/certify.py --env_name VanderPol --checkpoint apprfunc_2000.pkl --region -2 2 --inner 0.1 --max_depth 30

--dist_obs, --dist_act and --dist_state (half-widths: one value, or one per dimension) run it under bounded sensor noise,
actuator and process disturbances; the line then has a "disturbance" field.  --margin S_MAX bisects the largest scale
s in [0, S_MAX] of those boxes that is still proven invariant and adds a "margin" field (s_proven is null with
"nominal_proven": false when the undisturbed loop is not proven); the report is that of the run at s_proven:

    python tools/certify.py --env_name VanderPol --checkpoint apprfunc_2000.pkl --region -1 1 --dist_state 1e-3 --margin 0.1
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

import msacl_b200  # noqa: E402
from msacl_b200.algorithm import ApproxContainer  # noqa: E402
from msacl_b200.specs import get_spec  # noqa: E402


def network_kwargs(env_name, lyapunov_output_dim=256):
    """The ApproxContainer arguments of examples/msacl_train_b200.py (learning rates only size the unused optimisers)."""
    spec = get_spec(env_name)
    return dict(obs_dim=spec.obs_dim, act_dim=spec.act_dim, action_low_limit=spec.act_low, action_high_limit=spec.act_high,
                lyapunov_output_dim=lyapunov_output_dim, q_learning_rate=1e-3, lyapunov_learning_rate=1e-3,
                policy_learning_rate=3e-4, alpha_learning_rate=1e-3)


def main(argv=None):
    p = argparse.ArgumentParser()
    p.add_argument("--env_name", default="VanderPol")
    p.add_argument("--checkpoint", required=True, help="apprfunc_{iteration}.pkl written by the trainer")
    p.add_argument("--num_states", type=int, default=1 << 20)
    p.add_argument("--horizon", type=int, default=20, help="closed-loop steps per initial state (default: n_step = 20)")
    p.add_argument("--lya_eta", type=float, default=0.15)
    p.add_argument("--alpha1", type=float, default=1.0)
    p.add_argument("--alpha2", type=float, default=2.0)
    p.add_argument("--v_atol", type=float, default=0.0)
    p.add_argument("--seed", type=int, default=0)
    p.add_argument("--box", type=float, nargs=2, metavar=("LO", "HI"), help="uniform initial states in [LO, HI]^obs_dim "
                   "(box envs) instead of the env's reset distribution")
    p.add_argument("--lyapunov_output_dim", type=int, default=256)
    p.add_argument("--rollout_engine", default="tc")
    p.add_argument("--region", type=float, nargs=2, metavar=("LO", "HI"), help="run the sound region verifier over "
                   "[LO, HI]^obs_dim instead of the sampling check")
    p.add_argument("--inner", type=float, nargs="+", metavar="R", help="inner box B: a radius R, or LO HI (default 0.05 of "
                   "the box width)")
    p.add_argument("--steps", type=int, default=1, help="closed-loop steps m of the region verifier")
    p.add_argument("--max_depth", type=int, default=30, help="deepest cell of the region verifier")
    for key, what in (("obs", "sensor noise"), ("act", "actuator disturbance"), ("state", "process disturbance")):
        p.add_argument(f"--dist_{key}", type=float, nargs="+", metavar="R", help=f"region verifier: {what} half-widths")
    p.add_argument("--margin", type=float, metavar="S_MAX", help="region verifier: bisect the proven scale of the "
                   "disturbance in [0, S_MAX]")
    a = p.parse_args(argv)
    nets = ApproxContainer(**network_kwargs(a.env_name, a.lyapunov_output_dim)).cuda()
    nets.load_state_dict(torch.load(a.checkpoint, map_location="cuda", weights_only=True))
    if a.region:
        kw = dict(networks=nets, env_name=a.env_name, box=tuple(a.region), lya_eta=a.lya_eta, alpha1=a.alpha1, alpha2=a.alpha2,
                  steps=a.steps, max_depth=a.max_depth)
        if a.inner:
            kw["inner"] = a.inner[0] if len(a.inner) == 1 else tuple(a.inner[:2])
        dist = {k: getattr(a, f"dist_{k}") for k in ("obs", "act", "state") if getattr(a, f"dist_{k}") is not None}
        if dist:
            kw["disturbance"] = dist
        elif a.margin is not None:
            p.error("--margin needs --dist_obs, --dist_act or --dist_state")
        ver = msacl_b200.create_region_certifier(**kw)
        if a.margin is None:
            rep = ver.run()
            print(rep.to_json(), flush=True)
            return json.loads(rep.to_json())
        r = ver.robustness_margin(a.margin)
        out = json.loads(r.report.to_json())
        out["margin"] = dict(s_max=a.margin, s_proven=r.s_proven, s_failed=r.s_failed, runs=r.runs, nominal_proven=r.nominal_proven)
        print(json.dumps(out), flush=True)
        return out
    ver = msacl_b200.create_certifier(networks=nets, env_name=a.env_name, num_states=a.num_states, horizon=a.horizon,
                                      lya_eta=a.lya_eta, alpha1=a.alpha1, alpha2=a.alpha2, v_atol=a.v_atol, seed=a.seed,
                                      init=("box", a.box[0], a.box[1]) if a.box else "reset", rollout_engine=a.rollout_engine)
    rep = ver.run()
    print(rep.to_json(), flush=True)
    return json.loads(rep.to_json())


if __name__ == "__main__":
    main()
