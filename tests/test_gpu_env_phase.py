"""The env phase (noise, TanhGauss sample / clip / log-prob, env step, reward / cost, autoreset, n-step bookkeeping,
transition record) is one piece of code shared by all rollout kernels: given the same logits, the fused kernels and the
general engine's `rollout_step` must produce bit-identical transitions, env state and episode counts.

The fused kernel runs first and records the logits it sampled from; the general engine then replays the same K steps
from an identical initial state with an actor that returns exactly those logits."""
import numpy as np
import pytest
import torch

from oracle import actor as oactor
from oracle import envs as oenv

pytestmark = pytest.mark.gpu

STATE_FIELDS = ("sf", "sd", "step", "episode", "ep_len", "run", "ep_return")


def _replay_actor(w, logits, min_log_std, max_log_std):
    from msacl_b200.sampler import GeneralActor

    class ReplayActor(GeneralActor):
        """A GeneralActor whose k-th forward pass returns the logits a fused kernel recorded at step k."""

        def __init__(self):
            super().__init__(w, [torch.nn.ReLU(), torch.nn.ReLU(), torch.nn.Identity()], min_log_std=min_log_std,
                             max_log_std=max_log_std)
            self.k = 0

        def forward_state(self, state):
            out = logits[self.k].contiguous()
            self.k += 1
            return out

    return ReplayActor()


@pytest.mark.parametrize("noise", ["philox", "eps", "deterministic"])
@pytest.mark.parametrize("engine", ["tc", "ffma"])
@pytest.mark.parametrize("name", oenv.ENV_NAMES)
def test_fused_env_phase_matches_general_engine_bit_for_bit(name, engine, noise):
    from msacl_b200.sampler import ActorWeights, FusedRollout
    n, K, max_step, n_step, seed, env_base = 1000, 6, 4, 3, 11, 12345     # n is not a multiple of either tile size
    spec = oenv.SPECS[name]
    w = oactor.init_policy_weights(spec.obs_dim, spec.act_dim, seed=2)
    aw = ActorWeights(w, min_log_std=-5.0, max_log_std=0.5)
    eps = None
    if noise == "eps":
        eps = torch.as_tensor(np.random.default_rng(4).standard_normal((K, n, spec.act_dim)).astype(np.float32)).cuda()
    kw = dict(n_step=n_step, seed=seed, env_base=env_base, max_step=max_step, record_logits=True)
    a = FusedRollout(name, n, K, engine=engine, **kw)
    b = FusedRollout(name, n, K, **kw)
    a.state.reset(); b.state.reset()
    a.run(aw, eps=eps, deterministic=noise == "deterministic")
    ga = _replay_actor(w, a.tr.logits, aw.desc.min_log_std, aw.desc.max_log_std)
    b.run(ga, eps=eps, deterministic=noise == "deterministic")
    torch.cuda.synchronize()
    assert ga.k == K
    fa, fb = a.tr.fields(), b.tr.fields()
    for f in fa:
        assert torch.equal(fa[f][a.tr.H:], fb[f][b.tr.H:]), f
    assert torch.equal(a.tr.logits, b.tr.logits)
    for f in STATE_FIELDS:
        assert torch.equal(getattr(a.state, f), getattr(b.state, f)), f
    sa, sb = a.stats.cpu().numpy(), b.stats.cpu().numpy()
    assert np.array_equal(sa[[0, 2, 3, 4]], sb[[0, 2, 3, 4]])
    np.testing.assert_allclose(sa[1], sb[1], rtol=1e-5, atol=1e-3)     # sum of returns: per-launch vs per-step order
    assert sa[0] > 0
