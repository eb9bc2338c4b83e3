"""msacl_b200 -- B200-native (sm_100a) hot path of MSACL behind the reference's Python API.

Import name: `msacl_b200` (the repository keeps the package in a directory named after the
upstream project; `msacl_b200.py` at the repo root aliases it).
"""
from .specs import ENV_NAMES, SPECS, get_spec  # noqa: F401

__all__ = ["ENV_NAMES", "SPECS", "get_spec", "create_envs", "create_sampler", "create_buffer", "create_alg", "create_evaluator",
           "create_trainer", "create_certifier", "create_region_certifier", "load_library"]


def load_library():
    from . import _lib
    return _lib.load()


def create_envs(**args):
    from .envs import create_envs as f
    return f(**args)


def create_sampler(**kwargs):
    """Drop-in for RL/create_pkg/create_sampler.py:45-61 (sampler_name 'nstep_off_sampler')."""
    from .sampler import B200NstepOffSampler
    name = kwargs.get("sampler_name", "nstep_off_sampler")
    if name not in ("nstep_off_sampler", "b200_nstep_off_sampler"):
        raise KeyError(f"No registered sampler with id: {name}")
    return B200NstepOffSampler(**kwargs)


def create_buffer(**kwargs):
    """Drop-in for RL/create_pkg/create_buffer.py:44-66 (buffer_name 'nstep_replay_buffer')."""
    from .buffer import B200IndexedReplayBuffer, B200NstepReplayBuffer
    name = kwargs.get("buffer_name", "nstep_replay_buffer")
    if name == "b200_indexed_replay_buffer":          # index-based windows over the sampler's transition store
        return B200IndexedReplayBuffer(**kwargs)
    if name not in ("nstep_replay_buffer", "b200_nstep_replay_buffer"):
        raise KeyError(f"No registered buffer with id: {name}")
    return B200NstepReplayBuffer(**kwargs)


def create_alg(**kwargs):
    """Drop-in for RL/create_pkg/create_alg.py:50-79 (algorithm 'msacl')."""
    from .algorithm import B200MSACL
    name = kwargs.get("algorithm", "msacl")
    if name not in ("msacl", "msacl_b200"):
        raise KeyError(f"No registered algorithm with id: {name}")
    return B200MSACL(**kwargs)


def create_evaluator(**kwargs):
    """Drop-in for RL/create_pkg/create_evaluator.py (evaluator_name 'evaluator'): greedy evaluation on the fused kernel."""
    from .evaluator import B200Evaluator
    name = kwargs.get("evaluator_name", "evaluator")
    if name not in ("evaluator", "b200_evaluator"):
        raise KeyError(f"No registered evaluator with id: {name}")
    return B200Evaluator(**kwargs)


def create_trainer(alg, sampler, buffer, evaluator, **kwargs):
    """Drop-in for RL/create_pkg/create_trainer.py:41-61 (trainer 'nstep_off_serial_trainer')."""
    from .trainer import B200NstepOffSerialTrainer
    name = kwargs.get("trainer", "nstep_off_serial_trainer")
    if name not in ("nstep_off_serial_trainer", "b200_nstep_off_serial_trainer"):
        raise KeyError(f"No registered trainer with id: {name}")
    return B200NstepOffSerialTrainer(alg, sampler, buffer, evaluator, **kwargs)


def create_certifier(**kwargs):
    """Lyapunov-certificate verifier of a trained ApproxContainer (no counterpart in the reference): closed-loop checks of
    alpha1 |o|^2 <= V(o) <= alpha2 |o|^2 and of V's (1 - eta)^k decrease over many initial states -- an empirical check over
    the sampled states and horizon, not a proof.  `create_certifier(networks=..., env_name=..., num_states=N).run()`."""
    from .certify import B200CertificateVerifier
    return B200CertificateVerifier(**kwargs)


def create_region_certifier(**kwargs):
    """Sound region verifier of the Lyapunov certificate (no counterpart in the reference): interval branch-and-bound over
    the cells of a state box X0 \\ B, proving V's (1 - eta)^m decrease over m greedy closed-loop steps for every state of a
    verified cell, for the real-arithmetic closed loop.  `create_region_certifier(networks=..., env_name=..., box=(lo, hi),
    inner=r).run()` -> RegionReport.  With `disturbance=dict(obs=..., act=..., state=...)` (sensor noise, actuator and
    process disturbance boxes: a radius r for [-r, r] or a (lo, hi) tuple) every statement holds for every admissible
    disturbance sequence and run() returns a RobustRegionReport; `.robustness_margin(s_max)` bisects the largest proven scale
    of those boxes."""
    from .certify_region import B200RegionVerifier
    return B200RegionVerifier(**kwargs)
