"""Compact storage of MSACL network parameters in golden files, so that each file stays well under 1 MB.

Parameters at construction are stored as the seed that rebuilds them (torch's nn.Linear default initialisation, checked
against a SHA-256 digest), parameters after an update as float64 differences from the ones before it (exact for two
float32 arrays).  unpack_parameters restores the recorded float32 arrays bit for bit; rebuilding them needs torch (CPU
is enough), which the project depends on anyway.
"""
import hashlib

import numpy as np


def msacl_init_params(seed, obs_dim, act_dim):
    """State of the reference's MSACL networks right after construction under torch.manual_seed(seed): nn.Linear default
    initialisation in construction order q1, q2, lyapunov, policy; the target nets start as copies of q1 and q2."""
    import torch
    nets = {"q1.q": (obs_dim + act_dim, 256, 256, 1), "q2.q": (obs_dim + act_dim, 256, 256, 1),
            "lyapunov.lya": (obs_dim, 256, 256, 256), "policy.policy": (obs_dim, 256, 256, 2 * act_dim)}
    out = {}
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(seed)
        for net, dims in nets.items():
            for i, (a, b) in enumerate(zip(dims[:-1], dims[1:])):
                lin = torch.nn.Linear(a, b)
                out[f"{net}.{2 * i}.weight"] = lin.weight.detach().numpy().copy()
                out[f"{net}.{2 * i}.bias"] = lin.bias.detach().numpy().copy()
    for k in [k for k in out if k.startswith("q")]:
        out[k.replace(".", "_target.", 1)] = out[k].copy()
    return out


def _digest(arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def pack_parameters(g, seed, obs_dim, act_dim, init_keys, init_params, delta_keys, delta_bases):
    """The compact form of golden dict `g`: g[init_keys[i]] must equal msacl_init_params(...)[init_params[i]] and is
    dropped; g[delta_keys[i]] is stored as its float64 difference from g[delta_bases[i]]."""
    init = msacl_init_params(seed, obs_dim, act_dim)
    for k, p in zip(init_keys, init_params):
        assert np.array_equal(g[k], init[p]) and g[k].dtype == init[p].dtype, (k, p)
    out = dict(g)
    for k, b in zip(delta_keys, delta_bases):
        out["delta_" + k] = g[k].astype(np.float64) - g[b].astype(np.float64)
        assert np.array_equal((g[b].astype(np.float64) + out["delta_" + k]).astype(g[k].dtype), g[k]), k
        del out[k]
    for k in init_keys:
        del out[k]
    out.update(init_seed=np.int64(seed), init_dims=np.array([obs_dim, act_dim]), init_keys=np.array(init_keys),
               init_params=np.array(init_params), init_sha256=np.array(_digest(init[p] for p in init_params)),
               delta_keys=np.array(delta_keys), delta_bases=np.array(delta_bases))
    return out


def unpack_parameters(g):
    """Inverse of pack_parameters, in place."""
    obs_dim, act_dim = (int(x) for x in g.pop("init_dims"))
    init = msacl_init_params(int(g.pop("init_seed")), obs_dim, act_dim)
    params = [str(p) for p in g.pop("init_params")]
    assert _digest(init[p] for p in params) == str(g.pop("init_sha256")), \
        "torch's nn.Linear initialisation no longer reproduces the recorded network parameters"
    for k, p in zip(g.pop("init_keys"), params):
        g[str(k)] = init[p]
    for k, b in zip(g.pop("delta_keys"), g.pop("delta_bases")):
        k, b = str(k), str(b)
        g[k] = (g[b].astype(np.float64) + g.pop("delta_" + k)).astype(g[b].dtype)
