"""Float64 restatement of the REAL-ARITHMETIC greedy closed loop the region verifier encloses (csrc/interval_env.cuh,
csrc/certify_region.cu): policy mean -> a = half tanh(mu) + mid -> clip -> CONTROL_STEP explicit-Euler sub-steps with the
env's constants (the float32 values of env_dynamics.cuh, float64 in TwoLink's solve) read as reals, and V = sum z^2.

Written against an array namespace `xp` (numpy, or torch for float64 tensors on the GPU), rows = points.
"""
import numpy as np

from .envs import SPECS

F = lambda v: float(np.float32(v))
DT, DTD = F(0.01), 0.01


def _f(xp):
    if xp is np:
        return dict(sin=np.sin, cos=np.cos, tanh=np.tanh, stack=lambda a: np.stack(a, -1))
    import torch
    return dict(sin=torch.sin, cos=torch.cos, tanh=torch.tanh, stack=lambda a: torch.stack(a, -1))


def env_step(name, x, a, xp=np):
    """One env step (CONTROL_STEP sub-steps) of x [N, D] under a [N, A] in float64."""
    f = _f(xp)
    x = [x[:, j] for j in range(x.shape[1])]
    if name == "VanderPol":
        for _ in range(5):
            p, v = x
            dd = (1.0 - p * p) * v - p + a[:, 0]
            x = [p + v * DT, v + dd * DT]
    elif name == "Pendulum":
        mgl, ml2, c01 = F(0.15 * 9.81 * 0.5), F(0.15 * (0.5 * 0.5)), F(0.1)
        for _ in range(5):
            th, thd = x
            dd = (mgl * f["sin"](th) - c01 * thd + a[:, 0]) / ml2
            x = [th + thd * DT, thd + dd * DT]
    elif name == "DuctedFan":
        m, d, r, J = F(8.5), F(0.95), F(0.26), F(0.048)
        mg, nmg = F(8.5 * 9.81), F(-8.5 * 9.81)
        u1, u2 = a[:, 0], a[:, 1]
        for _ in range(5):
            sn, cs = f["sin"](x[2]), f["cos"](x[2])
            ddx = (nmg * sn - d * x[3] + u1 * cs - u2 * sn) / m
            ddy = (mg * (cs - 1.0) - d * x[4] + u1 * sn + u2 * cs) / m
            ddth = r * u1 / J
            x = [x[0] + x[3] * DT, x[1] + x[4] * DT, x[2] + x[5] * DT, x[3] + ddx * DT, x[4] + ddy * DT, x[5] + ddth * DT]
    elif name == "TwoLink":
        I = (1.0 / 12.0)
        p11, c125, c2l = F(I + I + 0.25), F(1.25), F(1.0)
        i2, lc2sq, l1lc2, M22 = F(I), F(0.25), F(0.5), I + 0.25
        hk, g1a, g1b, g2k = F(-0.5), F(-(0.5 + 1.0) * 9.81), F(0.5 * 9.81), F(-0.5 * 9.81)
        for _ in range(5):
            th1, th2, d1, d2 = x
            s2, c2 = f["sin"](th2), f["cos"](th2)
            m11 = p11 + (c125 + c2l * c2)
            m12 = i2 + (lc2sq + l1lc2 * c2)
            h = hk * s2
            Cq1 = (h * d2) * d1 + (h * d2 + h * d1) * d2
            Cq2 = (-h) * d1 * d1
            s12 = f["sin"](th1 + th2)
            G1 = g1a * f["sin"](th1) - g1b * s12
            G2 = g2k * s12
            b1, b2 = a[:, 0] - Cq1 - G1, a[:, 1] - Cq2 - G2
            det = m11 * M22 - m12 * m12
            x2 = (m11 * b2 - m12 * b1) / det
            x1 = (M22 * b1 - m12 * b2) / det
            x = [th1 + d1 * DTD, th2 + d2 * DTD, d1 + x1 * DTD, d2 + x2 * DTD]
    else:
        raise ValueError(f"region oracle: {name} is not supported")
    return f["stack"](x)


def policy_mean(layers, x, A, xp=np):
    (w1, b1), (w2, b2), (w3, b3) = layers
    relu = lambda z: z * (z > 0)
    h = relu(x @ w1.T + b1)
    h = relu(h @ w2.T + b2)
    return (h @ w3.T + b3)[:, :A]


def action(name, mu, xp=np):
    s = SPECS[name]
    lo, hi = s.act_low.astype(np.float64), s.act_high.astype(np.float64)
    half, mid = (hi - lo) / 2.0, (hi + lo) / 2.0
    if xp is not np:
        import torch
        half, mid, lo, hi = (torch.as_tensor(v, dtype=mu.dtype, device=mu.device) for v in (half, mid, lo, hi))
        return torch.maximum(torch.minimum(half * torch.tanh(mu) + mid, hi), lo)
    return np.clip(half * np.tanh(mu) + mid, lo, hi)


def lyapunov(layers, x, tanh_act=True, xp=np):
    (w1, b1), (w2, b2), (w3, b3) = layers
    act = _f(xp)["tanh"] if tanh_act else (lambda z: z * (z > 0))
    h = act(x @ w1.T + b1)
    h = act(h @ w2.T + b2)
    z = h @ w3.T + b3
    return (z * z).sum(-1)


def closed_loop(name, policy_layers, x, steps, xp=np, dist=None):
    """[(mu, a, F^j(x)) for j = 1..steps] of the greedy closed loop, disturbed as
    F_d(x) = Phi(x, clip(half tanh(mu(x + n)) + mid) + u) + w.  dist is None (no disturbance) or one (n, u, w) per step
    ([N, D], [N, A], [N, D] arrays, any of them None for {0})."""
    A = SPECS[name].act_dim
    out = []
    for j in range(steps):
        n, u, w = dist[j] if dist is not None else (None, None, None)
        mu = policy_mean(policy_layers, x if n is None else x + n, A, xp)
        a = action(name, mu, xp)
        if u is not None:
            a = a + u
        x = env_step(name, x, a, xp)
        if w is not None:
            x = x + w
        out.append((mu, a, x))
    return out
