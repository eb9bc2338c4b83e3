"""Region verifier on the GPU: enclosure of every layer against the float64 real-arithmetic oracle (oracle/region.py, run in
float64 on the GPU), soundness of "verified" cells and of counterexamples, an analytic VanderPol case that must verify and
its destabilised twin, determinism under re-chunking, and fresh weights on every run."""
import numpy as np
import pytest
import torch

from oracle import envs as oenv
from oracle import region as oreg

pytestmark = pytest.mark.gpu

ENVS = ["VanderPol", "Pendulum", "DuctedFan", "TwoLink"]
# slack for the float64 oracle's own rounding (the kernel's bounds are float32, >= 1 float32 ulp outside when rounded)
TOL = 1e-9
DEGENERATE_ULPS = 2 ** 15      # width of [c, c] enclosures, in float32 ulps of max(|value|, median |value| of the batch)
DEGENERATE_ULPS_VF = 2 ** 21   # the same for V(F(c)), m = 1


def _networks(name, seed=0, **kw):
    from msacl_b200.algorithm import ApproxContainer
    spec = oenv.SPECS[name]
    torch.manual_seed(seed)
    return ApproxContainer(obs_dim=spec.obs_dim, act_dim=spec.act_dim, action_low_limit=spec.act_low, action_high_limit=spec.act_high,
                           q_learning_rate=1e-3, lyapunov_learning_rate=1e-3, policy_learning_rate=3e-4, alpha_learning_rate=1e-3,
                           **kw).cuda()


def _layers(seq):
    lin = [m for m in seq if isinstance(m, torch.nn.Linear)]
    return [(m.weight.detach().double(), m.bias.detach().double()) for m in lin]


def _box(name):
    s = oenv.SPECS[name]
    return (s.obs_low * 0.5).astype(np.float32), (s.obs_high * 0.5).astype(np.float32)


def _inside(v, lo, hi):
    """#points with v outside [lo, hi] beyond the oracle slack."""
    slack = TOL * (1.0 + v.abs())
    lo, hi = lo.double(), hi.double()
    return int(((v < lo - slack) | (v > hi + slack) | lo.isnan() | hi.isnan()).sum())


@pytest.mark.parametrize("m", [1, 3])
@pytest.mark.parametrize("name", ENVS)
def test_enclosure_per_layer(name, m):
    import msacl_b200
    nets = _networks(name, seed=ENVS.index(name) + 10 * m)
    lo0, hi0 = _box(name)
    ver = msacl_b200.create_region_certifier(networks=nets, env_name=name, box=(lo0, hi0), steps=m)
    D, A = oenv.SPECS[name].obs_dim, oenv.SPECS[name].act_dim
    N, P = 100_000, 16
    g = torch.Generator(device="cuda").manual_seed(1)
    span = torch.as_tensor(hi0 - lo0, device="cuda", dtype=torch.float64)
    lo0t = torch.as_tensor(lo0, device="cuda", dtype=torch.float64)
    width = span * 10.0 ** (-6.0 * torch.rand(N, 1, device="cuda", generator=g, dtype=torch.float64))
    centre = lo0t + span * torch.rand(N, D, device="cuda", generator=g, dtype=torch.float64)
    lo = (centre - width / 2).float()
    hi = (centre + width / 2).float()
    deg = torch.arange(N, device="cuda") % 10 == 0                 # every tenth cell is degenerate [c, c]
    hi[deg] = lo[deg]
    o = ver.evaluate(lo, hi, trace=True)
    torch.cuda.synchronize()
    tr = o["trace"].double()
    pl, pv = _layers(nets.policy.policy), _layers(nets.lyapunov.lya)
    tanh = isinstance(nets.lyapunov.lya[1], torch.nn.Tanh)
    escapes = {}
    for p in range(P):
        if p == 0:
            u = torch.zeros(N, D, device="cuda", dtype=torch.float64)
        elif p == 1:
            u = torch.ones(N, D, device="cuda", dtype=torch.float64)
        elif p < 8:
            u = (torch.rand(N, D, device="cuda", generator=g) < 0.5).double()      # random corners
        else:
            u = torch.rand(N, D, device="cuda", generator=g, dtype=torch.float64)
        x = lo.double() + (hi.double() - lo.double()) * u
        x = torch.minimum(torch.maximum(x, lo.double()), hi.double())
        bump = lambda k, n: escapes.__setitem__(k, escapes.get(k, 0) + n)
        bump("V(x)", _inside(oreg.lyapunov(pv, x, tanh, torch), o["v_lo"], o["v_hi"]))
        steps = oreg.closed_loop(name, pl, x, m, torch)
        for j, (mu, a, xj) in enumerate(steps):
            t = tr[:, j]
            bump("mu", _inside(mu, t[:, :A], t[:, A:2 * A]))
            bump("a", _inside(a, t[:, 2 * A:3 * A], t[:, 3 * A:4 * A]))
            bump("F^j", _inside(xj, t[:, 4 * A:4 * A + D], t[:, 4 * A + D:]))
        xm = steps[-1][2]
        bump("F^m", _inside(xm, o["img_lo"], o["img_hi"]))
        bump("V(F^m x)", _inside(oreg.lyapunov(pv, xm, tanh, torch), o["vm_lo"], o["vm_hi"]))
    print(name, m, escapes)
    assert all(v == 0 for v in escapes.values()), escapes
    # degenerate cells [c, c]: the enclosures of V(c), mu, a and F(c) stay within a few thousand float32 ulps (256-term rd / ru
    # sums); V(F(c)) adds the interval amplification of the networks (the width of F(c) times the V net's interval Lipschitz
    # bound, ~sum |W| per layer), and every further step multiplies that again, so V(F^m(c)) is bounded for m = 1 only
    ulps = lambda a, b: float(((b - a) / (torch.maximum(b.abs(), b.abs().median()) * 2.0 ** -23)).max())
    t0 = tr[deg][:, 0]
    widths = {"V(c)": ulps(o["v_lo"][deg].double(), o["v_hi"][deg].double()),
              "mu": ulps(t0[:, :A], t0[:, A:2 * A]), "a": ulps(t0[:, 2 * A:3 * A], t0[:, 3 * A:4 * A]),
              "F(c)": ulps(t0[:, 4 * A:4 * A + D], t0[:, 4 * A + D:])}
    vm = ulps(o["vm_lo"][deg].double(), o["vm_hi"][deg].double())
    print(name, m, "max widths of degenerate enclosures in ulps", widths, "V(F^m(c))", vm)
    assert max(widths.values()) <= DEGENERATE_ULPS, widths
    if m == 1:
        assert vm <= DEGENERATE_ULPS_VF, vm


def _set_linear(lin, W, b):
    with torch.no_grad():
        lin.weight.zero_(); lin.bias.zero_()
        lin.weight[:W.shape[0], :W.shape[1]] = torch.as_tensor(W, dtype=torch.float32)
        lin.bias[:len(b)] = torch.as_tensor(b, dtype=torch.float32)


def _analytic_vanderpol(sign=1.0, eps=1e-2):
    """Policy mean k x (ReLU pair), action 5 tanh(k x); V = sum z^2 with z = L tanh(tanh(eps x)) / eps ~ L x, P = L^T L from
    the discrete Lyapunov equation of the linearised one-step map."""
    import scipy.linalg
    nets = _networks("VanderPol", lyapunov_hidden_activation="tanh")
    k = sign * np.array([-0.4, -0.8])
    pl = [m for m in nets.policy.policy if isinstance(m, torch.nn.Linear)]
    _set_linear(pl[0], np.stack([k, -k]), [0.0, 0.0])
    _set_linear(pl[1], np.eye(2), [0.0, 0.0])
    _set_linear(pl[2], np.array([[1.0, -1.0], [0.0, 0.0]]), [0.0, 0.0])
    Acl = np.array([[0.0, 1.0], [-1.0, 1.0]]) + np.array([[0.0], [1.0]]) @ (5.0 * k[None, :])
    Phi = np.linalg.matrix_power(np.eye(2) + 0.01 * Acl, 5)
    P = scipy.linalg.solve_discrete_lyapunov(Phi.T, np.eye(2))
    if sign > 0:
        L = np.linalg.cholesky(P).T
    else:
        L = np.linalg.cholesky(np.eye(2) * float(np.trace(P)) / 2).T
    L = L / np.sqrt(np.max(np.linalg.eigvalsh(L.T @ L)))
    vl = [m for m in nets.lyapunov.lya if isinstance(m, torch.nn.Linear)]
    _set_linear(vl[0], eps * np.eye(2), [0.0, 0.0])
    _set_linear(vl[1], np.eye(2), [0.0, 0.0])
    _set_linear(vl[2], L / eps, [0.0, 0.0])
    return nets


def _grid_ratio(nets, box, rin, n=801):
    """max over a dense float64 grid of X0 \\ B of V(F(x)) / V(x)."""
    t = torch.linspace(box[0], box[1], n, dtype=torch.float64, device="cuda")
    x = torch.stack(torch.meshgrid(t, t, indexing="ij"), -1).reshape(-1, 2)
    x = x[(x.abs() > rin).any(-1)]
    pl, pv = _layers(nets.policy.policy), _layers(nets.lyapunov.lya)
    v0 = oreg.lyapunov(pv, x, True, torch)
    v1 = oreg.lyapunov(pv, oreg.closed_loop("VanderPol", pl, x, 1, torch)[-1][2], True, torch)
    return float((v1 / v0).max())


BOX, RIN = (-1.0, 1.0), 0.1


def _analytic_run(sign, trace=None, **kw):
    import msacl_b200
    nets = _analytic_vanderpol(sign)
    rho = _grid_ratio(nets, BOX, RIN)
    eta = 1.0 - (1.0 + rho) / 2.0 if rho < 1 else 0.05
    args = dict(networks=nets, env_name="VanderPol", box=BOX, inner=RIN, lya_eta=eta, max_depth=24, trace=trace)
    args.update(kw)
    return msacl_b200.create_region_certifier(**args).run(), nets, eta, rho


def test_analytic_vanderpol_verifies_and_soundness_of_verified_cells():
    cells = []
    rep, nets, eta, rho = _analytic_run(1.0, trace=lambda lo, hi, st: cells.append((lo.clone(), hi.clone(), st.clone())))
    print(rep.to_json(), "rho", rho)
    assert rho < 1
    assert rep.verified_fraction_outside >= 0.95, rep.verified_fraction_outside
    assert rep.refuted == 0 and rep.invariant and rep.c_sound != "none" and rep.c_sound > 0
    # >= 1e6 points inside the verified cells satisfy DECREASE and ESCAPED in the float64 oracle
    lo = torch.cat([l[s == 1] for l, h, s in cells]).double()
    hi = torch.cat([h[s == 1] for l, h, s in cells]).double()
    assert lo.shape[0] == rep.verified
    g = torch.Generator(device="cuda").manual_seed(3)
    pl, pv = _layers(nets.policy.policy), _layers(nets.lyapunov.lya)
    total, bad = 0, 0
    while total < 1_000_000:
        x = lo + (hi - lo) * torch.rand(lo.shape, device="cuda", generator=g, dtype=torch.float64)
        v0 = oreg.lyapunov(pv, x, True, torch)
        x1 = oreg.closed_loop("VanderPol", pl, x, 1, torch)[-1][2]
        v1 = oreg.lyapunov(pv, x1, True, torch)
        bad += int((v1 > (1 - eta) * v0 * (1 + TOL)).sum()) + int((x1.abs() >= 10.0).any(-1).sum())
        total += x.shape[0]
    assert bad == 0


def test_destabilised_twin_is_refuted_with_sound_margins():
    rep, nets, eta, rho = _analytic_run(-1.0, max_depth=14, max_examples=64)
    print(rep.to_json())
    assert rep.refuted > 0 and not rep.invariant and rep.c_sound == "none"
    assert len(rep.counterexamples) == min(64, rep.refuted)
    pl, pv = _layers(nets.policy.policy), _layers(nets.lyapunov.lya)
    x = torch.tensor([c["x"] for c in rep.counterexamples], dtype=torch.float64, device="cuda")
    marg = torch.tensor([c["margin"] for c in rep.counterexamples], dtype=torch.float64, device="cuda")
    assert bool((marg > 0).all())
    x1 = oreg.closed_loop("VanderPol", pl, x, 1, torch)[-1][2]
    viol_dec = oreg.lyapunov(pv, x1, True, torch) - (1 - eta) * oreg.lyapunov(pv, x, True, torch)
    viol_esc = (x1.abs() - 10.0).max(-1).values
    kinds = [c["kind"] for c in rep.counterexamples]
    for i, kd in enumerate(kinds):
        v = float(viol_dec[i] if kd == "decrease" else viol_esc[i])
        assert v >= float(marg[i]) * (1 - 1e-9), (i, kd, v, float(marg[i]))
    assert all(not (abs(xi[0]) <= rep.inner[1][0] and abs(xi[1]) <= rep.inner[1][1]) for xi in x.tolist())


def test_random_network_counterexamples_are_sound():
    import msacl_b200
    name = "TwoLink"
    nets = _networks(name, seed=5)
    rep = msacl_b200.create_region_certifier(networks=nets, env_name=name, box=(-0.5, 0.5), inner=0.05, max_depth=12,
                                             max_examples=200).run()
    print(rep.to_json()[:2000])
    assert rep.refuted > 0
    pl, pv = _layers(nets.policy.policy), _layers(nets.lyapunov.lya)
    x = torch.tensor([c["x"] for c in rep.counterexamples], dtype=torch.float64, device="cuda")
    marg = np.array([c["margin"] for c in rep.counterexamples])
    x1 = oreg.closed_loop(name, pl, x, 1, torch)[-1][2]
    viol = (oreg.lyapunov(pv, x1, True, torch) - (1 - 0.15) * oreg.lyapunov(pv, x, True, torch)).cpu().numpy()
    hi = torch.as_tensor(oenv.SPECS[name].obs_high, dtype=torch.float64, device="cuda")
    esc = (x1.abs() - hi).max(-1).values.cpu().numpy()
    for c, vd, ve, mg in zip(rep.counterexamples, viol, esc, marg):
        assert (vd if c["kind"] == "decrease" else ve) >= mg * (1 - 1e-9)


def test_determinism_and_chunking_invariance():
    r1 = _analytic_run(1.0, max_depth=16)[0]
    r2 = _analytic_run(1.0, max_depth=16)[0]
    assert r1 == r2
    r3 = _analytic_run(1.0, max_depth=16, max_cells=256)[0]
    print(r1.to_json()[:600], r1.rounds, r3.rounds)
    assert r3.rounds > r1.rounds and r1.evaluated > 1000
    for k in ("verified", "refuted", "undecided", "inner_cells", "verified_fraction", "refuted_fraction", "undecided_fraction",
              "failed", "c_sound", "c_sound_candidate", "c_in", "v_inner", "invariant", "evaluated"):
        assert getattr(r1, k) == getattr(r3, k), k


def test_fresh_policy_weights_on_every_run():
    """FusedAdam writes the policy through raw pointers (torch's _version is unchanged): a second run() must see them."""
    import msacl_b200
    from msacl_b200.learner import FusedAdam
    name = "Pendulum"
    nets = _networks(name, seed=7)
    kw = dict(networks=nets, env_name=name, box=(-1.0, 1.0), inner=0.1, max_depth=10)
    ver = msacl_b200.create_region_certifier(**kw)
    first = ver.run()
    params = list(nets.policy.parameters())
    versions = [p._version for p in params]
    nets.policy_optimizer.param_groups[0]["lr"] = 0.05
    adam = FusedAdam(nets.policy_optimizer, params)
    g = torch.Generator(device="cuda").manual_seed(1)
    adam.step([(torch.randn((1,) + tuple(p.shape), device="cuda", generator=g), 1) for p in params])
    torch.cuda.synchronize()
    assert [p._version for p in params] == versions
    second = ver.run()
    fresh = msacl_b200.create_region_certifier(**kw).run()
    assert second == fresh and second != first
