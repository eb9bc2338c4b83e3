"""Region verifier under bounded disturbances on the GPU: explicit zero disturbances give the nominal verifier bit for bit;
enclosure of every layer against the float64 disturbed closed loop at corner and interior disturbance sequences; soundness
of verified cells and of counterexamples under disturbances; robustness_margin; chunking invariance."""
import dataclasses

import numpy as np
import pytest
import torch

from oracle import envs as oenv
from oracle import region as oreg
from test_gpu_certify_region import BOX, RIN, TOL, _analytic_run, _analytic_vanderpol, _box, _inside, _layers, _networks

pytestmark = pytest.mark.gpu

ENVS = ["VanderPol", "Pendulum", "DuctedFan", "TwoLink"]
ZERO = dict(obs=0.0, act=0.0, state=0.0)


def _cells(name, N, seed=1):
    """The enclosure test's cells: random centres in X0, widths 1e-6..1 of the box, every tenth cell degenerate."""
    lo0, hi0 = _box(name)
    D = oenv.SPECS[name].obs_dim
    g = torch.Generator(device="cuda").manual_seed(seed)
    span = torch.as_tensor(hi0 - lo0, device="cuda", dtype=torch.float64)
    lo0t = torch.as_tensor(lo0, device="cuda", dtype=torch.float64)
    width = span * 10.0 ** (-6.0 * torch.rand(N, 1, device="cuda", generator=g, dtype=torch.float64))
    centre = lo0t + span * torch.rand(N, D, device="cuda", generator=g, dtype=torch.float64)
    lo, hi = (centre - width / 2).float(), (centre + width / 2).float()
    deg = torch.arange(N, device="cuda") % 10 == 0
    hi[deg] = lo[deg]
    return lo, hi, g


def _base(rep):
    d = dataclasses.asdict(rep)
    d.pop("disturbance", None)
    return d


@pytest.mark.parametrize("m", [1, 3])
@pytest.mark.parametrize("name", ENVS)
def test_zero_disturbance_evaluate_is_bit_identical(name, m):
    import msacl_b200
    nets = _networks(name, seed=ENVS.index(name) + 10 * m)
    kw = dict(networks=nets, env_name=name, box=_box(name), steps=m)
    nom = msacl_b200.create_region_certifier(**kw)
    rob = msacl_b200.create_region_certifier(**kw, disturbance=ZERO)
    lo, hi, _ = _cells(name, 100_000)
    a, b = nom.evaluate(lo, hi, trace=True), rob.evaluate(lo, hi, trace=True)
    for k in a:
        assert torch.equal(a[k].view(torch.uint8), b[k].view(torch.uint8)), k


def test_zero_disturbance_reports_equal_nominal():
    import msacl_b200
    r_nom = _analytic_run(1.0)[0]
    r_rob = _analytic_run(1.0, disturbance=ZERO)[0]
    assert type(r_rob).__name__ == "RobustRegionReport" and _base(r_rob) == _base(r_nom)
    r_nom = _analytic_run(-1.0, max_depth=14, max_examples=64)[0]
    r_rob = _analytic_run(-1.0, max_depth=14, max_examples=64, disturbance=ZERO)[0]
    assert r_nom.refuted > 0 and _base(r_rob) == _base(r_nom)
    kw = dict(networks=_networks("TwoLink", seed=5), env_name="TwoLink", box=(-0.5, 0.5), inner=0.05, max_depth=12,
              max_examples=200)
    r_nom = msacl_b200.create_region_certifier(**kw).run()
    r_rob = msacl_b200.create_region_certifier(**kw, disturbance=ZERO).run()
    assert r_nom.refuted > 0 and _base(r_rob) == _base(r_nom)


def _dist_sets(name):
    """N symmetric, U asymmetric excluding 0 (a bias), W asymmetric containing 0; sizes relative to the box and action range."""
    s = oenv.SPECS[name]
    lo0, hi0 = _box(name)
    span = (hi0 - lo0).astype(np.float64)
    ar = (s.act_high - s.act_low).astype(np.float64)
    return dict(obs=1e-3 * span, act=(0.01 * ar, 0.03 * ar), state=(-2e-3 * span, 1e-3 * span))


def _draw(box, N, p, g):
    """[N, k] float64 draws from the float32 box (lo, hi): all lo (p = 0), all hi (p = 1), random corners (p < 8), interior."""
    lo = torch.as_tensor(box[0], dtype=torch.float64, device="cuda")
    hi = torch.as_tensor(box[1], dtype=torch.float64, device="cuda")
    k = lo.shape[0]
    if p == 0:
        t = torch.zeros(N, k, device="cuda", dtype=torch.float64)
    elif p == 1:
        t = torch.ones(N, k, device="cuda", dtype=torch.float64)
    elif p < 8:
        t = (torch.rand(N, k, device="cuda", generator=g) < 0.5).double()
    else:
        t = torch.rand(N, k, device="cuda", generator=g, dtype=torch.float64)
    return torch.minimum(torch.maximum(lo + (hi - lo) * t, lo), hi)


@pytest.mark.parametrize("m", [1, 3])
@pytest.mark.parametrize("name", ENVS)
def test_enclosure_under_disturbances(name, m):
    import msacl_b200
    nets = _networks(name, seed=ENVS.index(name) + 10 * m)
    ver = msacl_b200.create_region_certifier(networks=nets, env_name=name, box=_box(name), steps=m, disturbance=_dist_sets(name))
    assert 0.0 < float(ver.disturbance["act"][0].min())            # one set excludes 0
    D, A = oenv.SPECS[name].obs_dim, oenv.SPECS[name].act_dim
    N, P = 100_000, 16
    lo, hi, g = _cells(name, N)
    o = ver.evaluate(lo, hi, trace=True)
    torch.cuda.synchronize()
    tr = o["trace"].double()
    pl, pv = _layers(nets.policy.policy), _layers(nets.lyapunov.lya)
    tanh = isinstance(nets.lyapunov.lya[1], torch.nn.Tanh)
    escapes = {}
    bump = lambda k, n: escapes.__setitem__(k, escapes.get(k, 0) + n)
    for p in range(P):
        u = _draw((np.zeros(D), np.ones(D)), N, p, g)
        x = torch.minimum(torch.maximum(lo.double() + (hi.double() - lo.double()) * u, lo.double()), hi.double())
        seq = [tuple(_draw(ver.disturbance[k], N, p if j == 0 else (p + j) % P, g) for k in ("obs", "act", "state"))
               for j in range(m)]
        bump("V(x)", _inside(oreg.lyapunov(pv, x, tanh, torch), o["v_lo"], o["v_hi"]))
        steps = oreg.closed_loop(name, pl, x, m, torch, dist=seq)
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


W_SMALL = 1e-4          # process disturbance radius of the analytic case: small next to its decrease gap at the edge of B


def test_analytic_vanderpol_small_process_disturbance():
    cells = []
    rep, nets, eta, rho = _analytic_run(1.0, trace=lambda lo, hi, st: cells.append((lo.clone(), hi.clone(), st.clone())),
                                        disturbance=dict(state=W_SMALL))
    print(rep.to_json()[:1500], "rho", rho)
    assert rep.invariant and rep.c_sound != "none" and rep.c_sound > 0
    assert rep.verified_fraction_outside >= 0.95, rep.verified_fraction_outside
    lo = torch.cat([l[s == 1] for l, h, s in cells]).double()
    hi = torch.cat([h[s == 1] for l, h, s in cells]).double()
    assert lo.shape[0] == rep.verified
    wbox = [torch.as_tensor(b, dtype=torch.float64, device="cuda") for b in (rep.disturbance["state"][0], rep.disturbance["state"][1])]
    g = torch.Generator(device="cuda").manual_seed(3)
    pl, pv = _layers(nets.policy.policy), _layers(nets.lyapunov.lya)
    total, bad, p = 0, 0, 0
    while total < 1_000_000:
        x = lo + (hi - lo) * torch.rand(lo.shape, device="cuda", generator=g, dtype=torch.float64)
        w = _draw(wbox, x.shape[0], p % 16, g)
        v0 = oreg.lyapunov(pv, x, True, torch)
        x1 = oreg.closed_loop("VanderPol", pl, x, 1, torch, dist=[(None, None, w)])[-1][2]
        v1 = oreg.lyapunov(pv, x1, True, torch)
        bad += int((v1 > (1 - eta) * v0 * (1 + TOL)).sum()) + int((x1.abs() >= 10.0).any(-1).sum())
        total += x.shape[0]
        p += 1
    assert bad == 0


def test_large_constant_bias_is_refuted_with_sound_margins():
    dist = dict(act=(1.0, 1.5), state=(0.04, 0.06))
    rep, nets, eta, rho = _analytic_run(1.0, max_depth=14, max_examples=64, disturbance=dist)
    print(rep.to_json()[:1500])
    assert rep.refuted > 0 and not rep.invariant and rep.c_sound == "none"
    assert len(rep.counterexamples) == min(64, rep.refuted)
    pl, pv = _layers(nets.policy.policy), _layers(nets.lyapunov.lya)
    x = torch.tensor([c["x"] for c in rep.counterexamples], dtype=torch.float64, device="cuda")
    marg = torch.tensor([c["margin"] for c in rep.counterexamples], dtype=torch.float64, device="cuda")
    dec = torch.tensor([c["kind"] == "decrease" for c in rep.counterexamples], device="cuda")
    assert bool((marg > 0).all())
    boxes = {k: [np.asarray(b, np.float64) for b in rep.disturbance[k]] for k in ("act", "state")}
    g = torch.Generator(device="cuda").manual_seed(4)
    v0 = oreg.lyapunov(pv, x, True, torch)
    for p in range(64):                                   # the corners (p < 8 of _draw) and random interior draws
        u, w = _draw(boxes["act"], x.shape[0], p, g), _draw(boxes["state"], x.shape[0], p, g)
        x1 = oreg.closed_loop("VanderPol", pl, x, 1, torch, dist=[(None, u, w)])[-1][2]
        viol = torch.where(dec, oreg.lyapunov(pv, x1, True, torch) - (1 - eta) * v0, (x1.abs() - 10.0).max(-1).values)
        assert bool((viol >= marg * (1 - 1e-9)).all()), (p, float((viol - marg).min()))


def test_robustness_margin_on_the_analytic_case():
    import msacl_b200
    nets = _analytic_vanderpol(1.0)
    rep0, _, eta, _ = _analytic_run(1.0)
    kw = dict(networks=nets, env_name="VanderPol", box=BOX, inner=RIN, lya_eta=eta, max_depth=24, disturbance=dict(state=W_SMALL))
    ver = msacl_b200.create_region_certifier(**kw)
    r = ver.robustness_margin(100.0, iters=8)         # s = 1 is proven (the test above); s = 100 is far beyond the gap
    print(r.s_proven, r.s_failed, r.runs, r.report.to_json()[:600])
    assert rep0.invariant and r.nominal_proven and r.s_proven is not None and r.s_proven > 0 and r.s_failed is not None
    assert r.report.invariant and r.runs == 10
    assert r.report.disturbance["state"][1][0] >= r.s_proven * W_SMALL
    assert ver.run_scaled(r.s_proven) == r.report
    assert not ver.run_scaled(r.s_failed).invariant
    again = msacl_b200.create_region_certifier(**kw).robustness_margin(100.0, iters=8)
    assert (again.s_proven, again.s_failed, again.runs, again.report) == (r.s_proven, r.s_failed, r.runs, r.report)


def test_robust_report_independent_of_chunking():
    dist = dict(obs=5e-5, act=(-0.01, 0.02), state=1e-4)
    r1 = _analytic_run(1.0, max_depth=16, disturbance=dist)[0]
    r3 = _analytic_run(1.0, max_depth=16, max_cells=256, disturbance=dist)[0]
    print(r1.to_json()[:600], r1.rounds, r3.rounds)
    assert r3.rounds > r1.rounds and r1.evaluated > 1000
    for k in ("verified", "refuted", "undecided", "inner_cells", "verified_fraction", "refuted_fraction", "undecided_fraction",
              "failed", "c_sound", "c_sound_candidate", "c_in", "v_inner", "invariant", "evaluated", "disturbance"):
        assert getattr(r1, k) == getattr(r3, k), k
