"""The autograd-free learner (csrc/mlp_tc.cu, csrc/learner.cu, learner.py) against float64 / PyTorch fp32 references
of the same ops, the NumPy oracle and the reference's recorded tensors.

Stated tolerances: the default "bf16x6" GEMM (3-term bf16 operand split, 6 cross products, FP32 accumulation) is
FP32-class: <= 1.5e-6 * sum|a||b| per output (measured 7e-7); the optional "bf16x3" mode carries ~2^-16 per product (asserted 5e-5);
gradients through three layers 1e-4 relative to the gradient scale (backward kernels vs float64 through the kernel's own
activations); elementwise distribution kernels 2e-5 (CUDA tanhf/logf/atanhf vs torch / NumPy)."""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import actor as oactor

pytestmark = pytest.mark.gpu


def _gemm(**kw):
    import msacl_b200
    from msacl_b200 import _lib
    from msacl_b200.learner import _desc
    lib = msacl_b200.load_library()
    _lib.check(lib.msacl_gemm_tc(C.byref(_desc(**kw)), _lib.current_stream()))


def _rel(got, want):
    return float((got.double() - want).abs().max() / want.abs().max())


@pytest.mark.parametrize("prec,tol", [(6, 1.5e-6), (3, 5e-5)])
@pytest.mark.parametrize("m,n,k", [(128, 256, 256), (5120, 256, 4), (1000, 256, 6), (333, 1, 256), (4097, 4, 256), (260, 256, 16),
                                   (129, 8, 33), (640, 300, 100)])
def test_gemm_tc_forward_bias_act(m, n, k, prec, tol):
    """C = act(A B^T + bias) for the layer shapes of the learner (and ragged ones), all three activations, both precisions:
    bf16x6 (3-term operand split) is FP32-class (1.5e-6 of sum|a||b|: the tensor core aligns and truncates the addends of a k-step, measured 7e-7), bf16x3 5e-5."""
    g = torch.Generator(device="cuda").manual_seed(m + n + k)
    A = torch.randn(m, k, device="cuda", generator=g)
    Bm = torch.randn(n, k, device="cuda", generator=g) / max(1.0, k ** 0.5)
    bias = torch.randn(n, device="cuda", generator=g)
    for act, fn in ((0, lambda x: x), (1, torch.relu), (2, torch.tanh)):
        Cm = torch.full((m, n), 7.0, device="cuda")
        ss = torch.zeros(m, device="cuda") if n <= 256 else None
        _gemm(a=A, a_rs=k, a_ks=1, b=Bm, b_rs=k, b_ks=1, m=m, n=n, k=k, c=Cm, ldc=n, bias=bias, act=act, row_sumsq=ss, precision=prec)
        pre = A.double() @ Bm.double().t() + bias.double()
        want = fn(pre)
        scale = (A.double().abs() @ Bm.double().abs().t()).max()
        assert float((Cm.double() - want).abs().max()) <= tol * float(scale) + 2e-7 * float(want.abs().max()), (act, m, n, k)
        if ss is not None:
            np.testing.assert_allclose(ss.cpu().numpy(), (Cm.double() ** 2).sum(1).cpu().numpy(), rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("prec", [6, 3])
@pytest.mark.parametrize("transposed_b", [False, True])
def test_gemm_tc_prepacked_weights_bit_identical(prec, transposed_b):
    """Large row counts stream a pre-converted B operand (msacl_gemm_pack_b) with bulk copies: same bf16 images, so the result
    is bit-identical to the path that converts B inside every CTA -- forward (B = W) and dgrad (B = W^T read strided)."""
    import msacl_b200
    from msacl_b200 import _lib
    from msacl_b200.learner import _desc
    lib = msacl_b200.load_library()
    g = torch.Generator(device="cuda").manual_seed(11)
    m, n, k = 148 * 128 + 77, 256, 256
    A = torch.randn(m, k, device="cuda", generator=g)
    W = torch.randn(256, 256, device="cuda", generator=g) / 16
    bias = torch.randn(n, device="cuda", generator=g)
    b_rs, b_ks = (1, 256) if transposed_b else (256, 1)
    out = []
    for use_pack in (False, True):
        Cm = torch.empty(m, n, device="cuda")
        d = _desc(a=A, a_rs=k, a_ks=1, b=W, b_rs=b_rs, b_ks=b_ks, m=m, n=n, k=k, c=Cm, ldc=n, bias=bias, act=1, precision=prec)
        if use_pack:
            packed = torch.empty(int(lib.msacl_gemm_packed_b_bytes(k, prec)), dtype=torch.uint8, device="cuda")
            _lib.check(lib.msacl_gemm_pack_b(C.byref(d), packed.data_ptr(), _lib.current_stream()))
            d.b_packed = packed.data_ptr()
        _lib.check(lib.msacl_gemm_tc(C.byref(d), _lib.current_stream()))
        out.append(Cm)
    assert torch.equal(out[0], out[1])
    Wm = W.t() if transposed_b else W
    want = torch.relu(A.double() @ Wm.double().t() + bias.double())
    assert _rel(out[1], want) < (4e-6 if prec == 6 else 5e-5)


def test_gemm_tc_strided_operands_dgrad_mask_and_splitk_wgrad():
    """dgrad (B read transposed, activation-derivative mask in the epilogue) and wgrad (A and B read transposed, K = rows
    split over CTAs, partials reduced in order) vs float64."""
    import msacl_b200
    from msacl_b200 import _lib
    lib = msacl_b200.load_library()
    g = torch.Generator(device="cuda").manual_seed(5)
    rows, nin, nout = 3000, 256, 6
    dY = torch.randn(rows, nout, device="cuda", generator=g)
    W = torch.randn(nout, nin, device="cuda", generator=g) / 16
    H = torch.tanh(torch.randn(rows, nin, device="cuda", generator=g))
    dX = torch.empty(rows, nin, device="cuda")
    _gemm(a=dY, a_rs=nout, a_ks=1, b=W, b_rs=1, b_ks=nin, m=rows, n=nin, k=nout, c=dX, ldc=nin, mask=H, mask_ld=nin, mask_act=2)
    want = (dY.double() @ W.double()) * (1 - H.double() ** 2)
    assert _rel(dX, want) < 5e-5
    Hr = torch.relu(torch.randn(rows, nin, device="cuda", generator=g))
    _gemm(a=dY, a_rs=nout, a_ks=1, b=W, b_rs=1, b_ks=nin, m=rows, n=nin, k=nout, c=dX, ldc=nin, mask=Hr, mask_ld=nin, mask_act=1)
    want = (dY.double() @ W.double()) * (Hr.double() > 0)
    assert _rel(dX, want) < 5e-5
    # wgrad: dW[nout][nin] = dY^T X, split over 7 CTAs along the rows
    S = 7
    X = torch.randn(rows, nin, device="cuda", generator=g)
    parts = torch.full((S, nout, nin), 3.0, device="cuda")
    _gemm(a=dY, a_rs=1, a_ks=nout, b=X, b_rs=1, b_ks=nin, m=nout, n=nin, k=rows, c=parts, ldc=nin, split_k=S, c_split_stride=nout * nin)
    dW = torch.empty(nout, nin, device="cuda")
    _lib.check(lib.msacl_reduce_splits(parts.data_ptr(), nout * nin, S, dW.data_ptr(), _lib.current_stream()))
    want = dY.double().t() @ X.double()
    scale = (dY.double().abs().t() @ X.double().abs()).max()
    assert float((dW.double() - want).abs().max()) <= 5e-5 * float(scale)
    assert torch.equal(dW, parts.sum(0)) or _rel(dW, parts.double().sum(0)) < 1e-6
    # bias gradient: column sums over the same row splits
    cs = torch.empty(S, nout, device="cuda")
    _lib.check(lib.msacl_colsum(dY.data_ptr(), rows, nout, nout, S, cs.data_ptr(), _lib.current_stream()))
    np.testing.assert_allclose(cs.sum(0).cpu().numpy(), dY.double().sum(0).cpu().numpy(), rtol=1e-5, atol=1e-4)


@pytest.mark.parametrize("din,dout,act,rows,hidden", [(6, 1, "relu", 5120, (256, 256)), (4, 4, "relu", 777, (256, 256)),
                                                      (4, 256, "tanh", 2 * 640, (256, 256)), (16, 1, "relu", 130, (256, 256)),
                                                      (7, 2, "relu", 1500, (64, 128)), (12, 256, "tanh", 900, (300, 40)),
                                                      (3, 1, "relu", 20000, (512, 32))])
def test_fused_mlp_forward_backward_vs_autograd(din, dout, act, rows, hidden):
    """FusedMLP (three msacl_gemm_tc layers forward, dgrad + split-K wgrad backward) vs torch autograd on the same nn.Sequential;
    hidden widths are arbitrary (the reference builds them from `*_hidden_sizes`, mlp.py:18-33)."""
    from msacl_b200.algorithm import mlp
    from msacl_b200.learner import FusedMLP
    torch.manual_seed(rows)
    seq = mlp([din, *hidden, dout], {"relu": torch.nn.ReLU, "tanh": torch.nn.Tanh}[act]).cuda()
    x = torch.randn(rows, din, device="cuda")
    dy = torch.randn(rows, dout, device="cuda") / rows
    fm = FusedMLP(seq, "cuda")
    ws = fm.workspace("t", rows, train=True, need_dx=True, sumsq=(dout == 256))
    y = fm.forward(x, ws)
    xr = x.clone().requires_grad_(True)
    yr = seq(xr)
    assert _rel(y, yr.detach().double()) < 1e-4
    if dout == 256:
        np.testing.assert_allclose(ws.v.cpu().numpy(), (yr.detach() ** 2).sum(-1).cpu().numpy(), rtol=2e-4)
    dx = fm.backward(ws, dy, wgrad=True, need_dx=True)
    # (a) backward kernels vs float64 back-propagation through the kernel's OWN saved activations: same masks on both sides,
    #     so the comparison is not disturbed by hidden units whose pre-activation sits within round-off of the ReLU kink
    (W1, b1), (W2, b2), (W3, b3) = [(w.double(), b.double()) for w, b in fm.layers]
    h1, h2, xd, dyd = ws.h1.double(), ws.h2.double(), x.double(), dy.double()
    dact = (lambda h: (h > 0).double()) if act == "relu" else (lambda h: 1 - h * h)
    dA2 = (dyd @ W3) * dact(h2)
    dA1 = (dA2 @ W2) * dact(h1)
    want = [dA1.t() @ xd, dA1.sum(0), dA2.t() @ h1, dA2.sum(0), dyd.t() @ h2, dyd.sum(0)]
    assert _rel(dx, dA1 @ W1) < 1e-4
    for got, w, p in zip(fm.reduced_grads(ws), want, seq.parameters()):
        assert _rel(got, w) < 1e-4, tuple(p.shape)
    # (b) vs torch autograd end to end: all but the few rows with a unit on the kink agree to 2e-4 of the gradient scale
    yr.backward(dy)
    err = (dx.double() - xr.grad.double()).abs().max(dim=1).values / xr.grad.double().abs().max()
    assert float((err < 2e-4).double().mean()) > 0.99
    for got, p in zip(fm.reduced_grads(ws), seq.parameters()):
        assert _rel(got, p.grad.double()) < 2e-3, tuple(p.shape)


def test_tanh_gauss_kernels_vs_torch_oracle_and_reference_golden():
    """rsample / log_prob forward (a9: act_distribution_cls.py:59-84) vs the oracle and the reference's recorded log_prob;
    log_prob backward vs torch autograd of the same expression."""
    import msacl_b200
    from msacl_b200 import _lib
    from msacl_b200.algorithm import TanhGauss
    lib = msacl_b200.load_library()
    g = load_golden("msacl_targets_TwoLink.npz")
    lo, hi = torch.as_tensor(g["act_low"]).cuda(), torch.as_tensor(g["act_high"]).cuda()
    mean, std, act = (torch.as_tensor(g[k]).cuda().reshape(-1, 2) for k in ("pi_mean", "pi_std", "act"))
    rows, A = mean.shape
    logits = torch.cat([mean, std.log()], dim=-1).contiguous()
    st = _lib.current_stream()
    logp = torch.empty(rows, device="cuda")
    _lib.check(lib.msacl_tanh_gauss_log_prob(rows, A, logits.data_ptr(), act.contiguous().data_ptr(), lo.data_ptr(), hi.data_ptr(), -20.0, 1.0,
                                             logp.data_ptr(), st))
    np.testing.assert_allclose(logp.cpu().numpy(), g["logp_new"].reshape(-1), rtol=2e-5, atol=2e-5)       # the reference itself
    want = oactor.tanh_gauss_log_prob(mean.cpu().numpy(), std.cpu().numpy(), act.cpu().numpy(), g["act_low"], g["act_high"])
    np.testing.assert_allclose(logp.cpu().numpy(), want, rtol=2e-5, atol=2e-5)
    # backward vs autograd (torch fp32 reference of the same op)
    lg = logits.clone().requires_grad_(True)
    dist = TanhGauss(torch.cat([lg[:, :A], torch.clamp(lg[:, A:], -20.0, 1.0).exp()], dim=-1), lo, hi)
    gl = torch.randn(rows, device="cuda")
    (dist.log_prob(act) * gl).sum().backward()
    dlog = torch.empty_like(logits)
    _lib.check(lib.msacl_tanh_gauss_log_prob_bwd(rows, A, logits.data_ptr(), act.contiguous().data_ptr(), lo.data_ptr(), hi.data_ptr(),
                                                 -20.0, 1.0, gl.data_ptr(), 0, dlog.data_ptr(), st))
    np.testing.assert_allclose(dlog.cpu().numpy(), lg.grad.cpu().numpy(), rtol=2e-4, atol=2e-4 * float(lg.grad.abs().max()))
    # rsample forward vs the oracle
    eps = torch.randn(rows, A, device="cuda")
    a_out, lp_out = torch.empty(rows, A, device="cuda"), torch.empty(rows, device="cuda")
    _lib.check(lib.msacl_tanh_gauss_rsample(rows, A, logits.data_ptr(), eps.data_ptr(), lo.data_ptr(), hi.data_ptr(), -20.0, 1.0,
                                            a_out.data_ptr(), lp_out.data_ptr(), st))
    wa, wl, _ = oactor.tanh_gauss_sample(mean.cpu().numpy(), std.cpu().numpy(), eps.cpu().numpy(), g["act_low"], g["act_high"])
    np.testing.assert_allclose(a_out.cpu().numpy(), wa, rtol=0, atol=2e-5 * float((hi - lo).max()))
    ok = (np.abs(wa - (g["act_high"] + g["act_low"]) / 2) < 0.4995 * (g["act_high"] - g["act_low"])).all(axis=1)
    np.testing.assert_allclose(lp_out.cpu().numpy()[ok], wl[ok], rtol=1e-4, atol=1e-3)


def test_adam_multi_matches_torch_adam():
    """Three msacl_adam_multi steps (split gradient partials) vs torch.optim.Adam on identical gradients."""
    from msacl_b200.learner import FusedAdam
    torch.manual_seed(0)
    shapes = [(256, 6), (256,), (256, 256), (1, 256), (1,)]
    pa = [torch.nn.Parameter(torch.randn(*s, device="cuda")) for s in shapes]
    pb = [torch.nn.Parameter(p.detach().clone()) for p in pa]
    oa, ob = torch.optim.Adam(pa, lr=1e-3), torch.optim.Adam(pb, lr=1e-3)
    fa = FusedAdam(oa, pa)
    for step in range(3):
        S = 3
        parts = [torch.randn(S, *s, device="cuda") * (10.0 ** -step) for s in shapes]
        for p, g in zip(pb, parts):
            p.grad = (g[0] + g[1]) + g[2]
        ob.step()
        fa.step([(g, S) for g in parts])
        for a, b in zip(pa, pb):
            np.testing.assert_allclose(a.detach().cpu().numpy(), b.detach().cpu().numpy(), rtol=2e-6, atol=1e-7)
        assert float(oa.state[pa[0]]["step"]) == step + 1
    np.testing.assert_allclose(oa.state[pa[2]]["exp_avg_sq"].cpu().numpy(), ob.state[pb[2]]["exp_avg_sq"].cpu().numpy(), rtol=2e-6, atol=1e-12)


def test_learner_engine_falls_back_for_networks_outside_the_fused_family():
    """Three hidden layers / GELU: the default learner_engine switches to the autograd engine (with a warning) instead of
    failing at the first update; the reference accepts any `*_hidden_sizes` / `*_hidden_activation`."""
    import msacl_b200
    from msacl_b200.specs import get_spec
    spec = get_spec("VanderPol")
    D, A, n, B = spec.obs_dim, spec.act_dim, 5, 16
    alg = msacl_b200.create_alg(algorithm="msacl", env_name="VanderPol", obs_dim=D, act_dim=A, n_step=n, action_low_limit=spec.act_low,
                                action_high_limit=spec.act_high, q_learning_rate=1e-3, lyapunov_learning_rate=1e-3, policy_learning_rate=3e-4,
                                alpha_learning_rate=1e-3, value_hidden_sizes=[32, 32, 32], policy_hidden_activation="gelu")
    r = lambda *s: torch.randn(*s, device="cuda")
    data = dict(obs=r(B, n, D) * 0.3, obs2=r(B, n, D) * 0.3, act=torch.zeros(B, n, A, device="cuda"), rew=-torch.rand(B, n, device="cuda"),
                cost=torch.rand(B, n, device="cuda"), done=torch.zeros(B, n, device="cuda"), logp=r(B, n) - 1.0)
    with pytest.warns(UserWarning, match="learner_engine='torch'"):
        info = alg.model_update(data, 2)
    assert alg.engine_name == "torch" and info is not None and np.isfinite(list(info.values())).all()


@pytest.mark.parametrize("env,B,sizes", [("TwoLink", 48, None), ("QuadTracking", 20, None), ("DuctedFan", 33, None),
                                         ("SingleTrackCar", 24, dict(value_hidden_sizes=[128, 64], lyapunov_hidden_sizes=[64, 96],
                                                                     lyapunov_output_dim=32, policy_hidden_sizes=[96, 320]))])
def test_fused_learner_matches_torch_engine(env, B, sizes):
    """Two iterations (q + Lyapunov + 2 policy + alpha updates) of the fused learner vs the autograd engine from identical
    state, batch and rsample noise: same losses (2e-4) and the same parameters after the Adam steps."""
    import msacl_b200
    from msacl_b200.specs import get_spec
    spec = get_spec(env)
    D, A, n = spec.obs_dim, spec.act_dim, 20
    kw = dict(algorithm="msacl", env_name=env, obs_dim=D, act_dim=A, n_step=n, action_low_limit=spec.act_low, action_high_limit=spec.act_high,
              q_learning_rate=1e-3, lyapunov_learning_rate=1e-3, policy_learning_rate=3e-4, alpha_learning_rate=1e-3, lya_diff_scale=10.0,
              **(sizes or {}))
    torch.manual_seed(1)
    a = msacl_b200.create_alg(learner_engine="torch", **kw)
    b = msacl_b200.create_alg(learner_engine="fused", **kw)
    b.networks.load_state_dict(a.networks.state_dict())
    g = torch.Generator(device="cuda").manual_seed(2)
    r = lambda *s: torch.randn(*s, device="cuda", generator=g)
    lo, hi = (torch.as_tensor(x).cuda() for x in (spec.act_low, spec.act_high))
    obs = r(B, n, D) * 0.4
    data = dict(obs=obs, obs2=obs * 0.9 + 0.05 * r(B, n, D), act=(lo + (hi - lo) * torch.rand(B, n, A, device="cuda", generator=g)) * 0.97,
                rew=-torch.rand(B, n, device="cuda", generator=g) * 50, cost=torch.rand(B, n, device="cuda", generator=g),
                done=(torch.rand(B, n, device="cuda", generator=g) < 0.1).float(), logp=r(B, n) - 1.0)
    def compare_params(tag):
        sa, sb = a.networks.state_dict(), b.networks.state_dict()
        for k in sa:
            x, y = sa[k].cpu().numpy(), sb[k].cpu().numpy()
            bad = (~np.isclose(y, x, rtol=2e-4, atol=4e-6)).sum()
            # Adam's early steps are sign-like (lr * g / |g|): an entry whose gradient is at round-off level may step either
            # way, so a handful of entries per tensor is allowed to differ by up to 2 lr
            assert bad <= max(3, 0.002 * x.size), (tag, k, bad, x.size, np.abs(x - y).max())
            assert np.abs(x - y).max() <= 2.5e-3

    for it in (2, 3, 4):
        noise = [r(B, n, A) for _ in range(3)]
        ta = a.model_update(data, it, noise=[x.clone() for x in noise])
        tb = b.model_update(data, it, noise=[x.clone() for x in noise])
        assert (ta is None) == (tb is None)
        if ta is not None:
            for k in ta:
                if "time" not in k.lower():
                    np.testing.assert_allclose(tb[k], ta[k], rtol=1e-3, atol=1e-4, err_msg=f"{k} @ {it}")
        if it == 2:
            compare_params("after one update")
    # three updates later the two runs have drifted by a few sign-like steps at most
    sa, sb = a.networks.state_dict(), b.networks.state_dict()
    for k in sa:
        assert float((sa[k] - sb[k]).abs().max()) <= 4e-3, k


def _lib_st():
    import msacl_b200
    from msacl_b200 import _lib
    return msacl_b200.load_library(), _lib, _lib.current_stream()


@pytest.mark.parametrize("A", [1, 2, 8])
def test_policy_logits_grad_edges_vs_torch_autograd(A):
    """msacl_policy_logits_grad (critic path + entropy term + clipped surrogate on step 0 of each window) vs torch float32
    autograd of the same loss, at its edges: log_std exactly at min_log_std / max_log_std and beyond them (the clamp passes
    the gradient at the bounds), stored actions exactly at the action bounds (replay actions are clipped; the atanh argument
    is computed as the reference computes it, in float32), |u| > 9 where tanh is +-1 in float32, A = 1 and A = 8 (LA_MAX),
    and step-0 ratios on both sides of 1 - clip and 1 + clip."""
    from msacl_b200.algorithm import TanhGauss
    lib, _lib, st = _lib_st()
    g = torch.Generator(device="cuda").manual_seed(A)
    B, n, D, clip, min_ls, max_ls = 96, 4, 3, 0.1, -2.0, 0.5
    M = B * n
    r = lambda *s: torch.randn(*s, device="cuda", generator=g)
    lo = torch.tensor([-2.0, 0.0, -1.0, -5.0, -0.5, -3.0, 0.0, -1.0][:A], device="cuda")
    hi = torch.tensor([2.0, 3.0, 5.0, 5.0, 0.5, 1.0, 85.064, 1.0][:A], device="cuda")
    mean, ls = 0.5 * r(M, A), min_ls + (max_ls - min_ls) * torch.rand(M, A, device="cuda", generator=g)
    kind = torch.arange(M, device="cuda") % 8
    ls = torch.where(kind[:, None] == 1, torch.full_like(ls, min_ls), ls)        # exactly at the bounds ...
    ls = torch.where(kind[:, None] == 2, torch.full_like(ls, max_ls), ls)
    ls = torch.where(kind[:, None] == 3, min_ls - 0.5 - torch.rand_like(ls), ls)  # ... and beyond them
    ls = torch.where(kind[:, None] == 4, max_ls + 0.5 + torch.rand_like(ls), ls)
    eps = r(M, A)
    eps = torch.where(kind[:, None] == 5, torch.where(eps >= 0, 12.0, -12.0), eps)    # |u| > 9: tanh(u) = +-1 in float32
    mid, half = (hi + lo) / 2, (hi - lo) / 2
    act = mid + half * (1.9 * torch.rand(M, A, device="cuda", generator=g) - 0.95)
    at_bound = (kind == 6) | (kind == 7)
    act = torch.where(at_bound[:, None], torch.where(r(M, A) > 0, hi, lo), act)       # stored actions on the bounds
    logits = torch.cat([mean, ls], 1).contiguous()
    dxq1, dxq2 = r(M, D + A) / M, r(M, D + A) / M
    la = torch.tensor([-0.4], device="cuda")
    adv = r(B)

    def dist_of(lg):
        return TanhGauss(torch.cat([lg[:, :A], torch.clamp(lg[:, A:], min_ls, max_ls).exp()], 1), lo, hi)

    with torch.no_grad():
        lp0 = dist_of(logits).log_prob(act)
    log_ratio = torch.tensor([-0.5, -0.2, -0.05, 0.05, 0.2, 0.5], device="cuda")[torch.arange(M, device="cuda") % 6]
    old_logp = (lp0 - log_ratio).contiguous()
    first = torch.arange(M, device="cuda") % n == 0
    # torch float32 reference of the loss whose logits gradient the kernel writes
    lg = logits.clone().requires_grad_(True)
    dist = dist_of(lg)
    new_act, new_logp = dist.rsample(eps)
    ratio = torch.exp(dist.log_prob(act)[first] - old_logp[first])
    surr = torch.min(ratio * adv, torch.clamp(ratio, 1 - clip, 1 + clip) * adv)
    loss = (new_act * (dxq1 + dxq2)[:, D:]).sum() + la.exp() * new_logp.mean() - surr.mean()
    loss.backward()
    got = torch.full((M, 2 * A), float("nan"), device="cuda")
    sums = torch.zeros(3, dtype=torch.float64, device="cuda")
    _lib.check(lib.msacl_policy_logits_grad(M, n, D, A, logits.data_ptr(), eps.contiguous().data_ptr(), dxq1.data_ptr(), dxq2.data_ptr(),
                                            la.data_ptr(), act.contiguous().data_ptr(), old_logp.data_ptr(), adv.data_ptr(), clip,
                                            lo.data_ptr(), hi.data_ptr(), min_ls, max_ls, got.data_ptr(), sums.data_ptr(), st))
    want = lg.grad
    scale = float(want.abs().max())
    err = (got - want).abs() / scale
    print(f"A={A}: max err / max|g| {float(err.max()):.2e}, rows with actions on the bounds {float(err[at_bound].max()):.2e}")
    np.testing.assert_allclose(got.cpu().numpy(), want.cpu().numpy(), rtol=2e-4, atol=2e-5 * scale)
    # the kernel's ratios come from its own log_prob (float32, round-off apart): 1e-5 of the sum of |min(surr1, surr2)|
    assert abs(float(sums[2]) - float(surr.double().sum())) <= 1e-5 * float(surr.double().abs().sum())
    # every edge is exercised: clamped log_std columns get no gradient, the bound values do
    assert (got[kind == 3][:, A:] == 0).all() and (got[kind == 4][:, A:] == 0).all()
    assert (got[(kind == 1) | (kind == 2)][:, A:] != 0).all()
    r0 = ratio.detach()
    assert ((r0 < 1 - clip) & (adv > 0)).any() and ((r0 < 1 - clip) & (adv < 0)).any()
    assert ((r0 > 1 + clip) & (adv > 0)).any() and ((r0 > 1 + clip) & (adv < 0)).any() and ((r0 > 1 - clip) & (r0 < 1 + clip)).any()


def test_policy_q_route_exact_ties_vs_torch_minimum():
    """msacl_policy_q_route vs torch autograd of -mean(torch.minimum(q1, q2) - alpha logp): half the gradient to each critic
    on an exact tie; the two double-atomic sums vs float64."""
    lib, _lib, st = _lib_st()
    g = torch.Generator(device="cuda").manual_seed(4)
    rows = 3000
    q1 = torch.randn(rows, device="cuda", generator=g)
    q2 = torch.where(torch.arange(rows, device="cuda") % 3 == 0, q1, torch.randn(rows, device="cuda", generator=g))
    lp = torch.randn(rows, device="cuda", generator=g) - 2.0
    la = torch.tensor([0.3], device="cuda")
    a, b = q1.clone().requires_grad_(True), q2.clone().requires_grad_(True)
    (-(torch.minimum(a, b) - la.exp() * lp).mean()).backward()
    dq1, dq2 = torch.empty(rows, device="cuda"), torch.empty(rows, device="cuda")
    sums = torch.full((3,), 7.0, dtype=torch.float64, device="cuda")
    _lib.check(lib.msacl_policy_q_route(rows, q1.data_ptr(), q2.data_ptr(), lp.data_ptr(), la.data_ptr(), dq1.data_ptr(), dq2.data_ptr(),
                                        sums.data_ptr(), st))
    assert int((q1 == q2).sum()) == 1000
    np.testing.assert_allclose(dq1.cpu().numpy(), a.grad.cpu().numpy(), rtol=1e-6, atol=0)
    np.testing.assert_allclose(dq2.cpu().numpy(), b.grad.cpu().numpy(), rtol=1e-6, atol=0)
    alpha = float(torch.tensor(0.3).exp())
    np.testing.assert_allclose(float(sums[0]), float((torch.minimum(q1, q2).double() - alpha * lp.double()).sum()), rtol=1e-5)
    np.testing.assert_allclose(float(sums[1]), float(lp.double().sum()), rtol=1e-6)
    assert float(sums[2]) == 0.0


def test_q_backup_and_loss_grad_grid_stride_vs_float64():
    """msacl_q_backup_dev_alpha and msacl_q_loss_grad over more rows than one pass of the grid (148 * 8 * 256), so every
    thread strides; dq = 2 (q - y) / count and the four double-atomic sums vs float64."""
    lib, _lib, st = _lib_st()
    g = torch.Generator(device="cuda").manual_seed(9)
    count = 2 * 148 * 8 * 256 + 77
    r = lambda: torch.randn(count, device="cuda", generator=g)
    rew, nq1, nq2, nlp, q1, q2 = -torch.rand(count, device="cuda", generator=g) * 5, r(), r(), r() - 1, r(), r()
    done = (torch.rand(count, device="cuda", generator=g) < 0.2).float()
    la = torch.tensor([-0.25], device="cuda")
    backup = torch.empty(count, device="cuda")
    _lib.check(lib.msacl_q_backup_dev_alpha(count, rew.data_ptr(), done.data_ptr(), nq1.data_ptr(), nq2.data_ptr(), nlp.data_ptr(), 0.99,
                                            la.data_ptr(), backup.data_ptr(), st))
    alpha = float(np.exp(np.float32(-0.25)))
    want = rew.double() + (1 - done.double()) * 0.99 * (torch.minimum(nq1, nq2).double() - alpha * nlp.double())
    assert float((backup.double() - want).abs().max()) <= 2e-6 * float(want.abs().max())
    dq1, dq2 = torch.full_like(q1, float("nan")), torch.full_like(q2, float("nan"))
    sums = torch.full((4,), 7.0, dtype=torch.float64, device="cuda")
    _lib.check(lib.msacl_q_loss_grad(count, q1.data_ptr(), q2.data_ptr(), backup.data_ptr(), dq1.data_ptr(), dq2.data_ptr(), sums.data_ptr(), st))
    y = backup.double()
    for got, q in ((dq1, q1), (dq2, q2)):
        np.testing.assert_allclose(got.cpu().numpy(), (2 * (q.double() - y) / count).cpu().numpy(), rtol=1e-6, atol=0)
    want = [((q1.double() - y) ** 2).sum(), ((q2.double() - y) ** 2).sum(), q1.double().sum(), q2.double().sum()]
    scale = [want[0], want[1], q1.double().abs().sum(), q2.double().abs().sum()]
    for i in range(4):
        assert abs(float(sums[i] - want[i])) <= 1e-6 * float(scale[i]), (i, float(sums[i]), float(want[i]))


@pytest.mark.parametrize("cols", [32, 256])
def test_sumsq_bwd_vs_float64(cols):
    """msacl_sumsq_bwd: dz = 2 z dV for V = sum_j z_j^2 (the Lyapunov head), at 32 and 256 output columns."""
    lib, _lib, st = _lib_st()
    g = torch.Generator(device="cuda").manual_seed(cols)
    rows = 1234
    z, dv = torch.randn(rows, cols, device="cuda", generator=g), torch.randn(rows, device="cuda", generator=g)
    dz = torch.full_like(z, float("nan"))
    _lib.check(lib.msacl_sumsq_bwd(rows, cols, z.data_ptr(), dv.data_ptr(), dz.data_ptr(), st))
    zz = z.double().clone().requires_grad_(True)
    ((zz ** 2).sum(1) * dv.double()).sum().backward()
    np.testing.assert_allclose(dz.cpu().numpy(), zz.grad.cpu().numpy(), rtol=1e-7, atol=0)


@pytest.mark.parametrize("alpha_bound", [None, 0.72])
def test_alpha_update_steps_match_torch_adam(alpha_bound):
    """msacl_adam_tick + msacl_alpha_update, several steps, vs torch.optim.Adam on a float32 log_alpha with
    loss_alpha = exp(log_alpha) (entropy - target), with and without the alpha_bound clamp after the step."""
    import math
    lib, _lib, st = _lib_st()
    rows, target, lr = 1024, -2.0, 1e-2
    p = torch.nn.Parameter(torch.tensor(math.log(0.7)))
    opt = torch.optim.Adam([p], lr=lr)
    la = torch.tensor([math.log(0.7)], device="cuda")
    step, dyn = torch.zeros(1, dtype=torch.int32, device="cuda"), torch.zeros(2, device="cuda")
    state, ent_out = torch.zeros(2, device="cuda"), torch.zeros(1, device="cuda")
    clamp = math.log(alpha_bound) if alpha_bound else float("inf")
    for k, entropy in enumerate([-3.0, -2.5, -4.0, -2.25, -3.5, -1.5]):      # entropy below the target: log_alpha grows
        sums = torch.tensor([0.0, -entropy * rows, 0.0], dtype=torch.float64, device="cuda")
        _lib.check(lib.msacl_adam_tick(step.data_ptr(), dyn.data_ptr(), lr, 0.9, 0.999, st))
        _lib.check(lib.msacl_alpha_update(la.data_ptr(), sums.data_ptr(), rows, target, state.data_ptr(), 0.1, 0.999, 0.001, 0.0, 1.0, 1e-8,
                                          clamp, ent_out.data_ptr(), dyn.data_ptr(), st))
        opt.zero_grad()
        (p.exp() * (torch.tensor(entropy) - target)).backward()
        opt.step()
        if alpha_bound:
            with torch.no_grad():
                p.clamp_(max=math.log(alpha_bound))
        assert float(ent_out) == entropy
        np.testing.assert_allclose(float(la), float(p), rtol=2e-6, atol=1e-7, err_msg=f"step {k + 1}")
    assert int(step) == 6
    if alpha_bound:
        assert float(la) == float(np.float32(math.log(alpha_bound)))
