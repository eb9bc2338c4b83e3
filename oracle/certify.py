"""Oracle (test infrastructure): the Lyapunov-certificate verifier's contract over given trajectories.

NumPy restatement of csrc/certify.cu (include/msacl_b200.h, "Lyapunov-certificate verifier"); the reference has no
counterpart.  Inputs are the visited observations o [L, N, D] (float32; o[0] = initial state, o[k] = state after k greedy
steps), V [L, N] = V(o) (float32) and done [L, N] (done[k] = the step into o[k] terminated; done[0] is ignored), L >= T + 1.
Every comparison is in float64 on values that are exact in float64, so the kernel must agree bit for bit.
"""
import numpy as np

NONFINITE, BOUND_LO, BOUND_HI, DECREASE, ESCAPED, NOT_EXP_STABLE = 1, 2, 4, 8, 16, 32
FAIL_MASK = 31
FLAG_NAMES = ("nonfinite", "bound_lo", "bound_hi", "decrease", "escaped", "not_exp_stable")


def decay_table(T, lya_eta):
    """c_0 = 1, c_k = c_{k-1} (1 - eta), float64 by repeated multiplication (not pow)."""
    c = np.empty(T + 1, np.float64)
    c[0] = 1.0
    base = 1.0 - float(lya_eta)
    for k in range(1, T + 1):
        c[k] = c[k - 1] * base
    return c


def sumsq64(o):
    """sum_j o[..., j]^2 in float64, sequentially over j."""
    o = np.asarray(o, np.float32).astype(np.float64)
    s = np.zeros(o.shape[:-1], np.float64)
    for j in range(o.shape[-1]):
        s = s + o[..., j] * o[..., j]
    return s


def _visit(o, v, s, k, ck, v0, s0, alpha1, alpha2, v_atol):
    fin = np.isfinite(v) & np.all(np.isfinite(o), axis=-1)
    f = np.where(fin, 0, NONFINITE).astype(np.int64)
    vd = v.astype(np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        f |= np.where(vd < alpha1 * s - v_atol, BOUND_LO, 0)
        f |= np.where(vd > alpha2 * s + v_atol, BOUND_HI, 0)
        if k >= 1:
            f |= np.where(vd > ck * v0 + v_atol, DECREASE, 0)
            f |= np.where(s > (alpha2 / alpha1) * ck * s0, NOT_EXP_STABLE, 0)
    return f


def check(o, V, done, T, lya_eta=0.15, alpha1=1.0, alpha2=2.0, v_atol=0.0):
    """Per-state records: dict(v0, flags, first_violation, first_decrease, end_step, worst_ratio)."""
    o = np.asarray(o, np.float32)
    V = np.asarray(V, np.float32)
    done = np.asarray(done).astype(bool)
    assert o.shape[0] >= T + 1 and V.shape[0] >= T + 1 and done.shape[0] >= T + 1
    alpha1, alpha2, v_atol = float(alpha1), float(alpha2), float(v_atol)
    c = decay_table(T, lya_eta)
    N = o.shape[1]
    v0 = V[0].astype(np.float64)
    s0 = sumsq64(o[0])
    flags = _visit(o[0], V[0], s0, 0, 1.0, v0, s0, alpha1, alpha2, v_atol)
    fv = np.where(flags & FAIL_MASK, 0, -1)
    fd = np.full(N, -1, np.int64)
    end = np.full(N, T, np.int64)
    worst = np.zeros(N, np.float64)
    alive = np.ones(N, bool)
    for k in range(1, T + 1):
        if not alive.any():
            break
        s = sumsq64(o[k])
        f = _visit(o[k], V[k], s, k, c[k], v0, s0, alpha1, alpha2, v_atol)
        vd, den = V[k].astype(np.float64), c[k] * v0
        with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
            ratio = np.where(den == 0.0, np.where(vd > 0.0, np.inf, 0.0), vd / np.where(den == 0.0, 1.0, den))
            worst = np.where(alive & (ratio > worst), ratio, worst)
        f = np.where(done[k], f | ESCAPED, f)
        f = np.where(alive, f, 0)
        fv = np.where(((f & FAIL_MASK) != 0) & ((flags & FAIL_MASK) == 0), k, fv)
        fd = np.where(((f & DECREASE) != 0) & ((flags & DECREASE) == 0), k, fd)
        flags = flags | f
        ended = alive & done[k]
        end = np.where(ended, k, end)
        alive = alive & ~done[k]
    return dict(v0=V[0].copy(), flags=flags.astype(np.uint8), first_violation=fv.astype(np.int32),
                first_decrease=fd.astype(np.int32), end_step=end.astype(np.int32), worst_ratio=worst.astype(np.float32))


def summarize(rec, T):
    """Counts of every flag, certified and inconsistent (DECREASE != NOT_EXP_STABLE) states, the first-DECREASE histogram
    [T] (bin k - 1), c_star = min V_0 over uncertified states with V_0 not NaN (+inf if none) and roa_count =
    #{i : V_0,i < c_star}."""
    flags = rec["flags"].astype(np.int64)
    v0 = rec["v0"].astype(np.float32)
    out = {"states": int(flags.size)}
    for b, name in enumerate(FLAG_NAMES):
        out[name] = int(((flags >> b) & 1).sum())
    cert = (flags & FAIL_MASK) == 0
    out["certified"] = int(cert.sum())
    out["inconsistent"] = int((((flags >> 3) ^ (flags >> 5)) & 1).sum())
    fd = rec["first_decrease"]
    out["first_decrease_hist"] = np.bincount(fd[(fd >= 1) & (fd <= T)] - 1, minlength=T)[:T].astype(np.int64)
    cand = v0[~cert & ~np.isnan(v0)]
    out["c_star"] = float(cand.min()) if cand.size else float("inf")
    with np.errstate(invalid="ignore"):
        out["roa_count"] = int((v0 < np.float32(out["c_star"])).sum())
    return out
