"""A/B probe of msacl_lyapunov_risk over window lengths (constant element count 2^20 x 20): ms, GB/s, fraction of HBM."""
import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import msacl_b200  # noqa: F401
from msacl_b200 import targets as tg, _lib
lib = _lib.load(); st = _lib.current_stream()
HBM = 6551.0
try:
    HBM = float(json.load(open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "MEASURED_PEAKS.json"))).get("hbm_gbs", HBM))
except Exception:
    pass
D = int(os.environ.get("D", 4))
NS = [int(x) for x in os.environ.get("N", "8,16,20,24,32").split(",")]
for n in NS:
    B = (1 << 20) * 20 // n
    g = torch.Generator(device="cuda").manual_seed(0)
    r = lambda *s: torch.randn(*s, device="cuda", generator=g)
    obs, obs2, lpn, lpo, v1, v2 = r(B, n, D) * 0.5, r(B, n, D) * 0.5, r(B, n), r(B, n), r(B, n).abs(), r(B, n).abs()
    coef = tg.Coefficients(n)
    parts = torch.empty(3, dtype=torch.float64, device="cuda"); g1, g2 = torch.empty_like(v1), torch.empty_like(v2)
    fn = lambda: _lib.check(lib.msacl_lyapunov_risk(B, n, D, obs.data_ptr(), obs2.data_ptr(), lpn.data_ptr(), lpo.data_ptr(), v1.data_ptr(),
                                                    v2.data_ptr(), coef.son.data_ptr(), coef.diff.data_ptr(), coef.sl.data_ptr(), coef.alpha1,
                                                    coef.alpha2, 10.0, 1.0, parts.data_ptr(), g1.data_ptr(), g2.data_ptr(), None, None, st))
    for _ in range(3): fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(); a.record()
    for _ in range(20): fn()
    b.record(); torch.cuda.synchronize()
    ms = a.elapsed_time(b) / 20
    gbs = B * n * 4 * (2 * D + 6) / ms / 1e6
    print(f"n {n} D {D} ms {ms:.4f} GB/s {gbs:.0f} frac {gbs / HBM:.3f}", flush=True)
