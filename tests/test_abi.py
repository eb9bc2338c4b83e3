"""CPU-only checks of the C-ABI boundary: the library builds/loads, exports every symbol the
header declares, and the product path refuses to run without a GPU (no CPU fallback)."""
import os
import re

import pytest

import msacl_b200
from msacl_b200 import _lib, specs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    text = open(os.path.join(ROOT, "include", "msacl_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(msacl_[a-z0-9_]+)\s*\(", text)))


def test_library_loads_and_exports_every_declared_symbol_at_abi_3():
    lib = msacl_b200.load_library()
    syms = header_symbols()
    assert len(syms) >= 15
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/msacl_b200.h but not exported"
    assert sorted(_lib.SIGNATURES) == syms, "ctypes SIGNATURES and the header disagree"
    assert lib.msacl_abi_version() == 3


def test_env_dims_match_spec_table():
    import ctypes as C
    lib = msacl_b200.load_library()
    for name in specs.ENV_NAMES:
        s = specs.get_spec(name)
        dims = (C.c_int32 * 6)()
        assert lib.msacl_env_dims(s.env_id, dims) == 0
        assert list(dims) == [s.obs_dim, s.act_dim, s.sf_rows, s.sd_rows, s.obs_off, s.control_step]
    dims = (C.c_int32 * 6)()
    assert lib.msacl_env_dims(17, dims) == -1
    assert b"unknown env id" in lib.msacl_last_error()


def test_unknown_env_raises_like_reference():
    with pytest.raises(ValueError, match="Unknown custom env"):
        specs.get_spec("CartPole")


def test_product_never_imports_oracle():
    pkg = os.path.dirname(_lib.__file__)
    for root, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(root, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f


def test_no_cpu_fallback_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(Exception):
        msacl_b200.create_envs(env_name="VanderPol", env_num=4, env_seed=0)


def test_error_codes_without_gpu_work():
    """Argument validation happens on the host before any launch (no C++ exceptions across the ABI)."""
    import ctypes as C
    lib = msacl_b200.load_library()
    st = _lib.EnvState(env_id=0, max_step=1000, n=0, stride=0)
    assert lib.msacl_env_reset(C.byref(st), None) == -2 and b"invalid env state" in lib.msacl_last_error()
    assert lib.msacl_env_step(C.byref(st), None, None, None, None, None, None, None) == -2
    assert lib.msacl_q_backup(0, None, None, None, None, None, 0.99, 0.2, None, None) == -2
    assert lib.msacl_lyapunov_risk(4, 33, 2, *([None] * 9), 1.0, 2.0, 10.0, 1.0, *([None] * 5), None) == -2
    assert b"n_step must be <= 32" in lib.msacl_last_error()
    assert lib.msacl_action_noise(0, 0, 8, 5, 0, None, None) == -2
    n1, n2 = C.c_int64(0), C.c_int64(0)
    assert lib.msacl_tc_pack_bytes(C.byref(n1), C.byref(n2)) == 0 and n1.value == 16384 and n2.value == 262144


@pytest.mark.parametrize("n_envs,grid", [(65536, 148), (1 << 21, 148), (1 << 22, 148), (1000, 8), (128, 1), (129, 2), (70000, 148),
                                         (148 * 128 * 7 + 700, 148), (1 << 20, 140), (40001, 148), (5, 1)])
def test_tc_tile_shares_partition_the_tile_list(n_envs, grid):
    """msacl_rollout_fused_tc deals its 128-env tiles to the persistent CTAs in balanced contiguous shares, walked in rounds of at
    most 3 tiles (host-side arithmetic shared with the kernel: TcShare in csrc/rollout_tc.cu).  Every tile is owned exactly once,
    shares differ by at most one tile, round sizes are non-increasing (a warpgroup idle in one round stays idle: the kernel's
    X-operand counters rely on it) and the number of rounds is the minimum."""
    import ctypes as C
    lib = msacl_b200.load_library()
    tiles = (n_envs + 127) // 128
    nxt, shares = 0, []
    for cta in range(grid):
        out = (C.c_int64 * 5)()
        assert lib.msacl_tc_tile_share(n_envs, grid, cta, out) == 0
        first, share, rounds, per, ex = list(out)
        assert first == nxt, "shares are contiguous and in CTA order"
        sizes = [per + (1 if j < ex else 0) for j in range(rounds)]
        assert sum(sizes) == share and all(1 <= s <= 3 for s in sizes)
        assert sizes == sorted(sizes, reverse=True)
        assert rounds == -(-share // 3)
        nxt += share
        shares.append(share)
    assert nxt == tiles
    assert max(shares) - min(shares) <= 1
    out = (C.c_int64 * 5)()
    assert lib.msacl_tc_tile_share(n_envs, grid, grid, out) != 0          # cta out of range
    assert b"tc_tile_share" in lib.msacl_last_error()
