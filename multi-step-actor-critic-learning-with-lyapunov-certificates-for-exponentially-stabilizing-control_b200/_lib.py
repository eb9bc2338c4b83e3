"""ctypes binding of lib/libmsacl_b200.so (the C ABI declared in include/msacl_b200.h).

There is no CPU fallback: the library is (re)built with nvcc whenever its source digest does not match
the tree (build.py); if it cannot be built or loaded, importing the kernels raises.
"""
import ctypes as C
import os

from . import build as _build

_LIB = None
ABI_VERSION = 3      # MSACL_ABI_VERSION of include/msacl_b200.h this binding was written against

c_f32p = C.POINTER(C.c_float)
c_f64p = C.POINTER(C.c_double)
c_i32p = C.POINTER(C.c_int32)
c_i64p = C.POINTER(C.c_int64)
c_u8p = C.POINTER(C.c_uint8)
vp = C.c_void_p


class EnvState(C.Structure):
    _fields_ = [("env_id", C.c_int32), ("max_step", C.c_int32), ("n", C.c_int64), ("stride", C.c_int64),
                ("sf", vp), ("sd", vp), ("step", vp), ("episode", vp), ("ep_return", vp), ("ep_len", vp),
                ("run", vp), ("seed", C.c_uint64), ("env_base", C.c_uint64)]


class Actor(C.Structure):
    _fields_ = [("w1", vp), ("b1", vp), ("w2t", vp), ("b2", vp), ("w3", vp), ("b3", vp),
                ("min_log_std", C.c_float), ("max_log_std", C.c_float)]


class Transitions(C.Structure):
    _fields_ = [("obs", vp), ("act", vp), ("rew", vp), ("cost", vp), ("obs2", vp), ("done", vp), ("logp", vp),
                ("emit", vp), ("logits", vp)]


class Ring(C.Structure):
    _fields_ = [("max_size", C.c_int64), ("n_step", C.c_int32), ("obs_dim", C.c_int32), ("act_dim", C.c_int32),
                ("obs", vp), ("act", vp), ("rew", vp), ("cost", vp), ("obs2", vp), ("done", vp), ("logp", vp)]


class Gemm(C.Structure):
    _fields_ = [("a", vp), ("a_row_stride", C.c_int64), ("a_k_stride", C.c_int64),
                ("b", vp), ("b_row_stride", C.c_int64), ("b_k_stride", C.c_int64),
                ("m", C.c_int32), ("n", C.c_int32), ("k", C.c_int32),
                ("c", vp), ("ldc", C.c_int64), ("split_k", C.c_int32), ("c_split_stride", C.c_int64),
                ("bias", vp), ("act", C.c_int32), ("mask_src", vp), ("mask_ld", C.c_int64), ("mask_act", C.c_int32),
                ("row_sumsq", vp), ("precision", C.c_int32), ("b_packed", vp)]


class CertParams(C.Structure):
    _fields_ = [("horizon", C.c_int32), ("alpha1", C.c_double), ("alpha2", C.c_double), ("v_atol", C.c_double), ("decay", vp)]


class CertRecords(C.Structure):
    _fields_ = [("v0", vp), ("s0", vp), ("flags", vp), ("first_violation", vp), ("first_decrease", vp), ("end_step", vp),
                ("worst_ratio", vp)]


class RegionNets(C.Structure):
    _fields_ = [("env_id", C.c_int32), ("obs_dim", C.c_int32), ("act_dim", C.c_int32), ("p_h1", C.c_int32), ("p_h2", C.c_int32),
                ("p_w1", vp), ("p_b1", vp), ("p_w2", vp), ("p_b2", vp), ("p_w3", vp), ("p_b3", vp),
                ("v_h1", C.c_int32), ("v_h2", C.c_int32), ("v_out", C.c_int32),
                ("v_w1", vp), ("v_b1", vp), ("v_w2", vp), ("v_b2", vp), ("v_w3", vp), ("v_b3", vp)]


class RegionDisturbance(C.Structure):
    _fields_ = [("obs_lo", C.c_float * 16), ("obs_hi", C.c_float * 16), ("act_lo", C.c_float * 2), ("act_hi", C.c_float * 2),
                ("state_lo", C.c_float * 16), ("state_hi", C.c_float * 16)]


class RegionParams(C.Structure):
    _fields_ = [("env_id", C.c_int32), ("steps", C.c_int32), ("v_tanh", C.c_int32), ("decay_lo", C.c_double),
                ("decay_hi", C.c_double), ("alpha1", C.c_double), ("alpha2", C.c_double), ("x0_lo", C.c_float * 16),
                ("x0_hi", C.c_float * 16), ("dist", RegionDisturbance)]


class RegionOut(C.Structure):
    _fields_ = [("v_lo", vp), ("v_hi", vp), ("vm_lo", vp), ("vm_hi", vp), ("img_lo", vp), ("img_hi", vp), ("flags", vp),
                ("margin", vp), ("trace", vp)]


class RegionBnb(C.Structure):
    _fields_ = [("max_depth", C.c_int32), ("inner_level", C.c_int32), ("inner_lo", C.c_uint32 * 16), ("inner_hi", C.c_uint32 * 16),
                ("inner_box_lo", C.c_double * 16), ("inner_box_hi", C.c_double * 16), ("max_examples", C.c_int64)]


class RegionWs(C.Structure):
    _fields_ = [("cells", vp), ("lo", vp), ("hi", vp), ("res", RegionOut), ("plo", vp), ("phi", vp), ("pres", RegionOut),
                ("probe", vp), ("status", vp), ("scan", vp)]


f32 = C.c_float
i32, i64 = C.c_int32, C.c_int64

# name -> (restype, argtypes); must list every symbol of include/msacl_b200.h
SIGNATURES = {
    "msacl_last_error": (C.c_char_p, []),
    "msacl_abi_version": (C.c_int, []),
    "msacl_env_dims": (C.c_int, [C.c_int, c_i32p]),
    "msacl_env_bounds": (C.c_int, [C.c_int, c_f32p, c_f32p, c_f32p, c_f32p]),
    "msacl_env_reset": (C.c_int, [C.POINTER(EnvState), vp]),
    "msacl_quad_init_from_raw": (C.c_int, [C.POINTER(EnvState), vp]),
    "msacl_env_step": (C.c_int, [C.POINTER(EnvState), vp, vp, vp, vp, vp, vp, vp]),
    "msacl_rollout_fused": (C.c_int, [C.POINTER(EnvState), C.POINTER(Actor), C.c_int32, C.c_uint32, C.c_int32,
                                      C.c_float, C.c_float, vp, C.c_int32, C.POINTER(Transitions), vp, vp]),
    "msacl_tc_pack_bytes": (C.c_int, [c_i64p, c_i64p]),
    "msacl_rollout_tc_set_max_ctas": (C.c_int, [C.c_int32]),
    "msacl_tc_tile_share": (C.c_int, [i64, C.c_int32, C.c_int32, vp]),
    "msacl_tc_pack_actor": (C.c_int, [C.POINTER(Actor), C.c_int32, vp, vp, vp]),
    "msacl_rollout_fused_tc": (C.c_int, [C.POINTER(EnvState), C.POINTER(Actor), vp, vp, C.c_int32, C.c_uint32, C.c_int32,
                                         C.c_float, C.c_float, vp, C.c_int32, C.POINTER(Transitions), vp, vp]),
    "msacl_rollout_step": (C.c_int, [C.POINTER(EnvState), vp, C.c_float, C.c_float, C.c_uint32, C.c_int32, C.c_float, C.c_float, vp,
                                     C.c_int32, C.POINTER(Transitions), vp, vp]),
    "msacl_action_noise": (C.c_int, [C.c_uint64, C.c_uint64, C.c_int64, C.c_int32, C.c_uint32, vp, vp]),
    "msacl_window_store_scratch_elems": (C.c_int64, [C.c_int32, C.c_int64]),
    "msacl_selftest_quad_polar": (C.c_int, [vp, vp, C.c_int64, C.c_float, vp]),
    "msacl_window_store": (C.c_int, [C.POINTER(Transitions), C.c_int32, C.c_int32, C.c_int64, C.POINTER(Ring), vp, vp,
                                     vp, vp]),
    "msacl_window_index_store": (C.c_int, [vp, C.c_int32, C.c_int64, C.c_int64, vp, C.c_int64, vp, vp, vp, vp]),
    "msacl_window_gather_indexed": (C.c_int, [C.POINTER(Transitions), C.c_int64, vp, vp, C.c_int64, C.POINTER(Ring), vp]),
    "msacl_ring_sample": (C.c_int, [C.POINTER(Ring), vp, C.c_uint64, C.c_uint64, C.c_int64, C.POINTER(Ring), vp, vp]),
    "msacl_window_sample_indexed": (C.c_int, [C.POINTER(Transitions), C.c_int64, vp, C.c_int64, vp, vp, C.c_int32, C.c_uint64, C.c_uint64,
                                              C.c_int64, C.POINTER(Ring), vp, vp]),
    "msacl_ring_gather": (C.c_int, [C.POINTER(Ring), vp, C.c_int64, C.POINTER(Ring), vp]),
    "msacl_q_backup": (C.c_int, [C.c_int64, vp, vp, vp, vp, vp, C.c_float, C.c_float, vp, vp]),
    "msacl_lyapunov_risk": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, vp, vp, vp, vp, vp, vp, vp, vp, vp, C.c_float,
                                      C.c_float, C.c_float, C.c_float, vp, vp, vp, vp, vp, vp]),
    "msacl_stability_advantage": (C.c_int, [C.c_int64, C.c_int32, vp, vp, vp, vp, vp, vp, vp]),
    "msacl_advantage_normalize": (C.c_int, [C.c_int64, vp, vp, vp, vp]),
    "msacl_selftest_tc_gemm": (C.c_int, [vp, vp, vp, C.c_int32, vp]),
    "msacl_polyak_update": (C.c_int, [C.c_int32, vp, vp, vp, C.c_int64, C.c_float, C.c_float, vp]),
    "msacl_gemm_tc": (C.c_int, [C.POINTER(Gemm), vp]),
    "msacl_gemm_packed_b_bytes": (C.c_int64, [i32, i32]),
    "msacl_gemm_pack_b": (C.c_int, [C.POINTER(Gemm), vp, vp]),
    "msacl_colsum": (C.c_int, [vp, i64, i32, i64, i32, vp, vp]),
    "msacl_concat2": (C.c_int, [vp, i32, vp, i32, i64, vp, vp]),
    "msacl_reduce_splits": (C.c_int, [vp, i64, i32, vp, vp]),
    "msacl_tanh_gauss_rsample": (C.c_int, [i64, i32, vp, vp, vp, vp, f32, f32, vp, vp, vp]),
    "msacl_tanh_gauss_log_prob": (C.c_int, [i64, i32, vp, vp, vp, vp, f32, f32, vp, vp]),
    "msacl_tanh_gauss_log_prob_bwd": (C.c_int, [i64, i32, vp, vp, vp, vp, f32, f32, vp, i32, vp, vp]),
    "msacl_q_backup_dev_alpha": (C.c_int, [i64, vp, vp, vp, vp, vp, f32, vp, vp, vp]),
    "msacl_q_loss_grad": (C.c_int, [i64, vp, vp, vp, vp, vp, vp, vp]),
    "msacl_sumsq_bwd": (C.c_int, [i64, i32, vp, vp, vp, vp]),
    "msacl_policy_q_route": (C.c_int, [i64, vp, vp, vp, vp, vp, vp, vp, vp]),
    "msacl_policy_logits_grad": (C.c_int, [i64, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, f32, vp, vp, f32, f32, vp, vp, vp]),
    "msacl_alpha_update": (C.c_int, [vp, vp, i64, f32, vp, f32, f32, f32, f32, f32, f32, f32, vp, vp, vp]),
    "msacl_adam_multi": (C.c_int, [i32, vp, vp, vp, vp, vp, vp, i64, f32, f32, f32, f32, f32, f32, vp, vp]),
    "msacl_adam_tick": (C.c_int, [vp, vp, C.c_double, C.c_double, C.c_double, vp]),
    "msacl_ffma_probe": (C.c_int, [C.c_int32, C.c_int32, vp, c_f64p, vp]),
    "msacl_umma_probe": (C.c_int, [C.c_int32, C.c_int32, vp, vp]),
    "msacl_certify_box_init": (C.c_int, [C.POINTER(EnvState), c_f32p, c_f32p, vp]),
    "msacl_certify_begin": (C.c_int, [i64, i32, vp, vp, C.POINTER(CertParams), C.POINTER(CertRecords), vp]),
    "msacl_certify_steps": (C.c_int, [i64, i32, i32, i32, vp, vp, vp, C.POINTER(CertParams), C.POINTER(CertRecords), vp]),
    "msacl_certify_finish": (C.c_int, [i64, i32, C.POINTER(CertRecords), vp, vp]),
    "msacl_certify_roa": (C.c_int, [i64, vp, f32, vp, vp]),
    "msacl_region_image_bytes": (C.c_int64, []),
    "msacl_region_pack": (C.c_int, [C.POINTER(RegionNets), vp, vp]),
    "msacl_region_eval": (C.c_int, [C.POINTER(RegionParams), vp, i64, vp, vp, vp, C.POINTER(RegionOut), vp]),
    "msacl_region_round": (C.c_int, [C.POINTER(RegionParams), C.POINTER(RegionBnb), vp, vp, i64, i64, C.POINTER(RegionWs), vp, vp,
                                     vp, vp]),
}


def lib_path():
    return _build.LIB


def load():
    """Load (building first if needed) the CUDA library.  Raises on failure -- never falls back."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = _build.LIB
    try:
        _build.build()                  # sha256 of the sources vs the stamp: returns at once when the library is current
    except (OSError, RuntimeError) as e:
        # no usable nvcc on this host: an existing library may still be loaded, but never silently when it is stale
        if not os.path.exists(path):
            raise
        if not _build.is_current():
            import warnings
            warnings.warn(f"libmsacl_b200.so is older than its sources and could not be rebuilt ({e}); loading the stale binary")
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.msacl_abi_version() != ABI_VERSION:
        raise RuntimeError("libmsacl_b200.so ABI version mismatch")
    _LIB = lib
    return lib


class MsaclError(RuntimeError):
    pass


def check(rc):
    if rc != 0:
        msg = load().msacl_last_error().decode("utf-8", "replace")
        raise MsaclError(f"libmsacl_b200 error {rc}: {msg}")


def ptr(t):
    """Device pointer of a torch tensor (or None)."""
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous(), "libmsacl_b200 needs contiguous CUDA tensors"
    return t.data_ptr()


def current_stream():
    import torch
    return torch.cuda.current_stream().cuda_stream
