"""ctypes binding of libsaceo.so (include/saceo.h) - the only way the Python host code reaches CUDA.

There is no CPU fallback: if the shared library is missing the import of this module still works
(so layout arithmetic and the CPU tests can run), but every compute entry point raises
``SaceoError`` loudly, and ``load()`` raises if the library cannot be found.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SACEO_LIB") or os.path.join(_HERE, "libsaceo.so")     # SACEO_LIB: alternative build (experiments)

ABI_VERSION = 2
POLICY_MAX_HIDDEN = 8       # SACEO_POLICY_MAX_HIDDEN: most hidden layers of a dynamics model or an acted policy
ACT_IDS = {"relu": 0, "tanh": 1, "elu": 2}
GEMM_FP32_SIMT = 0
GEMM_TCGEN05_BF16X3 = 1


class SaceoError(RuntimeError):
    pass


class Config(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("device", C.c_int32), ("n_agents", C.c_int32),
        ("S", C.c_int32), ("A", C.c_int32),
        ("actor_hidden", C.c_int32 * 2), ("critic_hidden", C.c_int32 * 2),
        ("actor_act", C.c_int32 * 2), ("critic_act", C.c_int32 * 2),
        ("model_layers", C.c_int32), ("model_hidden", C.c_int32 * POLICY_MAX_HIDDEN),
        ("model_act", C.c_int32 * POLICY_MAX_HIDDEN),
        ("per_state_std", C.c_int32), ("separate_reward_nn", C.c_int32), ("num_models", C.c_int32),
        ("delta_clip_pred", C.c_float),
        ("B", C.c_int32), ("E", C.c_int32), ("target_update_int", C.c_int32),
        ("replay_capacity", C.c_int32), ("fvp_rows", C.c_int32), ("std_mult", C.c_float),
        ("gemm_mode", C.c_int32), ("use_graph", C.c_int32), ("reserved", C.c_int32 * 8),
    ]


class Layout(C.Structure):
    _fields_ = [
        ("na", C.c_int64), ("nc", C.c_int64), ("nm", C.c_int64),
        ("na_stride", C.c_int64), ("nc_stride", C.c_int64), ("nm_stride", C.c_int64),
        ("Ao", C.c_int32), ("model_out", C.c_int32),
        ("row_words", C.c_int32), ("off_s", C.c_int32), ("off_a", C.c_int32), ("off_sp", C.c_int32),
        ("off_r", C.c_int32), ("off_d", C.c_int32),
        ("norm_stride", C.c_int32), ("off_s_mean", C.c_int32), ("off_s_std", C.c_int32),
        ("off_a_mean", C.c_int32), ("off_a_std", C.c_int32), ("off_ret_std", C.c_int32),
        ("off_m_s_mean", C.c_int32), ("off_m_s_std", C.c_int32), ("off_m_a_mean", C.c_int32),
        ("off_m_a_std", C.c_int32), ("off_m_d_mean", C.c_int32), ("off_m_d_std", C.c_int32),
        ("off_act_limit", C.c_int32),
        ("hyper_stride", C.c_int32), ("n_losses", C.c_int32),
        ("workspace_bytes", C.c_int64),
    ]


class Tables(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "actor", "actor_m", "actor_v", "q", "q_m", "q_v", "qt", "model",
        "alpha", "alpha_m", "alpha_v", "adam_t", "norm", "hyper",
        "replay", "replay_size", "replay_start", "expert_s", "expert_sp", "fvp_states")]


class FitTables(C.Structure):
    """saceo_fit_tables (include/saceo.h): dynamics-model fitting state."""
    _fields_ = [(n, C.c_void_p) for n in ("model", "model_m", "model_v", "model_t", "fit_hyper",
                                          "model_logstd", "model_logstd_m", "model_logstd_v",
                                          "reward", "reward_m", "reward_v")] + \
               [("reward_hidden", C.c_int32 * 2), ("reward_act", C.c_int32 * 2), ("reward_stride", C.c_int64)]
    POINTERS = ("model", "model_m", "model_v", "model_t", "fit_hyper", "model_logstd", "model_logstd_m", "model_logstd_v",
                "reward", "reward_m", "reward_v")


class PolicyConfig(C.Structure):
    """saceo_policy_config (include/saceo.h): a set of policies of any depth, acted by ``saceo_policy_act``."""
    _fields_ = [
        ("abi_version", C.c_int32), ("device", C.c_int32), ("n_policies", C.c_int32), ("S", C.c_int32), ("A", C.c_int32),
        ("n_hidden", C.c_int32), ("hidden", C.c_int32 * POLICY_MAX_HIDDEN), ("act", C.c_int32 * POLICY_MAX_HIDDEN),
        ("squash", C.c_int32), ("per_state_std", C.c_int32), ("std_mult", C.c_float),
    ]


class GemmArgs(C.Structure):
    """saceo_gemm_args (include/saceo.h): one call of the GEMM dispatch, for saceo_test_gemm_ex."""
    _fields_ = [(n, C.c_int32) for n in ("gemm_mode", "n_agents", "nnet", "transA", "transB", "ones",
                                         "M", "N", "K", "lda", "ldb", "ldc")] + \
               [(n, C.c_int64) for n in ("sAa", "sAn", "sBa", "sBn", "sCa", "sCn", "sba", "sbn")] + \
               [(n, C.c_void_p) for n in ("A", "B", "C", "bias", "addend", "aux")] + \
               [(n, C.c_int32) for n in ("epi", "act", "f16")]


class GemmRoute(C.Structure):
    """saceo_gemm_route (include/saceo.h): which kernels a saceo_test_gemm_ex call launched."""
    _fields_ = [(n, C.c_int32) for n in ("n_tc", "n_skinny", "n_simt", "tc_rows", "tc_stream", "tc_akc", "tc_bkc",
                                         "tc_bn", "tc_stages", "tc_threads")]


class MlpWsArgs(C.Structure):
    """saceo_mlp_ws_args (include/saceo.h): one pass of the MLP dispatch, for saceo_test_mlp_ws."""
    _fields_ = [(n, C.c_int32) for n in ("n_agents", "nnet", "hnets", "in_", "nout", "kout")] + \
               [("hidden", C.c_int32 * 2), ("act", C.c_int32 * 2), ("rows", C.c_int32), ("rowsAllocH", C.c_int64),
                ("theta", C.c_void_p), ("sTa", C.c_int64), ("sTn", C.c_int64),
                ("X", C.c_void_p), ("ldx", C.c_int32), ("sXa", C.c_int64), ("sXn", C.c_int64),
                ("out", C.c_void_p), ("ldo", C.c_int32), ("sOa", C.c_int64), ("sOn", C.c_int64),
                ("dout", C.c_void_p), ("ldd", C.c_int32), ("sDa", C.c_int64), ("sDn", C.c_int64),
                ("H", C.c_void_p * 2), ("dH", C.c_void_p * 2)] + \
               [(n, C.c_void_p) for n in ("planes", "H1p", "dH2p", "dH1p")] + \
               [("sQa", C.c_int64), ("sQn", C.c_int64), ("dbpart", C.c_void_p), ("dbpart_cap", C.c_int64),
                ("grads", C.c_void_p), ("dXa", C.c_void_p), ("A_cols", C.c_int32), ("sXaA", C.c_int64),
                ("sXaN", C.c_int64), ("save_h", C.c_int32)]


class MlpWsRoute(C.Structure):
    """saceo_mlp_ws_route (include/saceo.h): which kernels a saceo_test_mlp_ws call launched."""
    _fields_ = [(n, C.c_int32) for n in ("plane_path", "n_fwd_ws", "n_bwd_ws", "n_dw_planes", "n_dw0_planes",
                                         "n_bias_finish", "n_tc", "n_skinny", "n_simt", "bwd_ng", "bwd_na", "bwd_mode")]


FIT_HYPER = 8
FIT_HYPER_NAMES = ("model_lr", "reward_loss_coef", "delta_clip_loss", "reward_clip_loss", "model_max_grad_norm",
                   "r_mean", "r_std", "scale_model_loss")

_lib: Optional[C.CDLL] = None

# every symbol include/saceo.h declares (tests/test_abi.py checks the library exports them all)
EXPORTS = [
    "saceo_query_layout", "saceo_create", "saceo_destroy", "saceo_bind", "saceo_weights_changed", "saceo_replay_append", "saceo_gather",
    "saceo_set_draws", "saceo_update", "saceo_update_host", "saceo_update_host_async", "saceo_update_phase", "saceo_bc_update", "saceo_profile_step",
    "saceo_actor_forward", "saceo_critic_forward", "saceo_model_eval", "saceo_fvp", "saceo_cg_solve",
    "saceo_fit_bind", "saceo_model_fit", "saceo_trpo_grad", "saceo_trpo_eval", "saceo_actor_step", "saceo_ppo_grad", "saceo_actor_adam", "saceo_onpolicy_expert_grad", "saceo_grad_blend",
    "saceo_policy_layout", "saceo_policy_act",
    "saceo_debug_ptr", "saceo_launch_count", "saceo_test_gemm", "saceo_test_gemm_ex", "saceo_test_mlp_ws", "saceo_last_error", "saceo_abi_version",
]


def load() -> C.CDLL:
    """Loads libsaceo.so (built in-tree by ``__graft_entry__.build()``); raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SaceoError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
            "sac_expert_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, u64, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64, C.c_float
    sig = {
        "saceo_query_layout": (C.c_int, [C.POINTER(Config), C.POINTER(Layout)]),
        "saceo_create": (C.c_int, [C.POINTER(Config), C.POINTER(vp)]),
        "saceo_destroy": (C.c_int, [vp]),
        "saceo_bind": (C.c_int, [vp, C.POINTER(Tables)]),
        "saceo_weights_changed": (C.c_int, [vp]),
        "saceo_replay_append": (C.c_int, [vp, vp, i32, vp]),
        "saceo_gather": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, vp]),
        "saceo_set_draws": (C.c_int, [vp, vp, vp, vp, vp]),
        "saceo_update": (C.c_int, [vp, i32, i64, i32, u64, vp, vp]),
        "saceo_update_host": (C.c_int, [vp, i64, u64, vp, vp, vp, vp]),
        "saceo_update_host_async": (C.c_int, [vp, i64, u64, vp, vp, vp, vp]),
        "saceo_update_phase": (C.c_int, [vp, i32, i64, vp]),
        "saceo_bc_update": (C.c_int, [vp, i32, i32, u64, vp, vp]),
        "saceo_profile_step": (C.c_int, [vp, i64, i32, u64, C.c_char_p, vp, i32, C.POINTER(i32), vp]),
        "saceo_actor_forward": (C.c_int, [vp, vp, i32, vp, vp, vp, vp]),
        "saceo_critic_forward": (C.c_int, [vp, i32, vp, vp, i32, i32, vp, vp]),
        "saceo_model_eval": (C.c_int, [vp, vp, vp, i32, vp, vp]),
        "saceo_fit_bind": (C.c_int, [vp, C.POINTER(FitTables), i32, i32]),
        "saceo_model_fit": (C.c_int, [vp, i32, vp, vp, vp]),
        "saceo_fvp": (C.c_int, [vp, vp, f32, vp, vp]),
        "saceo_cg_solve": (C.c_int, [vp, vp, i32, f32, f32, vp, vp, vp]),
        "saceo_trpo_grad": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, vp]),
        "saceo_trpo_eval": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, vp, vp]),
        "saceo_actor_step": (C.c_int, [vp, vp, vp, vp, vp]),
        "saceo_ppo_grad": (C.c_int, [vp, vp, vp, vp, vp, f32, f32, vp, vp, vp]),
        "saceo_actor_adam": (C.c_int, [vp, vp, vp]),
        "saceo_onpolicy_expert_grad": (C.c_int, [vp, C.c_int32, C.c_int32, vp, vp, vp]),
        "saceo_grad_blend": (C.c_int, [vp, vp, vp, vp, f32, vp, vp, vp]),
        "saceo_policy_layout": (C.c_int, [C.POINTER(PolicyConfig), C.POINTER(i64), C.POINTER(i64), C.POINTER(i32)]),
        "saceo_policy_act": (C.c_int, [C.POINTER(PolicyConfig), vp, vp, vp, i32, vp, vp, vp]),
        "saceo_debug_ptr": (vp, [vp, C.c_char_p, C.POINTER(i64)]),
        "saceo_launch_count": (i64, [vp]),
        "saceo_test_gemm": (C.c_int, [i32, i32, i32, i32, i32, i32, i32, vp, vp, vp, vp]),
        "saceo_test_gemm_ex": (C.c_int, [C.POINTER(GemmArgs), C.POINTER(GemmRoute), vp]),
        "saceo_test_mlp_ws": (C.c_int, [C.POINTER(MlpWsArgs), C.POINTER(MlpWsRoute), vp]),
        "saceo_last_error": (C.c_char_p, []),
        "saceo_abi_version": (C.c_int, []),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.saceo_abi_version() != ABI_VERSION:
        raise SaceoError("libsaceo ABI version mismatch")
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().saceo_last_error()
        raise SaceoError(f"libsaceo error {rc}: {msg.decode() if msg else '?'}")


def query_layout(cfg: Config) -> Layout:
    lay = Layout()
    check(load().saceo_query_layout(C.byref(cfg), C.byref(lay)))
    return lay
