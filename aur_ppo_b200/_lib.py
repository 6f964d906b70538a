"""ctypes binding of libaurppo.so (the C ABI declared in include/aur_ppo.h).

There is no fallback: if the library is missing or a call fails, an exception is
raised.  Build it with `python -c "import __graft_entry__ as g; g.build()"` or
`make -C aur_ppo_b200/csrc`.
"""
from __future__ import annotations

import ctypes
import os
import re
import subprocess
from ctypes import c_double, c_int, c_int32, c_int64, c_uint64, c_void_p, c_char_p

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("AUR_LIB_PATH", os.path.join(_PKG, "libaurppo.so"))
HEADER_PATH = os.path.join(os.path.dirname(_PKG), "include", "aur_ppo.h")

_lib = None
ABI_VERSION = 3          # AUR_ABI_VERSION of include/aur_ppo.h


class PolicyDesc(ctypes.Structure):
    _fields_ = [("obs_dim", c_int32), ("act_dim", c_int32), ("hidden_dim", c_int32), ("num_layers", c_int32),
                ("continuous", c_int32)]


class EnvState(ctypes.Structure):
    _fields_ = [("phys", c_void_p), ("pcg", c_void_p), ("elapsed", c_void_p), ("ep_return", c_void_p),
                ("ep_length", c_void_p), ("norm", c_void_p)]


class EpisodeLog(ctypes.Structure):
    _fields_ = [("entries", c_void_p), ("count", c_void_p), ("capacity", ctypes.c_uint32), ("_pad", ctypes.c_uint32),
                ("first_finished", c_void_p), ("totals", c_void_p)]


class RolloutArgs(ctypes.Structure):
    _fields_ = [("env_kind", c_int32), ("wrappers", c_int32), ("N", c_int64), ("T", c_int32), ("_pad", c_int32),
                ("policy", PolicyDesc), ("params", c_void_p), ("env", EnvState),
                ("obs_buf", c_void_p), ("act_buf", c_void_p), ("logp_buf", c_void_p), ("val_buf", c_void_p),
                ("rew_buf", c_void_p), ("done_buf", c_void_p), ("next_obs", c_void_p), ("next_done", c_void_p),
                ("next_value", c_void_p), ("actions_in", c_void_p), ("seed", c_uint64), ("step0", c_uint64),
                ("env_id0", c_uint64), ("log", EpisodeLog), ("gamma", c_double)]


class UpdateArgs(ctypes.Structure):
    _fields_ = [("policy", PolicyDesc), ("norm_adv", c_int32), ("clip_vloss", c_int32), ("mom_index", c_int32),
                ("m_local", c_int64), ("m_total", c_int64), ("idx", c_void_p), ("idx_offset", c_int64),
                ("obs", c_void_p), ("actions", c_void_p), ("logprobs", c_void_p), ("advantages", c_void_p),
                ("returns", c_void_p), ("values", c_void_p), ("params", c_void_p),
                ("clip_coeff", ctypes.c_float), ("entropy_coeff", ctypes.c_float), ("value_coeff", ctypes.c_float),
                ("_pad2", ctypes.c_float), ("adv_moments", c_void_p), ("workspace", c_void_p), ("grads_out", c_void_p),
                ("dp", c_void_p), ("dp_seq", ctypes.c_uint32), ("mom_seq", ctypes.c_uint32),
                ("rec_actor", c_void_p), ("rec_critic", c_void_p)]


class PopDesc(ctypes.Structure):
    _fields_ = [("K", c_int32), ("_pad", c_int32), ("n_member", c_int64), ("seeds", c_void_p)]


class PopHparams(ctypes.Structure):
    _fields_ = [("learning_rate", c_double), ("entropy_coeff", c_double), ("clip_coeff", c_double), ("value_coeff", c_double),
                ("max_grad_norm", c_double), ("target_kl", c_double)]


class PopUpdateArgs(ctypes.Structure):
    _fields_ = [("policy", PolicyDesc), ("norm_adv", c_int32), ("clip_vloss", c_int32), ("mb_index", c_int32), ("n_mb", c_int32),
                ("m", c_int64), ("idx", c_void_p), ("rec_actor", c_void_p), ("rec_critic", c_void_p), ("params", c_void_p),
                ("hparams", c_void_p), ("adv_moments", c_void_p), ("active", c_void_p), ("workspace", c_void_p),
                ("grads_out", c_void_p)]


class PopPbtArgs(ctypes.Structure):
    _fields_ = [("fitness", c_void_p), ("q", c_double), ("down", c_double), ("up", c_double), ("mask", ctypes.c_uint32),
                ("_pad", ctypes.c_uint32), ("seed", c_uint64), ("round", c_uint64), ("params", c_void_p), ("adam_m", c_void_p),
                ("adam_v", c_void_p), ("steps", c_void_p), ("hparams", c_void_p), ("norm", c_void_p), ("norm_ld", c_int64),
                ("rank_out", c_void_p), ("donor_out", c_void_p), ("order", c_void_p)]


DP_MAX_RANKS = 16
DP_HANDLE_BYTES = 64


class DpCtx(ctypes.Structure):
    _fields_ = [("world", c_int32), ("rank", c_int32), ("peer", c_void_p * DP_MAX_RANKS)]


class ConvArgs(ctypes.Structure):
    _fields_ = [("B", c_int32), ("Hb", c_int32), ("Wb", c_int32), ("Cin", c_int32), ("Cout", c_int32),
                ("epilogue", c_int32), ("out_Hb", c_int32), ("out_Wb", c_int32), ("out_off", c_int32), ("_pad", c_int32),
                ("inp", c_void_p), ("wmat", c_void_p), ("bias", c_void_p), ("out", c_void_p), ("pool_arg", c_void_p),
                ("relu_ref", c_void_p), ("ref_Hb", c_int32), ("ref_Wb", c_int32), ("ref_off", c_int32), ("_pad2", c_int32)]


class EquivHeadArgs(ctypes.Structure):
    _fields_ = [("B", c_int32), ("clip_vloss", c_int32), ("m_total", c_int64), ("a_out", c_void_p), ("a_bias", c_void_p),
                ("c_pre", c_void_p), ("c_bias1", c_void_p), ("c_w2", c_void_p), ("c_b2", c_void_p), ("action", c_void_p),
                ("oldlp", c_void_p), ("adv", c_void_p), ("ret", c_void_p), ("vold", c_void_p), ("adv_moments", c_void_p),
                ("clip_coeff", ctypes.c_float), ("entropy_coeff", ctypes.c_float), ("value_coeff", ctypes.c_float),
                ("_pad", ctypes.c_float), ("d_a_out", c_void_p), ("d_c_h", c_void_p), ("d_head", c_void_p),
                ("stats", c_void_p), ("value_out", c_void_p), ("logp_out", c_void_p)]


class PlainHeadArgs(ctypes.Structure):
    _fields_ = [("B", c_int32), ("clip_vloss", c_int32), ("m_total", c_int64), ("a_out", c_void_p), ("a_bias", c_void_p),
                ("actor_logstd", c_void_p), ("c_pre", c_void_p), ("c_bias1", c_void_p), ("c_w2", c_void_p), ("c_b2", c_void_p),
                ("action", c_void_p), ("oldlp", c_void_p), ("adv", c_void_p), ("ret", c_void_p), ("vold", c_void_p),
                ("adv_moments", c_void_p), ("clip_coeff", ctypes.c_float), ("entropy_coeff", ctypes.c_float),
                ("value_coeff", ctypes.c_float), ("_pad", ctypes.c_float), ("d_a_out", c_void_p), ("d_c_h", c_void_p),
                ("d_head", c_void_p), ("stats", c_void_p), ("value_out", c_void_p), ("logp_out", c_void_p)]


class AurError(RuntimeError):
    pass


def build(verbose: bool = False) -> str:
    """Compile csrc/*.cu for sm_100a into aur_ppo_b200/libaurppo.so (nvcc cross-compiles without a GPU)."""
    jobs = str(max(1, min(os.cpu_count() or 1, 8)))          # ~3.5 min serial, ~1 min on 8 cores
    r = subprocess.run(["make", "-j", jobs, "-C", os.path.join(_PKG, "csrc")], capture_output=True, text=True)
    if verbose or r.returncode != 0:
        print(r.stdout[-4000:])
        print(r.stderr[-4000:])
    if r.returncode != 0:
        raise AurError("building libaurppo.so failed")
    return LIB_PATH


def declared_symbols() -> list:
    """Every function include/aur_ppo.h declares (used by the export test)."""
    src = open(HEADER_PATH).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(aur_[a-z0-9_]+)\s*\(", src)))


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise AurError(f"{LIB_PATH} is missing: the CUDA extension has not been built and there is no CPU "
                       "fallback (run __graft_entry__.build())")
    L = ctypes.CDLL(LIB_PATH)
    L.aur_abi_version.restype = c_int
    if L.aur_abi_version() != ABI_VERSION:
        raise AurError(f"{LIB_PATH} has ABI version {L.aur_abi_version()}, this package binds version {ABI_VERSION}: rebuild it "
                       "(run __graft_entry__.build())")
    L.aur_last_error.restype = c_char_p
    L.aur_launch_count.restype = c_int64
    L.aur_launch_count_reset.restype = None
    L.aur_gae_f32.restype = c_int
    L.aur_gae_f32.argtypes = [c_int32, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_double, c_double,
                              c_int32, c_void_p, c_void_p, c_void_p]
    L.aur_gae_kernel_kind.restype = c_int
    L.aur_gae_kernel_kind.argtypes = [c_int32, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]
    L.aur_policy_param_count.restype = c_int64
    L.aur_policy_param_count.argtypes = [ctypes.POINTER(PolicyDesc)]
    L.aur_policy_evaluate.restype = c_int
    L.aur_policy_evaluate.argtypes = [ctypes.POINTER(PolicyDesc), c_void_p, c_int64, c_void_p, c_void_p, c_uint64,
                                      c_uint64, c_uint64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]
    L.aur_tc_set_precision.restype = c_int
    L.aur_tc_set_precision.argtypes = [c_int]
    L.aur_tc_get_precision.restype = c_int
    L.aur_policy_act.restype = c_int
    L.aur_policy_act.argtypes = [ctypes.POINTER(PolicyDesc), c_void_p, c_int64, c_void_p, c_void_p, c_int32, c_uint64,
                                 c_uint64, c_uint64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]
    L.aur_env_reset.restype = c_int
    L.aur_env_reset.argtypes = [c_int32, c_int64, c_int32, ctypes.POINTER(EnvState), c_void_p, c_void_p, c_void_p]
    L.aur_rollout.restype = c_int
    L.aur_rollout.argtypes = [ctypes.POINTER(RolloutArgs), c_void_p]
    L.aur_squashed_gaussian_sample.restype = c_int
    L.aur_squashed_gaussian_sample.argtypes = [c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_uint64, c_uint64, c_void_p, c_void_p,
                                               c_void_p, c_void_p, c_void_p, c_void_p]
    L.aur_ppo_pack_records.restype = c_int
    L.aur_ppo_pack_records.argtypes = [c_int64, c_int32, c_int32] + [c_void_p] * 9
    L.aur_shuffle_indices.restype = c_int
    L.aur_shuffle_indices.argtypes = [c_int64, c_uint64, c_uint64, c_void_p, c_void_p]
    L.aur_ppo_update_workspace_bytes.restype = c_int64
    L.aur_ppo_update_workspace_bytes.argtypes = [ctypes.POINTER(PolicyDesc)]
    L.aur_ppo_adv_moments.restype = c_int
    L.aur_ppo_adv_moments.argtypes = [c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p]
    L.aur_ppo_update_grad.restype = c_int
    L.aur_ppo_update_grad.argtypes = [ctypes.POINTER(UpdateArgs), c_void_p]
    L.aur_dp_area_bytes.restype = c_int64
    L.aur_dp_area_bytes.argtypes = [ctypes.POINTER(PolicyDesc)]
    L.aur_dp_alloc.restype = c_int
    L.aur_dp_alloc.argtypes = [c_int64, ctypes.POINTER(c_void_p), c_void_p]
    L.aur_dp_open.restype = c_int
    L.aur_dp_open.argtypes = [c_void_p, ctypes.POINTER(c_void_p)]
    L.aur_dp_close.restype = c_int
    L.aur_dp_close.argtypes = [c_void_p]
    L.aur_dp_free.restype = c_int
    L.aur_dp_free.argtypes = [c_void_p]
    L.aur_dp_status.restype = c_int
    L.aur_dp_status.argtypes = [c_void_p, c_void_p]
    L.aur_dp_wait_stats.restype = c_int
    L.aur_dp_wait_stats.argtypes = [c_void_p, c_void_p, c_int32, c_void_p]
    L.aur_ppo_adv_moments_multi.restype = c_int
    L.aur_ppo_adv_moments_multi.argtypes = [c_int32, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p,
                                            ctypes.c_uint32, c_void_p]
    L.aur_ppo_adv_moments_dp.restype = c_int
    L.aur_ppo_adv_moments_dp.argtypes = [c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, ctypes.c_uint32,
                                         c_void_p]
    L.aur_ppo_update_apply_dp.restype = c_int
    L.aur_ppo_update_apply_dp.argtypes = [ctypes.POINTER(PolicyDesc), c_void_p, c_void_p, c_void_p, c_void_p, c_double,
                                          c_double, c_double, c_double, c_int64, c_double, c_int64, c_double, c_double,
                                          c_void_p, c_void_p, ctypes.c_uint32, c_void_p]
    L.aur_rollout_set_impl.restype = c_int
    L.aur_rollout_set_impl.argtypes = [c_int]
    L.aur_rollout_get_impl.restype = c_int
    L.aur_ppo_update_set_impl.restype = c_int
    L.aur_ppo_update_set_impl.argtypes = [c_int]
    L.aur_ppo_update_get_impl.restype = c_int
    L.aur_ppo_update_set_wide.restype = c_int
    L.aur_ppo_update_set_wide.argtypes = [c_int]
    L.aur_ppo_update_get_wide.restype = c_int
    L.aur_ppo_update_apply.restype = c_int
    L.aur_ppo_update_apply.argtypes = [ctypes.POINTER(PolicyDesc), c_void_p, c_void_p, c_void_p, c_void_p, c_double,
                                       c_double, c_double, c_double, c_int64, c_double, c_int64, c_double, c_double,
                                       c_void_p, c_void_p]
    L.aur_tc_gemm_bf16.restype = c_int
    L.aur_tc_gemm_bf16.argtypes = [c_int64, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p]
    L.aur_conv3x3_bf16.restype = c_int
    L.aur_conv3x3_bf16.argtypes = [ctypes.POINTER(ConvArgs), c_void_p]
    L.aur_equiv_expand_regular.restype = c_int
    L.aur_equiv_expand_regular.argtypes = [c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]
    L.aur_equiv_conv0.restype = c_int
    L.aur_equiv_conv0.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_void_p, c_void_p, c_void_p]
    L.aur_wgrad3x3_bf16.restype = c_int
    L.aur_wgrad3x3_bf16.argtypes = [c_int32, c_int32, c_int64, c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_int32, c_void_p]
    L.aur_unpool_relu_bwd_colsum.restype = c_int
    L.aur_unpool_relu_bwd_colsum.argtypes = [c_int32] * 4 + [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p,
                                             c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p]
    L.aur_unpool_relu_bwd.restype = c_int
    L.aur_unpool_relu_bwd.argtypes = [c_int32] * 4 + [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p,
                                                      c_int32, c_int32, c_int32, c_void_p]
    L.aur_transpose_bf16.restype = c_int
    L.aur_transpose_bf16.argtypes = [c_int64, c_int32, c_void_p, c_void_p, c_void_p]
    L.aur_equiv_project_regular.restype = c_int
    L.aur_equiv_project_regular.argtypes = [c_void_p, c_int32, c_int32, c_void_p, c_void_p]
    L.aur_colsum_bf16.restype = c_int
    L.aur_colsum_bf16.argtypes = [c_int64, c_int32, c_void_p, c_int32, c_void_p, c_void_p]
    L.aur_equiv_conv0_wgrad.restype = c_int
    L.aur_equiv_conv0_wgrad.argtypes = [c_void_p] * 5 + [c_int32, c_void_p, c_void_p, c_void_p, c_void_p]
    L.aur_bias_relu_bf16.restype = c_int
    L.aur_bias_relu_bf16.argtypes = [c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p]
    L.aur_relu_mask_bf16.restype = c_int
    L.aur_relu_mask_bf16.argtypes = [c_int64, c_void_p, c_void_p, c_void_p, c_void_p]
    L.aur_equiv_head_loss.restype = c_int
    L.aur_equiv_head_loss.argtypes = [ctypes.POINTER(EquivHeadArgs), c_void_p]
    L.aur_equiv_head_eval.restype = c_int
    L.aur_equiv_head_eval.argtypes = [c_int32] + [c_void_p] * 7 + [c_uint64, c_uint64, ctypes.POINTER(ctypes.c_float)] + \
        [c_void_p] * 8
    L.aur_plain_conv0.restype = c_int
    L.aur_plain_conv0.argtypes = [c_void_p] * 4 + [c_int32, c_void_p, c_void_p, c_void_p]
    L.aur_plain_conv0_wgrad.restype = c_int
    L.aur_plain_conv0_wgrad.argtypes = [c_void_p] * 5 + [c_int32, c_void_p, c_void_p, c_void_p, c_void_p]
    L.aur_plain_head_eval.restype = c_int
    L.aur_plain_head_eval.argtypes = [c_int32] + [c_void_p] * 8 + [c_uint64, c_uint64, ctypes.POINTER(ctypes.c_float)] + \
        [c_void_p] * 8
    L.aur_plain_head_loss.restype = c_int
    L.aur_plain_head_loss.argtypes = [ctypes.POINTER(PlainHeadArgs), c_void_p]
    L.aur_sumsq_f32.restype = c_int
    L.aur_sumsq_f32.argtypes = [c_int64, c_void_p, c_void_p, c_void_p]
    L.aur_adam_flat.restype = c_int
    L.aur_adam_flat.argtypes = [c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_double, c_double, c_double, c_double,
                                c_int64, c_void_p, c_double, c_void_p]
    L.aur_pop_rollout.restype = c_int
    L.aur_pop_rollout.argtypes = [ctypes.POINTER(PopDesc), ctypes.POINTER(RolloutArgs), c_void_p]
    L.aur_pop_shuffle_indices.restype = c_int
    L.aur_pop_shuffle_indices.argtypes = [ctypes.POINTER(PopDesc), c_int32, c_int32, c_uint64, c_void_p, c_void_p]
    L.aur_pop_adv_moments_multi.restype = c_int
    L.aur_pop_adv_moments_multi.argtypes = [ctypes.POINTER(PopDesc), c_int32, c_int64, c_void_p, c_void_p, c_void_p, c_void_p,
                                            c_void_p]
    L.aur_pop_update_workspace_bytes.restype = c_int64
    L.aur_pop_update_workspace_bytes.argtypes = [ctypes.POINTER(PopDesc), ctypes.POINTER(PolicyDesc), c_int32, c_int64]
    L.aur_pop_update_grad.restype = c_int
    L.aur_pop_update_grad.argtypes = [ctypes.POINTER(PopDesc), ctypes.POINTER(PopUpdateArgs), c_void_p]
    L.aur_pop_update_apply.restype = c_int
    L.aur_pop_update_apply.argtypes = [ctypes.POINTER(PopDesc), ctypes.POINTER(PolicyDesc), c_void_p, c_void_p, c_void_p, c_void_p,
                                       c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_double, c_double, c_double, c_double,
                                       c_int64, c_void_p, c_int32, c_int32, c_int32, c_void_p]
    L.aur_pop_episode_fitness.restype = c_int
    L.aur_pop_episode_fitness.argtypes = [ctypes.POINTER(PopDesc), c_void_p, c_void_p, c_void_p, c_void_p]
    L.aur_pop_pbt_step.restype = c_int
    L.aur_pop_pbt_step.argtypes = [ctypes.POINTER(PopDesc), ctypes.POINTER(PolicyDesc), ctypes.POINTER(PopPbtArgs), c_void_p]
    L.aur_sincos_f64.restype = c_int
    L.aur_sincos_f64.argtypes = [c_int64, c_void_p, c_void_p, c_void_p, c_void_p]
    _lib = L
    return L


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().aur_last_error().decode(errors="replace")
        raise AurError(f"{what} failed (rc={rc}): {msg}")
