"""ctypes binding of libppx.so (the C ABI declared in include/ppx.h).

There is NO fallback: if the shared library is missing or a symbol is absent, importing the
compute path raises.  Build it with ``python -c "import __graft_entry__ as g; g.build()"`` or
``make -C ppo-exploration_b200/csrc``.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libppx.so")

c_p = C.c_void_p
c_i = C.c_int
c_l = C.c_int64
c_u = C.c_uint64
c_d = C.c_double


class PpoCfg(C.Structure):
    _fields_ = [("B", c_l), ("B_total", c_l), ("A", c_i), ("discrete", c_i), ("dual", c_i), ("clip_range", C.c_float),
                ("ent_coef", C.c_float), ("vf_coef", C.c_float), ("int_vf_coef", C.c_float),
                ("policy_weight", C.c_float), ("row_dev", c_p), ("row_hold", c_i), ("W", c_i), ("rank", c_i),
                ("peer_sums_host", c_p), ("seq_dev", c_p), ("status_dev", c_p)]


class GatherOpts(C.Structure):
    """ppx_gather_opts: sharded source decode, statistics range, device step cursor."""
    _fields_ = [("n_shard", c_i), ("stat_lo", c_l), ("stat_n", c_l), ("row_dev", c_p), ("n_mb", c_l), ("epoch_stride", c_l),
                ("mb_stride", c_l), ("W", c_i), ("rank", c_i), ("peer_moments_host", c_p), ("seq_dev", c_p), ("status_dev", c_p)]


class FusedAdam(C.Structure):
    """ppx_fused_adam: the optimiser tail of the fused MLP backward (clip_grad_norm_ + Adam in the reduce kernel's last block)."""
    _fields_ = [("params", c_p), ("grads", c_p), ("exp_avg", c_p), ("exp_avg_sq", c_p), ("n", c_l), ("max_norm", c_d), ("lr", c_d),
                ("beta1", c_d), ("beta2", c_d), ("eps", c_d), ("step_dev", c_p), ("norm_out", c_p), ("extra_grads", c_p),
                ("n_extra", c_i), ("ticket", c_p), ("W", c_i), ("rank", c_i), ("peer_xg_host", c_p),
                ("seq_dev", c_p), ("status_dev", c_p)]


class ValueHead(C.Structure):
    _fields_ = [("values", c_p), ("old_values", c_p), ("returns", c_p), ("branch", c_p), ("scale", C.c_float)]


# name -> (restype, argtypes).  Functions returning int are status codes checked by `call`.
SIGNATURES = {
    "ppx_last_error": (C.c_char_p, []),
    "ppx_version": (c_i, []),
    "ppx_launch_count": (c_u, []),
    "ppx_device_info": (c_i, [c_p, c_p, c_p]),
    "ppx_gae": (c_i, [c_p, c_p, c_p, c_p, c_p, c_d, c_d, c_i, c_i, c_p, c_p, c_p]),
    "ppx_gae_dual": (c_i, [c_p, c_p, c_p, c_p, c_p, c_d, c_d, c_p, c_p, c_p, c_d, c_i, c_i, c_p, c_p, c_p, c_p, c_p]),
    "ppx_discount": (c_i, [c_p, c_p, c_d, c_i, c_i, c_p, c_p]),
    "ppx_simhash_codes": (c_i, [c_p, c_p, c_i, c_i, c_l, c_p, c_p]),
    "ppx_count_table_create": (c_i, [c_u, C.POINTER(c_p)]),
    "ppx_count_table_destroy": (c_i, [c_p]),
    "ppx_count_table_clear": (c_i, [c_p, c_p]),
    "ppx_count_table_update": (c_i, [c_p, c_p, c_l, c_p, c_p]),
    "ppx_count_table_update_owned": (c_i, [c_p, c_p, c_l, c_p, c_i, c_i, c_p]),
    "ppx_simhash_update": (c_i, [c_p, c_p, c_p, c_i, c_i, c_l, c_d, c_p, c_i, c_p, c_p, c_p]),
    "ppx_simhash_bonus": (c_i, [c_p, c_l, c_d, c_p, c_i, c_p]),
    "ppx_count_table_size": (c_i, [c_p, C.POINTER(c_u)]),
    "ppx_count_table_dump": (c_i, [c_p, c_p, c_p, c_u, C.POINTER(c_u)]),
    "ppx_count_table_load": (c_i, [c_p, c_p, c_p, c_u, c_p]),
    "ppx_count_table_capacity": (c_i, [c_p, C.POINTER(c_u)]),
    "ppx_gather_minibatch": (c_i, [C.POINTER(c_p), C.POINTER(c_p), C.POINTER(c_i), c_i, c_p, c_l, c_i, c_i, c_p]),
    "ppx_gather_minibatch_stats": (c_i, [C.POINTER(c_p), C.POINTER(c_p), C.POINTER(c_i), c_i, c_p, c_l, c_i, c_i, C.POINTER(c_i),
                                         C.POINTER(c_p), c_i, c_p, c_p]),
    "ppx_loss_row_commit": (c_i, [c_p, c_p, c_p, c_i, c_i, c_p]),
    "ppx_mean_std": (c_i, [c_p, c_l, c_p, c_p]),
    "ppx_np_permutation": (c_i, [c_p, C.POINTER(c_i), c_l, c_p]),
    "ppx_np_shuffle_draws32": (c_i, [c_p, C.POINTER(c_i), c_l, c_p]),
    "ppx_np_shuffle_draws32_stream": (c_i, [c_p, C.POINTER(c_i), c_l, c_p]),
    "ppx_np_shuffle_apply_device_workspace": (c_l, [c_l]),
    "ppx_np_shuffle_apply_device": (c_i, [c_p, c_l, c_i, c_p, c_p, c_p]),
    "ppx_np_shuffle_stage": (c_i, [c_p, c_l, c_p, c_p, c_p, c_p, c_p, c_p]),
    "ppx_linear_fwd": (c_i, [c_p, c_i, c_p, c_p, c_i, c_i, c_i, c_i, c_p, c_i, c_i, c_l, c_l, c_l, c_l, c_p]),
    "ppx_linear_bwd_data": (c_i, [c_p, c_i, c_p, c_i, c_i, c_i, c_p, c_i, c_i, c_p, c_i, c_i, c_l, c_l, c_l, c_l, c_p]),
    "ppx_linear_bwd_weight_workspace": (c_l, [c_i, c_i, c_i, c_i]),
    "ppx_linear_bwd_weight": (c_i, [c_p, c_i, c_p, c_i, c_i, c_i, c_i, c_p, c_p, c_p, c_i, c_l, c_l, c_l, c_l, c_p]),
    "ppx_p2p_max_params": (c_l, []),
    "ppx_p2p_moments_merge": (c_i, [c_p, c_p, c_i, c_i, c_p, c_p, c_i, c_p, c_p]),
    "ppx_p2p_sums_allreduce": (c_i, [c_p, c_p, c_i, c_i, c_p, c_p, c_p, c_p]),
    "ppx_p2p_clip_adam": (c_i, [c_p, c_p, c_p, c_i, c_i, c_p, c_p, c_p, c_p, c_l, c_d, c_l, c_d, c_d, c_d, c_d, c_p, c_p, c_p, c_p]),
    "ppx_mlp3_fused_adam_blocks": (c_i, [c_i, c_i, c_i, c_p]),
    "ppx_mlp3_tc_bwd_probe": (c_i, [c_p]),
    "ppx_mlp3_supported": (c_i, [c_i, c_i, c_i, c_p]),
    "ppx_mlp3_fwd": (c_i, [c_p, c_i, c_i, c_i, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p]),
    "ppx_mlp3_bwd_workspace": (c_l, [c_i, c_i, c_i, c_i, c_p]),
    "ppx_mlp3_bwd": (c_i, [c_p, c_i, c_i, c_i, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_p, C.c_float, c_l, c_p, c_p, c_p, c_p, c_p, c_p, c_p,
                           c_p, c_p, c_p, c_p]),
    "ppx_mlp3_sumsq_partials": (c_i, [c_i, c_i, c_i, c_p]),
    "ppx_mlp3_tc_supported": (c_i, [c_i, c_i, c_i, c_p]),
    "ppx_mlp3_tc_act_elems": (c_l, [c_i, c_i, c_i]),
    "ppx_mlp3_tc_fwd": (c_i, [c_p, c_i, c_i, c_i, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p]),
    "ppx_mlp3_tc_bwd_workspace": (c_l, [c_i, c_i, c_i, c_i, c_p]),
    "ppx_mlp3_tc_bwd": (c_i, [c_p, c_i, c_i, c_i, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_p, C.c_float, c_l, c_p, c_p, c_p, c_p, c_p, c_p, c_p,
                              c_p, c_p, c_p, c_p]),
    "ppx_clip_adam_pre": (c_i, [c_p, c_p, c_p, c_p, c_l, c_d, c_d, c_d, c_d, c_d, c_p, c_p, c_p, c_i, c_p, c_i, c_p]),
    "ppx_tc_supported": (c_i, [c_i, c_i, c_i, c_i, c_i, c_p, c_p]),
    "ppx_tc_split": (c_i, [c_p, c_i, c_i, c_p, c_p, c_p, c_p, c_p]),
    "ppx_tc_linear": (c_i, [c_p, c_i, c_p, c_p, c_i, c_i, c_i, c_i, c_p, c_p, c_i, c_i, c_i, c_p, c_p, C.c_float, c_p, c_i, c_p]),
    "ppx_tc_linear_ws": (c_i, [c_p, c_i, c_p, c_p, c_i, c_i, c_i, c_i, c_p, c_p, c_i, c_i, c_i, c_p, c_p, C.c_float, c_p, c_i, c_p, c_l, c_p]),
    "ppx_tc_linear_workspace": (c_l, [c_i, c_i, c_i]),
    "ppx_im2col": (c_i, [c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_i, c_i, c_p, c_p]),
    "ppx_col2im": (c_i, [c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_i, c_i, c_p, c_p]),
    "ppx_act_bwd_mul": (c_i, [c_p, c_p, c_l, c_i, c_p, c_p]),
    "ppx_obs_istd": (c_i, [c_p, c_i, c_p, c_p]),
    "ppx_tc_wgrad_workspace": (c_l, [c_i, c_i, c_i]),
    "ppx_tc_wgrad_supported": (c_i, [c_i, c_i, c_i, c_p, c_p]),
    "ppx_tc_wgrad": (c_i, [c_p, c_i, c_p, c_i, c_i, c_i, c_i, c_p, c_p, c_p, c_p]),
    "ppx_ppo_loss_workspace": (c_l, [c_l, c_i]),
    "ppx_ppo_loss_fwd_bwd": (c_i, [C.POINTER(PpoCfg)] + [c_p] * 21),
    "ppx_ppo_loss_head_final": (c_i, [C.POINTER(PpoCfg)] + [c_p] * 20),
    "ppx_ppo_loss_finalize": (c_i, [C.POINTER(PpoCfg), c_p, c_p, c_p, c_p, c_p, c_p]),
    "ppx_moments_pack": (c_i, [c_p, c_l, c_p, c_p]),
    "ppx_moments_merge": (c_i, [c_p, c_i, c_p, c_p]),
    "ppx_ppo_loss_head": (c_i, [C.POINTER(PpoCfg)] + [c_p] * 18),
    "ppx_ppo_loss_finish": (c_i, [C.POINTER(PpoCfg)] + [c_p] * 14),
    "ppx_mse_fwd_bwd": (c_i, [c_p, c_p, c_l, c_d, c_p, c_p, c_p, c_p]),
    "ppx_xent_fwd_bwd": (c_i, [c_p, c_p, c_i, c_l, c_i, c_d, c_p, c_p, c_p]),
    "ppx_clip_adam": (c_i, [c_p, c_p, c_p, c_p, c_l, c_d, c_l, c_d, c_d, c_d, c_d, c_l, c_p, c_p, c_p, c_p]),
    "ppx_rms_update": (c_i, [c_p, c_i, c_l, c_i, c_p, c_p, c_p, c_p, c_p]),
    "ppx_normalize_obs": (c_i, [c_p, c_l, c_i, c_p, c_p, c_p, c_p]),
    "ppx_rnd_sqerr": (c_i, [c_p, c_p, c_l, c_p, c_p]),
    "ppx_rnd_normalize_rollout": (c_i, [c_p, c_i, c_i, c_p, c_p, c_p, c_p]),
    "ppx_icm_bonus_tail": (c_i, [c_p, c_p, c_l, c_i, c_d, c_p, c_p, c_p]),
    "ppx_embedding_fwd": (c_i, [c_p, c_i, c_p, c_i, c_i, c_l, c_p, c_i, c_p]),
    "ppx_embedding_bwd": (c_i, [c_p, c_i, c_p, c_i, c_i, c_l, c_i, c_p, c_p]),
    "ppx_vecnorm_obs": (c_i, [c_p, c_l, c_i, c_p, c_p, c_d, c_d, c_p, c_p]),
    "ppx_vecnorm_reward": (c_i, [c_p, c_p, c_p, c_i, c_d, c_p, c_p, c_p, c_d, c_d, c_i, c_p, c_p]),
    "ppx_policy_sample": (c_i, [c_p, c_p, c_l, c_i, c_i, c_u, c_u, c_p, c_p, c_p]),
    "ppx_policy_act_record": (c_i, [c_p, c_p, c_p, c_p, c_p, c_l, c_i, c_i, c_i, c_u, c_u, c_p, c_p, c_p, c_p, c_p, c_p, c_p]),
    "ppx_rollout_record_step": (c_i, [c_p, c_i, c_p, c_p, c_l, c_p, c_p, c_p, c_p, c_p, c_p]),
    "ppx_policy_act_eval": (c_i, [c_p, c_p, c_l, c_i, c_i, c_i, c_u, c_u, c_l, c_p, c_p]),
    "ppx_eval_episode_step": (c_i, [c_p, c_p, c_p, c_l, c_l, c_l, c_l, c_l, c_p, c_p, c_p, c_p, c_l, c_p, c_p]),
    "ppx_classic_step": (c_i, [c_i, c_l, c_l, c_u, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_p, c_p, c_p]),
    "ppx_classic_reset": (c_i, [c_i, c_l, c_l, c_u, c_p, c_p, c_p, c_p, c_p, c_p, c_p]),
    "ppx_episode_monitor_step": (c_i, [c_p, c_i, c_p, c_l, c_p, c_p, c_p, c_p, c_p]),
    "ppx_episode_log_record": (c_i, [c_p, c_p, c_p, c_l, c_p, c_p, c_p]),
    "ppx_episode_log_tail": (c_i, [c_p, c_p, c_p, c_l, c_l, c_p, c_p, c_p, c_p]),
    "ppx_noise_fill":(c_i, [c_p, c_l, c_u, c_p]),
    "ppx_es_perturb": (c_i, [c_p, c_p, c_p, c_d, c_i, c_i, c_p, c_i, c_p]),
    "ppx_es_forward": (c_i, [c_p, c_p, c_p, c_d, c_i, c_p, c_i, c_p, c_i, c_p, c_p]),
    "ppx_es_act": (c_i, [c_p, c_p, c_p, c_d, c_i, c_p, c_i, c_p, c_p, c_i, c_u, c_p, c_l, c_l, c_p, c_p, c_p]),
    "ppx_es_act_rows": (c_i, [c_p, c_p, c_i, c_p, c_i, c_p, c_p, c_i, c_u, c_p, c_l, c_p, c_p]),
    "ppx_es_episode_step": (c_i, [c_p, c_i, c_p, c_p, c_i, c_l, c_i, c_p, c_p, c_p, c_p, c_p, c_p]),
    "ppx_es_update_workspace": (c_l, [c_i, c_i]),
    "ppx_es_update": (c_i, [c_p, c_p, c_p, c_p, c_i, c_i, c_d, c_d, c_d, c_p, c_i, c_i, c_d, c_p, c_p, c_p, c_p]),
    "ppx_es_offsets": (c_i, [c_u, c_p, c_i, c_l, c_i, c_p, c_p]),
    "ppx_es_update_sharded": (c_i, [c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_d, c_d, c_d, c_p, c_i, c_d, c_p, c_p, c_p, c_p, c_p,
                                    c_p, c_i, c_i, c_p, c_p, c_p]),
    "ppx_rank_center": (c_i, [c_p, c_i, c_p, c_p, c_p]),
    "ppx_knn_novelty": (c_i, [c_p, c_l, c_p, c_i, c_i, c_i, c_p, c_p, c_p]),
    "ppx_knn_novelty_many": (c_i, [c_p, c_l, c_p, c_i, c_i, c_i, c_p, c_p, c_p]),
    "ppx_es_update_member_workspace": (c_l, [c_i, c_i]),
    "ppx_es_update_member": (c_i, [c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_d, c_d, c_i, c_d, c_p, c_p, c_p, c_p, c_p, c_p,
                                   c_i, c_i, c_p, c_p, c_p]),
}
_STATUS = {n for n, (r, _) in SIGNATURES.items() if r is c_i and n not in ("ppx_version", "ppx_tc_supported", "ppx_mlp3_supported", "ppx_mlp3_tc_supported", "ppx_tc_wgrad_supported", "ppx_mlp3_sumsq_partials", "ppx_mlp3_fused_adam_blocks")}

_lib = None


def load():
    """dlopen libppx.so and bind every declared symbol.  Works without a GPU (no CUDA call is made)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} not found: the CUDA extension is not built "
                           "(run __graft_entry__.build()); ppx has no CPU fallback")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is missing -> loud
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error():
    return load().ppx_last_error().decode()


def call(name, *args):
    fn = getattr(load(), name)
    rc = fn(*args)
    if name in _STATUS and rc != 0:
        raise RuntimeError(f"{name} failed ({rc}): {last_error()}")
    return rc


extra_launches = 0      # kernels launched through CUDA-graph replays (not seen by the C-side counter)


def launch_count():
    return int(load().ppx_launch_count()) + extra_launches


def stream():
    return torch.cuda.current_stream().cuda_stream


def ptr(t):
    """device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    return t.data_ptr()


def require_cuda(t, dtype=None, name="tensor"):
    if not t.is_cuda:
        raise RuntimeError(f"{name} must live on a CUDA device (ppx has no CPU path)")
    if dtype is not None and t.dtype != dtype:
        raise RuntimeError(f"{name} must be {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise RuntimeError(f"{name} must be contiguous")
    return t
