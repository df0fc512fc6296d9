"""ctypes signatures of the PPO rollout kernels (include/fwppo.h)."""
import ctypes as C

_P = C.c_void_p
_F = C.c_float
PPO_SYMBOLS = [
    ("ppo_param_count", C.c_int, [C.c_int32]),
    ("ppo_param_count_a", C.c_int, [C.c_int32, C.c_int32]),
    ("ppo_policy_forward_a", C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, _F, C.c_int32, C.c_uint64, C.c_uint32, C.c_uint32, _P,
                                       C.c_int32, _P, _P, _P, _P, _P, _P]),
    ("ppo_policy_forward_tc_a", C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, _F, C.c_int32, C.c_uint64, C.c_uint32, C.c_uint32, _P,
                                          C.c_int32, _P, _P, _P, _P, _P, _P]),
    ("ppo_value_forward_a", C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, _F, C.c_int32, _P, _P]),
    ("ppo_timeout_bootstrap_a", C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, _F, _P, C.c_int32, _F, _P, _P]),
    ("ppo_moments_update", C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    ("ppo_policy_forward", C.c_int, [_P, C.c_int32, _P, _P, _F, C.c_int32, C.c_uint64, C.c_uint32, C.c_uint32, _P,
                                     C.c_int32, _P, _P, _P, _P, _P, _P]),
    ("ppo_policy_forward_tc", C.c_int, [_P, C.c_int32, _P, _P, _F, C.c_int32, C.c_uint64, C.c_uint32, C.c_uint32, _P,
                                        C.c_int32, _P, _P, _P, _P, _P, _P]),
    ("ppo_counter_add", C.c_int, [_P, C.c_uint32, _P]),
    ("ppo_eval_ledger", C.c_int, [_P, _P, _P, C.c_int32, _P, _P, _P, _P, _P, C.c_uint32, _P, C.c_int32, _P, _P, _P, _P, _P, _P,
                                  _P]),
    ("ppo_moments_finalize", C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P]),
    ("ppo_random_permutation", C.c_int, [_P, C.c_int64, C.c_uint64, C.c_uint64, _P]),
    ("ppo_random_permutation_window", C.c_int, [_P, C.c_int64, C.c_uint64, _P, C.c_int64, _P]),
    ("ppo_value_forward", C.c_int, [_P, C.c_int32, _P, _P, _F, C.c_int32, _P, _P]),
    ("ppo_reward_normalize", C.c_int, [_P, _P, C.c_int32, _F, _F, _P, _P, _P, _P, _P, _P, _P]),
    ("ppo_timeout_bootstrap", C.c_int, [_P, C.c_int32, _P, _P, _F, _P, C.c_int32, _F, _P, _P, _P]),
    ("ppo_update_workspace_floats", C.c_int, [C.c_int32]),
    ("ppo_update_workspace_floats_a", C.c_int, [C.c_int32, C.c_int32]),
    ("ppo_minibatch_grad_a", C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P, C.c_int32, _F, _F, _F, _P, _P, _P, _P]),
    ("ppo_minibatch_steps_a", C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P, C.c_int32, C.c_int32, _F, _F, _F, _P, _P,
                                        _F, _F, _F, _F, _F, _P, _P, _P, _P, _P]),
    ("ppo_window_update_a", C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P, C.c_int32, C.c_int32, _F, _F, _F, _P, _P,
                                      _F, _F, _F, _F, _F, _P, _P, _P, _P, _P, _P]),
    ("ppo_window_update_p2p_a", C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P, C.c_int32, C.c_int32, _F, _F, _F, _P, _P,
                                          _F, _F, _F, _F, _F, _P, _P, _P, _P, _P, C.c_int32, C.c_int32, _P, _P, _P]),
    ("ppo_minibatch_steps_p2p_a", C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P, C.c_int32, C.c_int32, _F, _F, _F, _P, _P,
                                            _F, _F, _F, _F, _F, _P, _P, _P, _P, C.c_int32, C.c_int32, _P, _P, _P]),
    ("ppo_peer_bytes", C.c_int64, []),
    ("ppo_peer_alloc", C.c_int, [C.POINTER(C.c_void_p)]),
    ("ppo_peer_free", C.c_int, [_P]),
    ("ppo_peer_export", C.c_int, [_P, _P]),
    ("ppo_peer_import", C.c_int, [_P, C.POINTER(C.c_void_p)]),
    ("ppo_peer_close", C.c_int, [_P]),
    ("ppo_minibatch_grad", C.c_int, [_P, C.c_int32, _P, _P, _P, _P, _P, _P, C.c_int32, _F, _F, _F, _P, _P, _P, _P]),
    ("ppo_adam_step", C.c_int, [_P, _P, _P, _P, C.c_int32, _F, _F, _F, _F, _F, _F, _P, _P, _P]),
    ("ppo_gae", C.c_int, [_P, _P, _P, _P, C.c_int32, C.c_int32, _F, _F, _P, _P, _P]),
    # populations (members, rows_per_member, ...)
    ("ppo_pop_policy_forward_a", C.c_int, [C.c_int32, C.c_int32, _P, _P, C.c_int32, C.c_int32, _P, _P, _F, C.c_uint32, C.c_uint32,
                                           _P, C.c_int32, _P, _P, _P, _P, _P, _P]),
    ("ppo_pop_policy_forward_tc_a", C.c_int, [C.c_int32, C.c_int32, _P, _P, C.c_int32, C.c_int32, _P, _P, _F, C.c_uint32, C.c_uint32,
                                              _P, C.c_int32, _P, _P, _P, _P, _P, _P]),
    ("ppo_pop_value_forward_a", C.c_int, [C.c_int32, C.c_int32, _P, C.c_int32, C.c_int32, _P, _P, _F, _P, _P]),
    ("ppo_pop_timeout_bootstrap_a", C.c_int, [C.c_int32, C.c_int32, _P, _P, C.c_int32, C.c_int32, _P, _P, _F, _P, _P, _P]),
    ("ppo_pop_moments_update", C.c_int, [C.c_int32, C.c_int32, _P, C.c_int32, _P, _P, _P, _P]),
    ("ppo_pop_reward_normalize", C.c_int, [C.c_int32, C.c_int32, _P, _P, _P, _F, _P, _P, _P, _P, _P, _P, _P]),
    ("ppo_pop_gae", C.c_int, [C.c_int32, C.c_int32, _P, _P, _P, _P, _P, C.c_int32, _P, _P, _P]),
    ("ppo_pop_random_permutation", C.c_int, [C.c_int32, C.c_int32, _P, _P, C.c_int64, C.c_uint64, _P]),
    ("ppo_pop_minibatch_steps_a", C.c_int, [C.c_int32, _P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P, C.c_int64, C.c_int32,
                                            C.c_int32, _P, _P, _F, _F, _F, _P, _P, _P, _P, _P]),
    ("ppo_pop_episode_ledger", C.c_int, [C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P, _P]),
]


def bind(lib) -> None:
    for name, res, args in PPO_SYMBOLS:
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
