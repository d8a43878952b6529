"""ctypes binding of libpuffer_b200.so (include/pufferlib_b200.h).  No fallback: a missing library is an error.

Every wrapper takes raw device addresses (``tensor.data_ptr()``) and a raw ``cudaStream_t``; return codes are
turned into ``APIUsageError`` (misuse, as pufferlib/exceptions.py) or ``RuntimeError`` (CUDA).
"""
import ctypes as C
import os

from pufferlib_b200.exceptions import APIUsageError

HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get('PUFFERLIB_B200_SO', os.path.join(HERE, 'libpuffer_b200.so'))   # override: debug builds

PB_OK, PB_ERR_INVALID, PB_ERR_CUDA, PB_ERR_STATE, PB_ERR_UNSUPPORTED = 0, -1, -2, -3, -4
ENV_KINDS = {'squared': 0, 'breakout': 1, 'snake': 2, 'pong': 3, 'spaces': 4}
DTYPE_F32, DTYPE_U8 = 0, 1


class EnvConfig(C.Structure):
    _fields_ = [('kind', C.c_int32), ('num_envs', C.c_int32), ('device', C.c_int32), ('reserved', C.c_int32),
                ('env_index_offset', C.c_int64), ('iparam', C.c_int32 * 8)]


class EnvInfo(C.Structure):
    _fields_ = [('obs_dtype', C.c_int32), ('obs_ndim', C.c_int32), ('obs_shape', C.c_int32 * 4),
                ('obs_bytes', C.c_int64), ('num_actions', C.c_int32), ('num_envs', C.c_int32),
                ('obs_low', C.c_float), ('obs_high', C.c_float)]


class AdamTensor(C.Structure):
    _fields_ = [('param', C.c_void_p), ('exp_avg', C.c_void_p), ('exp_avg_sq', C.c_void_p), ('step', C.c_void_p),
                ('grad', C.c_void_p), ('numel', C.c_int64)]


class HeadPack(C.Structure):
    _fields_ = [('w_dec', C.c_void_p), ('b_dec', C.c_void_p), ('w_val', C.c_void_p), ('b_val', C.c_void_p),
                ('w_cat', C.c_void_p), ('b_cat', C.c_void_p), ('n_act', C.c_int32), ('hid', C.c_int32)]


class PeerComm(C.Structure):
    _fields_ = [('world', C.c_int32), ('rank', C.c_int32), ('base', C.c_void_p * 8), ('epoch', C.c_void_p),
                ('capacity', C.c_int64)]


class EnvOut(C.Structure):
    _fields_ = [('obs', C.c_void_p), ('obs_stride', C.c_int64), ('rewards', C.c_void_p), ('terminals', C.c_void_p),
                ('truncations', C.c_void_p), ('masks', C.c_void_p), ('dones_f32', C.c_void_p)]


# name -> (restype, argtypes); kept in one table so tests can check it against the header
SIGNATURES = {
    'pb_last_error': (C.c_char_p, []),
    'pb_abi_version': (C.c_int, []),
    'pb_device_count': (C.c_int, [C.POINTER(C.c_int)]),
    'pb_launch_count': (C.c_uint64, []),
    'pb_env_create': (C.c_int, [C.POINTER(EnvConfig), C.POINTER(C.c_void_p)]),
    'pb_env_destroy': (C.c_int, [C.c_void_p]),
    'pb_env_get_info': (C.c_int, [C.c_void_p, C.POINTER(EnvInfo)]),
    'pb_env_action_nvec': (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    'pb_env_reset': (C.c_int, [C.c_void_p, C.c_uint64, C.POINTER(EnvOut), C.c_void_p]),
    'pb_env_step': (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(EnvOut), C.c_void_p]),
    'pb_env_episode_rows': (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                      C.POINTER(C.c_void_p)]),
    'pb_env_stats_read': (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.c_int, C.c_void_p]),
    'pb_rollout_store': (C.c_int, [C.c_void_p] * 6 + [C.c_int64, C.c_void_p]),
    'pb_copy_rows': (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p]),
    'pb_gae_workspace_bytes': (C.c_size_t, [C.c_int64, C.c_int64]),
    'pb_gae': (C.c_int, [C.c_void_p] * 5 + [C.c_int64, C.c_int64, C.c_float, C.c_float, C.c_void_p, C.c_size_t,
                                            C.c_void_p]),
    'pb_flatten_batch': (C.c_int, [C.c_void_p] * 12 + [C.c_int64] * 5 + [C.c_void_p]),
    'pb_minibatch_gather': (C.c_int, [C.c_void_p, C.c_void_p] + [C.c_int64] * 8 + [C.c_void_p]),
    'pb_adv_norm_workspace_bytes': (C.c_size_t, [C.c_int64, C.c_int64]),
    'pb_adv_norm': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_size_t, C.c_void_p]),
    'pb_image_pack': (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p,
                                C.c_int64, C.c_int64, C.c_int32, C.c_void_p]),
    'pb_sample_logits': (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_uint64, C.c_uint64]
                         + [C.c_void_p] * 5 + [C.c_int64] + [C.c_void_p] * 3 + [C.c_void_p]),
    'pb_ppo_loss': (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64] + [C.c_void_p] * 5 + [C.c_int64, C.c_int32,
                    C.c_float, C.c_int32, C.c_float, C.c_float, C.c_float, C.c_void_p, C.c_int64, C.c_void_p,
                    C.c_int64, C.c_void_p, C.c_void_p]),
    'pb_sample_logits_multi': (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.POINTER(C.c_int32), C.c_int32, C.c_uint64,
                                         C.c_uint64] + [C.c_void_p] * 5 + [C.c_int64] + [C.c_void_p] * 3 + [C.c_void_p]),
    'pb_ppo_loss_multi': (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64] + [C.c_void_p] * 5 +
                          [C.c_int64, C.POINTER(C.c_int32), C.c_int32, C.c_float, C.c_int32, C.c_float, C.c_float, C.c_float,
                           C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    'pb_policy_mlp_sample': (C.c_int, [C.c_void_p, C.c_int64] + [C.c_void_p] * 4 + [C.c_int64, C.c_int32, C.c_int32,
                             C.c_int32, C.c_uint64] + [C.c_void_p] * 6 + [C.c_void_p]),
    'pb_mlp_tail_workspace_bytes': (C.c_size_t, [C.c_int64, C.c_int32]),
    'pb_mlp_tail_backward': (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p,
                             C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    'pb_rollout_breakout_mlp': (C.c_int, [C.c_void_p, C.c_int32] + [C.c_void_p] * 6 + [C.POINTER(EnvOut)] + [C.c_void_p] * 4 +
                                [C.c_int32, C.c_uint64, C.c_void_p, C.c_void_p]),
    'pb_rollout_debug_buffers': (C.c_int, [C.c_void_p, C.c_void_p]),
    'pb_mlp_update_workspace_bytes': (C.c_size_t, []),
    'pb_mlp_update_debug_clock': (C.c_int, [C.c_void_p]),
    'pb_mlp_update_fused': (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int32] + [C.c_void_p] * 10 +
                            [C.c_int64, C.c_int32, C.c_float, C.c_int32, C.c_float, C.c_float, C.c_float] + [C.c_void_p] * 3 +
                            [C.c_size_t] + [C.c_void_p] * 5),
    'pb_adv_stats_slabs': (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_size_t,
                                     C.c_void_p]),
    'pb_snake_set_variant': (C.c_int, [C.c_int32]),
    'pb_gae_set_variant': (C.c_int, [C.c_int32]),
    'pb_gae_time_major_supported': (C.c_int, [C.c_int64, C.c_int64]),
    'pb_gae_tm': (C.c_int, [C.c_void_p] * 6 + [C.c_int64, C.c_int64, C.c_float, C.c_float, C.c_void_p, C.c_size_t,
                                               C.c_void_p]),
    'pb_clip_adam': (C.c_int, [C.POINTER(AdamTensor), C.c_int32, C.c_float, C.c_float, C.c_float, C.c_void_p, C.c_float,
                               C.c_float, C.c_float, C.c_void_p, C.c_void_p]),
    'pb_clip_adam_peer': (C.c_int, [C.POINTER(AdamTensor), C.c_int32, C.c_float, C.c_float, C.c_float, C.c_void_p, C.c_float,
                                    C.c_float, C.c_float, C.c_void_p, C.POINTER(PeerComm), C.c_void_p, C.c_int64,
                                    C.c_void_p]),
    'pb_clip_adam_parts': (C.c_int, [C.POINTER(AdamTensor), C.c_int32, C.c_float, C.c_float, C.c_float, C.c_void_p, C.c_float,
                                     C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.POINTER(HeadPack),
                                     C.c_void_p]),
    'pb_clip_adam_peer_parts': (C.c_int, [C.POINTER(AdamTensor), C.c_int32, C.c_float, C.c_float, C.c_float, C.c_void_p, C.c_float,
                                          C.c_float, C.c_float, C.c_void_p, C.POINTER(PeerComm), C.c_void_p, C.c_int64, C.c_void_p,
                                          C.POINTER(HeadPack), C.c_void_p]),
    'pb_peer_allreduce_parts': (C.c_int, [C.POINTER(PeerComm), C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    'pb_peer_slices': (C.c_int32, []),
    'pb_mlp_update_sumsq_offset': (C.c_size_t, []),
    'pb_mlp_update_sumsq_parts': (C.c_int32, []),
    'pb_peer_buffer_bytes': (C.c_size_t, [C.c_int64]),
    'pb_peer_alloc': (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p), C.c_void_p]),
    'pb_peer_open': (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    'pb_peer_close': (C.c_int, [C.c_void_p]),
    'pb_peer_free': (C.c_int, [C.c_void_p]),
    'pb_peer_allreduce': (C.c_int, [C.POINTER(PeerComm), C.c_void_p, C.c_int64, C.c_void_p]),
    'pb_pack_heads': (C.c_int, [C.c_void_p] * 4 + [C.c_int32, C.c_int32] + [C.c_void_p] * 4 + [C.c_int64, C.c_void_p]),
    'pb_struct_pack': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p]),
    'pb_struct_unpack': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]),
}

_lib = None


def lib():
    """The loaded library.  Raises if it has not been built: the product path has no CPU fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise RuntimeError(
                f'{SO_PATH} is missing: build it with `python -m pufferlib_b200.build` (nvcc, sm_100a). '
                'pufferlib_b200 has no CPU fallback.')
        handle = C.CDLL(SO_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def last_error():
    return lib().pb_last_error().decode('utf-8', 'replace')


def check(rc):
    if rc == PB_OK:
        return
    msg = last_error()
    if rc in (PB_ERR_INVALID, PB_ERR_STATE):
        raise APIUsageError(msg)
    if rc == PB_ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise RuntimeError(f'libpuffer_b200: {msg}')


def ptr(t):
    """Device address of a torch tensor (or None)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr(stream=None):
    import torch
    s = torch.cuda.current_stream() if stream is None else stream
    return C.c_void_p(s.cuda_stream)
