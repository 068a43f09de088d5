"""
ctypes binding of libppoaf_b200.so (C ABI: include/ppoaf_b200.h).

This is the binding a PPO-AF maintainer would add behind the policy/dataset API (see
INTEGRATION.md).  There is NO CPU fallback: if the library is missing or no CUDA device is
visible, the compute entry points raise.  torch is used only for device memory and streams.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libppoaf_b200.so")

MAX_LAYERS = 8
ACT_IDS = {"identity": 0, "relu": 1, "leaky_relu": 2, "tanh": 3, "elu": 4, "selu": 5, "sigmoid": 6, "softplus": 7,
           "silu": 8, "gelu": 9, "gelu_tanh": 10, "mish": 11}
HEAD_GAUSSIAN_TANH, HEAD_CATEGORICAL, HEAD_MULTI_CATEGORICAL, HEAD_BERNOULLI = 0, 1, 2, 3

HP = dict(LR=0, ENTROPY_WEIGHT=1, SURR_CLIP=2, GRAD_CLIP=3, KL_WEIGHT=4, VF_CLIP=5, BETA1=6, BETA2=7,
          ADAM_EPS=8, INV_WORLD=9, COUNT=16)
ST = dict(ACTOR_LOSS=0, CRITIC_LOSS=1, ENTROPY=2, KL=3, COUNTER=4, BAD_RATIO=5, BAD_VALUE=6, COUNT=8)


class MlpDesc(C.Structure):
    _fields_ = [("n_layers", C.c_int32), ("dims", C.c_int32 * (MAX_LAYERS + 1)), ("activation", C.c_int32)]

    @classmethod
    def make(cls, dims, activation):
        assert 2 <= len(dims) <= MAX_LAYERS + 1
        d = cls()
        d.n_layers = len(dims) - 1
        for i, v in enumerate(dims):
            d.dims[i] = int(v)
        d.activation = ACT_IDS[activation] if isinstance(activation, str) else int(activation)
        return d


class UpdateCfg(C.Structure):
    _fields_ = [("actor", MlpDesc), ("critic", MlpDesc), ("head", C.c_int32), ("act_dim", C.c_int32),
                ("use_huber", C.c_int32), ("normalize_adv", C.c_int32), ("normalize_values", C.c_int32),
                ("vf_clip_enabled", C.c_int32), ("world_size", C.c_int32), ("reserved", C.c_int32 * 1), ("min_std", C.c_float),
                ("section_ends", C.c_uint32 * 2), ("reserved_f", C.c_float * 1)]


class UpdateBufs(C.Structure):
    _fields_ = [("critic_obs", C.c_void_p), ("obs", C.c_void_p), ("raw_actions", C.c_void_p),
                ("advantages", C.c_void_p), ("log_probs", C.c_void_p), ("rewards_to_go", C.c_void_p),
                ("values", C.c_void_p), ("perm", C.c_void_p), ("mb_adv_stats", C.c_void_p),
                ("mb_val_stats", C.c_void_p), ("params", C.c_void_p), ("grads", C.c_void_p),
                ("adam_m", C.c_void_p), ("adam_v", C.c_void_p), ("adam_step", C.c_void_p),
                ("hparams", C.c_void_p), ("epoch_stats", C.c_void_p), ("mb_cursor", C.c_void_p),
                ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t), ("n_flat", C.c_int64),
                ("batch", C.c_int32), ("batch_size", C.c_int32),
                ("n_mirror", C.c_int32), ("reserved0", C.c_int32), ("mirror_delta", C.c_int64 * 7)]


_P = C.c_void_p
_SIGNATURES = {
    "ppoaf_abi_version": (C.c_int, []),
    "ppoaf_last_error": (C.c_char_p, []),
    "ppoaf_device_info": (C.c_int, [C.POINTER(C.c_int)] * 3),
    "ppoaf_build_flat_map": (C.c_int, [_P, _P, _P, _P, _P, C.c_int32, C.c_int32, C.c_int64, _P, _P, _P]),
    "ppoaf_runtime_init": (C.c_int, []),
    "ppoaf_set_gemm_backend": (C.c_int, [C.c_int]),
    "ppoaf_get_gemm_backend": (C.c_int, []),
    "ppoaf_gather_rows": (C.c_int, [_P, C.c_int64, _P, C.c_int, _P, C.c_int64, C.c_int64, _P]),
    "ppoaf_segscan_workspace_bytes": (C.c_size_t, [C.c_int64]),
    "ppoaf_gae_rtg_segscan": (C.c_int, [_P, _P, _P, _P, _P, _P, C.c_int32, C.c_int64, C.c_double, C.c_double,
                                        C.c_int, _P, _P, _P, C.c_size_t, _P]),
    "ppoaf_moments_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int32]),
    "ppoaf_batch_moments": (C.c_int, [_P, C.c_int64, C.c_int32, _P, _P, C.c_size_t, _P]),
    "ppoaf_stats_merge": (C.c_int, [_P, _P, C.c_int32, C.c_int32, _P]),
    "ppoaf_normalize_clip": (C.c_int, [_P, C.c_int64, C.c_int32, _P, C.c_float, C.c_float, C.c_float, _P, _P]),
    "ppoaf_denormalize": (C.c_int, [_P, C.c_int64, C.c_int32, _P, C.c_float, _P, _P]),
    "ppoaf_reward_norm_triples": (C.c_int, [_P, _P, _P, C.c_int32, C.c_double, _P, _P]),
    "ppoaf_reward_scale_clip": (C.c_int, [_P, _P, C.c_float, C.c_float, C.c_float, _P, C.c_int32, _P]),
    "ppoaf_param_layout": (C.c_int64, [C.POINTER(MlpDesc), C.c_int32, C.POINTER(C.c_int64)]),
    "ppoaf_update_workspace_bytes": (C.c_size_t, [C.POINTER(UpdateCfg), C.c_int32]),
    "ppoaf_epoch_prepare": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int32, _P, _P, _P]),
    "ppoaf_value_stats_sequence": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_float, _P, _P]),
    "ppoaf_ppo_minibatch_grads": (C.c_int, [C.POINTER(UpdateCfg), C.POINTER(UpdateBufs), _P]),
    "ppoaf_ppo_minibatch_apply": (C.c_int, [C.POINTER(UpdateCfg), C.POINTER(UpdateBufs), _P]),
    "ppoaf_ppo_fused_supported": (C.c_int, [C.POINTER(UpdateCfg)]),
    "ppoaf_ppo_fused_workspace_bytes": (C.c_size_t, [C.POINTER(UpdateCfg), C.c_int32]),
    "ppoaf_ppo_fused_steps": (C.c_int, [C.POINTER(UpdateCfg), C.POINTER(UpdateBufs), C.c_int32, _P]),
    "ppoaf_mlp_forward_workspace_bytes": (C.c_size_t, [C.POINTER(MlpDesc), C.c_int32]),
    "ppoaf_mlp_forward": (C.c_int, [C.POINTER(MlpDesc), _P, _P, _P, C.c_int32, C.c_int, _P, _P, C.c_size_t, _P]),
    "ppoaf_head_evaluate": (C.c_int, [C.c_int32, _P, C.c_int32, _P, C.c_float, _P, C.c_int32, C.c_int32, _P, _P, _P]),
    "ppoaf_head_sample": (C.c_int, [C.c_int32, _P, C.c_int32, _P, C.c_float, _P, _P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    "ppoaf_multi_categorical_evaluate": (C.c_int, [_P, C.c_int32, C.c_uint32, C.c_uint32, _P, C.c_int32, C.c_int32, _P, _P, _P]),
    "ppoaf_multi_categorical_sample": (C.c_int, [_P, C.c_int32, C.c_uint32, C.c_uint32, _P, C.c_int32, C.c_int32, _P, _P, _P]),
    "ppoaf_nvls_ctrl_bytes": (C.c_size_t, []),
    "ppoaf_nvls_flag_block_bytes": (C.c_size_t, []),
    "ppoaf_nvls_allreduce_adam": (C.c_int, [_P, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int32, C.c_int32, _P, _P, _P,
                                            _P, _P, _P, C.c_int64, C.c_int64, _P, _P]),
    "ppoaf_peer_alloc": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p)]),
    "ppoaf_peer_free": (C.c_int, [_P]),
    "ppoaf_peer_export": (C.c_int, [_P, C.c_char_p]),
    "ppoaf_peer_import": (C.c_int, [C.c_char_p, C.POINTER(C.c_void_p)]),
    "ppoaf_peer_close": (C.c_int, [_P]),
    "ppoaf_peer_ctrl_bytes": (C.c_size_t, []),
    "ppoaf_peer_allreduce_adam": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int32, C.c_int32, _P, _P,
                                            _P, _P, _P, _P, C.c_int64, C.c_int64, _P, _P]),
    "ppoaf_clip_adam_step": (C.c_int, [_P, _P, _P, _P, _P, _P, C.c_int64, C.c_int64, _P, C.c_size_t, _P]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


class PpoafError(RuntimeError):
    pass


def load():
    """Load the shared library (building nothing: run `python -m ppo_and_friends_b200.build` first)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PpoafError(f"{LIB_PATH} is missing: the CUDA extension was not built "
                         f"(python -m ppo_and_friends_b200.build). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.ppoaf_abi_version() != 1:
        raise PpoafError("libppoaf_b200.so ABI version mismatch")
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        msg = load().ppoaf_last_error().decode(errors="replace")
        raise PpoafError(f"{what or 'ppoaf call'} failed (code {rc}): {msg}")


def require_cuda():
    if not torch.cuda.is_available():
        raise PpoafError("ppo_and_friends_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous(), "ppoaf kernels take contiguous CUDA tensors"
    return C.c_void_p(t.data_ptr())


def stream_ptr(stream=None):
    s = torch.cuda.current_stream() if stream is None else stream
    return C.c_void_p(s.cuda_stream)


def section_ends(nvec):
    """The multi-categorical section table of ppoaf_update_cfg: bit c set = actor output c ends a section."""
    mask = 0
    end = -1
    for n in nvec:
        end += int(n)
        mask |= 1 << end
    return mask


def param_layout(desc, log_std_dim=0):
    """(offsets[2L+1], total floats) of one network in the flat parameter buffer."""
    lib = load()
    offs = (C.c_int64 * (2 * desc.n_layers + 1))()
    total = lib.ppoaf_param_layout(C.byref(desc), int(log_std_dim), offs)
    if total < 0:
        check(1, "ppoaf_param_layout")
    return list(offs), int(total)
