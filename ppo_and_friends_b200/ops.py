"""
Torch-tensor front-ends of the C ABI (include/ppoaf_b200.h).  Each function only checks
shapes/dtypes, allocates outputs through torch and enqueues the kernel on torch's current
stream.  No arithmetic happens in Python and there is no CPU path.
"""
import ctypes as C

import torch

from . import _lib
from ._lib import check, load, ptr, stream_ptr

_ws_cache = {}


def _workspace(key, nbytes, device, zero=False):
    """Persistent per-(key, device) scratch buffers (uint8), grown on demand."""
    k = (key, str(device))
    buf = _ws_cache.get(k)
    if buf is None or buf.numel() < nbytes:
        buf = torch.zeros(max(int(nbytes), 256), dtype=torch.uint8, device=device)
        _ws_cache[k] = buf
    elif zero:
        buf.zero_()
    return buf


def runtime_init():
    _lib.require_cuda()
    check(load().ppoaf_runtime_init(), "ppoaf_runtime_init")


def set_gemm_backend(name):
    """GEMM tiles of mlp_forward: 'ffma' (default) or 'tcgen05' (3xTF32 tensor-core tiles); the update always runs FFMA."""
    check(load().ppoaf_set_gemm_backend({'ffma': 0, 'tcgen05': 1}[name]), 'ppoaf_set_gemm_backend')


def device_info():
    a, b, c = C.c_int(), C.c_int(), C.c_int()
    check(load().ppoaf_device_info(C.byref(a), C.byref(b), C.byref(c)), "ppoaf_device_info")
    return dict(sm_count=a.value, cc=(b.value, c.value))


# ---- A2/A5 ---------------------------------------------------------------------------------------
def build_flat_map(seg_col, seg_t0, seg_len, seg_off, seg_terminal, n_cols, n_flat):
    """Segment table (int32/int64/uint8 CUDA tensors) -> (src_row int32[N], seg_flag uint8[N])."""
    dev = seg_col.device
    n_seg = seg_col.numel()
    src_row = torch.empty(n_flat, dtype=torch.int32, device=dev)
    seg_flag = torch.empty(n_flat, dtype=torch.uint8, device=dev)
    check(load().ppoaf_build_flat_map(ptr(seg_col), ptr(seg_t0), ptr(seg_len), ptr(seg_off), ptr(seg_terminal),
                                      n_seg, int(n_cols), int(n_flat), ptr(src_row), ptr(seg_flag), stream_ptr()),
          "ppoaf_build_flat_map")
    return src_row, seg_flag


def gather_rows(src, idx, out=None, row_bytes=None, src_stride_bytes=0, src_offset_bytes=0, n_rows=None,
                out_shape=None, out_dtype=None):
    """dst[i] = src[idx[i]] (rows). With src_stride/offset: de-interleave a field of a packed ring."""
    assert idx.dtype in (torch.int32, torch.int64)
    n = idx.numel() if n_rows is None else n_rows
    if row_bytes is None:
        row_bytes = src[0].numel() * src.element_size()
    if out is None:
        shape = out_shape if out_shape is not None else (n,) + tuple(src.shape[1:])
        out = torch.empty(shape, dtype=out_dtype or src.dtype, device=src.device)
    sp = C.c_void_p(src.data_ptr() + int(src_offset_bytes))
    check(load().ppoaf_gather_rows(sp, int(src_stride_bytes), ptr(idx), int(idx.dtype == torch.int64), ptr(out), int(n),
                                   int(row_bytes), stream_ptr()), "ppoaf_gather_rows")
    return out


# ---- A3/A4 ---------------------------------------------------------------------------------------
def gae_rtg_segscan(rewards, values, seg_flag, seg_off, v_boot, r_boot, gamma, lambd, use_gae=True,
                    adv_out=None, rtg_out=None):
    n = rewards.numel()
    dev = rewards.device
    adv = adv_out if adv_out is not None else torch.empty(n, dtype=torch.float32, device=dev)
    rtg = rtg_out if rtg_out is not None else torch.empty(n, dtype=torch.float32, device=dev)
    if n == 0:
        return adv, rtg
    lib = load()
    nbytes = lib.ppoaf_segscan_workspace_bytes(n)
    ws = _workspace("segscan", nbytes, dev)
    check(lib.ppoaf_gae_rtg_segscan(ptr(rewards), ptr(values), ptr(seg_flag), ptr(seg_off), ptr(v_boot), ptr(r_boot),
                                    v_boot.numel(), n, float(gamma), float(lambd), int(bool(use_gae)), ptr(adv),
                                    ptr(rtg), ptr(ws), ws.numel(), stream_ptr()), "ppoaf_gae_rtg_segscan")
    return adv, rtg


# ---- N1/N2/N4 ------------------------------------------------------------------------------------
def batch_moments(x, dim, triple_out=None):
    """x: fp32 CUDA [n_rows, dim] (contiguous) -> fp64 [2*dim+1] = mean | M2 | n."""
    n_rows = x.numel() // dim
    dev = x.device
    out = triple_out if triple_out is not None else torch.empty(2 * dim + 1, dtype=torch.float64, device=dev)
    lib = load()
    ws = _workspace("moments", lib.ppoaf_moments_workspace_bytes(n_rows, dim), dev)
    check(lib.ppoaf_batch_moments(ptr(x), n_rows, dim, ptr(out), ptr(ws), ws.numel(), stream_ptr()),
          "ppoaf_batch_moments")
    return out


def stats_merge(state, triples, dim):
    n_triples = triples.numel() // (2 * dim + 1)
    check(load().ppoaf_stats_merge(ptr(state), ptr(triples), n_triples, dim, stream_ptr()), "ppoaf_stats_merge")


def normalize_clip(x, state, dim, eps=1e-8, lo=1.0, hi=-1.0, out=None):
    out = torch.empty_like(x) if out is None else out
    n_rows = x.numel() // dim
    check(load().ppoaf_normalize_clip(ptr(x), n_rows, dim, ptr(state), float(eps), float(lo), float(hi), ptr(out),
                                      stream_ptr()), "ppoaf_normalize_clip")
    return out


def denormalize(x, state, dim, eps=1e-8, out=None):
    out = torch.empty_like(x) if out is None else out
    n_rows = x.numel() // dim
    check(load().ppoaf_denormalize(ptr(x), n_rows, dim, ptr(state), float(eps), ptr(out), stream_ptr()),
          "ppoaf_denormalize")
    return out


# ---- P1/P2 ---------------------------------------------------------------------------------------
def mlp_forward(desc, params, x, idx=None, n_rows=None, softmax_out=False, out=None):
    n = int(n_rows if n_rows is not None else (idx.numel() if idx is not None else x.shape[0]))
    dev = x.device
    out_dim = desc.dims[desc.n_layers]
    y = out if out is not None else torch.empty((n, out_dim), dtype=torch.float32, device=dev)
    lib = load()
    ws = _workspace("mlp_fwd", lib.ppoaf_mlp_forward_workspace_bytes(C.byref(desc), n), dev)
    check(lib.ppoaf_mlp_forward(C.byref(desc), ptr(params), ptr(x), ptr(idx), n, int(bool(softmax_out)), ptr(y),
                                ptr(ws), ws.numel(), stream_ptr()), "ppoaf_mlp_forward")
    return y


def head_evaluate(head, actor_out, log_std, actions, min_std=0.01, want_entropy=True):
    n, pred = actor_out.shape
    act_dim = actions.shape[1] if actions.dim() > 1 else 1
    lp = torch.empty(n, dtype=torch.float32, device=actor_out.device)
    ent = torch.empty(n, dtype=torch.float32, device=actor_out.device) if want_entropy else None
    check(load().ppoaf_head_evaluate(int(head), ptr(actor_out), pred, ptr(log_std), float(min_std), ptr(actions),
                                     act_dim, n, ptr(lp), ptr(ent), stream_ptr()), "ppoaf_head_evaluate")
    return lp, ent


def head_sample(head, actor_out, log_std, noise, min_std=0.01, dist_min=None, dist_max=None, act_dim=1):
    """(raw_action, action, log_prob) from the actor output and host-drawn noise (see ppoaf_head_sample)."""
    n, pred = actor_out.shape
    dev = actor_out.device
    if head in (_lib.HEAD_GAUSSIAN_TANH, _lib.HEAD_BERNOULLI):
        raw = torch.empty((n, act_dim), dtype=torch.float32, device=dev)
        act = torch.empty((n, act_dim), dtype=torch.float32, device=dev)
    else:
        raw = torch.empty((n, 1), dtype=torch.int64, device=dev)
        act = torch.empty((n, 1), dtype=torch.int64, device=dev)
    lp = torch.empty(n, dtype=torch.float32, device=dev)
    check(load().ppoaf_head_sample(int(head), ptr(actor_out), pred, ptr(log_std), float(min_std), ptr(noise), ptr(dist_min),
                                   ptr(dist_max), int(act_dim), n, ptr(raw), ptr(act), ptr(lp), stream_ptr()),
          "ppoaf_head_sample")
    return raw, act, lp


def multi_categorical_evaluate(actor_out, section_ends, actions, want_entropy=True):
    """(log_prob, entropy) [n] of int64 actions [n, n_sections] under the multi-categorical head on logits actor_out."""
    n, pred = actor_out.shape
    lp = torch.empty(n, dtype=torch.float32, device=actor_out.device)
    ent = torch.empty(n, dtype=torch.float32, device=actor_out.device) if want_entropy else None
    check(load().ppoaf_multi_categorical_evaluate(ptr(actor_out), pred, section_ends & 0xFFFFFFFF, section_ends >> 32,
                                                  ptr(actions), actions.shape[1], n, ptr(lp), ptr(ent), stream_ptr()),
          "ppoaf_multi_categorical_evaluate")
    return lp, ent


def multi_categorical_sample(probs, section_ends, noise, n_sections):
    """(int64 actions [n, n_sections], log_prob [n]) from softmax probs and host-drawn Exp(1) noise laid out section after
    section (see ppoaf_multi_categorical_sample)."""
    n, pred = probs.shape
    act = torch.empty((n, n_sections), dtype=torch.int64, device=probs.device)
    lp = torch.empty(n, dtype=torch.float32, device=probs.device)
    check(load().ppoaf_multi_categorical_sample(ptr(probs), pred, section_ends & 0xFFFFFFFF, section_ends >> 32, ptr(noise),
                                                int(n_sections), n, ptr(act), ptr(lp), stream_ptr()),
          "ppoaf_multi_categorical_sample")
    return act, lp


def clip_adam_step(params, grads, m, v, adam_step, hparams, n_actor, n_critic):
    lib = load()
    ws = _workspace("adam", 1 << 16, params.device)
    check(lib.ppoaf_clip_adam_step(ptr(params), ptr(grads), ptr(m), ptr(v), ptr(adam_step), ptr(hparams), int(n_actor),
                                   int(n_critic), ptr(ws), ws.numel(), stream_ptr()), "ppoaf_clip_adam_step")
