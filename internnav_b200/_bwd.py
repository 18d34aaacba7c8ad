"""ctypes bindings of the backward primitives (include/n1b200.h, "training: backward primitives").

Validated on the B200 against PyTorch autograd / torch.optim (tests/test_bwd_ops_gpu.py, profiles/r2_bwd_ops_parity.log);
used by the training step (train_s1.py, train_step.py).  Nothing on the inference path imports this module.
"""
import ctypes
from ctypes import c_double, c_float, c_int, c_int64, c_void_p

import torch

from . import _lib
from ._lib import check, ptr, stream_ptr

_bound = False
BWD_SYMBOLS = ["n1_op_act_fwd", "n1_op_transpose", "n1_op_colsum", "n1_op_norm_bwd", "n1_op_act_bwd", "n1_op_swiglu_bwd",
               "n1_op_rope_transposed", "n1_op_attention_bwd", "n1_op_adamw", "n1_op_sgemm", "n1_op_scale_cols",
               "n1_op_patchify_depth", "n1_op_wgrad", "n1_op_dropout_add", "n1_op_dropout_bwd", "n1_op_dropout_mask",
               "n1_op_act_fwd_dropout", "n1_op_act_bwd_dropout", "n1_op_attention_dropout", "n1_op_attention_bwd_dropout"]


def _L():
    global _bound
    L = _lib.lib()
    if not _bound:
        vp = c_void_p
        L.n1_op_transpose.argtypes = [vp, c_int, c_int, c_int, vp, c_int, c_int, vp]
        L.n1_op_colsum.argtypes = [vp, vp, c_int, c_int, c_int, c_int, vp, c_int, vp]
        L.n1_op_norm_bwd.argtypes = [vp, c_int, vp, c_int, vp, vp, c_int, vp, c_int, vp, vp, c_int, c_int, c_float, c_int,
                                     c_int, vp]
        L.n1_op_act_fwd.argtypes = [vp, vp, c_int64, c_int, vp]
        L.n1_op_act_bwd.argtypes = [vp, vp, vp, c_int64, c_int, vp]
        L.n1_op_swiglu_bwd.argtypes = [vp, vp, vp, c_int64, c_int, vp]
        L.n1_op_rope_transposed.argtypes = [vp, c_int, vp, c_int64, c_int, c_int, vp]
        L.n1_op_attention_bwd.argtypes = [vp] * 8 + [c_int] * 12 + [vp, vp, c_int, c_int, c_int, c_float, vp, c_int, vp]
        L.n1_op_adamw.argtypes = [vp, vp, vp, vp, vp, c_int64, c_float, c_float, c_float, c_float, c_float, c_int, vp]
        L.n1_op_sgemm.argtypes = [vp, c_int, c_int, vp, c_int, c_int, vp, c_int, c_int, c_int, c_int, c_int, vp]
        L.n1_op_scale_cols.argtypes = [vp, c_int, vp, vp, c_int, vp, c_int, c_int64, c_int, vp]
        L.n1_op_patchify_depth.argtypes = [vp, vp, c_int, c_int, vp]
        L.n1_op_wgrad.argtypes = [vp, c_int, vp, c_int, c_int, c_int, c_int, vp, c_int, vp, ctypes.c_size_t, vp]
        L.n1_op_wgrad_workspace_bytes.argtypes = [c_int, c_int, c_int]
        d = [vp, c_int, c_double, vp]                       # dropout descriptor (rng, site, p) + stream
        L.n1_op_dropout_add.argtypes = [vp, vp, vp, c_int64] + d
        L.n1_op_dropout_bwd.argtypes = [vp, vp, c_int64] + d
        L.n1_op_dropout_mask.argtypes = [vp, c_int64] + d
        L.n1_op_act_fwd_dropout.argtypes = [vp, vp, c_int64, c_int] + d
        L.n1_op_act_bwd_dropout.argtypes = [vp, vp, vp, c_int64, c_int] + d
        L.n1_op_attention_dropout.argtypes = [vp] * 4 + [c_int] * 10 + [c_float] + d
        L.n1_op_attention_bwd_dropout.argtypes = [vp] * 8 + [c_int] * 12 + [c_float] + d
        L.n1_op_wgrad_workspace_bytes.restype = ctypes.c_size_t
        for n in BWD_SYMBOLS:
            getattr(L, n).restype = c_int
        _bound = True
    return L


def transpose(x, rows_pad=None):
    """x bf16 [rows, cols] -> [cols, rows_pad] with zero padding (rows_pad defaults to rows rounded up to 8)."""
    rows, cols = x.shape
    rows_pad = rows_pad or (rows + 7) // 8 * 8
    out = torch.empty(cols, rows_pad, dtype=torch.bfloat16, device=x.device)
    check(_L().n1_op_transpose(ptr(x), rows, cols, x.stride(0), ptr(out), rows_pad, rows_pad, stream_ptr()))
    return out


def colsum(a, b=None, out=None, accumulate=False):
    rows, cols = a.shape
    if out is None:
        out = torch.zeros(cols, dtype=torch.float32, device=a.device)
    check(_L().n1_op_colsum(ptr(a), ptr(b), rows, cols, a.stride(0), b.stride(0) if b is not None else 0, ptr(out),
                            1 if accumulate else 0, stream_ptr()))
    return out


def norm_bwd(dy, x, w, eps, rms=False, residual_grad=None, need_param_grads=True):
    rows, D = x.shape
    dx = torch.empty_like(x)
    dw = torch.zeros(D, dtype=torch.float32, device=x.device) if need_param_grads else None
    db = torch.zeros(D, dtype=torch.float32, device=x.device) if need_param_grads and not rms else None
    check(_L().n1_op_norm_bwd(ptr(dy), dy.stride(0), ptr(x), x.stride(0), ptr(w), ptr(residual_grad),
                              residual_grad.stride(0) if residual_grad is not None else 0, ptr(dx), dx.stride(0), ptr(dw),
                              ptr(db), rows, D, eps, 1 if rms else 0, 0, stream_ptr()))
    return dx, dw, db


def act_fwd(pre, act):
    out = torch.empty_like(pre)
    check(_L().n1_op_act_fwd(ptr(pre), ptr(out), pre.numel(), act, stream_ptr()))
    return out


def act_bwd(pre, dy, act):
    out = torch.empty_like(pre)
    check(_L().n1_op_act_bwd(ptr(pre), ptr(dy), ptr(out), pre.numel(), act, stream_ptr()))
    return out


def swiglu_bwd(pre, dact):
    out = torch.empty_like(pre)
    check(_L().n1_op_swiglu_bwd(ptr(pre), ptr(dact), ptr(out), dact.shape[0], dact.shape[1], stream_ptr()))
    return out


def rope_transposed(x, cos_sin, heads, head_dim):
    """in place on the first `heads` heads of every row of x [rows, >= heads * head_dim]; cos_sin fp32 [rows, hd/2, 2]"""
    check(_L().n1_op_rope_transposed(ptr(x), x.stride(0), ptr(cos_sin), x.shape[0], heads, head_dim, stream_ptr()))
    return x


def attention_bwd(q, k, v, o, dout, heads_q, heads_kv, head_dim, batch, seq_q, seq_k, causal=False, kv_div=1, scale=None,
                  cu_q=None, cu_k=None, max_seq_q=0, k_len=None, k_slot=0):
    dq = torch.zeros(q.shape[0], heads_q * head_dim, dtype=torch.bfloat16, device=q.device)
    dk = torch.zeros(k.shape[0], heads_kv * head_dim, dtype=torch.float32, device=q.device)
    dv = torch.zeros_like(dk)
    scale = head_dim ** -0.5 if scale is None else scale
    for t in (q, k, v, o, dout):   # column slices of packed projections are legal operands: row stride + unit inner stride
        assert t.is_cuda and t.dtype == torch.bfloat16 and t.stride(1) == 1
    vp = lambda t: c_void_p(t.data_ptr())
    check(_L().n1_op_attention_bwd(vp(q), vp(k), vp(v), vp(o), vp(dout), ptr(dq), ptr(dk), ptr(dv), q.stride(0),
                                   k.stride(0), v.stride(0), o.stride(0), dout.stride(0), dq.stride(0), heads_q, heads_kv,
                                   head_dim, batch, seq_q, seq_k, ptr(cu_q), ptr(cu_k), max_seq_q, kv_div,
                                   1 if causal else 0, scale, ptr(k_len), k_slot, stream_ptr()))
    return dq, dk, dv


def wgrad_supported(dy, x):
    """Operands the in-place weight-gradient kernel takes: bf16 rows with 16-byte aligned starts and pitches, Ko % 4 == 0."""
    import os
    if os.environ.get("N1_WGRAD_TN", "1") == "0":     # keep the transposing path (A/B comparison)
        return False
    return (dy.dtype == torch.bfloat16 and x.dtype == torch.bfloat16 and dy.dim() == 2 and x.dim() == 2
            and dy.shape[0] == x.shape[0] and dy.stride(1) == 1 and x.stride(1) == 1 and dy.stride(0) % 8 == 0
            and x.stride(0) % 8 == 0 and dy.data_ptr() % 16 == 0 and x.data_ptr() % 16 == 0 and x.shape[1] % 4 == 0
            and dy.shape[1] % 8 == 0 and x.shape[1] % 8 == 0)


def wgrad(dy, x, out=None, accumulate=False):
    """dW [No, Ko] fp32 (+)= dy[M, No]^T @ x[M, Ko], operands read in place (csrc/wgrad_tn.cu)."""
    assert wgrad_supported(dy, x), (dy.shape, dy.stride(), x.shape, x.stride())
    M, No, Ko = dy.shape[0], dy.shape[1], x.shape[1]
    if out is None:
        assert not accumulate
        out = torch.empty(No, Ko, dtype=torch.float32, device=dy.device)
    assert out.dtype == torch.float32 and out.is_contiguous() and tuple(out.shape) == (No, Ko)
    L = _L()
    nb = L.n1_op_wgrad_workspace_bytes(M, No, Ko)
    ws = torch.empty(nb + 16, dtype=torch.uint8, device=dy.device)
    check(L.n1_op_wgrad(c_void_p(dy.data_ptr()), dy.stride(0), c_void_p(x.data_ptr()), x.stride(0), M, No, Ko, ptr(out),
                        1 if accumulate else 0, c_void_p((ws.data_ptr() + 15) // 16 * 16), nb, stream_ptr()))
    return out


def sgemm(a, b, trans_a=False, trans_b=False, out=None, accumulate=False):
    """fp32 op(a) @ op(b): a [M, K] (or [K, M] with trans_a), b [K, N] (or [N, K] with trans_b) -> [M, N] fp32."""
    assert a.dtype == torch.float32 and b.dtype == torch.float32 and a.dim() == 2 and b.dim() == 2
    assert a.stride(1) == 1 and b.stride(1) == 1
    M, K = (a.shape[1], a.shape[0]) if trans_a else a.shape
    N = b.shape[0] if trans_b else b.shape[1]
    assert (b.shape[1] if trans_b else b.shape[0]) == K, (a.shape, b.shape, trans_a, trans_b)
    if out is None:
        out = torch.empty(M, N, dtype=torch.float32, device=a.device)
    check(_L().n1_op_sgemm(c_void_p(a.data_ptr()), a.stride(0), 1 if trans_a else 0, c_void_p(b.data_ptr()), b.stride(0),
                           1 if trans_b else 0, ptr(out), out.stride(0), M, N, K, 1 if accumulate else 0, stream_ptr()))
    return out


def scale_cols(x, gamma, add=None):
    """x [rows, cols] bf16 * gamma [cols] fp32 (+ add bf16) -> bf16."""
    assert x.dim() == 2 and x.stride(1) == 1 and x.dtype == torch.bfloat16 and gamma.dtype == torch.float32
    out = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
    check(_L().n1_op_scale_cols(c_void_p(x.data_ptr()), x.stride(0), ptr(gamma),
                                c_void_p(add.data_ptr()) if add is not None else None,
                                add.stride(0) if add is not None else 0, ptr(out), out.stride(0), x.shape[0], x.shape[1],
                                stream_ptr()))
    return out


def patchify_depth(frames, ldk=200):
    """frames fp32 [n, 224, 224] -> bf16 [n * 256, ldk]: im2col of the 14 x 14 patches of one channel."""
    assert frames.dtype == torch.float32 and tuple(frames.shape[1:]) == (224, 224)
    out = torch.empty(frames.shape[0] * 256, ldk, dtype=torch.bfloat16, device=frames.device)
    check(_L().n1_op_patchify_depth(ptr(frames), ptr(out), frames.shape[0], ldk, stream_ptr()))
    return out


def adamw(master, working, grad, m, v, lr, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, step=1):
    check(_L().n1_op_adamw(ptr(master), ptr(working), ptr(grad), ptr(m), ptr(v), master.numel(), lr, betas[0], betas[1], eps,
                           weight_decay, step, stream_ptr()))


# ------------------------------------------------------------------------------------------------ dropout (training)
# `rng`: the device int32 [4] state of internnav_b200.dropout.DropoutRNG; `site`: a site id of that module; 0 < p < 1.
def _rng(rng):
    assert rng.is_cuda and rng.dtype == torch.int32 and rng.numel() == 4 and rng.is_contiguous()
    return c_void_p(rng.data_ptr())


def _flat(t):
    assert t.dtype == torch.bfloat16 and t.is_contiguous(), (t.dtype, t.stride())
    return t


def dropout_add(residual, y, rng, site, p):
    """residual + Z y (bf16, same shape, contiguous)."""
    assert residual.shape == y.shape
    out = torch.empty_like(_flat(y))
    check(_L().n1_op_dropout_add(ptr(_flat(residual)), ptr(y), ptr(out), y.numel(), _rng(rng), site, p, stream_ptr()))
    return out


def dropout(x, rng, site, p):
    """Z x: a dropped tensor, and the backward of every dropout site (Z dy)."""
    out = torch.empty_like(_flat(x))
    check(_L().n1_op_dropout_bwd(ptr(x), ptr(out), x.numel(), _rng(rng), site, p, stream_ptr()))
    return out


def dropout_mask(shape, rng, site, p, device="cuda"):
    """The keep mask of a site as uint8 [shape] (1 = kept)."""
    out = torch.empty(shape, dtype=torch.uint8, device=device)
    check(_L().n1_op_dropout_mask(ptr(out), out.numel(), _rng(rng), site, p, stream_ptr()))
    return out


def act_fwd_dropout(pre, act, rng, site, p):
    out = torch.empty_like(_flat(pre))
    check(_L().n1_op_act_fwd_dropout(ptr(pre), ptr(out), pre.numel(), act, _rng(rng), site, p, stream_ptr()))
    return out


def act_bwd_dropout(pre, dy, act, rng, site, p):
    out = torch.empty_like(_flat(pre))
    check(_L().n1_op_act_bwd_dropout(ptr(pre), ptr(_flat(dy)), ptr(out), pre.numel(), act, _rng(rng), site, p, stream_ptr()))
    return out


def attention_dropout(q, k, v, heads, head_dim, batch, seq_q, seq_k, rng, site, p, causal=False, scale=None):
    """Fixed-length MHA (head_dim 48) with dropout on the probabilities: O = (softmax(S) o Z) V."""
    for t in (q, k, v):
        assert t.is_cuda and t.dtype == torch.bfloat16 and t.stride(1) == 1
    o = torch.empty(q.shape[0], heads * head_dim, device=q.device, dtype=torch.bfloat16)
    scale = head_dim ** -0.5 if scale is None else scale
    vp = lambda t: c_void_p(t.data_ptr())
    check(_L().n1_op_attention_dropout(vp(q), vp(k), vp(v), ptr(o), q.stride(0), k.stride(0), v.stride(0), o.stride(0), heads,
                                       head_dim, batch, seq_q, seq_k, 1 if causal else 0, scale, _rng(rng), site, p,
                                       stream_ptr()))
    return o


def attention_bwd_dropout(q, k, v, o, dout, heads, head_dim, batch, seq_q, seq_k, rng, site, p, causal=False, scale=None):
    """Backward of attention_dropout (the mask recomputed): dq bf16, dk / dv fp32."""
    dq = torch.zeros(q.shape[0], heads * head_dim, dtype=torch.bfloat16, device=q.device)
    dk = torch.zeros(k.shape[0], heads * head_dim, dtype=torch.float32, device=q.device)
    dv = torch.zeros_like(dk)
    scale = head_dim ** -0.5 if scale is None else scale
    for t in (q, k, v, o, dout):
        assert t.is_cuda and t.dtype == torch.bfloat16 and t.stride(1) == 1
    vp = lambda t: c_void_p(t.data_ptr())
    check(_L().n1_op_attention_bwd_dropout(vp(q), vp(k), vp(v), vp(o), vp(dout), ptr(dq), ptr(dk), ptr(dv), q.stride(0),
                                           k.stride(0), v.stride(0), o.stride(0), dout.stride(0), dq.stride(0), heads,
                                           head_dim, batch, seq_q, seq_k, 1 if causal else 0, scale, _rng(rng), site, p,
                                           stream_ptr()))
    return dq, dk, dv
