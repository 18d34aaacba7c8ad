"""System-1 half of the training step (SURVEY.md §8 row a13): forward with saves and hand-scheduled backward of
`forward_vlm_traj` + masked MSE (navdp.py L291-312, internvla_n1.py L287-303), as a sequence of kernel calls.

The schedule follows oracle/navdp_backward.py (the backward specification, equal to the reference's autograd) one
primitive at a time; every matrix product -- forward, dgrad (dY W) and wgrad (dY^T X) -- goes through the tcgen05 GEMM
(`ops.mm_nt`, operands transposed by a kernel where the contraction runs over rows), attention / LayerNorm / GELU / ReLU /
layer-scale forward and backward through the kernels of attention.cu, norm.cu and bwd_kernels.cu.  What stays in PyTorch
is tensor plumbing on bf16 buffers: slicing, concatenation, additions of equally shaped buffers.  The im2col of the
depth frames is the library's patchify kernel (three replicated channels folded into one, as at inference), and the
products too narrow for a tensor-core tile or held in fp32 (the 3-wide action embedding / action head, the 256 x 1369
position-table resample and their gradients) go through the library's small fp32 product (`ops.sgemm`).

`ops` is the kernel backend.  The product backend is `GpuOps` below (ctypes -> libn1b200.so; it refuses to run without
the library / a B200).  tests/test_train_s1_host.py drives this same schedule with a plain fp32 PyTorch implementation of
the `ops` contract on the CPU and checks every gradient against the oracle -- that validates the schedule, not the
kernels.  The kernels are validated on the B200 by tests/test_bwd_ops_gpu.py (op level, System-2 half, and the whole step
against the oracle chain; profiles/r2_bwd_ops_parity.log).

Train-mode dropout (`S1TrainStep(..., dropout=p)`, p > 0): at every site of internnav_b200/dropout.py the schedule calls the
dropout primitives of the backend with `drop = (DropoutRNG, site id, p)` -- `dropout_add` at the residual branches,
`dropout` on the cond / action embeddings and on the gradients flowing back through a site, `act_fwd` / `act_bwd` and
`attention` / `attention_bwd` with a `drop` argument.  With p == 0 the schedule issues exactly the calls it issues without.
"""
import math

import torch
import torch.nn.functional as F

from .dropout import (ACTION, COND, CROSS_PROBS, DROPOUT1, DROPOUT2, DROPOUT3, FF_INNER, SELF_PROBS, DropoutRNG, decoder_site,
                      qformer_site)

ACT_GELU, ACT_RELU = 1, 2


# ------------------------------------------------------------------------------------------------ kernel backend
class GpuOps:
    """The `ops` contract on libn1b200.so.  Activations bf16, parameter gradients fp32, everything on one CUDA device."""
    dtype = torch.bfloat16

    def __init__(self, device="cuda:0"):
        from . import _bwd, _lib
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("n1b200 has no CPU path: GpuOps needs device='cuda:N'")
        self._lib, self._bwd = _lib, _bwd
        _lib.lib()

    def cast(self, t):
        return t.to(self.device, self.dtype).contiguous()

    def mm_nt(self, a, w, bias=None, out_fp32=False):
        """a [M, K] @ w [N, K]^T (+ bias [N] fp32); K % 8 == 0."""
        return self._lib.gemm(a, w, bias=bias, out_fp32=out_fp32)

    def transpose(self, x):
        """[R, C] -> [C, R rounded up to 8] (zero padded): the operand layout of a product contracting over rows."""
        return self._bwd.transpose(x)

    def colsum(self, a, b=None):
        return self._bwd.colsum(a, b)

    def layernorm(self, x, w, b, eps):
        return self._lib.layernorm(x, w, b, eps)

    def norm_bwd(self, dy, x, w, eps):
        return self._bwd.norm_bwd(dy, x, w, eps)

    def attention(self, q, k, v, heads, hd, batch, sq, sk, causal, drop=None):
        if drop is not None:
            rng, site, p = drop
            return self._bwd.attention_dropout(q, k, v, heads, hd, batch, sq, sk, rng.dev, site, p, causal=causal)
        return self._lib.attention(q, k, v, heads, heads, hd, batch, sq, sk, causal=causal)

    def attention_bwd(self, q, k, v, o, do, heads, hd, batch, sq, sk, causal, drop=None):
        if drop is not None:
            rng, site, p = drop
            return self._bwd.attention_bwd_dropout(q, k, v, o, do, heads, hd, batch, sq, sk, rng.dev, site, p, causal=causal)
        return self._bwd.attention_bwd(q, k, v, o, do, heads, heads, hd, batch, sq, sk, causal=causal)

    def act_fwd(self, pre, kind, drop=None):
        if drop is not None:
            return self._bwd.act_fwd_dropout(pre, kind, drop[0].dev, drop[1], drop[2])
        return self._bwd.act_fwd(pre, kind)

    def act_bwd(self, pre, dy, kind, drop=None):
        if drop is not None:
            return self._bwd.act_bwd_dropout(pre, dy, kind, drop[0].dev, drop[1], drop[2])
        return self._bwd.act_bwd(pre, dy, kind)

    def dropout(self, x, drop):
        """Z x: a dropped tensor, or the gradient flowing back through a dropout site."""
        return self._bwd.dropout(x, drop[0].dev, drop[1], drop[2])

    def dropout_add(self, residual, y, drop):
        """residual + Z y: a residual branch with dropout."""
        return self._bwd.dropout_add(residual, y, drop[0].dev, drop[1], drop[2])

    def wgrad(self, dy, x):
        """dy [M, N]^T @ x [M, K] -> fp32 [N, K]: in place on MN-major operand tiles when the rows are aligned
        (csrc/wgrad_tn.cu), else through two operand transposes and the K-major GEMM."""
        if self._bwd.wgrad_supported(dy, x):
            return self._bwd.wgrad(dy, x)
        return self.mm_nt(self.transpose(dy), self.transpose(x), out_fp32=True)

    def sgemm(self, a, b, trans_a=False, trans_b=False):
        """fp32 op(a) @ op(b) on the CUDA cores (narrow / fp32-only products)."""
        return self._bwd.sgemm(a, b, trans_a, trans_b)

    def patchify_depth(self, frames):
        """[n, 224, 224] fp32 -> im2col rows [n * 256, 200] (196 columns + zero padding) in the kernel dtype."""
        return self._bwd.patchify_depth(frames)

    def scale_cols(self, x, gamma, add=None):
        """x * gamma (+ add), per column: LayerScale with the residual add."""
        return self._bwd.scale_cols(x, gamma, add)


# ------------------------------------------------------------------------------------------------ schedule
def _pad8(x):
    k = x.shape[-1]
    return x if k % 8 == 0 else F.pad(x, (0, 8 - k % 8))


class S1TrainStep:
    """params: {reference tensor name: fp32 tensor} (the state_dict keys of NavDP_Policy_DPT_CriticSum_DAT)."""

    def __init__(self, params, ops, heads=8, layers=16, frames=2, K=20, dropout=0.0, rng=None):
        """dropout: the reference's train-mode p (0.1) at every site of internnav_b200/dropout.py; rng: its DropoutRNG (the
        masks of micro-batch rng.step), by default seed 0 on the parameters' device."""
        self.ops, self.heads, self.layers, self.frames, self.K = ops, heads, layers, frames, K
        self.p32 = dict(params)
        self._alias_in_proj()
        self.w = {}           # working copies in the kernel dtype (refresh() after every optimizer step)
        self.refresh()
        self.dropout = float(dropout)
        if not 0.0 <= self.dropout < 1.0:
            raise ValueError("dropout must be in [0, 1)")
        self.rng = rng if rng is not None or self.dropout == 0 else DropoutRNG(0, device=self.w["layernorm.weight"].device)
        self._resample = {}
        self._touched = set()   # tensors that received a gradient in the current step (torch.optim skips the others)

    def refresh(self):
        """Working copies in the kernel dtype, refreshed IN PLACE after the first call: a captured CUDA graph of the step
        (DualSystemTrainer(graph_s1=True)) keeps reading the same buffers."""
        for k, v in self.p32.items():
            if not v.is_floating_point():
                continue
            cur = self.w.get(k)
            if cur is not None and cur.shape == v.shape and cur.device == v.device:
                cur.copy_(v)
            else:
                self.w[k] = self.ops.cast(v)

    # ---- primitives on the backend ----------------------------------------------------------------------------
    def _drop(self, site):
        """The dropout descriptor of a site, or None when the step runs without dropout."""
        return (self.rng, site, self.dropout) if self.dropout > 0 else None

    def _residual(self, x, y, site):
        """x + dropout(y) in the kernel dtype."""
        d = self._drop(site)
        if d is None:
            return self.ops.cast(x.float() + y.float())
        return self.ops.dropout_add(x.contiguous(), y.contiguous(), d)

    def _drop_grad(self, dy, site):
        """The gradient through a dropout site (dy itself without dropout)."""
        d = self._drop(site)
        return dy if d is None else self.ops.dropout(dy.contiguous(), d)

    def _act(self, pre, kind, site):
        d = self._drop(site)
        x = pre.reshape(-1, pre.shape[-1])
        return (self.ops.act_fwd(x, kind) if d is None else self.ops.act_fwd(x, kind, drop=d)).reshape(pre.shape)

    def _act_bwd(self, pre, dy, kind, site):
        d = self._drop(site)
        x, g = pre.reshape(-1, pre.shape[-1]).contiguous(), dy.reshape(-1, pre.shape[-1]).contiguous()
        return self.ops.act_bwd(x, g, kind) if d is None else self.ops.act_bwd(x, g, kind, drop=d)

    def _f32(self, name):
        return self.p32[name].to(self.w[name].device, torch.float32)

    def lin(self, name, x, rows=None):
        """y = x W^T + b for W = params[name + '.weight'] (optionally a row block of it, for packed in_proj)."""
        W, b = self.w[name + ".weight"], self.p32.get(name + ".bias")
        if rows is not None:
            W, b = W[rows], (b[rows] if b is not None else None)
        shp = x.shape
        y = self.ops.mm_nt(_pad8(x.reshape(-1, shp[-1])), _pad8(W), bias=None if b is None else b.to(W.device, torch.float32))
        return y.reshape(*shp[:-1], W.shape[0])

    def lin_bwd(self, name, x, dy, g, rows=None, need_dx=True):
        """wgrad dW = dy^T x and db = colsum(dy) into g (fp32), dgrad dx = dy W."""
        W = self.w[name + ".weight"]
        if rows is not None:
            W = W[rows]
        dy2, x2 = dy.reshape(-1, dy.shape[-1]), x.reshape(-1, x.shape[-1])
        dW = self.ops.wgrad(dy2, x2)                                        # [N, K] fp32
        self._acc(g, name + ".weight", dW, rows)
        if (name + ".bias") in self.p32:
            self._acc(g, name + ".bias", self.ops.colsum(dy2), rows)
        if not need_dx:
            return None
        Wt = self.ops.transpose(W)                                          # [K, Np]
        return self.ops.mm_nt(_pad8(dy2), Wt).reshape(*dy.shape[:-1], W.shape[1])

    def _acc(self, g, name, val, rows=None):
        full = self.p32[name]
        if name not in g:   # `g` may arrive pre-populated with views into the all-reduce buckets (forward_backward)
            g[name] = torch.zeros(full.shape, dtype=torch.float32, device=val.device)
        self._touched.add(name)
        tgt = g[name] if rows is None else g[name][rows]
        tgt += val.reshape(tgt.shape).float()

    def ln(self, name, x, eps):
        shp = x.shape
        y = self.ops.layernorm(x.reshape(-1, shp[-1]), self._f32(name + ".weight"), self._f32(name + ".bias"), eps)
        return y.reshape(shp)

    def ln_bwd(self, name, x, dy, g, eps):
        shp = x.shape
        dx, dw, db = self.ops.norm_bwd(dy.reshape(-1, shp[-1]).contiguous(), x.reshape(-1, shp[-1]).contiguous(),
                                       self._f32(name + ".weight"), eps)
        self._acc(g, name + ".weight", dw)
        self._acc(g, name + ".bias", db)
        return dx.reshape(shp)

    def mha(self, name, q_in, kv_in, causal=False, site=None):
        """nn.MultiheadAttention with packed in_proj; q_in [B, Sq, D], kv_in [B, Sk, D] (kv_in is q_in for self-attention)."""
        D = q_in.shape[-1]
        B, Sq, Sk = q_in.shape[0], q_in.shape[1], kv_in.shape[1]
        if kv_in is q_in:
            qkv = self.lin(name + ".in_proj", q_in).reshape(B * Sq, 3 * D)
            q, k, v = qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:]
        else:
            q = self.lin(name + ".in_proj", q_in, rows=slice(0, D)).reshape(B * Sq, D)
            kv = self.lin(name + ".in_proj", kv_in, rows=slice(D, 3 * D)).reshape(B * Sk, 2 * D)
            k, v = kv[:, :D], kv[:, D:]
        d = None if site is None else self._drop(site)
        if d is None:
            o = self.ops.attention(q, k, v, self.heads, D // self.heads, B, Sq, Sk, causal)
        else:
            o = self.ops.attention(q, k, v, self.heads, D // self.heads, B, Sq, Sk, causal, drop=d)
        y = self.lin(name + ".out_proj", o.reshape(B, Sq, D))
        return y, (q_in, kv_in, q, k, v, o, causal, d)

    def mha_bwd(self, name, saved, dy, g):
        q_in, kv_in, q, k, v, o, causal, d = saved
        D = q_in.shape[-1]
        B, Sq, Sk = q_in.shape[0], q_in.shape[1], kv_in.shape[1]
        do = self.lin_bwd(name + ".out_proj", o.reshape(B, Sq, D), dy, g).reshape(B * Sq, D).contiguous()
        if d is None:
            dq, dk, dv = self.ops.attention_bwd(q, k, v, o, do, self.heads, D // self.heads, B, Sq, Sk, causal)
        else:
            dq, dk, dv = self.ops.attention_bwd(q, k, v, o, do, self.heads, D // self.heads, B, Sq, Sk, causal, drop=d)
        dk, dv = dk.to(dq.dtype), dv.to(dq.dtype)
        if kv_in is q_in:
            dqkv = torch.cat((dq, dk, dv), dim=1).reshape(B, Sq, 3 * D)
            dx = self.lin_bwd(name + ".in_proj", q_in, dqkv, g)
            return dx, None
        dxq = self.lin_bwd(name + ".in_proj", q_in, dq.reshape(B, Sq, D), g, rows=slice(0, D))
        dkv = torch.cat((dk, dv), dim=1).reshape(B, Sk, 2 * D)
        dxkv = self.lin_bwd(name + ".in_proj", kv_in, dkv, g, rows=slice(D, 3 * D))
        return dxq, dxkv

    # nn.MultiheadAttention stores its packed projection as in_proj_weight / in_proj_bias (no ".weight" suffix)
    def _alias_in_proj(self):
        for k in list(self.p32):
            if k.endswith("in_proj_weight"):
                self.p32[k[:-len("in_proj_weight")] + "in_proj.weight"] = self.p32[k]
            elif k.endswith("in_proj_bias"):
                self.p32[k[:-len("in_proj_bias")] + "in_proj.bias"] = self.p32[k]

    # ---- DINOv2 ViT-S (depth branch; dinov2.py L180-322) ------------------------------------------------------
    def _R(self, src_side, dst_side, device):
        key = (src_side, dst_side, str(device))     # cached ON the device: a host copy could not be read under graph capture
        if key not in self._resample:
            n = src_side * src_side
            eye = torch.eye(n).reshape(n, 1, src_side, src_side)
            s = float(dst_side + 0.1) / src_side
            r = F.interpolate(eye, scale_factor=(s, s), mode="bicubic", antialias=False).reshape(n, -1).t().contiguous()
            self._resample[key] = r.to(device)
        return self._resample[key]

    def vit_fwd(self, p, frames):
        """frames: [n, 224, 224] fp32 depth frames.  The reference feeds the ViT three identical channels
        (navdp_backbone.py L176-181); the im2col keeps one and the patch-embed weight is summed over its channel axis."""
        ops, n = self.ops, frames.shape[0]
        patches = ops.patchify_depth(frames.float().contiguous())                               # [n * 256, 200]
        Wp = self.p32[p + "patch_embed.proj.weight"]
        Wf = ops.cast(_pad8(Wp.sum(1).reshape(Wp.shape[0], -1)).to(patches.device))              # [D, 196 -> 200]
        t = ops.mm_nt(patches, Wf, bias=self._f32(p + "patch_embed.proj.bias")).reshape(n, 256, -1)
        pe = self._f32(p + "pos_embed")
        src_side = int(math.isqrt(pe.shape[1] - 1))
        R = None if src_side == 16 else self._R(src_side, 16, pe.device)
        pe_patch = pe[0, 1:] if R is None else ops.sgemm(R, pe[0, 1:].contiguous())
        pos = torch.cat((pe[:, :1], pe_patch.unsqueeze(0)), dim=1)
        cls = self._f32(p + "cls_token").expand(n, -1, -1)
        t = ops.cast(torch.cat((cls, t.float()), dim=1) + pos)
        C, tape = t.shape[-1], []
        for i in range(12):
            b = "%sblocks.%d." % (p, i)
            h = self.ln(b + "norm1", t, 1e-6)
            qkv = self.lin(b + "attn.qkv", h).reshape(n * 257, 3 * C)
            q, k, v = qkv[:, :C], qkv[:, C:2 * C], qkv[:, 2 * C:]
            o = ops.attention(q, k, v, 6, C // 6, n, 257, 257, False)
            a = self.lin(b + "attn.proj", o.reshape(n, 257, C))
            t_mid = ops.scale_cols(a.reshape(-1, C), self._f32(b + "ls1.gamma"), t.reshape(-1, C)).reshape(t.shape)
            h2 = self.ln(b + "norm2", t_mid, 1e-6)
            f1 = self.lin(b + "mlp.fc1", h2)
            act = ops.act_fwd(f1.reshape(-1, f1.shape[-1]), ACT_GELU).reshape(f1.shape)
            f2 = self.lin(b + "mlp.fc2", act)
            t_out = ops.scale_cols(f2.reshape(-1, C), self._f32(b + "ls2.gamma"), t_mid.reshape(-1, C)).reshape(t.shape)
            tape.append((t, h, q, k, v, o, a, t_mid, h2, f1, act, f2))
            t = t_out
        y = self.ln(p + "norm", t, 1e-6)
        return y[:, 1:], (patches, R, tape, t, n)

    def vit_bwd(self, p, saved, dy, g):
        ops = self.ops
        patches, R, tape, t_last, n = saved
        C = dy.shape[-1]
        dyf = torch.cat((torch.zeros_like(dy[:, :1]), dy), dim=1)
        dt = self.ln_bwd(p + "norm", t_last, dyf, g, 1e-6)
        for i in reversed(range(12)):
            b = "%sblocks.%d." % (p, i)
            t_in, h, q, k, v, o, a, t_mid, h2, f1, act, f2 = tape[i]
            self._acc(g, b + "ls2.gamma", ops.colsum(dt.reshape(-1, C).contiguous(), f2.reshape(-1, C).contiguous()))
            df2 = ops.scale_cols(dt.reshape(-1, C), self._f32(b + "ls2.gamma")).reshape(dt.shape)
            dact = self.lin_bwd(b + "mlp.fc2", act, df2, g)
            df1 = ops.act_bwd(f1.reshape(-1, f1.shape[-1]).contiguous(), dact.reshape(-1, f1.shape[-1]).contiguous(), ACT_GELU)
            dh2 = self.lin_bwd(b + "mlp.fc1", h2, df1.reshape(f1.shape), g)
            dt = ops.cast(dt.float() + self.ln_bwd(b + "norm2", t_mid, dh2, g, 1e-6).float())
            self._acc(g, b + "ls1.gamma", ops.colsum(dt.reshape(-1, C).contiguous(), a.reshape(-1, C).contiguous()))
            da = ops.scale_cols(dt.reshape(-1, C), self._f32(b + "ls1.gamma")).reshape(dt.shape)
            do = self.lin_bwd(b + "attn.proj", o.reshape(n, 257, C), da, g).reshape(n * 257, C).contiguous()
            dq, dk, dv = ops.attention_bwd(q, k, v, o, do, 6, C // 6, n, 257, 257, False)
            dqkv = torch.cat((dq, dk.to(dq.dtype), dv.to(dq.dtype)), dim=1).reshape(n, 257, 3 * C)
            dh = self.lin_bwd(b + "attn.qkv", h, dqkv, g)
            dt = ops.cast(dt.float() + self.ln_bwd(b + "norm1", t_in, dh, g, 1e-6).float())
        dtf = dt.float()
        self._acc(g, p + "cls_token", dtf[:, :1].sum(0, keepdim=True))
        dpe_patch = dtf[:, 1:].sum(0).contiguous()
        dpe = torch.cat((dtf[:, :1].sum(0), dpe_patch if R is None else ops.sgemm(R, dpe_patch, trans_a=True)), dim=0).unsqueeze(0)
        self._acc(g, p + "pos_embed", dpe)
        dpatch = dt[:, 1:].reshape(-1, C).contiguous()
        Wp = self.p32[p + "patch_embed.proj.weight"]
        dWf = ops.wgrad(dpatch, patches)[:, :196]                                                # [D, 196], one channel
        # the three input channels are identical, so each channel of the Conv2d weight receives the same gradient
        self._acc(g, p + "patch_embed.proj.weight", dWf.reshape(Wp.shape[0], 1, 14, 14).expand(Wp.shape))
        self._acc(g, p + "patch_embed.proj.bias", ops.colsum(dpatch))

    # ---- Q-former layer (post-norm, ReLU; navdp_backbone.py L148) ---------------------------------------------
    def post_layer(self, p, x, mem, layer=0):
        site = lambda off: qformer_site(layer, off)                                       # noqa: E731
        a1, m1 = self.mha(p + "self_attn", x, x, site=site(SELF_PROBS))
        s1 = self._residual(x, a1, site(DROPOUT1))
        x1 = self.ln(p + "norm1", s1, 1e-5)
        a2, m2 = self.mha(p + "multihead_attn", x1, mem, site=site(CROSS_PROBS))
        s2 = self._residual(x1, a2, site(DROPOUT2))
        x2 = self.ln(p + "norm2", s2, 1e-5)
        f1 = self.lin(p + "linear1", x2)
        act = self._act(f1, ACT_RELU, site(FF_INNER))
        f2 = self.lin(p + "linear2", act)
        s3 = self._residual(x2, f2, site(DROPOUT3))
        return self.ln(p + "norm3", s3, 1e-5), (m1, s1, m2, s2, x2, f1, act, s3, layer)

    def post_layer_bwd(self, p, saved, dy, g):
        ops = self.ops
        m1, s1, m2, s2, x2, f1, act, s3, layer = saved
        site = lambda off: qformer_site(layer, off)                                       # noqa: E731
        d = self.ln_bwd(p + "norm3", s3, dy, g, 1e-5)
        dact = self.lin_bwd(p + "linear2", act, self._drop_grad(d, site(DROPOUT3)), g)
        df1 = self._act_bwd(f1, dact, ACT_RELU, site(FF_INNER))
        dx2 = ops.cast(d.float() + self.lin_bwd(p + "linear1", x2, df1.reshape(f1.shape), g).float())
        d = self.ln_bwd(p + "norm2", s2, dx2, g, 1e-5)
        dq, dmem = self.mha_bwd(p + "multihead_attn", m2, self._drop_grad(d, site(DROPOUT2)), g)
        dx1 = ops.cast(d.float() + dq.float())
        d = self.ln_bwd(p + "norm1", s1, dx1, g, 1e-5)
        dq, _ = self.mha_bwd(p + "self_attn", m1, self._drop_grad(d, site(DROPOUT1)), g)
        return ops.cast(d.float() + dq.float()), dmem

    # ---- model pieces ------------------------------------------------------------------------------------------
    def rgbd_fwd(self, rgb_tokens, depths, rgb_has_pe=False):
        """rgb_tokens: [B, T*256, D] from the frozen RGB ViT (detached in the reference, navdp_backbone.py L170-171);
        `rgb_has_pe`: they already carry former_pe (n1_rgb_tokens delivers them that way); depths [B, T, 224, 224, 1]."""
        ops, p = self.ops, "rgbd_encoder."
        B, T = depths.shape[:2]
        dtok, vsave = self.vit_fwd(p + "depth_model.", depths.reshape(-1, 224, 224))
        pe = self._f32(p + "former_pe.weight")[: self.frames * 512].clone()
        if rgb_has_pe:
            pe[: T * 256] = 0
        token = ops.cast(torch.cat((rgb_tokens.float(), dtok.reshape(B, T * 256, -1).float()), dim=1) + pe)
        x = ops.cast(self._f32(p + "former_query.weight")[: self.frames * 16].unsqueeze(0).expand(B, -1, -1))
        tape = []
        for i in range(2):
            x, s = self.post_layer("%sformer_net.layers.%d." % (p, i), x, token, layer=i)
            tape.append(s)
        return self.lin(p + "project_layer", x), (vsave, tape, x, B, T)

    def rgbd_bwd(self, saved, dy, g):
        p = "rgbd_encoder."
        vsave, tape, x_last, B, T = saved
        d = self.lin_bwd(p + "project_layer", x_last, dy, g)
        dtoken = 0
        for i in reversed(range(2)):
            d, dm = self.post_layer_bwd("%sformer_net.layers.%d." % (p, i), tape[i], d, g)
            dtoken = dtoken + dm.float()
        gq = torch.zeros_like(self.p32[p + "former_query.weight"], dtype=torch.float32, device=d.device)
        gq[: self.frames * 16] = d.float().sum(0)
        self._acc(g, p + "former_query.weight", gq)
        gpe = torch.zeros_like(self.p32[p + "former_pe.weight"], dtype=torch.float32, device=d.device)
        gpe[: self.frames * 512] = dtoken.sum(0)
        self._acc(g, p + "former_pe.weight", gpe)
        ddepth = self.ops.cast(dtoken[:, T * 256:].reshape(B * T, 256, -1))
        self.vit_bwd(p + "depth_model.", vsave, ddepth, g)

    def goal_fwd(self, vlm_tokens):
        ops, c = self.ops, "goal_compressor."
        x0 = ops.cast(vlm_tokens)
        h0 = self.lin("vlm_embed_mlp.0", x0)
        a0 = ops.act_fwd(h0.reshape(-1, h0.shape[-1]), ACT_RELU).reshape(h0.shape)
        h1 = self.lin("vlm_embed_mlp.2", a0)
        a1 = ops.act_fwd(h1.reshape(-1, h1.shape[-1]), ACT_RELU).reshape(h1.shape)
        h2 = self.lin("vlm_embed_mlp.4", a1)
        B, n, _ = h2.shape
        x = ops.cast(h2.float() + self._f32(c + "token_positional_encoding.position_embedding.weight")[:n])
        q = self._f32(c + "target_embedding.weight") + self._f32(c + "query_positional_encoding.position_embedding.weight")[:1]
        q = ops.cast(q.unsqueeze(0).expand(B, -1, -1))
        y, m = self.mha(c + "cross_attention", q, x)
        return y, (x0, h0, a0, h1, a1, m, n)

    def goal_bwd(self, saved, dy, g):
        ops, c = self.ops, "goal_compressor."
        x0, h0, a0, h1, a1, m, n = saved
        dq, dx = self.mha_bwd(c + "cross_attention", m, dy, g)
        dqs = dq.float().sum(0)
        self._acc(g, c + "target_embedding.weight", dqs)
        gqp = torch.zeros_like(self.p32[c + "query_positional_encoding.position_embedding.weight"], dtype=torch.float32, device=dqs.device)
        gqp[:1] = dqs
        self._acc(g, c + "query_positional_encoding.position_embedding.weight", gqp)
        gtp = torch.zeros_like(self.p32[c + "token_positional_encoding.position_embedding.weight"], dtype=torch.float32, device=dqs.device)
        gtp[:n] = dx.float().sum(0)
        self._acc(g, c + "token_positional_encoding.position_embedding.weight", gtp)
        d = self.lin_bwd("vlm_embed_mlp.4", a1, dx, g)
        d = ops.act_bwd(h1.reshape(-1, h1.shape[-1]).contiguous(), d.reshape(-1, h1.shape[-1]).contiguous(), ACT_RELU).reshape(h1.shape)
        d = self.lin_bwd("vlm_embed_mlp.2", a0, d, g)
        d = ops.act_bwd(h0.reshape(-1, h0.shape[-1]).contiguous(), d.reshape(-1, h0.shape[-1]).contiguous(), ACT_RELU).reshape(h0.shape)
        return self.lin_bwd("vlm_embed_mlp.0", x0, d, g)

    def decoder_fwd(self, noisy, timesteps, goal, rgbd):
        ops = self.ops
        R, T, _ = noisy.shape
        B = goal.shape[0]
        Ns = R // B
        # the 3 -> D action embedding is too narrow for a tensor-core tile: the small fp32 product, then the kernel dtype
        x = ops.sgemm(noisy.float().reshape(-1, 3).contiguous(), self._f32("input_embed.weight"), trans_b=True).reshape(R, T, -1) \
            + self._f32("input_embed.bias")
        half = 192
        freq = torch.exp(torch.arange(half, device=x.device) * -(math.log(10000) / (half - 1)))
        te = timesteps.to(x.device)[:, None].float() * freq[None, :]
        time_emb = torch.cat((te.sin(), te.cos()), dim=-1).unsqueeze(1)
        M = 2 + rgbd.shape[1]
        cond = torch.cat([time_emb, goal.float(), rgbd.float()], dim=1) + self._f32("cond_pos_embed")[:, :M]
        cond = ops.cast(cond.repeat_interleave(Ns, dim=0))
        x = ops.cast(x + self._f32("out_pos_embed")[:, :T])
        if self.dropout > 0:        # NavDP.drop on the condition and action embeddings (navdp.py L305-307)
            cond, x = ops.dropout(cond, self._drop(COND)), ops.dropout(x, self._drop(ACTION))
        tape = []
        for i in range(self.layers):
            p = "decoder.layers.%d." % i
            site = lambda off: decoder_site(i, off)                                        # noqa: E731
            h1 = self.ln(p + "norm1", x, 1e-5)
            a1, m1 = self.mha(p + "self_attn", h1, h1, causal=True, site=site(SELF_PROBS))
            x1 = self._residual(x, a1, site(DROPOUT1))
            h2 = self.ln(p + "norm2", x1, 1e-5)
            a2, m2 = self.mha(p + "multihead_attn", h2, cond, site=site(CROSS_PROBS))
            x2 = self._residual(x1, a2, site(DROPOUT2))
            h3 = self.ln(p + "norm3", x2, 1e-5)
            f1 = self.lin(p + "linear1", h3)
            act = self._act(f1, ACT_GELU, site(FF_INNER))
            f2 = self.lin(p + "linear2", act)
            tape.append((x, m1, x1, m2, x2, h3, f1, act))
            x = self._residual(x2, f2, site(DROPOUT3))
        hN = self.ln("layernorm", x, 1e-5)
        y = ops.sgemm(hN.float().reshape(-1, hN.shape[-1]), self._f32("action_head.weight"), trans_b=True).reshape(R, T, 3) \
            + self._f32("action_head.bias")                                                      # D -> 3
        return y, (noisy, tape, x, hN, B, Ns, M, T)

    def decoder_bwd(self, saved, dy, g):
        ops = self.ops
        noisy, tape, x_last, hN, B, Ns, M, T = saved
        dy2 = dy.reshape(-1, 3).float().contiguous()
        self._acc(g, "action_head.weight", ops.sgemm(dy2, hN.float().reshape(-1, hN.shape[-1]), trans_a=True))
        self._acc(g, "action_head.bias", dy2.sum(0))
        dx = self.ln_bwd("layernorm", x_last, ops.cast(ops.sgemm(dy2, self._f32("action_head.weight")).reshape(hN.shape)), g, 1e-5)
        dcond = 0
        for i in reversed(range(self.layers)):
            p = "decoder.layers.%d." % i
            x, m1, x1, m2, x2, h3, f1, act = tape[i]
            site = lambda off: decoder_site(i, off)                                        # noqa: E731
            dact = self.lin_bwd(p + "linear2", act, self._drop_grad(dx, site(DROPOUT3)), g)
            df1 = self._act_bwd(f1, dact, ACT_GELU, site(FF_INNER))
            dh3 = self.lin_bwd(p + "linear1", h3, df1.reshape(f1.shape), g)
            dx = ops.cast(dx.float() + self.ln_bwd(p + "norm3", x2, dh3, g, 1e-5).float())
            dq, dkv = self.mha_bwd(p + "multihead_attn", m2, self._drop_grad(dx, site(DROPOUT2)), g)
            dcond = dcond + dkv.float()
            dx = ops.cast(dx.float() + self.ln_bwd(p + "norm2", x1, dq, g, 1e-5).float())
            dq, _ = self.mha_bwd(p + "self_attn", m1, self._drop_grad(dx, site(DROPOUT1)), g)
            dx = ops.cast(dx.float() + self.ln_bwd(p + "norm1", x, dq, g, 1e-5).float())
        if self.dropout > 0:
            dx = ops.dropout(dx.contiguous(), self._drop(ACTION))
            dcond = ops.dropout(ops.cast(dcond), self._drop(COND)).float()
        dxf = dx.float()
        gop = torch.zeros_like(self.p32["out_pos_embed"], dtype=torch.float32, device=dxf.device)
        gop[:, :T] = dxf.sum(0, keepdim=True)
        self._acc(g, "out_pos_embed", gop)
        self._acc(g, "input_embed.weight", ops.sgemm(dxf.reshape(-1, dxf.shape[-1]).contiguous(),
                                                    noisy.float().reshape(-1, 3).contiguous(), trans_a=True))
        self._acc(g, "input_embed.bias", dxf.reshape(-1, dxf.shape[-1]).sum(0))
        dcond = dcond.reshape(B, Ns, M, -1).sum(1)
        gcp = torch.zeros_like(self.p32["cond_pos_embed"], dtype=torch.float32, device=dxf.device)
        gcp[:, :M] = dcond.sum(0, keepdim=True)
        self._acc(g, "cond_pos_embed", gcp)
        return ops.cast(dcond[:, 1:2]), ops.cast(dcond[:, 2:])

    # ---- the step ----------------------------------------------------------------------------------------------
    def forward_backward(self, traj_hidden_states, rgb_tokens, traj_depths, traj_poses, video_frame_num, noise, timesteps,
                         alphas_cumprod, rgb_has_pe=False, grads_into=None):
        """-> (loss, {name: fp32 gradient}, d loss / d traj_hidden_states [B, n_query, H]).
        rgb_tokens: [B*f, 2*256, D] RGB-ViT tokens of the [goal frame, current frame] pairs (frozen branch);
        traj_depths [B, f, 224, 224]; alphas_cumprod fp32 [K] (DDPMScheduler table, n1_ddpm_tables).
        grads_into: {reference tensor name: fp32 view}, e.g. the views into the all-reduce buckets (ddp.GradientBuckets):
        the gradients are ACCUMULATED there (the caller zeroes them), so nothing is copied or re-flattened afterwards."""
        dev = self.w["layernorm.weight"].device
        Bb, f = traj_depths.shape[:2]
        hs = traj_hidden_states.to(dev).unsqueeze(1).repeat(1, f, 1, 1).flatten(0, 1)
        if video_frame_num.device.type == "cuda":   # device-resident counts: no host round trip (CUDA-graph capturable)
            mask = (torch.arange(f, device=dev).expand(Bb, f) < video_frame_num.to(dev).unsqueeze(1))
            mask = mask.flatten(0, 1)[:, None, None].float()
        else:
            mask = (torch.arange(f).expand(Bb, f) < video_frame_num.cpu().unsqueeze(1)).flatten(0, 1)[:, None, None].float().to(dev)
        cur_d = traj_depths.to(dev).flatten(0, 1)
        g_d = traj_depths.to(dev)[:, 0:1].repeat(1, f, 1, 1).flatten(0, 1)
        depths_dp = torch.stack([g_d, cur_d], dim=1).unsqueeze(-1)
        poses = traj_poses.to(dev).flatten(0, 1).float()
        noise, timesteps = noise.to(dev).float(), timesteps.to(dev)
        acp = alphas_cumprod.to(dev)[timesteps]
        noisy = acp.sqrt()[:, None, None] * poses + (1 - acp).sqrt()[:, None, None] * noise       # add_noise, navdp.py L173
        goal, gsave = self.goal_fwd(hs)
        rgbd, rsave = self.rgbd_fwd(rgb_tokens.to(dev), depths_dp, rgb_has_pe)
        pred, dsave = self.decoder_fwd(noisy, timesteps, goal, rgbd)
        err = pred - noise
        denom = mask.sum() * err.shape[1] * err.shape[2]
        loss = (err.square() * mask).sum() / denom
        g = {}
        self._touched = set()
        if grads_into is not None:
            for k, view in grads_into.items():
                g[k.replace("in_proj_weight", "in_proj.weight").replace("in_proj_bias", "in_proj.bias")] = view
        dgoal, drgbd = self.decoder_bwd(dsave, 2.0 * err * mask / denom, g)
        self.rgbd_bwd(rsave, drgbd, g)
        dhs = self.goal_bwd(gsave, dgoal, g)
        grads = {}
        for k, v in g.items():   # report under the reference's tensor names
            k2 = k.replace("in_proj.weight", "in_proj_weight").replace("in_proj.bias", "in_proj_bias")
            if k in self._touched and (grads_into is None or k2 in grads_into):
                grads[k2] = v
        return loss, grads, dhs.float().reshape(Bb, f, *dhs.shape[1:]).sum(1)
