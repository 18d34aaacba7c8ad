"""Hand-written backward of the System-1 training loss in the reference's train() mode -- TEST INFRASTRUCTURE: the
specification of the dropout schedule of internnav_b200/train_s1.py.

oracle/navdp_backward.py with dropout: `masks(site, shape)` gives the multiplier of each dropout site (0 dropped,
1 / (1 - p) kept; site ids of internnav_b200/dropout.py), as in oracle/navdp_oracle_train.py.  A dropout multiplies the
value going forward and the gradient coming back by the same multiplier.  Attention with dropout on the probabilities,
o = (p o z) v:  dv = (p o z)^T do,  dp = (do v^T) o z,  and the softmax backward unchanged.  Everything without dropout
(linear, LayerNorm, GELU, the depth ViT, the goal compressor) is navdp_backward's own code.  tests/test_dropout_host.py
checks this file against autograd through navdp_oracle_train.
"""
import math

import torch
import torch.nn.functional as F

from . import ddpm
from . import navdp_backward as NB
from . import navdp_oracle as O


def _z(masks, site, shape):
    return masks(site, tuple(shape)).float()


def attn_core_fwd(q, k, v, causal, scale, z):
    s = (q @ k.transpose(-1, -2)) * scale
    if causal:
        s = s.masked_fill(torch.triu(torch.ones(s.shape[-2], s.shape[-1], dtype=torch.bool), diagonal=1), float("-inf"))
    p = s.softmax(-1)
    return (p * z) @ v, p


def attn_core_bwd(q, k, v, p, do, scale, z):
    dv = (p * z).transpose(-1, -2) @ do
    dp = (do @ v.transpose(-1, -2)) * z
    ds = p * (dp - (dp * p).sum(-1, keepdim=True))      # sum_j p dp = do . o: the D of the kernels
    return (ds @ k) * scale, (ds.transpose(-1, -2) @ q) * scale, dv


def mha_fwd(sd, p, q_in, k_in, v_in, heads, z, causal=False):
    D = q_in.shape[-1]
    w, b = sd[p + ".in_proj_weight"], sd[p + ".in_proj_bias"]
    q, k, v = F.linear(q_in, w[:D], b[:D]), F.linear(k_in, w[D:2 * D], b[D:2 * D]), F.linear(v_in, w[2 * D:], b[2 * D:])
    B, Sq, hd = q.shape[0], q.shape[1], D // heads
    qh, kh, vh = (t.view(B, -1, heads, hd).transpose(1, 2) for t in (q, k, v))
    oh, prob = attn_core_fwd(qh, kh, vh, causal, 1.0 / math.sqrt(hd), z)
    o = oh.transpose(1, 2).reshape(B, Sq, D)
    y = F.linear(o, sd[p + ".out_proj.weight"], sd[p + ".out_proj.bias"])
    return y, (q_in, k_in, v_in, qh, kh, vh, prob, o, z)


def mha_bwd(sd, p, saved, dy, g, heads):
    q_in, k_in, v_in, qh, kh, vh, prob, o, z = saved
    D = q_in.shape[-1]
    hd = D // heads
    dy2 = dy.reshape(-1, D)
    g.add(p + ".out_proj.weight", dy2.t() @ o.reshape(-1, D))
    g.add(p + ".out_proj.bias", dy2.sum(0))
    do = (dy @ sd[p + ".out_proj.weight"]).view(dy.shape[0], -1, heads, hd).transpose(1, 2)
    dqh, dkh, dvh = attn_core_bwd(qh, kh, vh, prob, do, 1.0 / math.sqrt(hd), z)
    dq, dk, dv = (t.transpose(1, 2).reshape(t.shape[0], -1, D) for t in (dqh, dkh, dvh))
    w = sd[p + ".in_proj_weight"]
    g.add(p + ".in_proj_weight", torch.cat([dq.reshape(-1, D).t() @ q_in.reshape(-1, D), dk.reshape(-1, D).t() @ k_in.reshape(-1, D),
                                            dv.reshape(-1, D).t() @ v_in.reshape(-1, D)]))
    g.add(p + ".in_proj_bias", torch.cat([dq.reshape(-1, D).sum(0), dk.reshape(-1, D).sum(0), dv.reshape(-1, D).sum(0)]))
    return dq @ w[:D], dk @ w[D:2 * D], dv @ w[2 * D:]


def _layer_masks(sd, p, masks, site0, R, heads, S, Sk, x_shape):
    shapes = ((R, heads, S, S), x_shape, (R, heads, S, Sk), x_shape, (R, S, sd[p + "linear1.weight"].shape[0]), x_shape)
    return [_z(masks, site0 + off, sh) for off, sh in enumerate(shapes)]


# ------------------------------------------------------------------------------------------------ Q-former (post-norm)
def _post_layer_fwd(sd, p, x, mem, heads, masks, site0):
    zs = _layer_masks(sd, p, masks, site0, x.shape[0], heads, x.shape[1], mem.shape[1], x.shape)
    a1, m1 = mha_fwd(sd, p + "self_attn", x, x, x, heads, zs[0])
    x1, n1 = NB.ln_fwd(sd, p + "norm1", x + a1 * zs[1], 1e-5)
    a2, m2 = mha_fwd(sd, p + "multihead_attn", x1, mem, mem, heads, zs[2])
    x2, n2 = NB.ln_fwd(sd, p + "norm2", x1 + a2 * zs[3], 1e-5)
    f1, _ = NB.lin_fwd(sd, p + "linear1", x2)
    f2, _ = NB.lin_fwd(sd, p + "linear2", F.relu(f1) * zs[4])
    x3, n3 = NB.ln_fwd(sd, p + "norm3", x2 + f2 * zs[5], 1e-5)
    return x3, (m1, n1, m2, n2, x2, f1, n3, zs)


def _post_layer_bwd(sd, p, saved, dy, g, heads):
    m1, n1, m2, n2, x2, f1, n3, zs = saved
    d = NB.ln_bwd(sd, p + "norm3", n3, dy, g)
    dact = NB.lin_bwd(sd, p + "linear2", F.relu(f1) * zs[4], d * zs[5], g)
    dx2 = d + NB.lin_bwd(sd, p + "linear1", x2, dact * zs[4] * (f1 > 0), g)
    d = NB.ln_bwd(sd, p + "norm2", n2, dx2, g)
    dq, dk, dv = mha_bwd(sd, p + "multihead_attn", m2, d * zs[3], g, heads)
    dx1, dmem = d + dq, dk + dv
    d = NB.ln_bwd(sd, p + "norm1", n1, dx1, g)
    dq, dk, dv = mha_bwd(sd, p + "self_attn", m1, d * zs[1], g, heads)
    return d + dq + dk + dv, dmem


def rgbd_fwd(sd, images, depths, masks, frames=2, p="rgbd_encoder."):
    B, T = images.shape[:2]
    with torch.no_grad():  # the RGB tokens are detached in the reference (navdp_backbone.py L170-171)
        mean = torch.tensor([0.485, 0.456, 0.406], dtype=torch.bfloat16).float().reshape(1, 3, 1, 1)
        std = torch.tensor([0.229, 0.224, 0.225], dtype=torch.bfloat16).float().reshape(1, 3, 1, 1)
        ti = images.permute(0, 1, 4, 2, 3).reshape(-1, 3, 224, 224)
        image_token = O.dinov2_vits(sd, p + "rgb_model.", (ti - mean) / std).reshape(B, T * 256, -1)
    td = depths.permute(0, 1, 4, 2, 3).reshape(-1, 1, 224, 224)
    dtok, vsave = NB.vit_fwd(sd, p + "depth_model.", torch.cat([td, td, td], dim=1))
    token = torch.cat((image_token, dtok.reshape(B, T * 256, -1)), dim=1) + sd[p + "former_pe.weight"][: frames * 512]
    x = sd[p + "former_query.weight"][: frames * 16].unsqueeze(0).expand(B, -1, -1)
    tape = []
    for i in range(2):
        x, s = _post_layer_fwd(sd, "%sformer_net.layers.%d." % (p, i), x, token, 8, masks, 256 + 8 * i)
        tape.append(s)
    y, _ = NB.lin_fwd(sd, p + "project_layer", x)
    return y, (vsave, tape, x, B, T, frames)


def rgbd_bwd(sd, saved, dy, g, p="rgbd_encoder."):
    vsave, tape, x_last, B, T, frames = saved
    d = NB.lin_bwd(sd, p + "project_layer", x_last, dy, g)
    dtoken = 0
    for i in reversed(range(2)):
        d, dm = _post_layer_bwd(sd, "%sformer_net.layers.%d." % (p, i), tape[i], d, g, 8)
        dtoken = dtoken + dm
    gq = torch.zeros_like(sd[p + "former_query.weight"])
    gq[: frames * 16] = d.sum(0)
    g.add(p + "former_query.weight", gq)
    gpe = torch.zeros_like(sd[p + "former_pe.weight"])
    gpe[: frames * 512] = dtoken.sum(0)
    g.add(p + "former_pe.weight", gpe)
    NB.vit_bwd(sd, p + "depth_model.", vsave, dtoken[:, T * 256:].reshape(B * T, 256, -1), g)


# ------------------------------------------------------------------------------------------------ decoder (pre-norm)
def decoder_fwd(sd, noisy, timestep, goal, rgbd, masks, layers=16, heads=8):
    R, T, _ = noisy.shape
    B = goal.shape[0]
    Ns = R // B
    x, _ = NB.lin_fwd(sd, "input_embed", noisy)
    M = 2 + rgbd.shape[1]
    cond = (torch.cat([O.sinusoidal_pos_emb(timestep).unsqueeze(1), goal, rgbd], dim=1)
            + sd["cond_pos_embed"][:, :M]).repeat_interleave(Ns, dim=0)
    x = x + sd["out_pos_embed"][:, :T]
    zc, za = _z(masks, 0, cond.shape), _z(masks, 1, x.shape)        # NavDP.drop (navdp.py L305-307)
    cond, x = cond * zc, x * za
    tape = []
    for i in range(layers):
        p = "decoder.layers.%d." % i
        zs = _layer_masks(sd, p, masks, 16 + 8 * i, R, heads, T, M, x.shape)
        h1, n1 = NB.ln_fwd(sd, p + "norm1", x, 1e-5)
        a1, m1 = mha_fwd(sd, p + "self_attn", h1, h1, h1, heads, zs[0], causal=True)
        x = x + a1 * zs[1]
        h2, n2 = NB.ln_fwd(sd, p + "norm2", x, 1e-5)
        a2, m2 = mha_fwd(sd, p + "multihead_attn", h2, cond, cond, heads, zs[2])
        x = x + a2 * zs[3]
        h3, n3 = NB.ln_fwd(sd, p + "norm3", x, 1e-5)
        f1, _ = NB.lin_fwd(sd, p + "linear1", h3)
        f2, _ = NB.lin_fwd(sd, p + "linear2", F.gelu(f1) * zs[4])
        x = x + f2 * zs[5]
        tape.append((n1, m1, n2, m2, n3, h3, f1, zs))
    hN, nN = NB.ln_fwd(sd, "layernorm", x, 1e-5)
    y, _ = NB.lin_fwd(sd, "action_head", hN)
    return y, (noisy, tape, nN, hN, B, Ns, M, T, zc, za)


def decoder_bwd(sd, saved, dy, g, layers=16, heads=8):
    noisy, tape, nN, hN, B, Ns, M, T, zc, za = saved
    dx = NB.ln_bwd(sd, "layernorm", nN, NB.lin_bwd(sd, "action_head", hN, dy, g), g)
    dcond = 0
    for i in reversed(range(layers)):
        p = "decoder.layers.%d." % i
        n1, m1, n2, m2, n3, h3, f1, zs = tape[i]
        dact = NB.lin_bwd(sd, p + "linear2", F.gelu(f1) * zs[4], dx * zs[5], g)
        dx = dx + NB.ln_bwd(sd, p + "norm3", n3, NB.lin_bwd(sd, p + "linear1", h3, NB.gelu_bwd(f1, dact * zs[4]), g), g)
        dq, dk, dv = mha_bwd(sd, p + "multihead_attn", m2, dx * zs[3], g, heads)
        dcond = dcond + dk + dv
        dx = dx + NB.ln_bwd(sd, p + "norm2", n2, dq, g)
        dq, dk, dv = mha_bwd(sd, p + "self_attn", m1, dx * zs[1], g, heads)
        dx = dx + NB.ln_bwd(sd, p + "norm1", n1, dq + dk + dv, g)
    dx, dcond = dx * za, dcond * zc
    gop = torch.zeros_like(sd["out_pos_embed"])
    gop[:, :T] = dx.sum(0, keepdim=True)
    g.add("out_pos_embed", gop)
    NB.lin_bwd(sd, "input_embed", noisy, dx, g, need_dx=False)
    dcond = dcond.reshape(B, Ns, M, -1).sum(1)
    gcp = torch.zeros_like(sd["cond_pos_embed"])
    gcp[:, :M] = dcond.sum(0, keepdim=True)
    g.add("cond_pos_embed", gcp)
    return dcond[:, 1:2], dcond[:, 2:]


def s1_training_backward(sd, traj_hidden_states, traj_images, traj_depths, traj_poses, video_frame_num, noise, timesteps,
                         masks, K=20):
    """navdp_backward.s1_training_backward in train() mode.  -> (loss, Grads, d loss / d hidden states)"""
    sd = {k: (v.float() if v.is_floating_point() else v) for k, v in sd.items()}
    Bb, f = traj_images.shape[:2]
    hs = traj_hidden_states.unsqueeze(1).repeat(1, f, 1, 1).flatten(0, 1)
    mask = (torch.arange(f).expand(Bb, f) < video_frame_num.unsqueeze(1)).flatten(0, 1)[:, None, None].float()
    g_i = traj_images[:, 0:1].repeat(1, f, 1, 1, 1).flatten(0, 1)
    g_d = traj_depths[:, 0:1].repeat(1, f, 1, 1).flatten(0, 1)
    images_dp = torch.stack([g_i, traj_images.flatten(0, 1)], dim=1)
    depths_dp = torch.stack([g_d, traj_depths.flatten(0, 1)], dim=1).unsqueeze(-1)
    goal, gsave = NB.goal_fwd(sd, hs)
    noisy = ddpm.DDPMScheduler(num_train_timesteps=K).add_noise(traj_poses.flatten(0, 1), noise, timesteps)
    rgbd, rsave = rgbd_fwd(sd, images_dp, depths_dp, masks)
    pred, dsave = decoder_fwd(sd, noisy, timesteps, goal, rgbd, masks)
    err = pred - noise
    denom = mask.sum() * err.shape[1] * err.shape[2]
    loss = (err.square() * mask).sum() / denom
    g = NB.Grads()
    dgoal, drgbd = decoder_bwd(sd, dsave, 2.0 * err * mask / denom, g)
    rgbd_bwd(sd, rsave, drgbd, g)
    dhs = NB.goal_bwd(sd, gsave, dgoal, g)
    return loss, g, dhs.reshape(Bb, f, *dhs.shape[1:]).sum(1)
