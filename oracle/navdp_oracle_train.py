"""The System-1 training forward of oracle/navdp_oracle.py in the reference's train() mode -- TEST INFRASTRUCTURE.

The reference trains with dropout p = 0.1 (navdp.py L27, L305-307; the decoder's and the Q-former's
nn.TransformerDecoderLayer, navdp_backbone.py L148).  torch's dropout draws cannot be reproduced by a kernel, so the masks
are an input here: `masks(site, shape)` returns the multiplier of a dropout site -- 0 where dropped, 1 / (1 - p) where
kept -- for the site ids of internnav_b200/dropout.py; `philox_masks` below gives the kernels' masks (oracle/philox.py).
Everything without dropout (DINOv2, goal compressor, linear / LayerNorm arithmetic) is navdp_oracle's own code.  Pinned
against the reference module in train() mode with the same masks: tests/golden/s1_training_dropout_reference.npz
(oracle/gen_golden_training_dropout.py).
"""
import math

import torch
import torch.nn.functional as F

from . import ddpm, philox
from . import navdp_oracle as O


def philox_masks(seed, p, step=0, rank=0):
    """The kernels' masks (oracle/philox.py) as a mask provider: masks(site, shape) -> fp32 multiplier."""
    def masks(site, shape):
        return torch.from_numpy(philox.multiplier(tuple(shape), seed, site, p, step, rank))
    return masks


def _z(masks, site, shape, like):
    return masks(site, tuple(shape)).to(like.device, like.dtype)


def _mha(sd, p, q_in, k_in, v_in, heads, z, causal=False):
    """navdp_oracle._mha (math path) with the dropout multiplier z [B, heads, Sq, Sk] on the probabilities."""
    D = q_in.shape[-1]
    w, b = sd[p + ".in_proj_weight"].to(q_in.dtype), sd[p + ".in_proj_bias"].to(q_in.dtype)
    q, k, v = F.linear(q_in, w[:D], b[:D]), F.linear(k_in, w[D:2 * D], b[D:2 * D]), F.linear(v_in, w[2 * D:], b[2 * D:])
    B, Sq, Sk, hd = q.shape[0], q.shape[1], k.shape[1], D // heads
    q, k, v = (t.view(B, -1, heads, hd).transpose(1, 2) for t in (q, k, v))
    s = (q @ k.transpose(-1, -2)) / math.sqrt(hd)
    if causal:
        s = s.masked_fill(torch.triu(torch.ones(Sq, Sk, dtype=torch.bool, device=q.device), diagonal=1), float("-inf"))
    o = ((s.softmax(-1) * z) @ v).transpose(1, 2).reshape(B, Sq, D)
    return F.linear(o, sd[p + ".out_proj.weight"].to(o.dtype), sd[p + ".out_proj.bias"].to(o.dtype))


def _decoder_layer_post(sd, p, x, mem, heads, masks, site0):
    """Post-norm Q-former layer (navdp_oracle._decoder_layer_post) with its six dropout sites from site0 on."""
    B, S, _ = x.shape
    z = lambda off, shape: _z(masks, site0 + off, shape, x)                 # noqa: E731
    x = O._ln(sd, p + "norm1", x + _mha(sd, p + "self_attn", x, x, x, heads, z(0, (B, heads, S, S))) * z(1, x.shape), 1e-5)
    x = O._ln(sd, p + "norm2", x + _mha(sd, p + "multihead_attn", x, mem, mem, heads, z(2, (B, heads, S, mem.shape[1])))
              * z(3, x.shape), 1e-5)
    h = O._lin(sd, p + "linear1", x)
    ff = O._lin(sd, p + "linear2", F.relu(h) * z(4, h.shape))
    return O._ln(sd, p + "norm3", x + ff * z(5, x.shape), 1e-5)


def rgbd_encoder(sd, images, depths, masks, frames=2, p="rgbd_encoder."):
    """navdp_oracle.rgbd_encoder (RGB tokens detached, as in training) with the Q-former's dropout."""
    B, T = images.shape[:2]
    with torch.no_grad():
        mean = torch.tensor([0.485, 0.456, 0.406], dtype=torch.bfloat16).to(images.device, images.dtype).reshape(1, 3, 1, 1)
        std = torch.tensor([0.229, 0.224, 0.225], dtype=torch.bfloat16).to(images.device, images.dtype).reshape(1, 3, 1, 1)
        ti = images.permute(0, 1, 4, 2, 3).reshape(-1, 3, 224, 224)
        image_token = O.dinov2_vits(sd, p + "rgb_model.", (ti - mean) / std).reshape(B, T * 256, -1)
    td = depths.permute(0, 1, 4, 2, 3).reshape(-1, 1, 224, 224)
    depth_token = O.dinov2_vits(sd, p + "depth_model.", torch.cat([td, td, td], dim=1)).reshape(B, T * 256, -1)
    token = torch.cat((image_token, depth_token), dim=1) + sd[p + "former_pe.weight"][: frames * 2 * 256].to(images.dtype)
    x = sd[p + "former_query.weight"][: frames * 16].to(images.dtype).unsqueeze(0).expand(B, -1, -1)
    for i in range(2):
        x = _decoder_layer_post(sd, "%sformer_net.layers.%d." % (p, i), x, token, 8, masks, 256 + 8 * i)
    return O._lin(sd, p + "project_layer", x)


def predict_noise(sd, last_actions, timestep, goal_embed, rgbd_embed, masks, layers=16, heads=8):
    """navdp_oracle.predict_noise with NavDP.drop on the condition / action embeddings (navdp.py L305-307) and the six
    dropout sites of every pre-norm decoder layer."""
    dt = last_actions.dtype
    R, T, _ = last_actions.shape
    B = goal_embed.shape[0]
    Ns = R // B
    x = O._lin(sd, "input_embed", last_actions)
    if timestep.numel() == 1:
        timestep = timestep.reshape(1).expand(B)
    time_emb = O.sinusoidal_pos_emb(timestep.to(last_actions.device)).unsqueeze(1).to(dt)
    M = 2 + rgbd_embed.shape[1]
    cond = (torch.cat([time_emb, goal_embed, rgbd_embed], dim=1) + sd["cond_pos_embed"][:, :M].to(dt)).repeat_interleave(Ns, dim=0)
    x = x + sd["out_pos_embed"][:, :T].to(dt)
    cond, x = cond * _z(masks, 0, cond.shape, cond), x * _z(masks, 1, x.shape, x)
    for i in range(layers):
        p = "decoder.layers.%d." % i
        z = lambda off, shape: _z(masks, 16 + 8 * i + off, shape, x)       # noqa: E731
        h = O._ln(sd, p + "norm1", x, 1e-5)
        x = x + _mha(sd, p + "self_attn", h, h, h, heads, z(0, (R, heads, T, T)), causal=True) * z(1, x.shape)
        h = O._ln(sd, p + "norm2", x, 1e-5)
        x = x + _mha(sd, p + "multihead_attn", h, cond, cond, heads, z(2, (R, heads, T, M))) * z(3, x.shape)
        h = O._ln(sd, p + "norm3", x, 1e-5)
        f1 = O._lin(sd, p + "linear1", h)
        x = x + O._lin(sd, p + "linear2", F.gelu(f1) * z(4, f1.shape)) * z(5, x.shape)
    return O._lin(sd, "action_head", O._ln(sd, "layernorm", x, 1e-5))


def s1_training_loss(sd, traj_hidden_states, traj_images, traj_depths, traj_poses, video_frame_num, noise, timesteps, masks,
                     K=20):
    """navdp_oracle.s1_training_loss in train() mode (forward_vlm_traj, navdp.py L291-312, with the given masks)."""
    B, f = traj_images.shape[:2]
    hs = traj_hidden_states.unsqueeze(1).repeat(1, f, 1, 1).flatten(0, 1)
    loss_mask = torch.arange(f, device=traj_images.device).expand(B, f) < video_frame_num.unsqueeze(1)
    g_i = traj_images[:, 0:1].repeat(1, f, 1, 1, 1).flatten(0, 1)
    g_d = traj_depths[:, 0:1].repeat(1, f, 1, 1).flatten(0, 1)
    images_dp = torch.stack([g_i, traj_images.flatten(0, 1)], dim=1)
    depths_dp = torch.stack([g_d, traj_depths.flatten(0, 1)], dim=1).unsqueeze(-1)
    goal = O.goal_token(sd, hs)
    noisy = ddpm.DDPMScheduler(num_train_timesteps=K).add_noise(traj_poses.flatten(0, 1), noise, timesteps)
    rgbd = rgbd_encoder(sd, images_dp, depths_dp, masks)
    err = (predict_noise(sd, noisy, timesteps, goal, rgbd, masks) - noise).square()
    mask = loss_mask.flatten(0, 1)[:, None, None]
    return (err * mask).sum() / mask.sum() / (err.shape[1] * err.shape[2])


def s1_training_grads(sd, traj_hidden_states, traj_images, traj_depths, traj_poses, video_frame_num, noise, timesteps, masks):
    """navdp_oracle.s1_training_grads in train() mode: -> (loss, {parameter: gradient}, d loss / d traj_hidden_states)."""
    leaf = {k: v.detach().clone().requires_grad_(True) for k, v in sd.items() if v.is_floating_point()}
    full = dict(sd)
    full.update(leaf)
    hs = traj_hidden_states.detach().clone().requires_grad_(True)
    loss = s1_training_loss(full, hs, traj_images, traj_depths, traj_poses, video_frame_num, noise, timesteps, masks)
    loss.backward()
    return loss.detach(), {k: v.grad for k, v in leaf.items() if v.grad is not None}, hs.grad
