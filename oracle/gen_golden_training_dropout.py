"""Generate tests/golden/s1_training_dropout_reference.npz from the REFERENCE's own NavDP module in train() mode.

    python -m oracle.gen_golden_training_dropout

The case of oracle/gen_golden_training.py (same weights, batch and injected `sample_noise` draws), but the module runs in
train() mode with dropout p = 0.1, as the reference trains it.  torch's own dropout draws cannot be reproduced by a
kernel, so the masks are injected: `torch.nn.functional.dropout` (what every nn.Dropout calls) and
`torch.nn.functional.scaled_dot_product_attention` (where F.multi_head_attention_forward applies the attention dropout
when need_weights=False) are patched to apply the masks of oracle/philox.py -- the kernels' contract.  Every intercepted
call with p > 0 is matched, in call order, to a site of internnav_b200/dropout.py and its shape is checked against the
site table; calls with p = 0 (goal compressor, DINOv2) pass through untouched.

Before that, the same patched module runs once with all-keep masks and must reproduce s1_training_reference.npz (the
eval-mode golden): nothing but dropout changes between eval() and train() mode (no BatchNorm, no other train-mode branch).

Stored: loss, prediction, per-parameter gradient norms and probe dots (as gen_golden_training), the gradient with respect
to the latent tokens, the seed, step, rank and p of the masks, and the number of dropped elements per site.
"""
import math
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from internnav_b200 import dropout as DS  # noqa: E402
from oracle import gen_golden_training as G, philox, ref_loader, weights  # noqa: E402

MASKS = dict(seed=0x5EED1234ABCD, step=7, rank=0, p=0.1)


def site_order(qformer_layers=2, layers=16):
    """The order in which the reference's forward reaches its dropout sites (post-norm Q-former layers, the two NavDP.drop
    calls, then the pre-norm decoder layers: attention probabilities before the dropout of their residual branch)."""
    order = []
    for q in range(qformer_layers):
        order += [DS.qformer_site(q, o) for o in range(6)]
    order += [DS.COND, DS.ACTION]
    for l in range(layers):
        order += [DS.decoder_site(l, o) for o in range(6)]
    return order


class Interceptor:
    """Patches F.dropout / F.scaled_dot_product_attention; `mult(site, shape)` -> fp32 multiplier tensor."""

    def __init__(self, R, mult):
        self.table, self.order, self.mult = DS.site_table(R), site_order(), mult
        self.i, self.dropped = 0, {}

    def _next(self, shape, p):
        site = self.order[self.i]
        self.i += 1
        name, want = self.table[site]
        assert tuple(shape) == tuple(want), (site, name, tuple(shape), want)
        assert abs(p - MASKS["p"]) < 1e-12, (site, p)
        z = self.mult(site, tuple(shape))
        self.dropped[site] = int((z == 0).sum())
        return z

    def dropout(self, x, p=0.5, training=True, inplace=False):
        if not training or p == 0:
            return x
        return x * self._next(x.shape, p)

    def sdpa(self, q, k, v, attn_mask=None, dropout_p=0.0, is_causal=False, scale=None, enable_gqa=False):
        s = (q @ k.transpose(-2, -1)) * (scale if scale is not None else 1.0 / math.sqrt(q.shape[-1]))
        if is_causal:
            s = s.masked_fill(torch.ones(s.shape[-2:], dtype=torch.bool).triu(1), float("-inf"))
        if attn_mask is not None:
            s = s.masked_fill(~attn_mask, float("-inf")) if attn_mask.dtype == torch.bool else s + attn_mask
        a = s.softmax(-1)
        if dropout_p > 0:
            a = a * self._next(a.shape, dropout_p)
        return a @ v

    def __enter__(self):
        self._saved = F.dropout, F.scaled_dot_product_attention
        F.dropout, F.scaled_dot_product_attention = self.dropout, self.sdpa
        return self

    def __exit__(self, *exc):
        F.dropout, F.scaled_dot_product_attention = self._saved
        return False


def run(mult):
    """One train()-mode forward / backward of the reference module with injected masks -> (gold dict, interceptor)."""
    m = ref_loader.build_reference_navdp(predict_size=32, memory_size=2, navdp_version=0.1)
    m.load_state_dict(weights.make_state_dict(0), strict=True)
    m.input_dtype = torch.float32
    m.train()
    for p in m.parameters():
        p.requires_grad_(True)
    batch = G.make_batch()
    B, f = batch["traj_images"].shape[:2]
    hs = batch["hs"].clone().requires_grad_(True)
    hs_rep = hs.unsqueeze(1).repeat(1, f, 1, 1).flatten(0, 1)
    images_dp, depths_dp = G.dp_inputs(batch)
    real_randn, real_randint = torch.randn, torch.randint
    torch.randn = lambda *a, **k: batch["noise"].clone()
    torch.randint = lambda *a, **k: batch["timesteps"].clone()
    try:
        with Interceptor(B * f, mult) as icpt:
            pred, eps = m.forward_vlm_traj(hs_rep, images_dp, depths_dp, tensor_label_actions=batch["traj_poses"])
    finally:
        torch.randn, torch.randint = real_randn, real_randint
    assert icpt.i == len(icpt.order), ("dropout sites reached", icpt.i, len(icpt.order))
    err = (pred - eps).square()
    mask = (torch.arange(f).expand(B, f) < batch["video_frame_num"].unsqueeze(1)).flatten(0, 1)[:, None, None]
    loss = (err * mask).sum() / mask.sum() / (err.shape[1] * err.shape[2])
    loss.backward()
    gold = {"pred": pred.detach().numpy(), "loss": np.float32(loss.item()), "grad_hs": hs.grad.numpy()}
    names, norms, dots = [], [], []
    for name, p in m.named_parameters():
        if p.grad is None:
            continue
        names.append(name)
        norms.append(float(p.grad.norm()))
        dots.append(float((p.grad * G.probe(name, tuple(p.shape))).sum()))
    gold["grad_names"] = np.array(names)
    gold["grad_norms"] = np.array(norms, dtype=np.float64)
    gold["grad_dots"] = np.array(dots, dtype=np.float64)
    return gold, icpt


def main():
    torch.set_num_threads(os.cpu_count())
    # 1. all-keep masks: train() mode must reproduce the eval-mode golden
    keep, _ = run(lambda site, shape: torch.ones(shape))
    ev = np.load(os.path.join(ROOT, "tests", "golden", "s1_training_reference.npz"))
    rel = lambda a, b: float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-30))   # noqa: E731
    e_loss, e_pred = abs(float(keep["loss"]) - float(ev["loss"])) / float(ev["loss"]), rel(keep["pred"], ev["pred"])
    e_norm, e_hs = rel(keep["grad_norms"], ev["grad_norms"]), rel(keep["grad_hs"], ev["grad_hs"])
    print("train() with all-keep masks vs eval golden: loss %.2e pred %.2e grad norms %.2e grad_hs %.2e" % (e_loss, e_pred, e_norm, e_hs))
    assert list(keep["grad_names"]) == list(ev["grad_names"]) and max(e_loss, e_pred, e_norm, e_hs) < 1e-5
    # 2. the kernels' masks
    c = MASKS
    gold, icpt = run(lambda site, shape: torch.from_numpy(philox.multiplier(shape, c["seed"], site, c["p"], c["step"], c["rank"])))
    sites = np.array(sorted(icpt.dropped), dtype=np.int32)
    gold.update(seed=np.uint64(c["seed"]), step=np.int64(c["step"]), rank=np.int64(c["rank"]), p=np.float64(c["p"]),
                sites=sites, dropped=np.array([icpt.dropped[s] for s in sites], dtype=np.int64),
                allkeep_vs_eval=np.array([e_loss, e_pred, e_norm, e_hs]))
    out = os.path.join(ROOT, "tests", "golden", "s1_training_dropout_reference.npz")
    np.savez_compressed(out, **gold)
    print("loss", float(gold["loss"]), "(eval mode %.6f)" % float(ev["loss"]), "sites", len(sites), "dropped",
          int(gold["dropped"].sum()), "bytes", os.path.getsize(out))


if __name__ == "__main__":
    main()
