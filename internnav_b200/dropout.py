"""Train-mode dropout of System 1: the site table and the trainer's RNG state.

The reference trains `NavDP_Policy_DPT_CriticSum_DAT` in train() mode with dropout p = 0.1 (navdp.py L27, L305-307; the
decoder's nn.TransformerDecoderLayer and the Q-former's, navdp_backbone.py L148).  Masks come from a counter-based
generator (csrc/dropout.cuh states the contract; oracle/philox.py restates it in numpy), so the backward recomputes the
forward's mask and a captured CUDA graph needs nothing but the device-resident state below.

This module imports nothing that loads the library.
"""
import math

import numpy as np
import torch

# site ids (< 2^16): the embedding sites, then 8 ids per decoder layer l at 16 + 8 l and per Q-former layer q at 256 + 8 q
COND, ACTION = 0, 1
SELF_PROBS, DROPOUT1, CROSS_PROBS, DROPOUT2, FF_INNER, DROPOUT3 = range(6)


def decoder_site(layer, offset):
    return 16 + 8 * layer + offset


def qformer_site(layer, offset):
    return 256 + 8 * layer + offset


def site_table(R, layers=16, qformer_layers=2, heads=8, D=384, T=32, M=34, Q=32, mem=1024):
    """{site id: (reference module, tensor shape)} for R samples: every tensor the reference drops in train() mode.
    T: predicted steps, M: condition tokens, Q: Q-former queries, mem: Q-former memory tokens."""
    t = {COND: ("NavDP.drop(cond)", (R, M, D)), ACTION: ("NavDP.drop(action)", (R, T, D))}
    for l in range(layers):
        p = "decoder.layers.%d." % l
        t[decoder_site(l, SELF_PROBS)] = (p + "self_attn", (R, heads, T, T))
        t[decoder_site(l, DROPOUT1)] = (p + "dropout1", (R, T, D))
        t[decoder_site(l, CROSS_PROBS)] = (p + "multihead_attn", (R, heads, T, M))
        t[decoder_site(l, DROPOUT2)] = (p + "dropout2", (R, T, D))
        t[decoder_site(l, FF_INNER)] = (p + "dropout", (R, T, 4 * D))
        t[decoder_site(l, DROPOUT3)] = (p + "dropout3", (R, T, D))
    for q in range(qformer_layers):
        p = "rgbd_encoder.former_net.layers.%d." % q
        t[qformer_site(q, SELF_PROBS)] = (p + "self_attn", (R, heads, Q, Q))
        t[qformer_site(q, DROPOUT1)] = (p + "dropout1", (R, Q, D))
        t[qformer_site(q, CROSS_PROBS)] = (p + "multihead_attn", (R, heads, Q, mem))
        t[qformer_site(q, DROPOUT2)] = (p + "dropout2", (R, Q, D))
        t[qformer_site(q, FF_INNER)] = (p + "dropout", (R, Q, 2048))
        t[qformer_site(q, DROPOUT3)] = (p + "dropout3", (R, Q, D))
    return t


def threshold(p):
    """Elements whose Philox word is below this are dropped: floor(p * 2^32) in double precision."""
    if not 0.0 <= p < 1.0:
        raise ValueError("dropout p must be in [0, 1), got %r" % (p,))
    return int(math.floor(float(p) * 4294967296.0))


def keep_scale(p):
    return float(np.float32(1.0 / (1.0 - float(p))))


class DropoutRNG:
    """{seed_lo, seed_hi, step, rank} as a device int32[4] that the kernels read at run time, with pinned host twins.
    `step` is the trainer's micro-batch counter; `rank` the data-parallel rank (ranks draw independent masks)."""
    SLOTS = 4   # host twins in rotation: an asynchronous copy never reads a twin that is being rewritten

    def __init__(self, seed=0, rank=0, device="cpu"):
        self.device = torch.device(device)
        self.seed, self.rank, self.step = int(seed) & (2 ** 64 - 1), int(rank), 0
        if not 0 <= self.rank < 2 ** 16:
            raise ValueError("rank must fit 16 bits")
        cuda = self.device.type == "cuda"
        self._host = [torch.zeros(4, dtype=torch.int32, pin_memory=cuda) for _ in range(self.SLOTS)]
        self._copied = [None] * self.SLOTS   # event after the copy out of each twin
        self._slot = 0
        self.dev = torch.zeros(4, dtype=torch.int32, device=self.device)
        self.set_step(0)

    def words(self):
        """(seed_lo, seed_hi, step, rank) as unsigned 32-bit integers."""
        return (self.seed & 0xFFFFFFFF, self.seed >> 32, self.step & 0xFFFFFFFF, self.rank)

    def set_step(self, step):
        """Point the device state at micro-batch `step` (stream-ordered: work enqueued after this call sees it)."""
        self.step = int(step)
        i = self._slot = (self._slot + 1) % self.SLOTS
        if self._copied[i] is not None:
            self._copied[i].synchronize()
        w = np.array(self.words(), dtype=np.uint32).view(np.int32)
        self._host[i].copy_(torch.from_numpy(w))
        self.dev.copy_(self._host[i], non_blocking=True)
        if self.device.type == "cuda":
            self._copied[i] = torch.cuda.Event()
            self._copied[i].record()

    def state(self):
        return {"seed": self.seed, "rank": self.rank, "step": self.step}
