"""Train-mode dropout of the System-1 training step on the CPU: the mask contract (oracle/philox.py), the mask-aware oracle
against the reference module's own train()-mode step (tests/golden/s1_training_dropout_reference.npz), the hand-written
backward with masks, and the dropout schedule of internnav_b200/train_s1.py on fp32 stand-in ops."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from ops_reference import TorchOps  # noqa: E402

from internnav_b200 import dropout as DS  # noqa: E402
from internnav_b200.train_s1 import S1TrainStep  # noqa: E402
from oracle import ddpm, gen_golden_training as G, navdp_oracle as O, philox, weights  # noqa: E402
from oracle import navdp_backward_train as NBT, navdp_oracle_train as OT  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden", "s1_training_dropout_reference.npz")


@pytest.fixture(scope="module")
def sd():
    return weights.make_state_dict(0)


def test_philox_known_answers():
    """The Random123 known-answer vectors of Philox4x32-10."""
    cases = [((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
             ((0xffffffff,) * 4, (0xffffffff, 0xffffffff), (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
             ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
              (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]
    for ctr, key, want in cases:
        got = philox.philox4x32_10(np.array([ctr], dtype=np.uint32), key)[0]
        assert [int(x) for x in got] == list(want), [hex(int(x)) for x in got]


def test_mask_statistics():
    """16 M elements: keep rate 1 - p; two sites or two steps are independent (agree on 0.9^2 + 0.1^2 of positions)."""
    n, seed, p = 1 << 24, 12345, 0.1
    a = philox.keep_mask((n,), seed, DS.decoder_site(3, DS.DROPOUT1), p, step=5)
    b = philox.keep_mask((n,), seed, DS.decoder_site(3, DS.DROPOUT2), p, step=5)
    c = philox.keep_mask((n,), seed, DS.decoder_site(3, DS.DROPOUT1), p, step=6)
    d = philox.keep_mask((n,), seed, DS.decoder_site(3, DS.DROPOUT1), p, step=5, rank=1)
    assert abs(a.mean() - 0.9) < 1e-3
    for other in (b, c, d):
        assert abs((a == other).mean() - 0.82) < 2e-3
    assert philox.threshold(0.1) == DS.threshold(0.1) == 429496729
    assert philox.scale(0.1) == np.float32(DS.keep_scale(0.1))
    # element e is decided by word e & 3 of block e >> 2: a prefix of a longer mask is the shorter mask
    assert np.array_equal(philox.keep_mask((1001,), seed, 7, 0.5), philox.keep_mask((4096,), seed, 7, 0.5)[:1001])


def test_rng_state_words():
    r = DS.DropoutRNG(seed=0x123456789ABCDEF0, rank=3)
    r.set_step(9)
    assert [int(x) & 0xFFFFFFFF for x in r.dev.tolist()] == [0x9ABCDEF0, 0x12345678, 9, 3]
    assert r.state() == {"seed": 0x123456789ABCDEF0, "rank": 3, "step": 9}


def test_site_table_matches_reference_golden():
    """Every site of the table was reached by the reference's train()-mode forward, with the mask of oracle/philox.py; the
    all-keep run of the same module reproduced the eval-mode golden (nothing else changes in train() mode)."""
    g = np.load(GOLD)
    table = DS.site_table(4)
    assert sorted(int(s) for s in g["sites"]) == sorted(table)
    for s, dropped in zip(g["sites"], g["dropped"]):
        z = philox.keep_mask(table[int(s)][1], int(g["seed"]), int(s), float(g["p"]), int(g["step"]), int(g["rank"]))
        assert int((~z).sum()) == int(dropped), int(s)
    assert float(np.max(g["allkeep_vs_eval"])) < 1e-5


def _masks_of_golden():
    g = np.load(GOLD)
    return OT.philox_masks(int(g["seed"]), float(g["p"]), int(g["step"]), int(g["rank"]))


def test_mask_aware_oracle_reproduces_reference_train_mode(sd):
    """oracle/navdp_oracle_train.py with the kernels' masks vs the reference module in train() mode with the same masks."""
    gold = np.load(GOLD)
    b = G.make_batch()
    loss, grads, g_hs = OT.s1_training_grads(sd, b["hs"], b["traj_images"], b["traj_depths"], b["traj_poses"],
                                            b["video_frame_num"], b["noise"], b["timesteps"], masks=_masks_of_golden())
    assert abs(float(loss) - float(gold["loss"])) < 1e-5 * max(1.0, float(gold["loss"]))
    names = [str(n) for n in gold["grad_names"]]
    assert sorted(grads) == sorted(names), set(grads) ^ set(names)
    for n, norm, dot in zip(names, gold["grad_norms"], gold["grad_dots"]):
        g = grads[n]
        assert abs(float(g.norm()) - norm) <= 1e-5 * norm + 1e-9, (n, float(g.norm()), norm)
        mine = float((g * G.probe(n, tuple(g.shape))).sum())
        assert abs(mine - dot) <= 1e-3 * norm + 2e-4 * abs(dot) + 1e-7, (n, mine, dot)
    assert np.allclose(g_hs.numpy(), gold["grad_hs"], atol=1e-7, rtol=2e-3)


def test_handwritten_backward_with_masks_matches_autograd(sd):
    """oracle/navdp_backward_train.py (the spec of the dropout schedule) vs autograd through navdp_oracle_train."""
    b = G.make_batch(dict(G.CASE, seed=204))
    args = (b["hs"], b["traj_images"], b["traj_depths"], b["traj_poses"], b["video_frame_num"], b["noise"], b["timesteps"])
    masks = OT.philox_masks(99, 0.1, step=3)
    loss_a, grads_a, dhs_a = OT.s1_training_grads(sd, *args, masks=masks)
    with torch.no_grad():
        loss_m, grads_m, dhs_m = NBT.s1_training_backward(sd, *args, masks=masks)
    assert abs(float(loss_a) - float(loss_m)) < 1e-6 * max(1.0, abs(float(loss_a)))
    assert sorted(grads_a) == sorted(grads_m)
    for k, ga in grads_a.items():
        gm = grads_m[k].reshape(ga.shape)
        rel = float((gm - ga).norm() / (ga.norm() + 1e-12))
        assert rel < 2e-3 or float((gm - ga).abs().max()) < 1e-8, (k, rel)
    assert float((dhs_m - dhs_a).norm() / dhs_a.norm()) < 2e-3


class DropoutTorchOps(TorchOps):
    """TorchOps with the dropout primitives of the GPU backend, built on oracle/philox.py."""

    def _z(self, drop, shape):
        rng, site, p = drop
        seed_lo, seed_hi, step, rank = rng.words()
        return torch.from_numpy(philox.multiplier(tuple(shape), seed_lo | (seed_hi << 32), site, p, step, rank))

    def dropout(self, x, drop):
        self._count("dropout")
        assert x.is_contiguous()
        return x * self._z(drop, x.shape)

    def dropout_add(self, residual, y, drop):
        self._count("dropout_add")
        assert residual.is_contiguous() and y.is_contiguous() and residual.shape == y.shape
        return residual + y * self._z(drop, y.shape)

    def act_fwd(self, pre, kind, drop=None):
        y = super().act_fwd(pre, kind)
        return y if drop is None else y * self._z(drop, y.shape)

    def act_bwd(self, pre, dy, kind, drop=None):
        return super().act_bwd(pre, dy if drop is None else dy * self._z(drop, dy.shape), kind)

    def _zp(self, drop, batch, heads, sq, sk):
        return None if drop is None else self._z(drop, (batch, heads, sq, sk))

    def attention(self, q, k, v, heads, hd, batch, sq, sk, causal, drop=None):
        if drop is None:
            return super().attention(q, k, v, heads, hd, batch, sq, sk, causal)
        self._count("attention")
        p = self._probs(q, k, heads, hd, batch, sq, sk, causal) * self._zp(drop, batch, heads, sq, sk)
        return (p @ self._heads(v, batch, sk, heads, hd)).transpose(1, 2).reshape(batch * sq, heads * hd)

    def attention_bwd(self, q, k, v, o, do, heads, hd, batch, sq, sk, causal, drop=None):
        if drop is None:
            return super().attention_bwd(q, k, v, o, do, heads, hd, batch, sq, sk, causal)
        self._count("attention_bwd")
        z = self._zp(drop, batch, heads, sq, sk)
        p = self._probs(q, k, heads, hd, batch, sq, sk, causal)
        qh, kh, vh = (self._heads(t, batch, n, heads, hd) for t, n in ((q, sq), (k, sk), (v, sk)))
        doh = self._heads(do, batch, sq, heads, hd)
        dv = (p * z).transpose(-1, -2) @ doh
        dp = (doh @ vh.transpose(-1, -2)) * z
        D = (doh * self._heads(o, batch, sq, heads, hd)).sum(-1, keepdim=True)
        ds = p * (dp - D) / hd ** 0.5
        back = lambda t, n: t.transpose(1, 2).reshape(batch * n, heads * hd)          # noqa: E731
        return back(ds @ kh, sq), back(ds.transpose(-1, -2) @ qh, sk), back(dv, sk)


def _schedule(sd, b, ops, **kw):
    imgs, _ = G.dp_inputs(b)
    with torch.no_grad():
        mean = torch.tensor([0.485, 0.456, 0.406], dtype=torch.bfloat16).float().reshape(1, 3, 1, 1)
        std = torch.tensor([0.229, 0.224, 0.225], dtype=torch.bfloat16).float().reshape(1, 3, 1, 1)
        ti = imgs.permute(0, 1, 4, 2, 3).reshape(-1, 3, 224, 224)
        rgb_tokens = O.dinov2_vits(sd, "rgbd_encoder.rgb_model.", (ti - mean) / std).reshape(imgs.shape[0], 2 * 256, -1)
        step = S1TrainStep({k: v.float() for k, v in sd.items() if v.is_floating_point()}, ops, **kw)
        acp = torch.as_tensor(ddpm.DDPMScheduler(num_train_timesteps=20).alphas_cumprod).float()
        return step.forward_backward(b["hs"], rgb_tokens, b["traj_depths"], b["traj_poses"], b["video_frame_num"],
                                     b["noise"], b["timesteps"], acp)


def test_dropout_schedule_reproduces_oracle_gradients(sd):
    torch.set_num_threads(os.cpu_count())
    b = G.make_batch(dict(G.CASE, seed=205))
    rng = DS.DropoutRNG(seed=0xC0FFEE, rank=1)
    rng.set_step(11)
    args = (b["hs"], b["traj_images"], b["traj_depths"], b["traj_poses"], b["video_frame_num"], b["noise"], b["timesteps"])
    loss_ref, grads_ref, dhs_ref = OT.s1_training_grads(sd, *args, masks=OT.philox_masks(0xC0FFEE, 0.1, step=11, rank=1))
    ops = DropoutTorchOps()
    loss, grads, dhs = _schedule(sd, b, ops, dropout=0.1, rng=rng)
    assert abs(float(loss) - float(loss_ref)) < 1e-5 * max(1.0, abs(float(loss_ref)))
    assert sorted(grads) == sorted(grads_ref)
    for k, gr in grads_ref.items():
        rel = float((grads[k].reshape(gr.shape) - gr).norm() / (gr.norm() + 1e-12))
        assert rel < 2e-3 or float((grads[k].reshape(gr.shape) - gr).abs().max()) < 1e-8, (k, rel)
    assert float((dhs - dhs_ref).norm() / dhs_ref.norm()) < 2e-3
    # every site went through the backend: 6 x (16 + 2) layer sites, 2 embedding sites
    assert ops.calls["dropout_add"] == 3 * 18 and ops.calls["dropout"] == 2 + 2 + 3 * 18
    # and with dropout the loss differs from the eval-mode step
    loss_eval, _, _ = O.s1_training_grads(sd, *args)
    assert abs(float(loss) - float(loss_eval)) > 1e-4


def test_zero_dropout_issues_the_plain_schedule(sd):
    """dropout=0 calls exactly the primitives (and computes exactly what) the step computes without the argument."""
    b = G.make_batch(dict(G.CASE, seed=206))
    o1, o2 = DropoutTorchOps(), DropoutTorchOps()
    l1, g1, d1 = _schedule(sd, b, o1)
    l2, g2, d2 = _schedule(sd, b, o2, dropout=0.0)
    assert o1.calls == o2.calls and "dropout" not in o1.calls
    assert torch.equal(l1, l2) and torch.equal(d1, d2) and all(torch.equal(g1[k], g2[k]) for k in g1)
