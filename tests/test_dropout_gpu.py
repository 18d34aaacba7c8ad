"""Train-mode dropout on the B200: the mask kernels against oracle/philox.py bit for bit, the elementwise and attention
kernels with dropout against PyTorch with the same masks, and the whole training step against the oracle chain."""
import numpy as np
import pytest
import torch

from internnav_b200 import dropout as DS
from oracle import philox

pytestmark = pytest.mark.gpu


def _rel(a, b):
    a, b = a.detach().float(), b.detach().float()
    return float((a - b).norm() / (b.norm() + 1e-12))


def _rng(seed, step=0, rank=0):
    r = DS.DropoutRNG(seed=seed, rank=rank, device="cuda")
    r.set_step(step)
    return r


def _z(shape, seed, site, p, step=0, rank=0):
    return torch.from_numpy(philox.multiplier(shape, seed, site, p, step, rank)).cuda()


@pytest.mark.parametrize("p", [0.1, 0.5])
def test_dropout_mask_bit_exact(p):
    from internnav_b200 import _bwd as K
    for seed, site, step, rank, n in [(0, 0, 0, 0, 1), (7, 17, 3, 0, 1001), (2 ** 40 + 5, 300, 9, 1, 4099 * 3),
                                      (123456789, DS.decoder_site(15, DS.FF_INNER), 2 ** 31 + 1, 7, 32 * 32 * 1536 + 3)]:
        m = K.dropout_mask((n,), _rng(seed, step, rank).dev, site, p).cpu().numpy().astype(bool)
        assert np.array_equal(m, philox.keep_mask((n,), seed, site, p, step, rank)), (seed, site, step, rank, n)


def test_elementwise_dropout_kernels():
    from internnav_b200 import _bwd as K
    torch.manual_seed(0)
    seed, p, step = 77, 0.1, 4
    rng = _rng(seed, step)
    x = torch.randn(96, 32, 384, device="cuda").bfloat16()
    r = torch.randn(96, 32, 384, device="cuda").bfloat16()
    z = _z(x.shape, seed, 5, p, step)
    assert _rel(K.dropout_add(r, x, rng.dev, 5, p), r.float() + z * x.float()) < 5e-3
    assert torch.equal(K.dropout(x, rng.dev, 5, p), (z * x.float()).bfloat16())
    pre = (2 * torch.randn(96 * 32, 1536, device="cuda")).bfloat16()
    dy = torch.randn(96 * 32, 1536, device="cuda").bfloat16()
    for act, fn in [(1, torch.nn.functional.gelu), (2, torch.relu)]:
        zz = _z(pre.shape, seed, 20, p, step)
        pf = pre.float().requires_grad_(True)
        y = fn(pf) * zz
        y.backward(dy.float())
        assert _rel(K.act_fwd_dropout(pre, act, rng.dev, 20, p), y) < 5e-3
        assert _rel(K.act_bwd_dropout(pre, dy, act, rng.dev, 20, p), pf.grad) < 5e-3


@pytest.mark.parametrize("B,Sq,Sk,causal,p", [(6, 32, 32, True, 0.1), (6, 32, 34, False, 0.1), (6, 32, 32, False, 0.1),
                                              (2, 32, 1024, False, 0.1), (6, 32, 32, True, 0.5), (6, 32, 34, False, 0.5),
                                              (3, 32, 1024, False, 0.5), (5, 17, 30, False, 0.5)])
def test_attention_with_dropout(B, Sq, Sk, causal, p):
    """The four training shapes of the table (decoder self / cross, Q-former self / cross; 8 heads x 48) and an odd one,
    forward and backward, vs autograd of (softmax(S) o Z) V with Z from oracle/philox.py."""
    from internnav_b200 import _bwd as K
    H, hd, seed, site, step = 8, 48, 31337, DS.qformer_site(1, DS.CROSS_PROBS), 2
    torch.manual_seed(B * Sq + Sk)
    q = torch.randn(B * Sq, H * hd, device="cuda").bfloat16()
    k = torch.randn(B * Sk, H * hd, device="cuda").bfloat16()
    v = torch.randn(B * Sk, H * hd, device="cuda").bfloat16()
    do = torch.randn(B * Sq, H * hd, device="cuda").bfloat16()
    z = _z((B, H, Sq, Sk), seed, site, p, step)
    qf, kf, vf = (t.float().requires_grad_(True) for t in (q, k, v))
    qh, kh, vh = (t.view(B, -1, H, hd).transpose(1, 2) for t in (qf, kf, vf))
    s = qh @ kh.transpose(-1, -2) * hd ** -0.5
    if causal:
        i, j = torch.arange(Sq, device="cuda")[:, None], torch.arange(Sk, device="cuda")[None, :]
        s = s.masked_fill(j > i + (Sk - Sq), float("-inf"))
    o_ref = ((s.softmax(-1) * z) @ vh).transpose(1, 2).reshape(B * Sq, H * hd)
    o_ref.backward(do.float())
    rng = _rng(seed, step)
    o = K.attention_dropout(q, k, v, H, hd, B, Sq, Sk, rng.dev, site, p, causal=causal)
    assert _rel(o, o_ref) < 1.5e-2, _rel(o, o_ref)
    dq, dk, dv = K.attention_bwd_dropout(q, k, v, o, do, H, hd, B, Sq, Sk, rng.dev, site, p, causal=causal)
    errs = (_rel(dq, qf.grad), _rel(dk, kf.grad), _rel(dv, vf.grad))
    assert max(errs) < 1.5e-2, errs


def _training_case():
    from internnav_b200.internvla_n1 import InternVLAN1ForCausalLM
    from internnav_b200.manifest import random_navdp_state_dict
    from internnav_b200.training import collate_traj_batch
    from oracle import qwen_oracle as Q
    cfg = Q.tiny_cfg()
    s2_sd = Q.make_s2_state_dict(cfg, seed=31, vocab_rows=512)
    s1_sd = {k: v.float() for k, v in random_navdp_state_dict(seed=32, vlm_token_dim=cfg["hidden"]).items()}
    model = InternVLAN1ForCausalLM(cfg, device="cuda:0")
    model.load_parts(s2_sd, s1_sd)
    rng = np.random.Generator(np.random.PCG64(33))
    g = torch.Generator().manual_seed(34)
    gpp, frames = [[(1, 8, 12)], [(1, 4, 8)]], [2, 1]
    inst = []
    for gs, f in zip(gpp, frames):
        ids = torch.tensor([Q.make_prompt(rng, 6, gs, 11)])
        n_p = sum(t * h * w for t, h, w in gs)
        inst.append(dict(input_ids=ids, labels=torch.full_like(ids, -100), pixel_values=torch.randn(n_p, 1176, generator=g).bfloat16(),
                         image_grid_thw=torch.tensor(gs), traj_images=torch.rand(f, 224, 224, 3, generator=g),
                         traj_depths=torch.rand(f, 224, 224, generator=g) * 5, traj_poses=torch.randn(f, 32, 3, generator=g) * 0.5))
    batch = collate_traj_batch(inst)
    B, fmax = len(inst), max(frames)
    noise = torch.randn(B * fmax, 32, 3, generator=g)
    ts = torch.randint(0, 20, (B * fmax,), generator=g)
    return cfg, s2_sd, s1_sd, model, batch, noise, ts


def test_training_step_with_dropout_vs_oracle():
    """The whole step at p = 0.1 against the oracle chain with the same masks (fp32, CPU), with the bounds of the step
    without dropout; a bf16 autograd run of the oracle with the same masks is reported as the error class."""
    from internnav_b200.train_step import DualSystemTrainer
    from oracle import navdp_oracle as O, navdp_oracle_train as OT, qwen_oracle as Q
    cfg, s2_sd, s1_sd, model, batch, noise, ts = _training_case()
    seed, step = 4242, 5
    tr = DualSystemTrainer(model, s1_sd, s2_sd["model.latent_queries"], lr=1e-3, dropout=0.1, dropout_seed=seed)
    loss, grads, hs = tr.loss_and_grads(batch, noise, ts, dropout_step=step)
    with torch.no_grad():
        hs_ref = Q.training_traj_states(s2_sd, cfg, batch["input_ids"], batch["attention_mask"], batch["pixel_values"].float(),
                                        batch["image_grid_thw"], batch["t_s_pos"])
    masks = OT.philox_masks(seed, 0.1, step=step)
    args = (batch["traj_images"], batch["traj_depths"], batch["traj_poses"], batch["video_frame_num"], noise, ts)
    loss_ref, grads_ref, dhs_ref = OT.s1_training_grads(s1_sd, hs_ref, *args, masks=masks)
    loss_nodrop, _, _ = O.s1_training_grads(s1_sd, hs_ref, *args)
    glat_ref = Q.latent_query_grads(s2_sd, cfg, batch["input_ids"], batch["attention_mask"], batch["pixel_values"].float(),
                                    batch["image_grid_thw"], batch["t_s_pos"], dhs_ref)
    sd16 = {k: (v.bfloat16() if v.is_floating_point() else v) for k, v in s1_sd.items()}
    a16 = tuple(t.bfloat16() if t.is_floating_point() else t for t in args)
    loss16, grads16, _ = OT.s1_training_grads(sd16, hs_ref.bfloat16(), *a16, masks=masks)
    e_loss, e16 = abs(float(loss) - float(loss_ref)) / float(loss_ref), abs(float(loss16) - float(loss_ref)) / float(loss_ref)
    print("dropout train step: loss %.6f oracle %.6f (no dropout %.6f) rel %.2e, bf16 autograd rel %.2e"
          % (float(loss), float(loss_ref), float(loss_nodrop), e_loss, e16))
    assert abs(float(loss_ref) - float(loss_nodrop)) > 1e-4            # the masks changed the step
    assert e_loss < 1e-2
    bad, beyond_class = [], []
    for k, gr in grads_ref.items():
        rel = _rel(grads[k].cpu().reshape(gr.shape), gr)
        rel16 = _rel(grads16[k].float().reshape(gr.shape), gr)
        if rel > 0.08 and float(gr.norm()) > 1e-6:
            bad.append((k, rel))
        if rel > 2 * max(rel16, 1e-3):
            beyond_class.append((k, round(rel, 4), round(rel16, 4)))
    print("parameter gradients beyond 8 %:", bad[:10], "of", len(grads_ref))
    print("tensors whose error exceeds 2x the bf16 autograd error:", beyond_class)
    assert len(bad) <= len(grads_ref) // 50
    assert _rel(grads["model.latent_queries"].cpu(), glat_ref) < 0.1


def test_graph_replay_mask_stream_and_state():
    from internnav_b200 import _bwd as K
    from internnav_b200.train_step import DualSystemTrainer
    cfg, s2_sd, s1_sd, model, batch, noise, ts = _training_case()
    lat = s2_sd["model.latent_queries"]
    dev_batch = {k: (v.cuda() if torch.is_tensor(v) and k in ("traj_images", "traj_depths", "traj_poses", "video_frame_num")
                     else v) for k, v in batch.items()}
    n, t = noise.cuda(), ts.cuda()
    # successive micro-batches draw different masks; the same micro-batch the same
    t0 = DualSystemTrainer(model, s1_sd, lat, lr=1e-3, dropout=0.1, dropout_seed=9)
    l0, l1, l0b = (float(t0.loss_and_grads(batch, noise, ts, dropout_step=s)[0]) for s in (0, 1, 0))
    assert l0 != l1 and l0 == l0b
    # ranks draw different masks
    site = DS.decoder_site(0, DS.DROPOUT1)
    m0 = K.dropout_mask((4096,), _rng(9, 0, 0).dev, site, 0.1)
    m1 = K.dropout_mask((4096,), _rng(9, 0, 1).dev, site, 0.1)
    assert not torch.equal(m0, m1)
    # a resumed trainer continues the stream
    t1 = DualSystemTrainer(model, s1_sd, lat, lr=1e-3, dropout=0.1, dropout_seed=9)
    t1.load_dropout_state({"p": 0.1, "seed": 9, "step": 1})
    assert float(t1.loss_and_grads(batch, noise, ts)[0]) == l1 and t1.dropout_state()["step"] == 1
    # graph replay == eager, bit for bit, over two steps
    ta = DualSystemTrainer(model, s1_sd, lat, lr=1e-3, max_grad_norm=1.0, dropout=0.1, dropout_seed=9)
    tb = DualSystemTrainer(model, s1_sd, lat, lr=1e-3, max_grad_norm=1.0, dropout=0.1, dropout_seed=9, graph_s1=True)
    losses = []
    for _ in range(2):
        model._s2.set_latent_queries(ta.latent)
        la = float(ta.step(dev_batch, n, t))
        model._s2.set_latent_queries(tb.latent)
        lb = float(tb.step(dev_batch, n, t))
        assert la == lb, (la, lb)
        losses.append(la)
    assert losses[0] != losses[1] and ta.dropout_state()["step"] == tb.dropout_state()["step"] == 2
    assert all(torch.equal(ta.masters[k], tb.masters[k]) for k in ta.masters)
    # dropout = 0 is the trainer without the argument
    tc = DualSystemTrainer(model, s1_sd, lat, lr=1e-3)
    td = DualSystemTrainer(model, s1_sd, lat, lr=1e-3, dropout=0.0)
    model._s2.set_latent_queries(tc.latent)
    lc = float(tc.step(dev_batch, n, t))
    model._s2.set_latent_queries(td.latent)
    ld = float(td.step(dev_batch, n, t))
    assert lc == ld and all(torch.equal(tc.masters[k], td.masters[k]) for k in tc.masters)
