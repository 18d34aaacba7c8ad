"""Pins the System-2 oracle (oracle/qwen_oracle.py) and the C++ integer planners -- CPU only.

  * vision tower / decoder restatements vs the container's transformers implementation of the same Qwen2.5-VL blocks
    (seeded tiny configs, fp32, eager attention);
  * rope_index vs the committed fixture tests/golden/rope_index.json, the output of the reference's own
    internnav/dataset/rope2d.py;
  * libn1b200's host-only planners (n1_rope_index, n1_vit_window_index) bit-exact vs the oracle.
"""
import ctypes
import json
import os

import numpy as np
import pytest
import torch

from oracle import qwen_oracle as Q

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
GOLD = os.path.join(GOLDEN, "rope_index.json")


def _cases():
    rng = np.random.Generator(np.random.PCG64(7))
    cases = []
    for pre, grids, post in [(24, [(1, 28, 28)], 80), (5, [(1, 16, 16), (1, 16, 16)], 9), (0, [(1, 28, 20)], 1),
                             (12, [(1, 8, 12), (1, 28, 28), (1, 4, 4)], 30), (40, [], 7),
                             (3, [(1, 28, 28)] * 9, 60)]:
        ids = Q.make_prompt(rng, pre, grids, post) + [Q.TRAJ_TOKEN_INDEX] * 4
        cases.append((ids, [list(g) for g in grids]))
    return cases


def test_rope_index_golden():
    with open(GOLD) as fh:
        gold = json.load(fh)
    for (ids, grids), g in zip(_cases(), gold):
        assert ids == g["input_ids"]
        pos, delta = Q.rope_index(torch.tensor([ids]), torch.tensor(grids).reshape(-1, 3))
        assert pos[:, 0].tolist() == g["position_ids"] and int(delta) == g["delta"]


def test_rope_index_vs_reference():
    """The oracle's full position tensor [3, 1, S] and delta against the reference's get_rope_index_25 on the same cases,
    whose outputs tests/golden/rope_index.json records."""
    with open(GOLD) as fh:
        gold = json.load(fh)
    for (ids, grids), g in zip(_cases(), gold):
        t = torch.tensor([ids])
        pos, delta = Q.rope_index(t, torch.tensor(grids).reshape(-1, 3) if grids else torch.zeros(0, 3, dtype=torch.long))
        assert torch.equal(pos, torch.tensor(g["position_ids"]).unsqueeze(1)) and int(delta) == g["delta"]


def _lib():
    from internnav_b200 import _lib
    return _lib.lib()


def test_cxx_rope_index_bit_exact():
    L = _lib()
    for ids, grids in _cases():
        n = len(ids)
        a = (ctypes.c_int32 * n)(*ids)
        g = (ctypes.c_int32 * max(1, 3 * len(grids)))(*[v for gr in grids for v in gr])
        out = (ctypes.c_int32 * (3 * n))()
        d = ctypes.c_int32()
        rc = L.n1_rope_index(a, n, g, len(grids), 2, out, ctypes.byref(d))
        assert rc == 0, L.n1_last_error()
        pos, delta = Q.rope_index(torch.tensor([ids]), torch.tensor(grids).reshape(-1, 3))
        assert list(out) == pos[:, 0].reshape(-1).tolist() and d.value == int(delta)


@pytest.mark.parametrize("grids", [[(1, 28, 28)], [(1, 16, 16), (1, 28, 20)], [(1, 8, 8)], [(2, 12, 20)],
                                   [(1, 32, 32), (1, 4, 4), (1, 28, 28)]])
def test_cxx_window_index_bit_exact(grids):
    L = _lib()
    n_p = sum(t * h * w for t, h, w in grids)
    g = (ctypes.c_int32 * (3 * len(grids)))(*[v for gr in grids for v in gr])
    widx = (ctypes.c_int32 * (n_p // 4))()
    cu = (ctypes.c_int32 * (n_p // 4 + 2))()
    ncu = ctypes.c_int32()
    pos = (ctypes.c_int32 * (2 * n_p))()
    assert L.n1_vit_window_index(g, len(grids), 2, 4, widx, cu, ctypes.byref(ncu), pos) == 0, L.n1_last_error()
    pos_ids, window_index, cu_window, _ = Q.vit_indices(grids)
    assert list(widx) == window_index.tolist()
    assert list(cu)[: ncu.value] == cu_window.tolist()
    reordered = pos_ids.reshape(n_p // 4, 4, 2)[window_index].reshape(-1).tolist()
    assert list(pos) == reordered


def _hf_cfgs(cfg):
    from transformers.models.qwen2_5_vl.configuration_qwen2_5_vl import Qwen2_5_VLTextConfig, Qwen2_5_VLVisionConfig
    vc = Qwen2_5_VLVisionConfig(depth=cfg["v_depth"], hidden_size=cfg["v_hidden"], num_heads=cfg["v_heads"],
                                intermediate_size=cfg["v_inter"], out_hidden_size=cfg["v_out"],
                                fullatt_block_indexes=cfg["fullatt"], window_size=cfg["v_window"], hidden_act="silu")
    tc = Qwen2_5_VLTextConfig(hidden_size=cfg["hidden"], num_hidden_layers=cfg["layers"],
                              num_attention_heads=cfg["heads"], num_key_value_heads=cfg["kv_heads"],
                              intermediate_size=cfg["inter"], vocab_size=cfg["vocab"], rms_norm_eps=cfg["rms_eps"],
                              rope_parameters={"rope_type": "default", "rope_theta": cfg["rope_theta"],
                                               "mrope_section": cfg["mrope"]}, use_sliding_window=False)
    return vc, tc


def test_vision_tower_vs_transformers():
    from transformers.models.qwen2_5_vl.modeling_qwen2_5_vl import Qwen2_5_VisionTransformerPretrainedModel as VT
    cfg = Q.tiny_cfg()
    sd = Q.make_s2_state_dict(cfg, seed=1, vocab_rows=64)
    vc, _ = _hf_cfgs(cfg)
    m = VT._from_config(vc, attn_implementation="eager").float().eval()
    missing = m.load_state_dict({k[len("visual."):]: v for k, v in sd.items() if k.startswith("visual.")}, strict=True)
    grids = [(1, 16, 20), (1, 28, 28)]
    n_p = sum(t * h * w for t, h, w in grids)
    torch.manual_seed(0)
    px = torch.randn(n_p, 1176)
    with torch.no_grad():
        ref = m(px, grid_thw=torch.tensor(grids))
        ref = ref.pooler_output if hasattr(ref, "pooler_output") else ref
        mine = Q.vit_forward(sd, cfg, px, grids)
    assert torch.allclose(ref, mine, atol=2e-4, rtol=1e-4), (ref - mine).abs().max()


def test_decoder_vs_transformers():
    from transformers.models.qwen2_5_vl.modeling_qwen2_5_vl import Qwen2_5_VLTextModel as TM
    cfg = Q.tiny_cfg(vocab=2048)
    sd = Q.make_s2_state_dict(cfg, seed=2)
    _, tc = _hf_cfgs(cfg)
    m = TM._from_config(tc, attn_implementation="eager").float().eval()
    tsd = {k[len("model."):]: v for k, v in sd.items() if k.startswith("model.") and "latent_queries" not in k}
    m.load_state_dict(tsd, strict=True)
    rng = np.random.Generator(np.random.PCG64(3))
    grids = [(1, 8, 12)]
    ids = torch.tensor([Q.make_prompt(rng, 6, grids, 10, vocab_text=2000) + [5] * 4])
    # image / vision_start ids exceed the tiny vocabulary: position ids come from the real ids, embeddings are random
    pos, _ = Q.rope_index(ids, torch.tensor(grids))
    torch.manual_seed(1)
    emb = torch.randn(1, ids.shape[1], cfg["hidden"])
    with torch.no_grad():
        ref = m(inputs_embeds=emb, position_ids=pos).last_hidden_state
        mine = Q.text_forward(sd, cfg, emb, pos)
    assert torch.allclose(ref, mine, atol=3e-4, rtol=1e-4), (ref - mine).abs().max()


# ------------------------------------------------------------------------------------------------ greedy decode
GEN_CASE = dict(seed=5, prompt_seed=3, grids=[(1, 8, 12)], n_pre=6, n_post=10, pixel_seed=0, max_new=12)


def _gen_case():
    cfg = Q.tiny_cfg()
    sd = Q.make_s2_state_dict(cfg, seed=GEN_CASE["seed"], lm_head=True)
    rng = np.random.Generator(np.random.PCG64(GEN_CASE["prompt_seed"]))
    grids = GEN_CASE["grids"]
    ids = torch.tensor([Q.make_prompt(rng, GEN_CASE["n_pre"], grids, GEN_CASE["n_post"])])
    torch.manual_seed(GEN_CASE["pixel_seed"])
    px = torch.randn(sum(t * h * w for t, h, w in grids), 1176)
    return cfg, sd, ids, px, grids


def test_greedy_generate_golden():
    """The oracle's greedy decode reproduces the committed token ids (tests/golden/greedy_generate.json, written by
    this file's __main__ after the transformers check below passed in the build container)."""
    with open(os.path.join(GOLDEN, "greedy_generate.json")) as fh:
        gold = json.load(fh)
    cfg, sd, ids, px, grids = _gen_case()
    with torch.no_grad():
        assert Q.greedy_generate(sd, cfg, ids, px, grids, max_new_tokens=GEN_CASE["max_new"]) == gold["tokens"]
        stop = gold["tokens"][3]
        got = Q.greedy_generate(sd, cfg, ids, px, grids, max_new_tokens=GEN_CASE["max_new"], eos_token_ids=(stop,))
        assert got == gold["tokens"][:4]


def test_greedy_generate_vs_transformers():
    """`model.generate(do_sample=False)` of the container's transformers (KV cache, GenerationMixin stop rules) against
    the oracle's cache-free loop, token for token.  transformers 5.x computes a different temporal position for image
    tokens than the reference's pin (4.51) and in-tree rope2d.get_rope_index_25; the reference-equal `rope_index`
    (pinned bit-exactly above) is substituted so that the comparison is about the decode loop."""
    from transformers.models.qwen2_5_vl.configuration_qwen2_5_vl import Qwen2_5_VLConfig
    from transformers.models.qwen2_5_vl.modeling_qwen2_5_vl import Qwen2_5_VLForConditionalGeneration as M
    cfg, sd, ids, px, grids = _gen_case()
    vc, tc = _hf_cfgs(cfg)
    c = Qwen2_5_VLConfig(text_config=tc.to_dict(), vision_config=vc.to_dict(), image_token_id=151655,
                         video_token_id=151656, vision_start_token_id=151652, tie_word_embeddings=False)
    m = M._from_config(c, attn_implementation="eager").float().eval()
    msd = {}
    for k, v in sd.items():
        if k.startswith("visual."):
            msd["model." + k] = v
        elif k == "model.latent_queries":
            continue
        elif k.startswith("model."):
            msd["model.language_model." + k[len("model."):]] = v
        else:
            msd[k] = v
    m.load_state_dict(msd, strict=True)
    m.model.get_rope_index = lambda input_ids, **kw: Q.rope_index(input_ids, kw["image_grid_thw"])
    kw = dict(input_ids=ids, attention_mask=torch.ones_like(ids), pixel_values=px, image_grid_thw=torch.tensor(grids),
              do_sample=False, pad_token_id=151643, mm_token_type_ids=(ids == 151655).int())
    with torch.no_grad():
        ref = m.generate(max_new_tokens=GEN_CASE["max_new"], eos_token_id=[151645, 151643], **kw)[0, ids.shape[1]:].tolist()
        mine = Q.greedy_generate(sd, cfg, ids, px, grids, max_new_tokens=GEN_CASE["max_new"])
        assert ref == mine
        stop = mine[3]  # stop rule: the eos id is emitted, then generation ends
        ref2 = m.generate(max_new_tokens=GEN_CASE["max_new"], eos_token_id=[stop], **kw)[0, ids.shape[1]:].tolist()
        assert ref2 == mine[:4] == Q.greedy_generate(sd, cfg, ids, px, grids, max_new_tokens=GEN_CASE["max_new"],
                                                      eos_token_ids=(stop,))


if __name__ == "__main__":
    # refresh tests/golden/greedy_generate.json (build container; run the transformers check first)
    test_greedy_generate_vs_transformers()
    cfg, sd, ids, px, grids = _gen_case()
    with torch.no_grad():
        toks = Q.greedy_generate(sd, cfg, ids, px, grids, max_new_tokens=GEN_CASE["max_new"])
    with open(os.path.join(GOLDEN, "greedy_generate.json"), "w") as fh:
        json.dump({"case": GEN_CASE, "tokens": toks}, fh)
    print("wrote greedy_generate.json", toks)


# ------------------------------------------------------------------------------------------------ training forward
def collate(prompts, pad=151643, nq=4):
    """process_input_with_traj_tokens + pad_sequence of the reference collator (internvla_n1_lerobot_dataset.py
    L1155-1215): TRAJ tokens appended, right padding, attention_mask = input_ids != pad."""
    rows = [list(p) + [Q.TRAJ_TOKEN_INDEX] * nq for p in prompts]
    S = max(len(r) for r in rows)
    ids = torch.tensor([r + [pad] * (S - len(r)) for r in rows])
    return ids, ids.ne(pad), [len(p) for p in prompts]


def test_training_states_equal_latent_prefill():
    """The padded-batch training forward (TRAJ tokens inside the sequence, key padding mask, masked get_rope_index)
    yields, at the TRAJ positions, exactly what generate_latents yields for each unpadded prompt -- the identity the
    CUDA path's forward() relies on.  One prompt also holds the pad id in its middle (masked there, as the collator's
    `input_ids.ne(pad)` does)."""
    cfg = Q.tiny_cfg()
    sd = Q.make_s2_state_dict(cfg, seed=7, vocab_rows=256)
    rng = np.random.Generator(np.random.PCG64(21))
    gpp = [[(1, 8, 12)], [(1, 4, 8), (1, 8, 8)], [(1, 4, 4)]]
    prompts = [Q.make_prompt(rng, 5 + 4 * i, gs, 18 - 6 * i) for i, gs in enumerate(gpp)]
    prompts[2][3] = 151643
    grids = [g for gs in gpp for g in gs]
    torch.manual_seed(3)
    px = torch.randn(sum(t * h * w for t, h, w in grids), 1176)
    ids, mask, t_s_pos = collate(prompts)
    with torch.no_grad():
        full = Q.training_traj_states(sd, cfg, ids, mask, px, grids, t_s_pos)
        off = 0
        for b, (p, gs) in enumerate(zip(prompts, gpp)):
            n = sum(t * h * w for t, h, w in gs)
            kept = [t for t in p if t != 151643]
            ref = Q.generate_latents(sd, cfg, torch.tensor([kept]), px[off:off + n], gs)
            off += n
            assert torch.allclose(full[b], ref[0], atol=2e-5, rtol=1e-5), (b, (full[b] - ref[0]).abs().max())


def test_decoder_padding_mask_vs_transformers():
    """text_forward(key_mask=...) against the transformers text model driven with a 2-D attention_mask (right padding),
    compared on the unpadded positions."""
    from transformers.models.qwen2_5_vl.modeling_qwen2_5_vl import Qwen2_5_VLTextModel as TM
    cfg = Q.tiny_cfg(vocab=2048)
    sd = Q.make_s2_state_dict(cfg, seed=2)
    _, tc = _hf_cfgs(cfg)
    m = TM._from_config(tc, attn_implementation="eager").float().eval()
    m.load_state_dict({k[len("model."):]: v for k, v in sd.items() if k.startswith("model.") and "latent_queries" not in k},
                      strict=True)
    torch.manual_seed(4)
    B, S = 2, 24
    emb = torch.randn(B, S, cfg["hidden"])
    mask = torch.ones(B, S, dtype=torch.bool)
    mask[1, 17:] = False
    pos = torch.arange(S).view(1, 1, S).expand(3, B, S).clone()
    pos[:, 1, 17:] = 1
    with torch.no_grad():
        ref = m(inputs_embeds=emb, position_ids=pos, attention_mask=mask.long()).last_hidden_state
        mine = Q.text_forward(sd, cfg, emb, pos, key_mask=mask)
    assert torch.allclose(ref[mask], mine[mask], atol=3e-4, rtol=1e-4), (ref[mask] - mine[mask]).abs().max()


def test_latent_query_gradient_vs_transformers():
    """Backward oracle of the System-2 half (row a13): d loss / d latent_queries through the frozen decoder, against
    autograd through the transformers text model fed the same embeddings / positions / padding mask (the gradient of
    the embedding rows at the TRAJ positions, summed over the batch, is the gradient of the shared latent_queries)."""
    from transformers.models.qwen2_5_vl.modeling_qwen2_5_vl import Qwen2_5_VLTextModel as TM
    cfg = Q.tiny_cfg()
    sd = Q.make_s2_state_dict(cfg, seed=9, vocab_rows=256)
    _, tc = _hf_cfgs(cfg)
    m = TM._from_config(tc, attn_implementation="eager").float().eval()
    m.load_state_dict({k[len("model."):]: v for k, v in sd.items() if k.startswith("model.") and "latent_queries" not in k},
                      strict=True)
    rng = np.random.Generator(np.random.PCG64(31))
    gpp = [[(1, 8, 12)], [(1, 4, 8)]]
    prompts = [Q.make_prompt(rng, 5 + 6 * i, gs, 14 - 5 * i) for i, gs in enumerate(gpp)]
    grids = [g for gs in gpp for g in gs]
    torch.manual_seed(5)
    px = torch.randn(sum(t * h * w for t, h, w in grids), 1176)
    ids, mask, t_s_pos = collate(prompts)
    G = torch.randn(len(prompts), cfg["n_query"], cfg["hidden"])
    mine = Q.latent_query_grads(sd, cfg, ids, mask, px, grids, t_s_pos, G)
    # transformers side: same embeddings and positions, autograd w.r.t. the embedding rows
    with torch.no_grad():
        emb = sd["model.embed_tokens.weight"][ids].clone()
        emb[ids == Q.IMAGE_TOKEN_INDEX] = Q.vit_forward(sd, cfg, px, grids)
        emb[ids == Q.TRAJ_TOKEN_INDEX] = sd["model.latent_queries"].reshape(cfg["n_query"], -1).repeat(len(prompts), 1)
        pos = torch.ones(3, *ids.shape, dtype=torch.long)
        img = 0
        for b, gs in enumerate(gpp):
            keep = mask[b]
            pb, _ = Q.rope_index(ids[b][keep].unsqueeze(0), torch.tensor(gs))
            pos[:, b, keep] = pb[:, 0]
    emb.requires_grad_(True)
    hs = m(inputs_embeds=emb, position_ids=pos, attention_mask=mask.long()).last_hidden_state
    sel = torch.stack([hs[b, t:t + cfg["n_query"]] for b, t in enumerate(t_s_pos)])
    (sel * G).sum().backward()
    ref = torch.stack([emb.grad[b, t:t + cfg["n_query"]] for b, t in enumerate(t_s_pos)]).sum(0, keepdim=True)
    assert mine.shape == ref.shape == (1, cfg["n_query"], cfg["hidden"])
    assert torch.allclose(mine, ref, atol=2e-5, rtol=2e-3), (mine - ref).abs().max()


def test_handwritten_latent_query_backward_matches_autograd():
    """oracle/qwen_backward.py (backward restricted to the TRAJ rows against the per-layer K/V cache; no autograd)
    equals autograd through the padded-batch forward."""
    from oracle import qwen_backward as QB
    cfg = Q.tiny_cfg()
    sd = Q.make_s2_state_dict(cfg, seed=10, vocab_rows=256)
    rng = np.random.Generator(np.random.PCG64(41))
    gpp = [[(1, 8, 12)], [(1, 4, 8), (1, 4, 4)], [(1, 4, 4)]]
    prompts = [Q.make_prompt(rng, 4 + 5 * i, gs, 13 - 4 * i) for i, gs in enumerate(gpp)]
    grids = [g for gs in gpp for g in gs]
    torch.manual_seed(6)
    px = torch.randn(sum(t * h * w for t, h, w in grids), 1176)
    ids, mask, t_s_pos = collate(prompts)
    G = torch.randn(len(prompts), cfg["n_query"], cfg["hidden"])
    ref = Q.latent_query_grads(sd, cfg, ids, mask, px, grids, t_s_pos, G)
    with torch.no_grad():
        mine = QB.latent_query_backward(sd, cfg, ids, mask, px, grids, t_s_pos, G)
    rel = float((mine - ref).norm() / ref.norm())
    print("latent_queries gradient rel err (TRAJ-row backward vs autograd)", rel)
    assert mine.shape == ref.shape and rel < 1e-4
