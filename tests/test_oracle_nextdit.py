"""oracle/nextdit_oracle.py against (a) the committed output of the REFERENCE's own generate_traj (nextdit_async branch;
tests/golden/nextdit_reference.npz from oracle/gen_golden_nextdit.py) and (b) the reference's DiT classes (shapes and
output recorded by oracle/gen_golden_checks.py).  In both the `diffusers` leaf modules are the stand-ins of oracle/diffusers_standin.py (the package
is absent from the image), so what is pinned is the reference's wiring -- generate_traj, LuminaNextDiTBlock,
LuminaNextDiT2DModel, MemoryEncoder, QFormer, the DINOv2 ViT -- not the third-party leaves (see the oracle's header)."""
import os

import numpy as np
import torch

GOLD = os.path.join(os.path.dirname(__file__), "golden", "nextdit_reference.npz")


def _rel(a, b):
    a, b = torch.as_tensor(a).float(), torch.as_tensor(b).float()
    return float((a - b).norm() / (b.norm() + 1e-12))


def test_generate_traj_matches_the_reference_run():
    from internnav_b200.manifest import random_nextdit_state_dict
    from oracle import nextdit_oracle as O
    from oracle.gen_golden_nextdit import make_inputs
    g = np.load(GOLD)
    sd = random_nextdit_state_dict(int(g["seed"]))
    inp = make_inputs(int(g["seed"]), int(g["batch"]), int(g["ns"]))
    with torch.no_grad():
        cond = O.condition_tokens(sd, inp["traj_latents"], inp["images_dp"])
        assert _rel(cond, g["condition_tokens"]) < 2e-5
        for scale, key in ((1.0, "traj_scale_1"), (2.5, "traj_scale_2p5")):
            out = O.generate_traj(sd, inp["traj_latents"], inp["images_dp"], inp["x_init"], guidance_scale=scale,
                                  num_sample_trajs=int(g["ns"]))
            assert out.shape == (3, 32, 3)
            assert _rel(out, g[key]) < 5e-5, (scale, _rel(out, g[key]))
    assert _rel(g["traj_scale_1"], g["traj_scale_2p5"]) > 1e-3      # the guidance branch is live in the fixture


def test_flow_match_schedule():
    from oracle import nextdit_oracle as O
    ts, sig = O.flow_match_schedule(10)
    assert ts.to(torch.long).tolist() == [1000, 900, 800, 700, 600, 500, 400, 300, 200, 100]
    assert sig.shape == (11,) and float(sig[-1]) == 0.0 and abs(float(sig[3]) - 0.7) < 1e-6


def test_manifest_and_dit_match_the_reference_classes():
    """State-dict shapes of the reference's NextDiTCrossAttn / MemoryEncoder / QFormer and its DiT output on seeded inputs
    (a fixed sample of its trajectory tokens), recorded in tests/golden/reference_traces.json and reference_checks.npz (oracle/gen_golden_checks.py)."""
    import json
    from internnav_b200.manifest import nextdit_shapes, random_nextdit_state_dict
    from oracle import nextdit_oracle as O
    from oracle.gen_golden_checks import NEXTDIT_ROWS, NEXTDIT_SEED, nextdit_inputs
    golden = os.path.dirname(GOLD)
    with open(os.path.join(golden, "reference_traces.json"), encoding="utf-8") as fh:
        ref = {k: tuple(v) for k, v in json.load(fh)["nextdit_shapes"].items()}
    mine = {k: tuple(v) for k, v in nextdit_shapes().items() if k.startswith(("traj_dit.", "memory_encoder.", "rgb_resampler."))}
    assert mine == ref
    sd = random_nextdit_state_dict(NEXTDIT_SEED)
    with torch.no_grad():
        out = O.traj_dit(sd, *nextdit_inputs())[:, NEXTDIT_ROWS]
        assert _rel(out, np.load(os.path.join(golden, "reference_checks.npz"))["nextdit_dit"]) < 1e-5
