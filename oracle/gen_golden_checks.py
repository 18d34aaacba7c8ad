"""Generate tests/golden/reference_traces.json and tests/golden/reference_checks.npz from the original InternNav tree.

    N1_REFERENCE_ROOT=<InternNav checkout> python -m oracle.gen_golden_checks

Runs the REFERENCE's own classes (through oracle/ref_loader.py) on the seeded scripts, weights and inputs of the tests
that compare against them, and records what those tests compare:

  * tests/test_vs_live_reference.py -- InternVLAN1Net host logic (s2_step / step_no_infer / s1_step_latent / reset) and
    InternVLAN1Agent (real S2 worker thread) step by step: the call sequence and every result the test asserts on;
  * tests/test_oracle_s1.py -- NavDP RGB-D encoder, goal token and predict_noise on inputs of seed 107;
  * tests/test_oracle_nextdit.py -- the state-dict shapes of NextDiTCrossAttn / MemoryEncoder / QFormer and the DiT
    output on seeded inputs (a fixed sample of 8 of its 32 trajectory tokens);
  * tests/test_oracle_navdp_policy.py -- the state-dict shapes of the stand-alone NavDPNet.
"""
import contextlib
import io
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import agent_script, policy_script, ref_loader, weights  # noqa: E402

POLICY_SEEDS = [101, 102, 103]
AGENT_CASES = [(201, "partial_async"), (202, "sync"), (203, "partial_async")]
NEXTDIT_SEED = 3
NEXTDIT_ROWS = sorted(int(r) for r in np.random.Generator(np.random.PCG64(0)).choice(32, 8, replace=False))  # stored sample
NAVDP_INPUT_SEED = 107


def policy_script_of(seed):
    """-> (rng, answers, trajs, num_history): the seeded script of one policy trace; `rng` continues into the ops."""
    rng = np.random.Generator(np.random.PCG64(seed))
    answers, trajs = policy_script.random_answers(rng, n=40), policy_script.random_trajs(rng, n=8)
    return rng, answers, trajs, int(rng.choice([2, 4, 8]))


def agent_script_of(seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    return agent_script.random_script(rng, p_latent=float(rng.uniform(0.3, 0.9)), p_raise=0.05)


def _json(x):
    return json.loads(json.dumps(x))


def policy_trace(seed):
    """45 frames of one environment; S2 on frame 0, after a look-down answer and at random, S1 after some latent answers,
    reset before frame 20.  One record per call with the reference's results."""
    rng, answers, trajs, num_history = policy_script_of(seed)
    _, Net = ref_loader.load_reference_policy()
    proc, llm = policy_script.FakeProcessor(), policy_script.ScriptedLLM(answers, trajs)
    ref = Net(llm, proc, num_history=num_history)
    ref.reset()
    look, steps = False, []
    for k in range(45):
        o = agent_script.make_obs(k, size=(24, 32))
        u = rng.random()
        if k == 20:
            ref.reset()
            steps.append({"op": "reset"})
            look = False
        if k == 0 or look or u < 0.5:
            a = ref.s2_step(o["rgb"], o["depth"], None, o["instruction"], None, look_down=look)
            rec = {"op": "s2", "k": k, "look_down": look, "processor": _json(proc.log.pop()), "llm_output": ref.llm_output,
                   "pixel": None if a.output_pixel is None else [int(v) for v in a.output_pixel],
                   "actions": None if a.output_action is None else [int(v) for v in a.output_action],
                   "episode_idx": int(ref.episode_idx), "n_rgb": len(ref.rgb_list), "s1_idx": None}
            look = a.output_action is not None and 5 in a.output_action[:1]
            if a.output_latent is not None and rng.random() < 0.6:
                rec["s1_idx"] = [int(v) for v in ref.s1_step_latent(None, None, torch.zeros(1)).idx]
            steps.append(rec)
        else:
            ref.step_no_infer(o["rgb"], o["depth"], None)
            steps.append({"op": "noinfer", "k": k})
    return {"seed": seed, "steps": steps}


def agent_trace(seed, mode):
    """40 frames of one environment through the reference agent (reset before frame 17): per frame the action, the
    policy calls it made, dual_forward_step and look_down."""
    script = agent_script_of(seed)
    holder = {}

    def factory(config=None):
        holder["policy"] = agent_script.ScriptedPolicy(script, s2_output_cls=holder["mod"].S2Output,
                                                       s1_output_cls=holder["mod"].S1Output)
        return holder["policy"]
    mod = holder["mod"] = ref_loader.load_reference_agent(factory)
    settings = dict(policy_name="InternVLAN1_Policy", state_encoder=None, device="cpu", infer_mode=mode,
                    sys2_max_forward_step=8, width=640, height=480, hfov=79, vis_debug=False)
    ref = mod.InternVLAN1Agent(mod.AgentCfg(model_name="internvla_n1", model_settings=settings))
    rpol = holder["policy"]
    ref.reset()
    rpol.drain()
    steps = []
    for k in range(40):
        if k == 17:
            ref.reset(reset_index=[0])
        a = ref.step([agent_script.make_obs(k)])
        steps.append({"k": k, "action": [int(v) for v in a[0]["action"]], "calls": _json(rpol.drain()),
                      "dual_forward_step": int(ref.dual_forward_step), "look_down": bool(ref.look_down)})
    return {"seed": seed, "mode": mode, "steps": steps}


def navdp_modules():
    """RGB-D encoder, goal token and predict_noise of the reference NavDP on weights.make_state_dict(0)."""
    m = ref_loader.build_reference_navdp()
    m.load_state_dict(weights.make_state_dict(0), strict=True)
    inp = weights.make_inputs(NAVDP_INPUT_SEED, B=1)
    with torch.no_grad():
        r = m.rgbd_encoder(inp["rgb"], inp["depth"])
        g = m.goal_compressor(m.vlm_embed_mlp(inp["latents"]), None)
        eps = m.predict_noise(inp["x_init"], torch.tensor([3]), g, r)
    return {"navdp_rgbd": r.numpy(), "navdp_goal": g.numpy(), "navdp_eps": eps.numpy()}


def nextdit_inputs():
    gen = torch.Generator().manual_seed(0)
    x, z = torch.randn(4, 32, 384, generator=gen), torch.randn(4, 36, 768, generator=gen)
    return x, torch.tensor([1000, 700, 100, 100]), z


def nextdit_modules():
    """-> (state-dict shapes of NextDiTCrossAttn / MemoryEncoder / QFormer, DiT output on nextdit_inputs() at the
    trajectory tokens NEXTDIT_ROWS)."""
    import importlib

    from internnav_b200.manifest import random_nextdit_state_dict
    _, cross = ref_loader.load_reference_nextdit()
    arch = importlib.import_module("internnav.model.basemodel.internvla_n1.internvla_n1_arch")
    m = cross.NextDiTCrossAttn(cross.NextDiTCrossAttnConfig(latent_embedding_size=768, _gradient_checkpointing=False)).eval()
    shapes = {"traj_dit." + k: list(v.shape) for k, v in m.state_dict().items()}
    shapes.update({"memory_encoder." + k: list(v.shape) for k, v in arch.MemoryEncoder().state_dict().items()})
    shapes.update({"rgb_resampler." + k: list(v.shape) for k, v in arch.QFormer().state_dict().items()})
    sd = random_nextdit_state_dict(NEXTDIT_SEED)
    m.load_state_dict({k[len("traj_dit."):]: v for k, v in sd.items() if k.startswith("traj_dit.")}, strict=True)
    with torch.no_grad():
        out = m(*nextdit_inputs())
    return shapes, out[:, NEXTDIT_ROWS].numpy()


def navdp_policy_shapes():
    net = ref_loader.build_reference_navdp_policy()
    return {k: list(v.shape) for k, v in net.state_dict().items()
            if not k.startswith(("image_encoder.", "pixel_encoder.", "pixel_aux_head.", "image_aux_head."))}


def main():
    assert ref_loader.available(), "needs the reference tree (N1_REFERENCE_ROOT)"
    torch.set_num_threads(os.cpu_count())
    with contextlib.redirect_stdout(io.StringIO()):   # the reference classes print every step
        policy = [policy_trace(s) for s in POLICY_SEEDS]
        agent = [agent_trace(s, m) for s, m in AGENT_CASES]
    nextdit_shapes, dit_out = nextdit_modules()
    traces = {"policy": policy, "agent": agent, "nextdit_shapes": nextdit_shapes,
              "navdp_policy_shapes": navdp_policy_shapes()}
    out = os.path.join(ROOT, "tests", "golden", "reference_traces.json")
    with open(out, "w", encoding="utf-8") as fh:
        json.dump(traces, fh, ensure_ascii=False)
    print("wrote", out, os.path.getsize(out), "bytes")
    arrays = dict(navdp_modules(), nextdit_dit=dit_out)
    out = os.path.join(ROOT, "tests", "golden", "reference_checks.npz")
    np.savez_compressed(out, **{k: v.astype(np.float32) for k, v in arrays.items()})
    print("wrote", out, os.path.getsize(out), "bytes")


if __name__ == "__main__":
    main()
