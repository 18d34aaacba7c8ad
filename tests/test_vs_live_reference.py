"""Differential tests against the reference's OWN classes on seeded random scripts, beyond the committed goldens of
tests/test_policy.py and tests/test_agent.py: tests/golden/reference_traces.json holds, call by call, what the reference
returned on these scripts (oracle/gen_golden_checks.py ran it), and the mirrors here must return the same.

  * InternVLAN1Net host logic (s2_step / step_no_infer / s1_step_latent / reset) vs internnav_b200.policy.InternVLAN1Policy
  * InternVLAN1Agent (real S2 worker thread) vs internnav_b200.agent.InternVLAN1Agent
"""
import contextlib
import io
import json
import os
from types import SimpleNamespace

import pytest
import torch

from oracle import agent_script, policy_script
from oracle.gen_golden_checks import agent_script_of, policy_script_of

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
with open(os.path.join(ROOT, "tests", "golden", "reference_traces.json"), encoding="utf-8") as fh:
    GOLD = json.load(fh)


def _json(x):
    return json.loads(json.dumps(x))


@pytest.mark.parametrize("seed", [101, 102, 103])
def test_policy_host_logic_vs_live_reference(seed):
    from internnav_b200.policy import InternVLAN1Policy
    _, answers, trajs, num_history = policy_script_of(seed)
    steps = next(t["steps"] for t in GOLD["policy"] if t["seed"] == seed)

    class Model:  # the n1b200 model mirror's two calls, answering from the same script
        def __init__(self):
            self.n, self.nt = 0, 0

        def generate_with_latents(self, prompts, pixel_values, image_grid_thw, max_new_tokens=128):
            ans = answers[self.n % len(answers)]
            self.n += 1
            return SimpleNamespace(generated=[policy_script.encode(ans) + [151645]], latents=torch.zeros(1, 1, 1))

        def generate_traj(self, traj_latents=None, images_dp=None, depths_dp=None):
            t = trajs[self.nt % len(trajs)]
            self.nt += 1
            return torch.tensor(t, dtype=torch.float32)
    mproc = policy_script.FakeProcessor()
    mine = InternVLAN1Policy(Model(), mproc, num_envs=1, num_history=num_history)
    mine.reset()
    with contextlib.redirect_stdout(io.StringIO()):
        for ref in steps:
            if ref["op"] == "reset":
                mine.reset([0])
                continue
            k = ref["k"]
            o = agent_script.make_obs(k, size=(24, 32))
            if ref["op"] == "s2":
                b = mine.s2_step([0], [o["rgb"]], [o["depth"]], [None], [o["instruction"]], None, [ref["look_down"]])[0]
                assert _json(mproc.log.pop()) == ref["processor"], k
                assert mine.episodes[0].llm_output == ref["llm_output"]
                assert (None if b.output_pixel is None else [int(v) for v in b.output_pixel]) == ref["pixel"]
                assert (None if b.output_action is None else [int(v) for v in b.output_action]) == ref["actions"]
                assert (mine.episodes[0].episode_idx, len(mine.episodes[0].rgb_list)) == (ref["episode_idx"], ref["n_rgb"])
                if ref["s1_idx"] is not None:
                    rb = mine.s1_step_latent([0], [torch.zeros(1, 2, 4, 4, 3)], [torch.zeros(1, 2, 4, 4, 1)], [torch.zeros(1, 1, 1)])[0]
                    assert [int(v) for v in rb.idx] == ref["s1_idx"], k
            else:
                mine.step_no_infer([0], [o["rgb"]])


@pytest.mark.parametrize("seed,mode", [(201, "partial_async"), (202, "sync"), (203, "partial_async")])
def test_agent_vs_live_reference(seed, mode):
    from internnav_b200.agent import InternVLAN1Agent, PerEnvPolicies
    steps = next(t["steps"] for t in GOLD["agent"] if (t["seed"], t["mode"]) == (seed, mode))
    with contextlib.redirect_stdout(io.StringIO()):
        mpol = agent_script.ScriptedPolicy(agent_script_of(seed))
        mine = InternVLAN1Agent(PerEnvPolicies([mpol]), num_envs=1, infer_mode=mode, sys2_max_forward_step=8)
        mine.reset()
        mpol.drain()
        for ref in steps:
            k = ref["k"]
            if k == 17:
                mine.reset([0])
            b = mine.step([agent_script.make_obs(k)])
            assert [int(v) for v in b[0]["action"]] == ref["action"], k
            assert _json(mpol.drain()) == ref["calls"], k
            assert int(mine.dual_forward_step[0]) == ref["dual_forward_step"] and bool(mine.look_down[0]) == ref["look_down"]
