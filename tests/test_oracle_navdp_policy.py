"""Stand-alone NavDP policy (SURVEY.md §8f-3): the oracle restatement (oracle/navdp_policy_oracle.py) against outputs of the
REFERENCE's own NavDPNet (tests/golden/navdp_policy_reference.npz, produced by oracle/gen_golden_navdp_policy.py from
internnav/model/basemodel/navdp/navdp_policy.py), same seeded weights and inputs; and the manifest against the state-dict shapes of the reference class (tests/golden/reference_traces.json)."""
import os

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = dict(atol=2e-4, rtol=2e-4)


@pytest.fixture(scope="module")
def setup():
    from internnav_b200.manifest import random_navdp_policy_state_dict
    from oracle.gen_golden_navdp_policy import make_inputs
    torch.set_num_threads(os.cpu_count())
    gold = dict(np.load(os.path.join(ROOT, "tests", "golden", "navdp_policy_reference.npz")))
    return random_navdp_policy_state_dict(seed=7), make_inputs(), gold


def test_oracle_equals_reference_outputs(setup):
    from oracle import navdp_policy_oracle as P, navdp_oracle as O
    sd, inp, gold = setup
    with torch.no_grad():
        rgbd = P.rgbd_backbone(sd, inp["images"], inp["depths"])
        assert torch.allclose(rgbd, torch.from_numpy(gold["rgbd"]), **TOL)
        goal = O._lin(sd, "point_encoder", inp["goal"]).unsqueeze(1)
        eps = P.predict_noise(sd, inp["x_init"], torch.tensor([7]), goal, rgbd)
        assert torch.allclose(eps, torch.from_numpy(gold["eps"]), **TOL)
        cr = P.predict_critic(sd, inp["x_init"], rgbd)
        assert torch.allclose(cr, torch.from_numpy(gold["critic_of_x_init"]), **TOL)
        neg, pos, _, _ = P.predict_pointgoal_batch_action_vel(sd, inp["goal"], inp["images"], inp["depths"], inp["x_init"],
                                                              inp["step_noise"])
        assert torch.allclose(neg, torch.from_numpy(gold["pointgoal_negative"]), atol=2e-3, rtol=2e-3)
        assert torch.allclose(pos, torch.from_numpy(gold["pointgoal_positive"]), atol=2e-3, rtol=2e-3)
        neg, pos, _, _ = P.predict_nogoal_batch_action_vel(sd, inp["images"], inp["depths"], inp["x_init"], inp["step_noise"])
        assert torch.allclose(neg, torch.from_numpy(gold["nogoal_negative"]), atol=2e-3, rtol=2e-3)
        assert torch.allclose(pos, torch.from_numpy(gold["nogoal_positive"]), atol=2e-3, rtol=2e-3)


def test_manifest_matches_reference_class():
    """The shape manifest used for random initialisation equals the reference class's own state_dict, whose shapes
    tests/golden/reference_traces.json records (oracle/gen_golden_checks.py)."""
    import json
    from internnav_b200.manifest import navdp_policy_shapes
    with open(os.path.join(ROOT, "tests", "golden", "reference_traces.json"), encoding="utf-8") as fh:
        ref = {k: tuple(v) for k, v in json.load(fh)["navdp_policy_shapes"].items()}
    mine = {k: tuple(v) for k, v in navdp_policy_shapes().items()}
    assert mine == ref, (set(mine) ^ set(ref))
