"""Pins the System-1 oracle (oracle/navdp_oracle.py) -- CPU only.

tests/golden/s1_reference_outputs.npz and traj_to_actions.json hold OUTPUTS of the reference's own modules
(/root/reference imported by oracle/gen_golden.py) on seeded weights/inputs that this test regenerates from their seeds.
"""
import json
import os

import numpy as np
import pytest
import torch

from oracle import navdp_oracle as O, weights

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = np.load(os.path.join(ROOT, "tests", "golden", "s1_reference_outputs.npz"))
TOL = dict(atol=5e-5, rtol=1e-4)  # fp32 CPU vs fp32 CPU, different summation orders


@pytest.fixture(scope="module")
def sd():
    torch.set_num_threads(os.cpu_count())
    return weights.make_state_dict(0)


def test_rgbd_encoder_golden(sd):
    inp = weights.make_inputs(101, B=2)
    with torch.no_grad():
        out = O.rgbd_encoder(sd, inp["rgb"], inp["depth"])
    assert np.allclose(out.numpy(), GOLD["rgbd_B2"], **TOL), np.abs(out.numpy() - GOLD["rgbd_B2"]).max()


def test_goal_token_golden(sd):
    inp = weights.make_inputs(102, B=3)
    with torch.no_grad():
        out = O.goal_token(sd, inp["latents"])  # batched call == the reference's per-env bs=1 calls
    assert np.allclose(out.numpy(), GOLD["goal_B3"], **TOL)


@pytest.mark.parametrize("tag,T,k", [("T32", 32, 7), ("T8", 8, 13)])
def test_predict_noise_golden(sd, tag, T, k):
    inp = weights.make_inputs(103, B=1, T=T, Ns=32)
    with torch.no_grad():
        out = O.predict_noise(sd, inp["x_init"], torch.tensor([k]), inp["goal"], inp["rgbd"])
    assert np.allclose(out.numpy(), GOLD["eps_" + tag], **TOL), np.abs(out.numpy() - GOLD["eps_" + tag]).max()


def test_full_sampling_golden(sd):
    inp = weights.make_inputs(104, B=1, K=20)
    with torch.no_grad():
        out = O.predict_pointgoal_action_async(sd, inp["latents"], inp["rgb"], inp["depth"], inp["x_init"],
                                               inp["step_noise"], K=20)
    assert np.allclose(out.numpy(), GOLD["traj_full"], atol=2e-4, rtol=1e-3), np.abs(out.numpy() - GOLD["traj_full"]).max()


def test_batched_equals_per_env(sd):
    """The B-environment generalisation equals the bs=1 reference semantics applied per environment (SURVEY.md F4)."""
    inp = weights.make_inputs(106, B=2, T=8, Ns=4)
    k = torch.tensor([5])
    with torch.no_grad():
        both = O.predict_noise(sd, inp["x_init"], k, inp["goal"], inp["rgbd"])
        for b in range(2):
            one = O.predict_noise(sd, inp["x_init"][b * 4:(b + 1) * 4], k, inp["goal"][b:b + 1], inp["rgbd"][b:b + 1])
            assert torch.allclose(both[b * 4:(b + 1) * 4], one, atol=1e-5)


def _action_cases():
    rng = np.random.Generator(np.random.PCG64(105))
    out = []
    for i in range(12):
        out.append(torch.from_numpy(rng.standard_normal((32, 32, 3), dtype=np.float32) * 0.15 +
                                    np.array([0.5 * np.cos(i), 0.5 * np.sin(i), 0.0], dtype=np.float32)))
    out.append(torch.from_numpy(GOLD["traj_full"].copy()))
    return out


def test_traj_to_actions_golden_bit_exact():
    with open(os.path.join(ROOT, "tests", "golden", "traj_to_actions.json")) as fh:
        gold = json.load(fh)
    from internnav_b200 import postprocess as P
    cases = _action_cases()
    assert len(cases) == len(gold)
    for tr, g in zip(cases, gold):
        assert O.traj_to_actions(tr) == g                       # oracle restatement
        assert P.traj_to_actions(tr.clone()) == g               # product host code
        assert P.batched_traj_to_actions(tr, 1)[0] == g
        # early-exit variant keeps exactly the entries s1_step_latent consumes
        assert P.s1_action_list(P.batched_traj_to_actions(tr, 1, max_actions=4)[0]) == P.s1_action_list(g)
    # empty / degenerate trajectories: the reference returns [] -> action -1 upstream
    z = torch.zeros(32, 8, 3)
    assert O.traj_to_actions(z) == [] and P.traj_to_actions(z.clone()) == []
    # in-place contract of the reference function (vln_utils.py L129)
    t = cases[0].clone()
    P.traj_to_actions(t)
    assert torch.allclose(t[:, :, :2], cases[0][:, :, :2] / 4.0)


def test_ddpm_properties():
    """Known answers of the scheduler restatement: cosine ᾱ endpoints, last step has zero variance and returns the
    clipped x0 prediction, add_noise/step consistency at t = 0."""
    from oracle import ddpm
    s = ddpm.DDPMScheduler(num_train_timesteps=20)
    import math
    abar = lambda u: math.cos((u + 0.008) / 1.008 * math.pi / 2) ** 2  # noqa: E731
    assert abs(float(s.alphas_cumprod[0]) - abar(1 / 20) / abar(0.0)) < 1e-6
    assert abs(float(s.alphas_cumprod[9]) - abar(10 / 20) / abar(0.0)) < 1e-5 and float(s.alphas_cumprod[-1]) < 1e-4
    assert float(s.betas.max()) <= 0.999 + 1e-6
    s.set_timesteps(20)
    assert s.timesteps.tolist() == list(range(19, -1, -1))
    x = torch.randn(4, 8, 3)
    eps = torch.randn(4, 8, 3)
    out = s.step(eps, 0, x).prev_sample
    a0 = s.alphas_cumprod[0]
    x0 = ((x - (1 - a0) ** 0.5 * eps) / a0 ** 0.5).clamp(-1, 1)
    assert torch.allclose(out, x0, atol=1e-6)


def test_ddpm_step_is_the_gaussian_posterior_of_the_forward_process():
    """Independent known-answer check of oracle/ddpm.py (the one unpinned oracle piece: diffusers is neither vendored
    nor installed).  Nothing here uses the scheduler's own formulas: the forward process q(x_t | x_{t-1}) =
    N(sqrt(1 - beta_t) x_{t-1}, beta_t) and q(x_{t-1} | x_0) = N(sqrt(abar_{t-1}) x_0, 1 - abar_{t-1}) are combined with
    the textbook product-of-Gaussians rule (precision-weighted mean) in float64.  The ancestral step with the true x_0
    substituted must reproduce that posterior's mean, and its injected-noise scale must be the posterior's standard
    deviation (variance_type 'fixed_small' == Ho et al. 2020 eq. 7); the kernel's tables (n1_ddpm_tables, checked
    against this scheduler in tests/test_abi_symbols.py / test_s1_gpu.py) inherit the check.  Also pins the constructor
    arguments the reference's own tree documents for this class
    (internnav/model/encoder/diffusion_policy/config/*.yaml: variance_type fixed_small, clip_sample True,
    prediction_type epsilon, beta_schedule squaredcos_cap_v2)."""
    import math
    from oracle import ddpm
    N = 20
    s = ddpm.DDPMScheduler(num_train_timesteps=N)
    s.set_timesteps(N)
    abar_fn = lambda u: math.cos((u + 0.008) / 1.008 * math.pi / 2) ** 2  # noqa: E731  (Nichol & Dhariwal 2021, eq. 17)
    beta = [min(1 - abar_fn((i + 1) / N) / abar_fn(i / N), 0.999) for i in range(N)]
    abar = [1.0]
    for b in beta:
        abar.append(abar[-1] * (1 - b))          # abar[t + 1] = prod_{j <= t} (1 - beta_j); abar[0] = 1 is "t = -1"
    g = torch.Generator().manual_seed(0)
    x0 = torch.rand(5, 8, 3, generator=g, dtype=torch.float64) * 1.6 - 0.8      # inside the clip range
    for t in range(N - 1, 0, -1):
        eps = torch.randn(5, 8, 3, generator=g, dtype=torch.float64)
        a_t, a_prev = abar[t + 1], abar[t]
        x_t = math.sqrt(a_t) * x0 + math.sqrt(1 - a_t) * eps                   # forward marginal (add_noise)
        assert torch.allclose(s.add_noise(x0.float(), eps.float(), torch.tensor([t])).double(), x_t, atol=2e-6)
        # product of N(x_{t-1}; sqrt(a_prev) x0, 1 - a_prev) and the likelihood of x_t given x_{t-1}
        prec_prior = 1.0 / (1 - a_prev)
        prec_lik = (1 - beta[t]) / beta[t]                                     # (sqrt(1-beta))^2 / beta
        var_post = 1.0 / (prec_prior + prec_lik)
        mean_post = var_post * (prec_prior * math.sqrt(a_prev) * x0 + math.sqrt(1 - beta[t]) / beta[t] * x_t)
        z = torch.randn(5, 8, 3, generator=g)
        s.noise_queue = [z.clone()]
        out = s.step(eps.float(), t, x_t.float()).prev_sample.double()         # eps is the true noise -> x0 recovered
        assert torch.allclose(out, mean_post + math.sqrt(var_post) * z.double(), atol=5e-5), t
    # t = 0: no noise is added and the clipped x0 prediction is returned
    eps = torch.randn(5, 8, 3, generator=g, dtype=torch.float64)
    x_t = math.sqrt(abar[1]) * x0 + math.sqrt(1 - abar[1]) * eps
    s.noise_queue = []
    assert torch.allclose(s.step(eps.float(), 0, x_t.float()).prev_sample.double(), x0, atol=5e-6)


def test_oracle_vs_reference_modules(sd):
    """Direct comparison with the reference classes on inputs of seed 107: their outputs are recorded in
    tests/golden/reference_checks.npz (oracle/gen_golden_checks.py)."""
    ref = np.load(os.path.join(ROOT, "tests", "golden", "reference_checks.npz"))
    inp = weights.make_inputs(107, B=1)
    with torch.no_grad():
        o = O.rgbd_encoder(sd, inp["rgb"], inp["depth"])
        assert torch.allclose(torch.from_numpy(ref["navdp_rgbd"]), o, **TOL)
        g = O.goal_token(sd, inp["latents"])
        assert torch.allclose(torch.from_numpy(ref["navdp_goal"]), g, **TOL)
        k = torch.tensor([3])
        assert torch.allclose(torch.from_numpy(ref["navdp_eps"]), O.predict_noise(sd, inp["x_init"], k, g, o), **TOL)


def test_training_branch_forward_and_gradients_vs_reference(sd):
    """Row a13, System-1 half: the oracle's forward_vlm_traj + masked MSE and ONE autograd backward through it against
    tests/golden/s1_training_reference.npz -- prediction, loss, per-parameter gradient norms and seeded projections,
    and the gradient w.r.t. the latent tokens, all produced by the reference's own module (oracle/gen_golden_training.py).
    Also pins which parameters train at all: the RGB ViT is detached in the reference (navdp_backbone.py L170-171)."""
    from oracle import gen_golden_training as G
    gold = np.load(os.path.join(ROOT, "tests", "golden", "s1_training_reference.npz"))
    b = G.make_batch()
    with torch.no_grad():
        imgs, deps = G.dp_inputs(b)
        f = b["traj_images"].shape[1]
        hs_rep = b["hs"].unsqueeze(1).repeat(1, f, 1, 1).flatten(0, 1)
        pred, _ = O.forward_vlm_traj(sd, hs_rep, imgs, deps, b["traj_poses"].flatten(0, 1), b["noise"], b["timesteps"])
    assert np.allclose(pred.numpy(), gold["pred"], **TOL), np.abs(pred.numpy() - gold["pred"]).max()
    loss, grads, g_hs = O.s1_training_grads(sd, b["hs"], b["traj_images"], b["traj_depths"], b["traj_poses"],
                                            b["video_frame_num"], b["noise"], b["timesteps"])
    assert abs(float(loss) - float(gold["loss"])) < 1e-5 * max(1.0, float(gold["loss"]))
    names = [str(n) for n in gold["grad_names"]]
    assert sorted(grads) == sorted(names), set(grads) ^ set(names)
    assert not any(k.startswith("rgbd_encoder.rgb_model.") for k in grads)
    for n, norm, dot in zip(names, gold["grad_norms"], gold["grad_dots"]):
        g = grads[n]
        assert abs(float(g.norm()) - norm) <= 2e-4 * norm + 1e-9, (n, float(g.norm()), norm)
        mine = float((g * G.probe(n, tuple(g.shape))).sum())
        assert abs(mine - dot) <= 1e-3 * norm + 2e-4 * abs(dot) + 1e-7, (n, mine, dot)   # |g . probe| ~ |g|
    assert np.allclose(g_hs.numpy(), gold["grad_hs"], atol=1e-7, rtol=2e-3), np.abs(g_hs.numpy() - gold["grad_hs"]).max()


def test_handwritten_backward_matches_autograd(sd):
    """oracle/navdp_backward.py (explicit dgrad / wgrad / LayerNorm / GELU / softmax-attention backward, the spec of the
    backward kernels) against autograd through the restated forward: loss, every parameter gradient, d loss / d latents."""
    from oracle import gen_golden_training as G, navdp_backward as NB
    b = G.make_batch(dict(G.CASE, seed=202))
    args = (b["hs"], b["traj_images"], b["traj_depths"], b["traj_poses"], b["video_frame_num"], b["noise"], b["timesteps"])
    loss_a, grads_a, dhs_a = O.s1_training_grads(sd, *args)
    with torch.no_grad():
        loss_m, grads_m, dhs_m = NB.s1_training_backward(sd, *args)
    assert abs(float(loss_a) - float(loss_m)) < 1e-6 * max(1.0, abs(float(loss_a)))
    assert sorted(grads_a) == sorted(grads_m), set(grads_a) ^ set(grads_m)
    worst = ("", 0.0)
    for k, ga in grads_a.items():
        gm = grads_m[k].reshape(ga.shape)
        rel = float((gm - ga).norm() / (ga.norm() + 1e-12))
        if rel > worst[1]:
            worst = (k, rel)
        assert rel < 2e-3 or float((gm - ga).abs().max()) < 1e-8, (k, rel)
    rel_h = float((dhs_m - dhs_a).norm() / dhs_a.norm())
    print("worst parameter gradient rel err", worst, "latent gradient rel err", rel_h)
    assert rel_h < 2e-3
