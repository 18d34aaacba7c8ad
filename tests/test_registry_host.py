"""Registry-level drop-in (SURVEY.md §8b) and checkpoint reading -- CPU only."""
import json
import os
import subprocess
import sys
from types import SimpleNamespace

import pytest
import torch

from internnav_b200.checkpoint import cfg_from_hf, read_checkpoint
from internnav_b200.qwen import QWEN25VL_7B
from oracle import agent_script

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _rerun_without_gpu(name):
    """Runs test `name` of this file in a child pytest that sees no CUDA device, so the no-device path is also checked on a
    machine that has one."""
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", "%s::%s" % (__file__, name)],
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), cwd=os.path.dirname(__file__), capture_output=True,
                       text=True)
    assert r.returncode == 0 and " passed" in r.stdout, r.stdout + r.stderr


FLAT_451 = dict(  # the released config.json layout (transformers 4.51): text fields at the top level
    architectures=["InternVLAN1ForCausalLM"], model_type="internvla_n1", hidden_size=3584, num_hidden_layers=28,
    num_attention_heads=28, num_key_value_heads=4, intermediate_size=18944, vocab_size=152064, rms_norm_eps=1e-6,
    rope_theta=1000000.0, rope_scaling={"type": "mrope", "mrope_section": [16, 24, 24]}, n_query=4, system1="navdp_async",
    vision_config=dict(depth=32, hidden_size=1280, num_heads=16, intermediate_size=3420, out_hidden_size=3584, patch_size=14,
                       temporal_patch_size=2, spatial_merge_size=2, window_size=112, fullatt_block_indexes=[7, 15, 23, 31]))


def test_config_translation_both_layouts():
    assert cfg_from_hf(FLAT_451) == QWEN25VL_7B
    nested = {k: v for k, v in FLAT_451.items() if k in ("vision_config", "n_query", "system1")}
    nested["text_config"] = {k: v for k, v in FLAT_451.items() if k not in ("vision_config", "n_query", "system1")}
    nested["text_config"]["rope_parameters"] = {"rope_type": "default", "rope_theta": 1000000.0, "mrope_section": [16, 24, 24]}
    del nested["text_config"]["rope_scaling"]
    assert cfg_from_hf(nested) == QWEN25VL_7B
    tiny = dict(FLAT_451, hidden_size=256, num_hidden_layers=2, num_attention_heads=2, num_key_value_heads=1,
                intermediate_size=512)
    c = cfg_from_hf(tiny)
    assert (c["hidden"], c["layers"], c["heads"], c["kv_heads"], c["head_dim"], c["inter"]) == (256, 2, 2, 1, 128, 512)


def test_read_sharded_safetensors(tmp_path):
    from safetensors.torch import save_file
    a = {"model.embed_tokens.weight": torch.randn(8, 4), "visual.merger.ln_q.weight": torch.ones(4).bfloat16()}
    b = {"model.navdp.layernorm.weight": torch.randn(3), "lm_head.weight": torch.randn(8, 4)}
    save_file(a, str(tmp_path / "model-00001-of-00002.safetensors"))
    save_file(b, str(tmp_path / "model-00002-of-00002.safetensors"))
    wm = {k: "model-00001-of-00002.safetensors" for k in a}
    wm.update({k: "model-00002-of-00002.safetensors" for k in b})
    (tmp_path / "model.safetensors.index.json").write_text(json.dumps({"weight_map": wm}))
    (tmp_path / "config.json").write_text(json.dumps(FLAT_451))
    cfg, conf, sd = read_checkpoint(str(tmp_path))
    assert cfg == QWEN25VL_7B and conf["system1"] == "navdp_async"
    assert set(sd) == set(a) | set(b)
    assert torch.equal(sd["lm_head.weight"], b["lm_head.weight"]) and sd["visual.merger.ln_q.weight"].dtype == torch.bfloat16
    (tmp_path / "empty").mkdir()
    (tmp_path / "empty" / "config.json").write_text(json.dumps(FLAT_451))
    with pytest.raises(FileNotFoundError):
        read_checkpoint(str(tmp_path / "empty"))


def test_from_pretrained_needs_a_gpu(tmp_path):
    """No CPU path: the checkpoint is parsed, then construction refuses a CPU device."""
    from safetensors.torch import save_file
    from internnav_b200.internvla_n1 import InternVLAN1ForCausalLM
    if torch.cuda.is_available():
        _rerun_without_gpu("test_from_pretrained_needs_a_gpu")
        return
    save_file({"model.norm.weight": torch.ones(4)}, str(tmp_path / "model.safetensors"))
    (tmp_path / "config.json").write_text(json.dumps(FLAT_451))
    with pytest.raises((RuntimeError, ImportError)):
        InternVLAN1ForCausalLM.from_pretrained(str(tmp_path), torch_dtype=torch.bfloat16,
                                               attn_implementation="flash_attention_2", device_map={"": "cpu"})


def test_registries_build_the_agent_from_config():
    from internnav_b200 import registry
    from internnav_b200.agent import PerEnvPolicies
    assert registry.get_policy("InternVLAN1_Policy") is registry.InternVLAN1Net
    assert registry.get_config("InternVLAN1_Policy") is registry.InternVLAN1ModelConfig
    with pytest.raises(ValueError):
        registry.get_policy("CMA_Policy")
    settings = dict(policy_name="InternVLAN1_Policy", env_num=2, infer_mode="partial_async", sys2_max_forward_step=8,
                    width=640, height=480, hfov=79, device="cuda:0", model_path="unused")
    cfg = SimpleNamespace(model_name="internvla_n1", model_settings=settings)        # AgentCfg's two fields that matter
    pols = [agent_script.ScriptedPolicy({"s2": [{"actions": [1, 2]}], "s1": [[1]]}) for _ in range(2)]
    ag = registry.Agent.init(cfg, policy=PerEnvPolicies(pols))
    assert isinstance(ag, registry.ConfiguredInternVLAN1Agent) and ag.num_envs == 2 and ag.mode == "partial_async"
    ag.reset()
    out = ag.step([agent_script.make_obs(0), agent_script.make_obs(0)])
    assert [o["action"] for o in out] == [[1], [1]] and all(o["ideal_flag"] for o in out)
    with pytest.raises(ValueError):
        registry.Agent.register("internvla_n1")(object)


def test_policy_from_config_uses_injected_collaborators():
    from internnav_b200 import registry
    from oracle import policy_script
    conf = registry.InternVLAN1ModelConfig(model_cfg={"model": dict(model_path="unused", device="cuda:0", num_history=4,
                                                                    resize_w=56, resize_h=56, env_num=3)})
    net = registry.InternVLAN1Net(conf, model=SimpleNamespace(device="cpu"), processor=policy_script.FakeProcessor())
    assert (net.num_history, net.resize_w, len(net.episodes)) == (4, 56, 3) and net.model_config.model_path == "unused"
