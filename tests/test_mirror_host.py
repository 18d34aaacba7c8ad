"""Host-side behaviour of the mirror classes that needs no GPU: argument handling, padding rules, error paths."""
import ctypes
import os
import subprocess
import sys
from types import SimpleNamespace

import pytest
import torch

from internnav_b200.internvla_n1 import IMAGE_TOKEN_INDEX, TRAJ_TOKEN_INDEX, InternVLAN1ForCausalLM


def _rerun_without_gpu(name):
    """Runs test `name` of this file in a child pytest that sees no CUDA device, so the no-device path is also checked on a
    machine that has one."""
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", "%s::%s" % (__file__, name)],
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), cwd=os.path.dirname(__file__), capture_output=True,
                       text=True)
    assert r.returncode == 0 and " passed" in r.stdout, r.stdout + r.stderr


class FakeS2:
    def __init__(self, gens):
        self.gens, self.calls = gens, []

    def generate(self, prompts, pixel_values, grid, max_new_tokens=128, eos_token_ids=(), pad_token_id=0,
                 with_latents=False):
        self.calls.append(dict(prompts=prompts, max_new=max_new_tokens, eos=tuple(eos_token_ids), pad=pad_token_id,
                               with_latents=with_latents))
        lat = torch.zeros(len(prompts), 4, 8) if with_latents else None
        return self.gens[: len(prompts)], lat, 3

    def generate_latents(self, prompts, pixel_values, grid):
        self.calls.append(dict(latent_prompts=prompts))
        return torch.arange(len(prompts) * 4 * 8, dtype=torch.float32).view(len(prompts), 4, 8)


def _model(gens=None):
    m = InternVLAN1ForCausalLM.__new__(InternVLAN1ForCausalLM)
    m.device = torch.device("cpu")
    m.config = SimpleNamespace(n_query=4, system1="navdp_async")
    m._s2 = FakeS2(gens or [])
    return m


def test_generate_sequences_layout_and_defaults():
    m = _model([[7, 8, 151645], [9, 151645]])
    prompts = [[1, 2, 3, 4], [5, 6]]                                     # ragged: left-padded like the HF processor does
    out = m.generate(prompts, None, [], max_new_tokens=5, return_dict_in_generate=True, use_cache=True,
                     past_key_values=None, attention_mask=None)
    assert out.sequences.tolist() == [[1, 2, 3, 4, 7, 8, 151645], [151643, 151643, 5, 6, 9, 151645, 151643]]
    assert out.generated == [[7, 8, 151645], [9, 151645]] and out.decode_passes == 3
    call = m._s2.calls[-1]
    assert call["eos"] == (151645, 151643) and call["pad"] == 151643 and call["max_new"] == 5 and not call["with_latents"]
    seq = m.generate(torch.tensor([[1, 2, 3, 4]]), None, [], eos_token_id=7, pad_token_id=0)
    assert torch.is_tensor(seq) and m._s2.calls[-1]["eos"] == (7,) and m._s2.calls[-1]["pad"] == 0
    both = m.generate_with_latents(prompts, None, [])
    assert both.latents.shape == (2, 4, 8) and m._s2.calls[-1]["with_latents"]


def test_generate_refuses_sampling():
    m = _model([[1]])
    with pytest.raises(NotImplementedError):
        m.generate([[1, 2]], None, [], do_sample=True)
    with pytest.raises(NotImplementedError):
        m.generate([[1, 2]], None, [], num_beams=4)


def test_training_prefix_extraction():
    m = _model()
    T, P, I = TRAJ_TOKEN_INDEX, 151643, IMAGE_TOKEN_INDEX
    ids = torch.tensor([[11, 12, I, 13, T, T, T, T, P, P],
                        [21, P, 22, 23, 24, 25, T, T, T, T]])            # a pad id inside sample 1 is masked, as the
    mask = ids.ne(P)                                                     # collator's input_ids.ne(pad) does
    hs = m.traj_hidden_states(ids, mask, None, [], [4, 6])
    assert m._s2.calls[-1]["latent_prompts"] == [[11, 12, I, 13], [21, 22, 23, 24, 25]]
    assert hs.shape == (2, 4, 8)
    with pytest.raises(ValueError):
        m.traj_hidden_states(ids, mask, None, [], [3, 6])
    bad = torch.tensor([[11, T, T, T, T, I, 12, P]])
    with pytest.raises(NotImplementedError):
        m.traj_hidden_states(bad, bad.ne(P), None, [], [1])
    with pytest.raises(NotImplementedError):
        m.forward(input_ids=ids)                                         # inference-style call: use generate*()


def test_resize_plan_needs_a_device():
    """Compute entry points fail loudly without a B200 (no host fallback behind the C ABI)."""
    from internnav_b200 import _lib
    from internnav_b200.preprocess import FramePreprocessor, _bind
    if torch.cuda.is_available():
        _rerun_without_gpu("test_resize_plan_needs_a_device")
        return
    L = _lib.lib()
    _bind(L)
    p = ctypes.c_void_p()
    assert L.n1_resize_plan_create(480, 640, 224, 224, ctypes.byref(p), None) != 0
    assert len(L.n1_last_error()) > 0
    with pytest.raises(RuntimeError):
        FramePreprocessor("cpu")
