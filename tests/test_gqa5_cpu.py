"""Qwen3-14B (40 q / 8 kv heads, GQA group 5) and Qwen3-32B (64 / 8): the registered specs
against transformers' own config and model classes, the groups that stay refused, and the
oracle on the group-5 parity model against its golden transformers logits."""
import os

import numpy as np
import pytest

from oracle.model_ref import RefModel
from sutro_b200 import modelspec as MS
from sutro_b200 import pretrained as PT

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# public model-card values (config.json of Qwen/Qwen3-14B and Qwen/Qwen3-32B)
CARDS = {
    "qwen-3-14b": dict(num_hidden_layers=40, hidden_size=5120, num_attention_heads=40,
                       num_key_value_heads=8, intermediate_size=17408),
    "qwen-3-32b": dict(num_hidden_layers=64, hidden_size=5120, num_attention_heads=64,
                       num_key_value_heads=8, intermediate_size=25600),
}


def qwen3_config(name, **over):
    from transformers import Qwen3Config
    kw = dict(CARDS[name], vocab_size=151936, head_dim=128, max_position_embeddings=40960,
              rms_norm_eps=1e-6, rope_theta=1e6, tie_word_embeddings=False)
    kw.update(over)
    return Qwen3Config(**kw)


@pytest.mark.parametrize("name", ["qwen-3-14b", "qwen-3-32b"])
def test_spec_from_transformers_config_equals_the_registered_spec(name):
    spec = MS.get_spec(name)
    assert PT.spec_from_hf_config(qwen3_config(name).to_dict(), name) == spec
    assert MS.get_spec(name + "-thinking") is spec
    assert spec.n_q_heads // spec.n_kv_heads == (5 if name == "qwen-3-14b" else 8)


@pytest.mark.parametrize("name", ["qwen-3-14b", "qwen-3-32b"])
def test_parameter_count_equals_transformers(name):
    import torch
    from transformers import Qwen3ForCausalLM
    with torch.device("meta"):
        m = Qwen3ForCausalLM(qwen3_config(name))
    assert MS.get_spec(name).n_params() == sum(p.numel() for p in m.parameters())


@pytest.mark.parametrize("hq,hkv", [(24, 8), (48, 8), (128, 8)])   # groups 3, 6, 16
def test_other_groups_are_still_refused(hq, hkv):
    cfg = qwen3_config("qwen-3-14b", num_attention_heads=hq, num_key_value_heads=hkv).to_dict()
    with pytest.raises(ValueError, match="GQA group"):
        PT.spec_from_hf_config(cfg, "x")


def test_rope_theta_is_read_from_either_config_layout():
    flat = dict(qwen3_config("qwen-3-14b").to_dict(), rope_theta=5e5)
    flat.pop("rope_parameters")
    assert PT.spec_from_hf_config(flat, "x").rope_theta == 5e5
    assert PT.spec_from_hf_config(qwen3_config("qwen-3-14b", rope_theta=5e5).to_dict(),
                                  "x").rope_theta == 5e5


def test_oracle_logits_match_golden_transformers_logits_group5():
    # same fixture recipe and bars as test_golden.py
    name = "tiny-qwen3-g5"
    z = np.load(os.path.join(G, f"hf_logits_{name}.npz"))
    spec = MS.get_spec(name)
    assert spec.n_q_heads // spec.n_kv_heads == 5
    w = MS.make_weights(spec, seed=3, std=0.05)
    got = RefModel(spec, w).logits(z["ids"].tolist())[-4:].numpy()
    want = z["logits_last4"]
    scale = want.std()
    assert np.abs(got - want).max() < 0.1 * scale
    assert np.abs(got - want).mean() < 0.015 * scale
    top2 = np.sort(want, axis=-1)[:, -2:]
    decided = (top2[:, 1] - top2[:, 0]) > 0.05 * scale
    assert (got.argmax(-1)[decided] == want.argmax(-1)[decided]).all()
