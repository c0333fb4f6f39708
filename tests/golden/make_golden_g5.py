"""Generates hf_logits_tiny-qwen3-g5.npz, the golden logits of the GQA-group-5 parity model
(10 q / 2 kv heads), with the recipe of make_golden.py: transformers 5.5.0 fp32 logits (last 4
positions) of the seeded tiny architecture on the same fixed id sequence.

    python tests/golden/make_golden_g5.py     # writes only this fixture

It is a separate script so that regenerating it leaves the other fixtures alone (a re-saved
zip differs byte for byte from the committed one even when its arrays are equal).
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))

from sutro_b200 import modelspec as MS  # noqa: E402

NAME = "tiny-qwen3-g5"


def main():
    import transformers
    from test_oracle_vs_hf import hf_model
    spec = MS.get_spec(NAME)
    w = MS.make_weights(spec, seed=3, std=0.05)
    ids = torch.randint(0, spec.vocab_size, (40,), generator=torch.Generator().manual_seed(1))
    with torch.no_grad():
        lg = hf_model(spec, w)(ids[None]).logits[0, -4:].float().numpy()
    path = os.path.join(HERE, f"hf_logits_{NAME}.npz")
    np.savez_compressed(path, ids=ids.numpy(), logits_last4=lg.astype(np.float32),
                        transformers=np.array(transformers.__version__))
    print("golden fixture written to", path)


if __name__ == "__main__":
    main()
