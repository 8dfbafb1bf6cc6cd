"""Generates tests/golden/clip_text_small.npz by running the REFERENCE'S OWN src/utils/encode_text_word_embedding.py
(imported unmodified) on oracle/ladi_oracle/clip.py:ClipTextEncoder (which exposes the transformers-4.27 attribute surface that file
touches; its layer arithmetic is pinned against the installed transformers CLIPTextModel in tests/test_oracle_pins.py), CPU fp32,
seeded small-config weights.  Needs a checkout of miccunifi/ladi-vton:

    python tests/golden/make_golden_clip.py <ladi-vton checkout>

tests/test_oracle_pins.py imports this module for build(); only main() reads the checkout.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    sys.path.insert(0, p)

from ladi_oracle.clip import ClipTextEncoder  # noqa: E402

CFG = dict(vocab=1000, dim=64, heads=2, layers=2, mlp=128, max_pos=77)


def build(seed=1234):
    torch.manual_seed(seed)
    enc = ClipTextEncoder(**CFG).eval()
    g = torch.Generator().manual_seed(seed + 1)
    ids = torch.randint(1, 250, (4, 77), generator=g)
    ids[:, 0] = 998
    for b in range(4):
        ids[b, 12 + 5 * b:] = 999
    ids[0, 3:7] = 259   # 4 pseudo-words in the middle
    ids[2, 20:24] = 259
    ids[3, 9:11] = 259  # FIRST '$' at 9: window 9..12 (only 2 '$' tokens written, window still num_vstar wide)
    we = torch.randn((4, 4, CFG["dim"]), generator=g)
    return enc, ids, we


def main(reference):
    sys.path.insert(0, reference)
    from src.utils.encode_text_word_embedding import encode_text_word_embedding  # the reference file, unmodified
    enc, ids, we = build()
    with torch.no_grad():
        out = encode_text_word_embedding(enc, ids.clone(), we.clone(), 4)
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "clip_text_small.npz"), last_hidden_state=out.last_hidden_state.numpy(),
                        pooler_output=out.pooler_output.numpy(), input_ids=ids.numpy(), word_embeddings=we.numpy())
    print("wrote clip_text_small.npz", out.last_hidden_state.shape)


if __name__ == "__main__":
    main(sys.argv[1])
