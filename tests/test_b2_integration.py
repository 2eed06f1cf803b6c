"""Module boundary (SURVEY.md §8 b2): QAHeadV1 keeps the reference head's state_dict contract and output.
The golden tests/golden/model_qa_head.npz is the UNMODIFIED reference head run on CPU in fp32 on the same seeded weights
and inputs (oracle/make_golden_model.py::golden_qa_head)."""
import json
import os

import numpy as np
import torch

from sceneverse_b200 import weights

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def test_qa_head_matches_reference():
    from sceneverse_b200.modules import heads
    z = np.load(os.path.join(GOLDEN, "model_qa_head.npz"))
    mine = heads.QAHeadV1(None, num_answers=200).eval()
    ref_shapes = json.loads(str(z["state_dict_shapes"]))
    mine.load_state_dict(weights.synthetic_state_dict(ref_shapes, seed=int(z["weight_seed"])), strict=True)  # same keys and shapes
    g = torch.Generator().manual_seed(int(z["input_seed"]))
    obj, txt = torch.randn(3, 20, 768, generator=g), torch.randn(3, 12, 768, generator=g)
    om = torch.rand(3, 20, generator=g) > 0.3
    om[:, 0] = True
    tm = torch.arange(12)[None, :] < torch.tensor([12, 5, 9])[:, None]
    with torch.no_grad():
        got = mine(obj, om, txt, tm)
    want = z["out"]
    assert got.shape == want.shape
    assert np.abs(got.numpy() - want).max() <= 1e-5 * np.abs(want).max()
