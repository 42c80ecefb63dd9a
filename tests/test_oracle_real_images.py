"""CPU: the oracle port on two committed stills of the reference's test video reproduces what the UNMODIFIED reference
modules produced on them in the build container (tests/golden/real/*.npz, scripts/make_real_golden.py)."""
import os

import numpy as np
import pytest
import torch
from PIL import Image

from oracle import net, synth

REAL = os.path.join(synth.GOLDEN_DIR, "real")
# The goldens were computed with 8 CPU threads.  fp32 CPU convolutions and reductions sum in an order that depends on
# the thread count, and on still 0 (an all-black frame) the SceneSeg logits amplify that to several times the gate
# below, so the oracle runs with the same thread count whatever the host's default.
GOLDEN_THREADS = 8


@pytest.fixture
def golden_threads():
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(n)


@pytest.mark.parametrize("model", ["scene_seg", "ego_lanes"])
def test_oracle_equals_reference_on_real_stills(model, golden_threads):
    sd = synth.synth_state_dict(model)
    gold = np.load(os.path.join(REAL, f"{model}_real.npz"))
    for i in (0, 28):
        small = np.asarray(Image.open(os.path.join(REAL, f"frame_{i:02d}.png")).convert("RGB"))
        out = net.forward(model, sd, net.to_tensor_normalize(small))
        o = out[0].numpy()
        assert np.abs(o[:, ::8, ::8] - gold[f"sample_{i}"]).max() <= 1e-4 * max(1.0, float(gold[f"std_{i}"]))
        post = np.asarray(net.postprocess(model, out)) if model == "scene_seg" else net.ego_lanes_masks(o)[1]
        bad = post.astype(np.uint8) != gold[f"post_{i}"]
        assert bad.mean() <= 1e-5          # identical up to exact ties between thread counts
