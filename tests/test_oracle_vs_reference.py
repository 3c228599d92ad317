"""Pins the oracle's wiring restatement (oracle/unet3d_ref.py) against the reference's OWN models/*.py: the outputs and
parameter shapes in tests/golden/oracle_vs_reference.pt come from those files imported unmodified
(tests/golden/make_golden_reference.py), on weights the test redraws with helpers.seeded_state_dict."""
import os

import pytest
import torch

from helpers import seeded_state_dict
from oracle import unet3d_ref as R

GOLDEN = torch.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "oracle_vs_reference.pt"), weights_only=False)
SMALL = dict(block_out_channels=(64, 128, 128, 128), attention_head_dim=32, cross_attention_dim=64)


def _weights():
    from t2v_b200.models.unet_3d_condition import UNet3DConditionModel
    assert GOLDEN["cfg"] == SMALL
    with torch.device("meta"):
        m = UNet3DConditionModel(**SMALL)
    return seeded_state_dict(m, GOLDEN["weight_seed"], conv4_std=GOLDEN["conv4_std"])


@pytest.mark.parametrize("frames,hw", [(4, 16), (1, 8), (3, 12)])
def test_wiring_matches_reference(frames, hw):
    c = GOLDEN["wiring"][f"{frames}x{hw}"]
    y_ref = c["y"]
    assert c["x"].shape == (2, 4, frames, hw, hw)
    with torch.no_grad():
        y = R.unet3d_forward(_weights(), R.full_config(**SMALL), c["x"], c["t"], c["ehs"])
    assert y.shape == y_ref.shape
    assert (y - y_ref).abs().max().item() <= 2e-5 * y_ref.abs().max().item()


def test_checkpointed_reference_equals_plain():
    """The reference with gradient checkpointing gives its plain output bit for bit, and the oracle reproduces both."""
    c = GOLDEN["checkpointed"]
    assert torch.equal(c["y_plain"], c["y_checkpointed"])
    with torch.no_grad():
        y = R.unet3d_forward(_weights(), R.full_config(**SMALL), c["x"], c["t"], c["ehs"])
    assert (y - c["y_checkpointed"]).abs().max().item() <= 2e-5 * c["y_checkpointed"].abs().max().item()


def test_structural_pins_full_size():
    """1,411,233,860 parameters / 1,480 tensors for the ms-1.7b configuration, same keys+shapes as the product model."""
    from t2v_b200.models.unet_3d_condition import UNet3DConditionModel
    with torch.device("meta"):
        mine = UNet3DConditionModel()
    a = dict(GOLDEN["full_size_shapes"])
    b = {k: tuple(v.shape) for k, v in mine.state_dict().items()}
    assert len(a) == 1480 and sum(torch.Size(s).numel() for s in a.values()) == 1_411_233_860
    assert a == b
