"""Constructor behaviour of the UNet3DConditionModel mirror without a GPU: the three configuration checks of
models/unet_3d_condition_mask.py:118-131 raise the same ValueError as the verbatim reference class (whose outcome
tests/golden/unet_config_errors_ref.json records: `python tests/golden/make_golden.py config_errors`), the config object
exposes what callers read (train.py:91 `unet.config.in_channels`, models/pipeline.py:107 `unet.config.sample_size`),
`conv_in.weight/bias` are nn.Parameters (train.py:98-101), and unknown block types are rejected
(models/unet_3d_blocks.py:96,172)."""
import json
import os
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

TINY = dict(sample_size=16, block_out_channels=(64, 64, 64, 64), attention_head_dim=64, cross_attention_dim=32,
            motion_mask=True, motion_strength=True)
BAD = [
    dict(TINY, up_block_types=("UpBlock3D", "CrossAttnUpBlock3D", "CrossAttnUpBlock3D")),
    dict(TINY, block_out_channels=(64, 64, 64)),
    dict(TINY, attention_head_dim=(64, 64)),
]


def _reference_outcome(i):
    """What the reference's own class raised for BAD[i] (tests/golden/unet_config_errors_ref.json)."""
    with open(os.path.join(HERE, "golden", "unet_config_errors_ref.json")) as f:
        case = json.load(f)["cases"][i]
    assert case["config"] == json.loads(json.dumps(BAD[i])), "fixture was generated from a different config"
    return case["error"]


@pytest.mark.parametrize("i", range(len(BAD)))
def test_inconsistent_configs_raise_like_the_reference(i):
    from animate_anything_b200.unet_3d_condition_mask import UNet3DConditionModel
    ref = _reference_outcome(i)
    assert ref is not None and ref["type"] == "ValueError"
    with pytest.raises(ValueError) as e:
        UNet3DConditionModel(**BAD[i])
    assert str(e.value) == ref["message"]


def test_config_surface_and_parameters():
    from animate_anything_b200.unet_3d_condition_mask import UNet3DConditionModel
    m = UNet3DConditionModel(**TINY)
    assert m.config.in_channels == 4 and m.config.sample_size == 16
    assert isinstance(m.conv_in.weight, torch.nn.Parameter) and isinstance(m.conv_in.bias, torch.nn.Parameter)
    assert m.conv_in2.weight.shape[1] == 5                         # 4 latent channels + 1 mask channel (:140-142)
    assert hasattr(m, "motion_proj") or hasattr(m, "motion_embedding")
    m.requires_grad_(False).eval()
    assert m.dtype == torch.float32
    assert any(n.endswith("attn1.to_q.weight") for n in m.state_dict())


def test_unknown_block_type_rejected():
    from animate_anything_b200.unet_3d_condition_mask import UNet3DConditionModel
    with pytest.raises(ValueError):
        UNet3DConditionModel(**dict(TINY, down_block_types=("NoSuchBlock3D", "CrossAttnDownBlock3D", "CrossAttnDownBlock3D",
                                                            "DownBlock3D")))
