"""C2FTracker host side (no GPU): the two encoder levels of the eval backbone, the backbone check, and the config keys
the coarse-to-fine path does not implement."""
import pytest
import torch
import torch.nn as nn

BACKBONE = dict(type="ResNet", depth=18, strides=(1, 1, 1, 4), out_indices=(2, 3), pool_type="none")
CFG = dict(precede_frames=5, topk=10, temperature=0.07, neighbor_range=24, radius_fine=12)


class _Levels(nn.Module):
    """a backbone that returns zero feature maps of the given [C, H, W] shapes"""

    def __init__(self, *shapes):
        super().__init__()
        self.shapes = shapes

    def forward(self, x):
        out = tuple(torch.zeros(x.shape[0], *s) for s in self.shapes)
        return out[0] if len(out) == 1 else out


def test_eval_backbone_gives_the_config_3_levels():
    from fgvc_b200.encoder import ResNetEncoder
    enc = ResNetEncoder(depth=18, strides=(1, 1, 1, 4), out_indices=(2, 3), pool_type="none").eval()
    with torch.no_grad():
        fine, coarse = enc(torch.randn(2, 3, 256, 256))
    assert fine.shape == (2, 256, 128, 128) and coarse.shape == (2, 512, 32, 32)


def test_model_takes_fine_then_coarse_from_one_encoder_pass():
    import fgvc_b200
    model = fgvc_b200.B200C2FTracker(backbone=dict(BACKBONE), test_cfg=dict(CFG)).eval()
    assert fgvc_b200.B200C2FTracker is fgvc_b200.C2FTracker and model.two_phase_sharding
    with torch.no_grad():
        fine, coarse = model.extract_feat(torch.randn(1, 3, 64, 96))
    assert fine.shape == (1, 256, 32, 48) and coarse.shape == (1, 512, 8, 12)


@pytest.mark.parametrize("shapes", [
    [(256, 32, 32)],                                     # one level
    [(256, 32, 32), (512, 8, 8), (512, 4, 4)],           # three levels
    [(256, 30, 30), (512, 8, 8)],                        # non-integer ratio
    [(256, 32, 64), (512, 8, 8)],                        # unequal ratios in H and W
    [(512, 8, 8), (256, 32, 32)],                        # coarse level first
])
def test_backbone_without_two_nested_levels_raises_value_error(shapes):
    import fgvc_b200
    model = fgvc_b200.C2FTracker(backbone=_Levels(*shapes), test_cfg=dict(CFG))
    with pytest.raises(ValueError, match="out_indices=\\(2, 3\\)"):
        model.extract_feat(torch.zeros(1, 3, 64, 64))


@pytest.mark.parametrize("key,value", [("test_mode", "v2"), ("sim_mode", "l2-distance"), ("hard_prop", True),
                                       ("stride_sample", 2), ("topk", None), ("neighbor_range", None)])
def test_keys_the_c2f_path_does_not_implement_raise(key, value):
    import fgvc_b200
    with pytest.raises(NotImplementedError, match=key):
        fgvc_b200.C2FTracker(backbone=dict(BACKBONE), test_cfg=dict(CFG, **{key: value}))


def test_default_values_of_those_keys_are_accepted():
    import fgvc_b200
    fgvc_b200.C2FTracker(backbone=dict(BACKBONE), test_cfg=dict(CFG, test_mode="v1", sim_mode="dot_product",
                                                                hard_prop=False, stride_sample=False))
