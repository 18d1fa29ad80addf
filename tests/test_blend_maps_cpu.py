"""CPU: the restatement of the per-pixel blend (tests/blend_maps_oracle.py) against scipy and
F.interpolate, and MultiStyleStylizer's argument validation for weight maps (raised before any device work)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import restate as R
from tests import blend_maps_oracle as BM

scipy_ndimage = pytest.importorskip("scipy.ndimage")


@pytest.mark.parametrize("hw", [(1, 1), (3, 50), (64, 48), (17, 300)])
@pytest.mark.parametrize("sigma", [0.5, 2.0, 6.3])
def test_gaussian_blur_matches_scipy(hw, sigma):
    """includes radii >= the plane size (reflection folded more than once)"""
    g = torch.Generator().manual_seed(hash((hw, sigma)) % 2 ** 31)
    planes = torch.rand(2, 3, *hw, generator=g, dtype=torch.float64)
    got = BM.gaussian_blur(planes, sigma)
    for idx in np.ndindex(2, 3):
        ref = scipy_ndimage.gaussian_filter(planes[idx].numpy(), sigma, mode="reflect", truncate=4.0)
        assert np.abs(got[idx].numpy() - ref).max() <= 1e-12, (hw, sigma, idx)


def test_gaussian_blur_sigma_zero_is_identity():
    planes = torch.rand(2, 4, 9, 13, dtype=torch.float64)
    assert torch.equal(BM.gaussian_blur(planes, 0.0), planes)


@pytest.mark.parametrize("hw,HW", [((1, 1), (8, 12)), ((5, 7), (40, 56)), ((16, 16), (64, 64)), ((7, 9), (7, 9)),
                                   ((13, 10), (50, 31))])
def test_sample_maps_matches_interpolate(hw, HW):
    g = torch.Generator().manual_seed(3)
    maps = torch.rand(2, 4, *hw, generator=g)
    got = BM.sample_maps(maps, *HW)
    ref = F.interpolate(maps, size=HW, mode="bilinear", align_corners=False)
    assert (got - ref).abs().max() <= 1e-6
    const = torch.full((1, 3, *hw), 0.3)
    assert torch.equal(BM.sample_maps(const, *HW), torch.full((1, 3, *HW), 0.3))


def test_blend_maps_with_constant_maps_is_blend_outputs():
    g = torch.Generator().manual_seed(5)
    ys = [torch.rand(2, 3, 10, 14, generator=g) * 2 - 1 for _ in range(3)]
    x = torch.rand(2, 3, 10, 14, generator=g) * 2 - 1
    w, w_x = [0.2, 0.3, 0.5], 0.4
    maps = torch.tensor(w + [w_x]).view(1, 4, 1, 1).expand(1, 4, 3, 5).contiguous()
    assert torch.equal(BM.blend_maps(ys, maps[:, :3], gain=1.1, clip=(-1, 1)), R.blend_outputs(ys, w, gain=1.1, clip=(-1, 1)))
    assert torch.equal(BM.blend_maps(ys, maps, x=x), R.blend_outputs(ys, w, x=x, w_x=w_x))


def test_blend_maps_normalize():
    ys = [torch.full((1, 3, 4, 4), float(s + 1)) for s in range(2)]
    maps = torch.zeros(1, 2, 4, 4)
    maps[0, 0, :, :2] = 3.0
    maps[0, 1, :, :2] = 1.0                     # left half: weights 0.75 / 0.25; right half: all zero
    out = BM.blend_maps(ys, maps, normalize=True)
    assert torch.allclose(out[..., :2], torch.full((1, 3, 4, 2), 1.25))
    assert torch.equal(out[..., 2:], torch.zeros(1, 3, 4, 2))


# ---- MultiStyleStylizer argument validation -------------------------------------------------------------------------------
S, B, H, W = 3, 4, 32, 48


def check(weights=None, w_x=0.0, weight_maps=None, feather_sigma=0.0):
    from multi_style_transfer_gan_b200.stylize import check_blend_args
    check_blend_args(S, B, H, W, weights, w_x, weight_maps, feather_sigma)


def test_blend_args_accept_valid_inputs():
    check(weights=[0.2, 0.3, 0.5], w_x=0.1)
    check(weight_maps=torch.rand(1, S, 1, 1))
    check(weight_maps=torch.rand(B, S + 1, H, W), feather_sigma=2.0)
    check(weight_maps=torch.rand(B, S, 8, 12).double())


@pytest.mark.parametrize("kwargs", [
    dict(),                                                                      # neither
    dict(weights=[0.2, 0.3, 0.5], weight_maps=torch.rand(1, S, 1, 1)),           # both
    dict(weights=[0.5, 0.5]),                                                    # wrong number of global weights
    dict(weight_maps=torch.rand(1, S, 1, 1), w_x=0.5),                           # w_x with maps
    dict(weight_maps=torch.rand(1, S + 2, 1, 1)),                                # wrong K
    dict(weight_maps=torch.rand(1, S - 1, 1, 1)),
    dict(weight_maps=torch.rand(2, S, 1, 1)),                                    # Bm not in {1, B}
    dict(weight_maps=torch.rand(1, S, H + 1, W)),                                # larger than the image
    dict(weight_maps=torch.rand(1, S, H, W + 1)),
    dict(weight_maps=torch.ones(1, S, 4, 4, dtype=torch.int32)),                 # integer maps
    dict(weight_maps=torch.rand(S, 4, 4)),                                       # not 4-D
    dict(weight_maps=torch.rand(1, S, 4, 4), feather_sigma=-1.0),                # negative sigma
    dict(weight_maps=torch.rand(1, S, 4, 4), feather_sigma=float("nan")),
], ids=["neither", "both", "n_weights", "w_x", "K_high", "K_low", "Bm", "h", "w", "int", "dim", "sigma", "sigma_nan"])
def test_blend_args_reject(kwargs):
    with pytest.raises(ValueError):
        check(**kwargs)


def test_stylizer_validates_before_device_work():
    """the stylizer raises ValueError on bad maps even on a machine without a GPU (before any device call)"""
    from multi_style_transfer_gan_b200.enhanced_generator import EnhancedGenerator
    from multi_style_transfer_gan_b200.stylize import MultiStyleStylizer
    st = MultiStyleStylizer.__new__(MultiStyleStylizer)
    st.generators = [EnhancedGenerator(8, 1) for _ in range(S)]
    x = torch.zeros(B, 3, H, W)
    with pytest.raises(ValueError):
        st(x, weight_maps=torch.rand(1, S + 2, 4, 4))
    with pytest.raises(ValueError):
        st(x, [0.2, 0.3, 0.5], weight_maps=torch.rand(1, S, 4, 4))
