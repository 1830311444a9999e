"""Argument checks of the drop-in surface: the same exceptions and messages as the reference's
diff_gaussian_rasterization/__init__.py:191-195 (misspelling included), raised before any native call."""
import pytest
import torch

import frosting_b200 as fb


def test_invalid_combinations_raise_like_the_reference():
    r = fb.GaussianRasterizer(None)
    m = torch.zeros(4, 3)
    with pytest.raises(Exception, match="excatly one of either SHs or precomputed colors"):
        r(means3D=m, means2D=m, opacities=m[:, :1], scales=m, rotations=torch.zeros(4, 4))
    with pytest.raises(Exception, match="exactly one of either scale/rotation pair"):
        r(means3D=m, means2D=m, opacities=m[:, :1], shs=torch.zeros(4, 16, 3))
