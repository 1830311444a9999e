"""Row f4: extra feature channels blended in the same traversal == the reference's SECOND rasterizer pass with the
features as colors_precomp (frosting_scene/sugar_model.py:2343-2387), forward and backward."""
import pytest
import torch

import frosting_b200 as fb
from tests.util import scene, golden_case, check_inputs, check_forward, check_grad

pytestmark = pytest.mark.gpu

PARAMS = [(3, 0.0), (3, 0.25), (1, 0.0), (2, 1.0)]


def _features(P, E, cam_like_depth, gen, device):
    # depth-like channel + signed normal-like channels, as render_depth_and_normal builds them
    f = torch.randn(P, E, generator=gen)
    f[:, 0] = f[:, 0].abs() * 3.0 + 0.5
    return f.to(device)


def extra_inputs(E, device):
    P, W, H, D = 60_000, 400, 304, 3
    cam, g, rs = scene(P, W, H, 21, D, device, 0.5)
    gen = torch.Generator().manual_seed(8)
    feats = _features(P, E, None, gen, device)
    cot_c = torch.randn(3, H, W, generator=gen).to(device)
    cot_e = torch.randn(E, H, W, generator=gen).to(device)
    return rs, g, feats, cot_c, cot_e


@pytest.mark.parametrize("E,bg_e", PARAMS)
def test_extra_pass_matches_second_reference_pass(E, bg_e, cuda_device):
    """The reference's outputs (tests/golden/make_ref_golden.py): pass 1 with the SH colours, pass 2 with the features
    as colors_precomp padded to 3 channels over a background of bg_e; gradients are the sum of both passes'."""
    dev = cuda_device
    rs, g, feats, cot_c, cot_e = extra_inputs(E, dev)
    P, H, W = feats.shape[0], rs.image_height, rs.image_width
    bg_extra = torch.full((E,), bg_e, device=dev)
    kw = dict(scales=g["scales"], rotations=g["rotations"])
    case = golden_case(f"extra_E{E}_bg{bg_e:g}")
    check_inputs(case, *(g[k] for k in ("means3D", "opacities", "shs", "scales", "rotations")), feats, cot_c, cot_e)

    leaves = {k: g[k].clone().requires_grad_(True) for k in ("means3D", "opacities", "shs", "scales", "rotations")}
    fl = feats.clone().requires_grad_(True)
    m2 = torch.zeros(P, 3, device=dev, requires_grad=True)
    color, radii, extra = fb.GaussianRasterizer(rs)(
        means3D=leaves["means3D"], means2D=m2, opacities=leaves["opacities"], shs=leaves["shs"],
        scales=leaves["scales"], rotations=leaves["rotations"], extra_features=fl, extra_background=bg_extra)
    assert extra.shape == (E, H, W)
    # colour is untouched by the extension: bit-identical to the colour-only call
    c0, _ = fb.GaussianRasterizer(rs)(means3D=g["means3D"], means2D=torch.zeros(P, 3, device=dev),
                                      opacities=g["opacities"], shs=g["shs"], **kw)
    assert torch.equal(color.detach().view(torch.int32), c0.view(torch.int32))
    check_forward(case, {"radii": radii, "color": extra.detach()}, color_tol=2e-6 * max(1.0, float(feats.abs().max())))

    ((color * cot_c).sum() + (extra * cot_e).sum()).backward()
    got = dict(means3D=leaves["means3D"].grad, means2D=m2.grad, opacities=leaves["opacities"].grad,
               scales=leaves["scales"].grad, rotations=leaves["rotations"].grad, sh=leaves["shs"].grad, features=fl.grad)
    for k, v in got.items():
        check_grad(case, k, v, radii, frac_bar=5e-3, tag=f"extra E{E}")
    assert torch.equal(fl.grad[radii <= 0], torch.zeros_like(fl.grad[radii <= 0]))


def test_extra_only_loss_and_argument_checks(cuda_device):
    dev = cuda_device
    P, W, H = 5_000, 160, 96
    cam, g, rs = scene(P, W, H, 2, 1, dev, 0.0)
    f = torch.rand(P, 2, device=dev, requires_grad=True)
    op = g["opacities"].clone().requires_grad_(True)
    color, radii, extra = fb.GaussianRasterizer(rs)(
        means3D=g["means3D"], means2D=torch.zeros(P, 3, device=dev), opacities=op, shs=g["shs"],
        scales=g["scales"], rotations=g["rotations"], extra_features=f)
    extra.sum().backward()                          # loss on the extra image only
    assert f.grad is not None and torch.isfinite(f.grad).all() and float(f.grad.abs().sum()) > 0
    assert op.grad is not None and float(op.grad.abs().sum()) > 0
    # with a constant feature of 1 the extra image is the accumulated alpha: 1 - final_T
    ones = torch.ones(P, 1, device=dev)
    _, _, acc = fb.GaussianRasterizer(rs)(
        means3D=g["means3D"], means2D=torch.zeros(P, 3, device=dev), opacities=g["opacities"], shs=g["shs"],
        scales=g["scales"], rotations=g["rotations"], extra_features=ones)
    st = fb.forward_with_state(rs, g["means3D"], g["opacities"], shs=g["shs"], scales=g["scales"], rotations=g["rotations"])
    assert (acc[0] - (1.0 - st["final_T"].view(H, W))).abs().max().item() <= 2e-6
    with pytest.raises(RuntimeError):
        fb.GaussianRasterizer(rs)(means3D=g["means3D"], means2D=torch.zeros(P, 3, device=dev), opacities=g["opacities"],
                                  shs=g["shs"], scales=g["scales"], rotations=g["rotations"],
                                  extra_features=torch.zeros(P, 4, device=dev))
    # empty scene: the extra image is its background
    e = torch.zeros(0, 3, device=dev)
    _, _, ex0 = fb.GaussianRasterizer(rs)(means3D=e, means2D=e, opacities=torch.zeros(0, 1, device=dev),
                                          shs=torch.zeros(0, 4, 3, device=dev), scales=e,
                                          rotations=torch.zeros(0, 4, device=dev),
                                          extra_features=torch.zeros(0, 3, device=dev),
                                          extra_background=torch.tensor([0.5, 0.25, 1.0], device=dev))
    assert torch.equal(ex0[:, 0, 0].cpu(), torch.tensor([0.5, 0.25, 1.0]))
