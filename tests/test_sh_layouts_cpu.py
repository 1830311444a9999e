"""The float64 SH statement of tests/util.py pinned to the C oracle at every SH layout the kernels accept: rows of
M = 1, 4, 9, 16 coefficients, every degree D with (D + 1)^2 <= M.  The GPU tests of tests/test_sh_layouts_gpu.py use
that statement as their independent reference for the SH colour and its gradients."""
import ctypes as C

import numpy as np
import pytest
import torch

from frosting_b200 import scenes
from oracle import cpu
from tests.util import sh_layouts, sh_dirs64, sh_color64

P, W, H = 3011, 241, 133


def _scene(M, D, seed=5):
    cam = scenes.make_camera(W, H)
    g = {k: v.numpy() for k, v in scenes.random_gaussians(P, cam, seed + M, sh_coeffs=M).items()}
    rs = scenes.settings_for(cam, D)
    return rs, g


def _oracle_sh_backward(rs, g, pre, dL_dcolor):
    """oracle_geom_bwd with only a colour cotangent (dL/dmeans2D = dL/dconic = 0): dL/dmeans3D is then the view-direction
    term of the SH backward alone."""
    cam = cpu.Camera(rs)
    M = g["shs"].shape[1]
    f32 = lambda a: np.ascontiguousarray(a, dtype=np.float32)
    z2, z3 = np.zeros((P, 2), np.float32), np.zeros((P, 3), np.float32)
    dcol = f32(dL_dcolor)
    out = dict(means3D=np.zeros((P, 3), np.float32), cov3D=np.zeros((P, 6), np.float32), sh=np.zeros((P, M, 3), np.float32),
               scales=np.zeros((P, 3), np.float32), rotations=np.zeros((P, 4), np.float32))
    keep = [f32(g["means3D"]), f32(g["shs"]), f32(g["scales"]), f32(g["rotations"]), f32(pre["cov3D"])]
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    cpu.lib().oracle_geom_bwd(C.c_int(P), C.c_int(cam.D), C.c_int(M), p(keep[0]), p(pre["radii"]), p(keep[1]),
                              p(pre["clamped"]), p(keep[2]), p(keep[3]), C.c_float(cam.mod), p(keep[4]), p(cam.view),
                              p(cam.proj), p(cam.campos), C.c_int(cam.W), C.c_int(cam.H), C.c_float(cam.tanx),
                              C.c_float(cam.tany), p(z2), p(z3), p(dcol), p(out["means3D"]), p(out["cov3D"]), p(out["sh"]),
                              p(out["scales"]), p(out["rotations"]))
    return out


@pytest.mark.parametrize("M,D", sh_layouts())
def test_float64_sh_colour_matches_the_oracle(M, D):
    rs, g = _scene(M, D)
    pre = cpu.preprocess(cpu.Camera(rs), g["means3D"], g["opacities"], shs=g["shs"], scales=g["scales"],
                         rots=g["rotations"])
    vis = pre["radii"] > 0
    assert 100 < vis.sum() < P
    raw, clamped = sh_color64(g["shs"][vis], sh_dirs64(g["means3D"][vis], rs.campos), D)
    assert np.array_equal(clamped.numpy(), pre["clamped"][vis].astype(bool))
    assert 0 < int(clamped.sum()) or D == 0 or M == 1      # the clamp is exercised (random rows clamp a few channels)
    err = np.abs(raw.clamp_min(0).numpy() - pre["rgb"][vis].astype(np.float64)).max()
    assert err <= 3e-7, err


@pytest.mark.parametrize("M,D", sh_layouts())
def test_float64_sh_gradients_match_the_oracle(M, D):
    """dL/dsh = b_k(dir) dL/drgb on unclamped channels, zero on clamped channels, unrendered rows and every column past
    (D + 1)^2; dL/dmeans3D through the normalised view direction equals the float64 autograd of the statement."""
    rs, g = _scene(M, D)
    pre = cpu.preprocess(cpu.Camera(rs), g["means3D"], g["opacities"], shs=g["shs"], scales=g["scales"],
                         rots=g["rotations"])
    vis = pre["radii"] > 0
    dcol = torch.randn(P, 3, generator=torch.Generator().manual_seed(M * 4 + D)).numpy().astype(np.float32)
    out = _oracle_sh_backward(rs, g, pre, dcol)
    n = (D + 1) ** 2
    assert not out["sh"][~vis].any() and not out["sh"][:, n:].any() and not out["means3D"][~vis].any()

    means = torch.from_numpy(g["means3D"][vis]).double().requires_grad_(True)
    shs = torch.from_numpy(g["shs"][vis]).double().requires_grad_(True)
    raw, _ = sh_color64(shs, sh_dirs64(means, rs.campos), D)
    live = torch.from_numpy(~pre["clamped"][vis].astype(bool))
    dRGB = torch.from_numpy(dcol[vis]).double() * live
    (raw * dRGB).sum().backward()
    if D == 0:                       # a constant colour: no view-direction term
        assert means.grad is None and not out["means3D"].any()
    for name, ref in (("sh", shs.grad), ("means3D", means.grad))[:1 if D == 0 else 2]:
        mine = torch.from_numpy(out[name][vis]).double()
        scale = ref.abs().max().item()
        assert scale > 0
        err = (mine - ref).abs().max().item() / scale
        assert err <= (1e-6 if name == "sh" else 1e-5), (name, err)
    # clamped channels get exactly zero in every coefficient
    assert not np.where(live.numpy()[:, None, :], 0.0, out["sh"][vis]).any()
