"""The C ABI used the way a foreign host would use it (no Python shim): the ONE-phase fb200_forward with a caller-chosen
capacity, its overflow protocol, fb200_backward with the accumulators cleared by the library, and a frame larger than the
tile-scan's shared-memory staging (> 10240 tiles)."""
import ctypes as C

import pytest
import torch

import frosting_b200 as fb
from frosting_b200 import _lib
from frosting_b200._lib import Params, Inputs, Workspace, Grads
from tests.util import scene, rel_err_stats, golden_case, check_inputs, check_forward, ours_forward_fields

pytestmark = pytest.mark.gpu


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _one_phase(rs, g, P, W, H, D, capacity, dev):
    L = _lib.lib()
    prm = Params(P=P, sh_degree=D, sh_coeffs=g["shs"].shape[1], image_width=W, image_height=H, tanfovx=float(rs.tanfovx),
                 tanfovy=float(rs.tanfovy), scale_modifier=1.0, prefiltered=0, debug=0, extra=None)
    t = dict(bg=rs.bg.contiguous(), view=rs.viewmatrix.contiguous(), proj=rs.projmatrix.contiguous(),
             campos=rs.campos.contiguous())
    inp = Inputs(d_background=_p(t["bg"]), d_means3D=_p(g["means3D"]), d_shs=_p(g["shs"]), d_colors_precomp=None,
                 d_opacities=_p(g["opacities"]), d_scales=_p(g["scales"]), d_rotations=_p(g["rotations"]),
                 d_cov3D_precomp=None, d_viewmatrix=_p(t["view"]), d_projmatrix=_p(t["proj"]), d_campos=_p(t["campos"]),
                 d_visibility=None)
    geom = torch.empty(L.fb200_geom_bytes(P), dtype=torch.uint8, device=dev)
    image = torch.empty(L.fb200_image_bytes(W, H), dtype=torch.uint8, device=dev)
    binning = torch.empty(L.fb200_binning_bytes(capacity), dtype=torch.uint8, device=dev)
    status = torch.zeros(_lib.FB200_STATUS_WORDS, dtype=torch.int32, device=dev)
    ws = Workspace(d_geom=geom.data_ptr(), geom_bytes=geom.numel(), d_image=image.data_ptr(), image_bytes=image.numel(),
                   d_binning=binning.data_ptr(), binning_bytes=binning.numel(), binning_capacity=capacity,
                   d_status=status.data_ptr(), acc_zeroed_by_forward=0, h_status=None)
    color = torch.full((3, H, W), -7.0, device=dev)
    radii = torch.empty(P, dtype=torch.int32, device=dev)
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    _lib.check(L.fb200_forward(C.byref(prm), C.byref(inp), C.byref(ws), _p(color), _p(radii), stream))
    torch.cuda.synchronize(dev)
    keep = (t, geom, image, binning, status)
    return prm, inp, ws, color, radii, status.cpu(), keep


def test_one_phase_forward_overflow_protocol_and_backward(cuda_device):
    dev = cuda_device
    P, W, H, D = 30_000, 320, 208, 2
    cam, g, rs = scene(P, W, H, 4, D, dev, 0.25)
    two = fb.forward_with_state(rs, g["means3D"], g["opacities"], shs=g["shs"], scales=g["scales"], rotations=g["rotations"])
    R = two["num_rendered"]
    # capacity too small: the count and the radii are valid, the overflow word is set, nothing is rendered
    prm, inp, ws, color, radii, st, keep = _one_phase(rs, g, P, W, H, D, max(R // 2, 1), dev)
    assert st[_lib.ST_NUM_RENDERED] == R and st[_lib.ST_OVERFLOW] == 1
    assert torch.equal(radii, two["radii"])
    assert float(color.min()) == -7.0 and float(color.max()) == -7.0
    # grown as the header prescribes: bit-identical to the two-phase path of the Python shim
    prm, inp, ws, color, radii, st, keep = _one_phase(rs, g, P, W, H, D, R + 17, dev)
    assert st[_lib.ST_NUM_RENDERED] == R and st[_lib.ST_OVERFLOW] == 0
    assert torch.equal(color.view(torch.int32), two["color"].view(torch.int32))
    # backward straight through the ABI (the library clears its accumulators: acc_zeroed_by_forward = 0)
    L = _lib.lib()
    cot = torch.randn(3, H, W, generator=torch.Generator().manual_seed(2)).to(dev)
    M = g["shs"].shape[1]
    outs = dict(m2=torch.empty(P, 3, device=dev), op=torch.empty(P, 1, device=dev), m3=torch.empty(P, 3, device=dev),
                sh=torch.empty(P, M, 3, device=dev), sc=torch.empty(P, 3, device=dev), ro=torch.empty(P, 4, device=dev))
    grads = Grads(d_dL_dmeans2D=_p(outs["m2"]), d_dL_dcolors=None, d_dL_dopacity=_p(outs["op"]), d_dL_dmeans3D=_p(outs["m3"]),
                  d_dL_dcov3D=None, d_dL_dsh=_p(outs["sh"]), d_dL_dscales=_p(outs["sc"]), d_dL_drotations=_p(outs["ro"]))
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    for _ in range(2):      # twice: the second call must clear the accumulators again
        _lib.check(L.fb200_backward(C.byref(prm), C.byref(inp), C.byref(ws), _p(radii), _p(cot), C.byref(grads), stream))
    torch.cuda.synchronize(dev)
    leaves = {k: g[k].clone().requires_grad_(True) for k in ("means3D", "opacities", "shs", "scales", "rotations")}
    m2 = torch.zeros(P, 3, device=dev, requires_grad=True)
    c, _ = fb.GaussianRasterizer(rs)(means3D=leaves["means3D"], means2D=m2, opacities=leaves["opacities"], shs=leaves["shs"],
                                     scales=leaves["scales"], rotations=leaves["rotations"])
    (c * cot).sum().backward()
    for mine, ref in ((outs["m3"], leaves["means3D"].grad), (outs["op"], leaves["opacities"].grad), (outs["sh"], leaves["shs"].grad),
                      (outs["sc"], leaves["scales"].grad), (outs["ro"], leaves["rotations"].grad), (outs["m2"], m2.grad)):
        m, _ = rel_err_stats(mine, ref)
        assert m <= 1e-3, m          # two runs of one frame differ by the order of the blend backward's float atomics
    # a missing required gradient pointer is refused, not dereferenced
    bad = Grads(d_dL_dmeans2D=None, d_dL_dcolors=None, d_dL_dopacity=_p(outs["op"]), d_dL_dmeans3D=_p(outs["m3"]),
                d_dL_dcov3D=None, d_dL_dsh=_p(outs["sh"]), d_dL_dscales=_p(outs["sc"]), d_dL_drotations=_p(outs["ro"]))
    assert L.fb200_backward(C.byref(prm), C.byref(inp), C.byref(ws), _p(radii), _p(cot), C.byref(bad), stream) == -1


def many_tiles_scene(device):
    P, W, H, D = 40_000, 2608, 1712, 1
    cam, g, rs = scene(P, W, H, 12, D, device, 0.0)
    return P, rs, g


def test_frame_with_more_tiles_than_the_scan_stages(cuda_device):
    """2608 x 1712 = 163 x 107 = 17 441 tiles > 10 240: the tile scan reads its counts from global memory."""
    P, rs, g = many_tiles_scene(cuda_device)
    case = golden_case("cabi_many_tiles")
    check_inputs(case, *(g[k] for k in ("means3D", "opacities", "shs", "scales", "rotations")))
    st = fb.forward_with_state(rs, g["means3D"], g["opacities"], shs=g["shs"], scales=g["scales"], rotations=g["rotations"])
    f = ours_forward_fields(st)
    check_forward(case, {k: f[k] for k in ("num_rendered", "radii", "point_list", "n_contrib", "color")})
