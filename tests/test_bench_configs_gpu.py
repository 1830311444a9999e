"""Parity ON THE CONFIGS THE NUMBERS ARE QUOTED ON (VERDICT r1, task 1).

bench.py's own workloads -- built by frosting_b200.camera_batch.build_workload, the function bench.py calls -- are
rendered through the C ABI and compared with the UNMODIFIED reference's outputs for the same inputs, recorded in
tests/golden/ref_outputs.npz (tests/golden/make_ref_golden.py):
  C3  2 M frosting-layer Gaussians, ring cameras, 1920x1080, occlusion mask ON  (fused `visibility_mask` AND the plain
      drop-in with Frosting's boolean gathers, frosting_model.py:1578-1586)
  C5  6 M free Gaussians, 1600x1200
  C2  500 k, 800x800, backward (forward is in test_parity_gpu.py)
plus the SURVEY 7.2-3b sweep: >= 1e8 random Gaussians through preprocess, zero mismatches of depth bits / radius / rect.
Bars: radii, depth bits, rect, point_list, ranges, n_contrib, final_T bit-exact; colour <= 1e-4 abs; the 8 gradients
<= 1e-3 relative (tests/util.py::check_grad, against the reference's own atomic-order noise).
Reference: CR/forward.cu:155-374, CR/backward.cu:399-557, CR/rasterizer_impl.cu:70-138.
"""
import os

import pytest
import torch

import frosting_b200 as fb
from frosting_b200 import camera_batch as cbm
from frosting_b200 import scenes
from tests.util import golden_case, check_inputs, check_forward, check_grad, ours_forward_fields

pytestmark = pytest.mark.gpu

KEYS = ("means3D", "opacities", "shs", "scales", "rotations")
FWD_FIELDS = ("num_rendered", "radii", "depth", "touched", "means2D", "conic", "rgb", "ranges", "point_list",
              "n_contrib", "final_T", "color")
C3_CAMS = (0, 3)
SWEEP_CHUNKS = 13


def _compare_forward(case, st, P, index_map=None, vis_rows=None):
    """st: ours (forward_with_state); case: the reference forward on the (possibly gathered) inputs.
    index_map: ours' Gaussian index -> reference row (masked variant), vis_rows: rows of ours present in ref."""
    f = ours_forward_fields(st, rows=vis_rows, index_map=index_map)
    check_forward(case, {k: f[k] for k in FWD_FIELDS})
    if vis_rows is not None:
        dropped = torch.ones(P, dtype=torch.bool, device=st["radii"].device)
        dropped[vis_rows] = False
        assert int(st["radii"][dropped].abs().sum()) == 0
    return st["num_rendered"]


def _compare_grads(case, mine, radii, tag):
    for k, v in mine.items():
        assert v is not None and v.shape[0] == radii.shape[0], (tag, k)
        check_grad(case, k, v, radii, tag=tag)


def _ours_backward(rs, a, cot, P, device, mask=None):
    leaves = {k: a[k].detach().clone().requires_grad_(True) for k in KEYS}
    m2 = torch.zeros(leaves["means3D"].shape[0], 3, device=device, requires_grad=True)
    color, radii = fb.GaussianRasterizer(rs)(
        means3D=leaves["means3D"], means2D=m2, opacities=leaves["opacities"], shs=leaves["shs"],
        scales=leaves["scales"], rotations=leaves["rotations"], visibility_mask=mask)
    (color * cot).sum().backward()
    return dict(means3D=leaves["means3D"].grad, means2D=m2.grad, sh=leaves["shs"].grad,
                opacities=leaves["opacities"].grad, scales=leaves["scales"].grad, rotations=leaves["rotations"].grad), radii


@pytest.mark.parametrize("cam_index", C3_CAMS)
def test_c3_bench_workload_mask_on(cam_index, cuda_device):
    """bench.py's C3 frame: fused mask == reference with boolean gathers, forward integers bit-exact + 8 gradients;
    then the plain drop-in (gathers in torch + our rasterizer) against the same reference call."""
    dev = cuda_device
    wl = cbm.build_workload("c3", dev)
    cbm.visible_faces(wl)
    P, W, H, D = wl["P"], wl["W"], wl["H"], wl["D"]
    cam = wl["cams"][cam_index]
    rs = scenes.settings_for(cam, D, device=dev)
    a = wl["attrs"]
    mask = fb.gaussian_render_mask(wl["face_visible"][cam_index], wl["mesh"]["cells"], P)
    keep = mask.bool()
    # torch restatement of the mask (frosting_model.py:1564-1576)
    assert torch.equal(keep, wl["face_visible"][cam_index].bool()[wl["mesh"]["cells"]])
    rows = torch.nonzero(keep).squeeze(1)
    index_map = torch.cumsum(keep.long(), 0) - 1
    g = {k: a[k][keep].contiguous() for k in KEYS}
    cot = wl["cot_host"][cam_index].to(dev)
    case = golden_case(f"bench_c3_cam{cam_index}")
    check_inputs(case, *(g[k] for k in KEYS), cot)
    st = fb.forward_with_state(rs, a["means3D"], a["opacities"], shs=a["shs"], scales=a["scales"],
                               rotations=a["rotations"], visibility_mask=mask)
    R = _compare_forward(case, st, P, index_map=index_map, vis_rows=rows)
    print(f"C3 cam {cam_index}: kept {rows.numel()} of {P}, visible {int((st['radii'] > 0).sum())}, R = {R}")
    del st
    mine, radii = _ours_backward(rs, a, cot, P, dev, mask=mask)
    for k, v in mine.items():
        assert float(v[~keep].abs().sum()) == 0.0, f"masked rows of {k} must get zero gradient"
    _compare_grads(case, {k: v[keep] for k, v in mine.items()}, radii[keep], "c3-fused-mask")
    # plain drop-in: same gathers as the reference, our rasterizer, no API extension
    st2 = fb.forward_with_state(rs, g["means3D"], g["opacities"], shs=g["shs"], scales=g["scales"], rotations=g["rotations"])
    _compare_forward(case, st2, rows.numel())
    del st2
    mine, radii = _ours_backward(rs, g, cot, rows.numel(), dev)
    _compare_grads(case, mine, radii, "c3-dropin")


def test_c5_bench_workload(cuda_device):
    dev = cuda_device
    wl = cbm.build_workload("c5", dev, cams_per_gpu=1)
    P, W, H, D = wl["P"], wl["W"], wl["H"], wl["D"]
    rs = scenes.settings_for(wl["cams"][0], D, device=dev)
    a = wl["attrs"]
    cot = wl["cot_host"][0].to(dev)
    case = golden_case("bench_c5")
    check_inputs(case, *(a[k] for k in KEYS), cot)
    st = fb.forward_with_state(rs, a["means3D"], a["opacities"], shs=a["shs"], scales=a["scales"], rotations=a["rotations"])
    R = _compare_forward(case, st, P)
    print(f"C5: visible {int((st['radii'] > 0).sum())} of {P}, R = {R}, longest tile list {int(st['tile_count'].max())}")
    del st
    mine, radii = _ours_backward(rs, a, cot, P, dev)
    _compare_grads(case, mine, radii, "c5")


def test_c2_bench_workload_backward(cuda_device):
    dev = cuda_device
    wl = cbm.build_workload("c2", dev, cams_per_gpu=1)
    P, W, H, D = wl["P"], wl["W"], wl["H"], wl["D"]
    rs = scenes.settings_for(wl["cams"][0], D, device=dev)
    a = wl["attrs"]
    cot = wl["cot_host"][0].to(dev)
    case = golden_case("bench_c2")
    check_inputs(case, *(a[k] for k in KEYS), cot)
    st = fb.forward_with_state(rs, a["means3D"], a["opacities"], shs=a["shs"], scales=a["scales"], rotations=a["rotations"])
    _compare_forward(case, st, P)
    del st
    mine, radii = _ours_backward(rs, a, cot, P, dev)
    _compare_grads(case, mine, radii, "c2")


def sweep_chunk(c, device):
    """Chunk c of the preprocess sweep: 8 M random Gaussians with their own seed, image size and SH degree 0."""
    chunk = 8_000_000
    sizes = [(1920, 1080), (1600, 1200), (800, 800), (803, 597), (640, 360)]
    W, H = sizes[c % len(sizes)]
    cam = scenes.make_camera(W, H, device=device, fovx_deg=(50.0, 60.0, 75.0)[c % 3])
    gen = torch.Generator(device=device).manual_seed(1000 + c)
    z = torch.rand(chunk, generator=gen, device=device) * 9.9 + 0.1
    z[: chunk // 50] = torch.rand(chunk // 50, generator=gen, device=device) * 1.2 - 1.0          # near-plane cull
    xy = (torch.rand(chunk, 2, generator=gen, device=device) * 2 - 1) * 1.2
    means = torch.stack([xy[:, 0] * z.abs() * cam.tanfovx, xy[:, 1] * z.abs() * cam.tanfovy, z], 1).contiguous()
    fx = W / (2 * cam.tanfovx)
    scales = (1.5 * 6.0 / fx) * torch.exp(0.5 * torch.randn(chunk, 3, generator=gen, device=device))
    scales[: chunk // 400] *= 12
    q = torch.randn(chunk, 4, generator=gen, device=device)
    # NOT normalised (the reference uses quaternions as given, forward.cu:127): norms in [0.7, 1.3]
    q = q / q.norm(dim=1, keepdim=True) * (0.7 + 0.6 * torch.rand(chunk, 1, generator=gen, device=device))
    op = torch.rand(chunk, 1, generator=gen, device=device)
    col = torch.rand(chunk, 3, generator=gen, device=device)
    rs = scenes.settings_for(cam, 0, device=device, scale_modifier=(1.0, 0.7, 1.3)[c % 3])
    return rs, means, op, col, scales, q


def test_preprocess_sweep_1e8_gaussians(cuda_device):
    """SURVEY 7.2-3b: zero mismatches of (depth bits, radius, rect) over >= 1e8 random Gaussians: 13 chunks of 8 M,
    each with its own seed, image size and SH degree 0 (the integer path does not depend on the colour)."""
    dev = cuda_device
    n_chunks = int(os.environ.get("FB200_SWEEP_CHUNKS", str(SWEEP_CHUNKS)))
    total = 0
    for c in range(n_chunks):
        rs, means, op, col, scales, q = sweep_chunk(c, dev)
        # preprocess only: geometry phase through the C ABI
        st = fb.rasterizer.geometry_state(rs, means, op, colors_precomp=col, scales=scales, rotations=q)
        vis = st["radii"] > 0
        rect = st["rect"]
        touched = ((rect[:, 1] & 0xffff) - (rect[:, 0] & 0xffff)) * (((rect[:, 1] >> 16) & 0xffff) - ((rect[:, 0] >> 16) & 0xffff))
        # the rect itself against the reference's getRect from ITS means2D / radius (auxiliary.h:46-56)
        check_forward(golden_case(f"sweep_{c}"), dict(
            num_rendered=st["num_rendered"], radii=st["radii"], depth=st["depth"][vis].view(torch.int32),
            touched=touched[vis], rect_minx=rect[vis][:, 0] & 0xffff, rect_miny=(rect[vis][:, 0] >> 16) & 0xffff))
        total += means.shape[0]
        del st, means, op, col, scales, q
    print(f"preprocess sweep: {total} Gaussians, no mismatches")
    assert total >= 100_000_000 or n_chunks < SWEEP_CHUNKS
