"""GPU tests of the host shim's round-2 behaviour: speculative one-phase forward and its overflow protocol, the
in-kernel visible-face lookup (row f1), unaligned views, per-thread host state, the alpha output."""
import threading

import pytest
import torch

import frosting_b200 as fb
from frosting_b200 import rasterizer as fbr
from frosting_b200 import scenes
from tests.util import scene, rel_err_stats

pytestmark = pytest.mark.gpu

KEYS = ("means3D", "opacities", "shs", "scales", "rotations")


def _fwd_bwd(rs, g, cot, **kw):
    leaves = {k: g[k].detach().clone().requires_grad_(True) for k in KEYS}
    m2 = torch.zeros(leaves["means3D"].shape[0], 3, device=cot.device, requires_grad=True)
    out = fb.GaussianRasterizer(rs)(means3D=leaves["means3D"], means2D=m2, opacities=leaves["opacities"],
                                    shs=leaves["shs"], scales=leaves["scales"], rotations=leaves["rotations"], **kw)
    (out[0] * cot).sum().backward()
    return out, {k: v.grad for k, v in leaves.items()}


def test_speculative_forward_equals_exact_and_overflow_is_loud(cuda_device):
    dev = cuda_device
    P, W, H = 60_000, 400, 304
    cam, g, rs = scene(P, W, H, 31, 3, dev)
    cot = torch.randn(3, H, W, generator=torch.Generator().manual_seed(2)).to(dev)
    host = fbr._host_state(dev)
    host.hints.pop((P, W, H), None)
    (c0, r0), g0 = _fwd_bwd(rs, g, cot)             # first frame of this size: exact two-phase path
    assert (P, W, H) in host.hints
    (c1, r1), g1 = _fwd_bwd(rs, g, cot)             # second frame: speculative one-phase path, no host wait
    assert torch.equal(c0.view(torch.int32), c1.view(torch.int32)) and torch.equal(r0, r1)
    for k in g0:
        assert rel_err_stats(g1[k], g0[k])[0] <= 1e-3, k      # two runs: atomic-order noise (typ. 1e-6, tail 1.7e-4)
    R = fbr.last_num_rendered(dev)
    assert R > 1000
    # force an overflow: pretend earlier frames of this size were almost empty.  The frame's backward is enqueued without
    # waiting for its status words (every kernel of the frame exits on the overflow word: its gradients are zeros) and the
    # NEXT call on this thread raises
    host.hints[(P, W, H)] = R // 2
    (_cx, _rx), gx = _fwd_bwd(rs, g, cot)
    torch.cuda.synchronize(dev)
    for k in gx:
        assert float(gx[k].abs().sum()) == 0.0, k
    with pytest.raises(fbr.BinningOverflow):
        _fwd_bwd(rs, g, cot)
    assert host.hints[(P, W, H)] >= R                # the count that overflowed sized the next frame
    (c2, r2), g2 = _fwd_bwd(rs, g, cot)
    assert torch.equal(c0.view(torch.int32), c2.view(torch.int32))
    # FB200_CHECK_BEFORE_BACKWARD=1: the overflow is raised from the frame's own backward (one host wait per frame)
    fbr.last_num_rendered(dev)                       # look at every earlier frame first (they would re-grow the hint)
    host.hints[(P, W, H)] = R // 2
    fbr.CHECK_BEFORE_BACKWARD = True
    try:
        with pytest.raises(fbr.BinningOverflow):
            _fwd_bwd(rs, g, cot)
    finally:
        fbr.CHECK_BEFORE_BACKWARD = False
    (c3, r3), g3 = _fwd_bwd(rs, g, cot)
    assert torch.equal(c0.view(torch.int32), c3.view(torch.int32))
    # an overflow nobody differentiates is reported by the next call on this thread
    fbr.last_num_rendered(dev)
    host.hints[(P, W, H)] = R // 2
    with torch.no_grad():
        fb.GaussianRasterizer(rs)(means3D=g["means3D"], means2D=None, opacities=g["opacities"], shs=g["shs"],
                                  scales=g["scales"], rotations=g["rotations"])
    torch.cuda.synchronize(dev)
    with pytest.raises(fbr.BinningOverflow):
        with torch.no_grad():
            fb.GaussianRasterizer(rs)(means3D=g["means3D"], means2D=None, opacities=g["opacities"], shs=g["shs"],
                                      scales=g["scales"], rotations=g["rotations"])
    torch.cuda.synchronize(dev)
    host.pending.clear(); host.overflowed.clear()


def test_visible_face_lookup_equals_mask_tensor(cuda_device):
    dev = cuda_device
    W, H, P = 320, 200, 40_000
    cam = scenes.make_camera(W, H, device=dev)
    params, mesh = scenes.frosting_layer(P, cam, 3, n_faces_target=6000, device=dev, view_distance=4.5)
    a = scenes.frosting_attributes(params, mesh)
    # 500 background Gaussians behind the mesh-bound ones: they always render (frosting_model.py:1573-1576)
    nbg = 500
    bgg = scenes.random_gaussians(nbg, cam, 8, device=dev)
    a = {k: torch.cat([a[k], bgg[k]]).contiguous() for k in KEYS}
    rs = scenes.settings_for(cam, 3, device=dev)
    _, fv, _ = fb.rasterize_mesh(mesh["verts"], mesh["faces"], cam.full_proj_transform, H, W, mark_last_on_bg=True)
    mask = fb.gaussian_render_mask(fv, mesh["cells"], P + nbg)
    assert int(mask[P:].sum()) == nbg and 0 < int(mask[:P].sum()) < P
    cot = torch.randn(3, H, W, generator=torch.Generator().manual_seed(5)).to(dev)
    (c1, r1), g1 = _fwd_bwd(rs, a, cot, visibility_mask=mask)
    (c2, r2), g2 = _fwd_bwd(rs, a, cot, face_visibility=(fv, mesh["cells"]))
    assert torch.equal(c1.view(torch.int32), c2.view(torch.int32)) and torch.equal(r1, r2)
    for k in g1:
        assert rel_err_stats(g2[k], g1[k])[0] <= 1e-3, k
    # the fused attribute kernel takes the same marks
    a1 = fb.frosting_attributes_fused(params, mesh, mask[:P])
    a2 = fb.frosting_attributes_fused(params, mesh, face_visible=fv)
    for k in a1:
        assert torch.equal(a1[k], a2[k]), k


def test_views_at_odd_storage_offsets_are_accepted(cuda_device):
    """A contiguous view whose storage offset is not a multiple of 4 floats is legal for the reference (scalar
    loads); the shim copies it to an aligned allocation instead of faulting in a 128-bit load."""
    dev = cuda_device
    P, W, H = 5_000, 160, 96
    cam, g, rs = scene(P, W, H, 4, 3, dev)
    flat = torch.zeros(3 + 4 * P, device=dev)
    flat[3:] = g["rotations"].reshape(-1)
    rot_view = flat[3:].view(P, 4)
    assert rot_view.is_contiguous() and rot_view.data_ptr() % 16 != 0
    flat_sh = torch.zeros(1 + 48 * P, device=dev)
    flat_sh[1:] = g["shs"].reshape(-1)
    sh_view = flat_sh[1:].view(P, 16, 3)
    with torch.no_grad():
        c_ref, r_ref = fb.GaussianRasterizer(rs)(means3D=g["means3D"], means2D=None, opacities=g["opacities"],
                                                 shs=g["shs"], scales=g["scales"], rotations=g["rotations"])
        c, r = fb.GaussianRasterizer(rs)(means3D=g["means3D"], means2D=None, opacities=g["opacities"], shs=sh_view,
                                         scales=g["scales"], rotations=rot_view)
    assert torch.equal(c.view(torch.int32), c_ref.view(torch.int32)) and torch.equal(r, r_ref)


def test_two_host_threads_share_a_device(cuda_device):
    """Host state (capacity hints, status mailboxes, pending frames) is per thread: two threads rendering different
    problem sizes on one GPU, each on its own stream, get what a single thread gets."""
    dev = cuda_device
    cfgs = [(30_000, 256, 160, 1), (45_000, 320, 208, 2)]
    expect, got, errs = {}, {}, []
    for i, (P, W, H, seed) in enumerate(cfgs):
        cam, g, rs = scene(P, W, H, seed, 2, dev)
        with torch.no_grad():
            expect[i] = fb.GaussianRasterizer(rs)(means3D=g["means3D"], means2D=None, opacities=g["opacities"],
                                                  shs=g["shs"], scales=g["scales"], rotations=g["rotations"])[0].clone()
    torch.cuda.synchronize(dev)

    def work(i):
        try:
            P, W, H, seed = cfgs[i]
            torch.cuda.set_device(dev)
            cam, g, rs = scene(P, W, H, seed, 2, dev)
            with torch.cuda.stream(torch.cuda.Stream(dev)), torch.no_grad():
                for _ in range(6):
                    c = fb.GaussianRasterizer(rs)(means3D=g["means3D"], means2D=None, opacities=g["opacities"],
                                                  shs=g["shs"], scales=g["scales"], rotations=g["rotations"])[0]
                torch.cuda.current_stream(dev).synchronize()
                got[i] = c.clone()
        except Exception as ex:   # surfaced below
            errs.append(repr(ex))

    ts = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errs, errs
    for i in range(2):
        assert torch.equal(got[i].view(torch.int32), expect[i].view(torch.int32))


def test_alpha_output(cuda_device):
    dev = cuda_device
    P, W, H = 20_000, 200, 120
    cam, g, rs = scene(P, W, H, 6, 1, dev)
    with torch.no_grad():
        color, radii, alpha = fb.GaussianRasterizer(rs)(
            means3D=g["means3D"], means2D=None, opacities=g["opacities"], shs=g["shs"], scales=g["scales"],
            rotations=g["rotations"], return_alpha=True)
        # the differentiable route: one extra channel of ones, background 0 -> sum alpha_i T_i = 1 - final_T
        _, _, ones_img = fb.GaussianRasterizer(rs)(
            means3D=g["means3D"], means2D=None, opacities=g["opacities"], shs=g["shs"], scales=g["scales"],
            rotations=g["rotations"], extra_features=torch.ones(P, 1, device=dev))
    st = fb.forward_with_state(rs, g["means3D"], g["opacities"], shs=g["shs"], scales=g["scales"], rotations=g["rotations"])
    assert alpha.shape == (H, W) and torch.equal(alpha, 1.0 - st["final_T"])
    assert (alpha - ones_img[0]).abs().max().item() <= 2e-5
    assert 0.0 <= float(alpha.min()) and float(alpha.max()) <= 1.0


def test_frosting_render_equals_the_two_step_path(cuda_device):
    """Row f1: the single fused op (attribute kernel -> rasterizer with the in-kernel face lookup -> sparse-row backward ->
    attribute backward) against the same frame built from the separate pieces (torch property chain of
    frosting_model.py:713-799 + mask tensor + rasterizer): identical image, equal parameter gradients."""
    dev = cuda_device
    W, H, P = 320, 200, 50_000
    cam = scenes.make_camera(W, H, device=dev)
    params, mesh = scenes.frosting_layer(P, cam, 9, n_faces_target=8000, device=dev, view_distance=4.5)
    rs = scenes.settings_for(cam, 3, device=dev)
    _, fv, _ = fb.rasterize_mesh(mesh["verts"], mesh["faces"], cam.full_proj_transform, H, W, mark_last_on_bg=True)
    cot = torch.randn(3, H, W, generator=torch.Generator().manual_seed(7)).to(dev)

    p1 = {k: v.detach().clone().requires_grad_(True) for k, v in params.items()}
    m1 = dict(mesh); m1["inner"] = mesh["inner"].clone().requires_grad_(True); m1["outer"] = mesh["outer"].clone().requires_grad_(True)
    color1, radii1 = fb.frosting_render(p1, m1, rs, face_visible=fv)
    (color1 * cot).sum().backward()

    # (a) the same frame from the separate kernels with the SAME attribute values (fused attribute kernel + rasterizer,
    # dense gradient rows): identical image, gradients equal up to the order of the float atomics
    p2 = {k: v.detach().clone().requires_grad_(True) for k, v in params.items()}
    m2 = dict(mesh); m2["inner"] = mesh["inner"].clone().requires_grad_(True); m2["outer"] = mesh["outer"].clone().requires_grad_(True)
    a = fb.frosting_attributes_fused(p2, m2, face_visible=fv)
    z = torch.zeros(P, 3, device=dev, requires_grad=True)
    color2, radii2 = fb.GaussianRasterizer(rs)(means3D=a["means3D"], means2D=z, opacities=a["opacities"], shs=a["shs"],
                                               scales=a["scales"], rotations=a["rotations"],
                                               face_visibility=(fv, mesh["cells"]))
    (color2 * cot).sum().backward()
    assert torch.equal(radii1, radii2) and 0 < int((radii1 > 0).sum()) < P
    assert torch.equal(color1.view(torch.int32), color2.view(torch.int32))
    # the two frames' blend backwards accumulate with float atomics in different orders: typically 1e-6 of the tensor's
    # scale, but the scale / rotation gradients cancel large terms -- tools/dbg_frost.py saw 1.7e-4 once in 60 repeats
    for k in p1:
        m, frac = rel_err_stats(p1[k].grad, p2[k].grad)
        assert m <= 1e-3 and frac <= 1e-3, (k, m, frac)
    for k in ("inner", "outer"):
        m, frac = rel_err_stats(m1[k].grad, m2[k].grad)
        assert m <= 1e-3, (k, m)
    # (b) against Frosting's torch property chain (frosting_model.py:713-799) + mask tensor: the attribute values agree
    # to ~1 ulp, which flips a handful of alpha >= 1/255 / tile-rect decisions -- statistical comparison
    p3 = {k: v.detach().clone().requires_grad_(True) for k, v in params.items()}
    a3 = scenes.frosting_attributes(p3, mesh)
    mask = fb.gaussian_render_mask(fv, mesh["cells"], P)
    color3, radii3 = fb.GaussianRasterizer(rs)(means3D=a3["means3D"], means2D=torch.zeros(P, 3, device=dev),
                                               opacities=a3["opacities"], shs=a3["shs"], scales=a3["scales"],
                                               rotations=a3["rotations"], visibility_mask=mask)
    (color3 * cot).sum().backward()
    d = (color1 - color3).abs()
    assert (d > 1e-4).float().mean().item() < 1e-3 and d.max().item() < 2e-2
    for k in p1:
        m, frac = rel_err_stats(p1[k].grad, p3[k].grad)
        assert m <= 2e-2 and frac <= 2e-2, (k, m, frac)
    # unrendered Gaussians get exact zeros although the rasterizer never wrote their rows
    dead = radii1 <= 0
    for k in p1:
        assert float(p1[k].grad[dead].abs().sum()) == 0.0, k


# (SH rest coefficients R, degree D): checkpoints trained at degree 0-3 (R = 0, 3, 8, 15), and Frosting's SH warm-up,
# which renders a degree-3 layout at degree 0, 1, 2 first.  (15, 3) is the full layout.
FROSTING_SH = [(0, 0), (3, 0), (3, 1), (8, 0), (8, 2), (15, 0), (15, 1), (15, 2), (15, 3)]


def test_frosting_mode_equals_the_attribute_kernel_route(cuda_device):
    """Row f1 proper: `frosting_render` (the rasterizer reads the parameters itself, nothing materialised, parameter
    gradients written by the per-Gaussian backward for rendered rows only) against `frosting_render_two_step` (attribute
    kernel -> rasterizer -> attribute backward): bit-identical image and radii, gradients equal up to the order of the
    blend backward's float atomics; the optimizer-sink route gives the same numbers as the autograd route."""
    _frosting_mode_against_the_attribute_kernel_route(cuda_device, 15, 3)


@pytest.mark.parametrize("R,D", [rd for rd in FROSTING_SH if rd != (15, 3)])
def test_frosting_mode_equals_the_attribute_kernel_route_at_lower_sh_layouts(cuda_device, R, D):
    """The same comparison with fewer rest coefficients per row (R < 15: narrower rows, R = 0: no rest tensor) and at
    degrees below the row's (D < 3: coefficients past (D + 1)^2 are not read and get zero gradients)."""
    _frosting_mode_against_the_attribute_kernel_route(cuda_device, R, D)


def _frosting_mode_against_the_attribute_kernel_route(dev, R, D):
    for (W, H, P, faces, occl) in ((320, 200, 50_000, 8000, True), (200, 120, 3001, 500, False)):
        cam = scenes.make_camera(W, H, device=dev)
        params, mesh = scenes.frosting_layer(P, cam, 11, n_faces_target=faces, device=dev, view_distance=4.5,
                                             sh_coeffs=R + 1)
        rs = scenes.settings_for(cam, D, device=dev)
        fv = None
        if occl:
            _, fv, _ = fb.rasterize_mesh(mesh["verts"], mesh["faces"], cam.full_proj_transform, H, W, mark_last_on_bg=True)
        cot = torch.randn(3, H, W, generator=torch.Generator().manual_seed(3)).to(dev)
        res = []
        for fn in (fb.frosting_render, fb.frosting_render_two_step):
            p = {k: v.detach().clone().requires_grad_(True) for k, v in params.items()}
            m = dict(mesh); m["inner"] = mesh["inner"].clone().requires_grad_(True); m["outer"] = mesh["outer"].clone().requires_grad_(True)
            color, radii = fn(p, m, rs, face_visible=fv)
            (color * cot).sum().backward()
            res.append((color, radii, p, m))
        (c1, r1, p1, m1), (c2, r2, p2, m2) = res
        assert torch.equal(r1, r2) and 0 < int((r1 > 0).sum()) <= P
        assert torch.equal(c1.view(torch.int32), c2.view(torch.int32))
        for k in p1:
            mx, frac = rel_err_stats(p1[k].grad, p2[k].grad)
            assert mx <= 1e-3 and frac <= 1e-3, (k, mx, frac)     # atomic-order noise of two blend backwards, see above
            assert float(p1[k].grad[r1 <= 0].abs().sum()) == 0.0, k
        for k in ("inner", "outer"):
            mx, _ = rel_err_stats(m1[k].grad, m2[k].grad)
            assert mx <= 1e-3, (k, mx)
        # gradients straight into a caller-owned sink (dirty on entry: rows of unrendered Gaussians must come out zero)
        sink = {k: torch.full_like(v, 7.0) for k, v in params.items()}
        p3 = {k: v.detach().clone().requires_grad_(True) for k, v in params.items()}
        color, radii = fb.frosting_render(p3, mesh, rs, face_visible=fv, grad_sink=sink)
        (color * cot).sum().backward()
        for k in p1:
            mx, _ = rel_err_stats(sink[k].view_as(p1[k].grad), p1[k].grad)
            assert mx <= 1e-3 and p3[k].grad is None, (k, mx)


def test_fused_attribute_kernels_against_reference_property_goldens(cuda_device):
    """The fused attribute kernels against vectors produced by executing the reference's own property source
    (tests/golden/make_frosting_attr_golden.py): values 1e-6, gradients 2e-5 of scale, shell-vertex gradients included."""
    import os
    import numpy as np
    dev = cuda_device
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "frosting_attrs.npz"))
    params = {k[len("param_"):]: torch.from_numpy(z[k]).to(dev).requires_grad_(True) for k in z.files if k.startswith("param_")}
    mesh = {k[len("mesh_"):]: torch.from_numpy(z[k]).to(dev) for k in z.files if k.startswith("mesh_")}
    mesh["inner"].requires_grad_(True); mesh["outer"].requires_grad_(True)
    out = fb.frosting_attributes_fused(params, mesh)
    for k, v in out.items():
        ref = torch.from_numpy(z[f"out_{k}"]).to(dev)
        assert (v - ref).abs().max().item() <= 1e-6 * max(1.0, ref.abs().max().item()), k
    sum((out[k] * torch.from_numpy(z[f"cot_{k}"]).to(dev)).sum() for k in out).backward()
    for k, v in params.items():
        ref = torch.from_numpy(z[f"grad_{k}"]).to(dev)
        assert (v.grad - ref).abs().max().item() <= 2e-5 * ref.abs().max().item(), k
    ref = torch.from_numpy(z["grad_base_verts"]).to(dev)
    assert ((mesh["inner"].grad + mesh["outer"].grad) - ref).abs().max().item() <= 2e-5 * ref.abs().max().item()
