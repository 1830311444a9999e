"""Every SH layout the kernels accept, on the GPU.

Plain path: rows of M = 1, 4, 9, 16 coefficients at every degree D with (D + 1)^2 <= M -- a 3DGS checkpoint trained at a
lower degree.  Frosting mode and the fused attribute kernels: R = 0, 3, 8, 15 rest coefficients, also rendered below
their full degree (Frosting's SH warm-up starts a degree-3 layout at degree 0).  The kernels branch on these values
(vector or scalar SH loads, the 16-coefficient staging path or the generic loop, staged or unstaged rest rows), so
each branch is checked against the C oracle, the float64 SH statement of tests/util.py or a twin run.

The scenes have a ragged image (241 x 133), P not a multiple of 32, whole 32-row runs of unrendered Gaussians next to
partly rendered runs, and an all-unrendered tail run of 23 rows."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

import frosting_b200 as fb
from frosting_b200 import _lib, scenes
from frosting_b200 import rasterizer as fbr
from frosting_b200._lib import Grads
from frosting_b200.frosting_render import _params_block
from oracle import cpu
from tests.test_c_abi_gpu import _one_phase, _p
from tests.test_shim_gpu import FROSTING_SH
from tests.util import SH_C0, rel_err_stats, sh_basis64, sh_dirs64, sh_layouts

pytestmark = pytest.mark.gpu

P, W, H = 6007, 241, 133
KEYS = ("means3D", "opacities", "shs", "scales", "rotations")
PARAM_KEYS = ("bary_logits", "opacity_logits", "log_scales", "quats", "sh_dc", "sh_rest")


def _scene(M, D, dev, seed=21):
    """random_gaussians puts rows 0..119 at or behind the near plane (three whole runs of 32 and a partial one); rows
    3200..3279 (two whole runs and half of a third) and the 23-row tail run are moved behind the camera as well."""
    cam = scenes.make_camera(W, H)
    g = scenes.random_gaussians(P, cam, seed + M, sh_coeffs=M)
    g["means3D"][3200:3280, 2] = -1.0
    g["means3D"][P - 23:, 2] = -1.0
    rs = scenes.settings_for(cam, D, device=dev)
    return rs, {k: v.to(dev) for k, v in g.items()}


def _check_unrendered_pattern(radii):
    dead = (radii <= 0).cpu()
    assert dead[:96].all() and not dead[96:128].all() and dead[96:128].any()
    assert dead[3200:3264].all() and not dead[3264:3296].all()
    assert dead[P - 23:].all() and 1000 < int((~dead).sum()) < P - 200


def _grads(rs, g, cot, shs=None):
    leaves = {k: (shs if (k == "shs" and shs is not None) else g[k]).detach().clone().requires_grad_(True) for k in KEYS}
    m2 = torch.zeros(P, 3, device=cot.device, requires_grad=True)
    color, radii = fb.GaussianRasterizer(rs)(means3D=leaves["means3D"], means2D=m2, opacities=leaves["opacities"],
                                             shs=leaves["shs"], scales=leaves["scales"], rotations=leaves["rotations"])
    (color * cot).sum().backward()
    out = {k: leaves[k].grad for k in KEYS}
    out["means2D"] = m2.grad
    return color, radii, out


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.int32)


def _cot(dev, seed=3):
    return torch.randn(3, H, W, generator=torch.Generator().manual_seed(seed)).to(dev)


# ---- plain path ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,D", sh_layouts())
def test_plain_preprocess_is_bit_exact_with_the_oracle(cuda_device, M, D):
    rs, g = _scene(M, D, cuda_device)
    st = fb.forward_with_state(rs, g["means3D"], g["opacities"], shs=g["shs"], scales=g["scales"], rotations=g["rotations"])
    _check_unrendered_pattern(st["radii"])
    A = {k: v.cpu().numpy() for k, v in g.items()}
    pre = cpu.preprocess(cpu.Camera(rs), A["means3D"], A["opacities"], shs=A["shs"], scales=A["scales"],
                         rots=A["rotations"])
    radii = st["radii"].cpu().numpy()
    assert np.array_equal(radii, pre["radii"])
    vis = radii > 0
    rec = st["rec"].cpu().numpy()[vis]
    assert np.array_equal(st["depth"].cpu().numpy()[vis].view(np.int32), _bits(pre["depths"][vis]))
    assert np.array_equal(rec[:, 0:2].view(np.int32), _bits(pre["xy"][vis]))
    assert np.array_equal(rec[:, 2:6].view(np.int32), _bits(pre["conic_opacity"][vis]))
    assert np.array_equal(rec[:, 6:9].view(np.int32), _bits(pre["rgb"][vis]))
    cl = st["clamped"].cpu().numpy()[vis]
    assert np.array_equal(np.stack([cl & 1, (cl >> 1) & 1, (cl >> 2) & 1], 1), pre["clamped"][vis])


@pytest.mark.parametrize("M,D", [(M, D) for (M, D) in sh_layouts() if M < 16])
def test_plain_path_never_reads_coefficients_past_the_degree(cuda_device, M, D):
    """The same coefficients as [P, M, 3] rows and padded to [P, 16, 3], NaN at every index >= (D + 1)^2 in both."""
    dev = cuda_device
    rs, g = _scene(M, D, dev)
    n = (D + 1) ** 2
    narrow = g["shs"].clone()
    narrow[:, n:] = float("nan")
    wide = torch.full((P, 16, 3), float("nan"), device=dev)
    wide[:, :n] = g["shs"][:, :n]
    st = [fb.forward_with_state(rs, g["means3D"], g["opacities"], shs=s, scales=g["scales"], rotations=g["rotations"])
          for s in (narrow, wide)]
    for k in ("color", "final_T"):
        assert torch.equal(st[0][k].view(torch.int32), st[1][k].view(torch.int32)), k
    for k in ("radii", "n_contrib"):
        assert torch.equal(st[0][k], st[1][k]), k
    assert torch.isfinite(st[0]["color"]).all()
    cot = _cot(dev)
    c0, r0, g0 = _grads(rs, g, cot, narrow)
    c1, r1, g1 = _grads(rs, g, cot, wide)
    assert torch.equal(c0.view(torch.int32), c1.view(torch.int32)) and torch.equal(r0, r1)
    for k in g0:
        assert torch.isfinite(g0[k]).all() and torch.isfinite(g1[k]).all(), k
    for k in ("means3D", "means2D", "opacities", "scales", "rotations"):
        assert rel_err_stats(g0[k], g1[k])[0] <= 1e-3, k       # two blend backwards: atomic-order noise
    assert rel_err_stats(g0["shs"][:, :n], g1["shs"][:, :n])[0] <= 1e-3
    assert float(g0["shs"][:, :n].abs().max()) > 0
    assert not g0["shs"][:, n:].any() and not g1["shs"][:, n:].any()


@pytest.mark.parametrize("M,D", sh_layouts())
def test_plain_sh_gradient_is_the_basis_times_the_colour_gradient(cuda_device, M, D):
    """On every rendered row: dL/dsh[k, c] = b_k(dir) dL/dsh[0, c] / C0 with the float64 basis (independent of the blend
    backward's summation order), exact zeros on clamped channels and past (D + 1)^2; dL/dmeans3D against the oracle."""
    dev = cuda_device
    rs, g = _scene(M, D, dev)
    cot = _cot(dev, 4)
    color, radii, gr = _grads(rs, g, cot)
    st = fb.forward_with_state(rs, g["means3D"], g["opacities"], shs=g["shs"], scales=g["scales"], rotations=g["rotations"])
    assert torch.equal(st["radii"], radii)
    vis = (radii > 0).cpu()
    n = (D + 1) ** 2
    dsh = gr["shs"].cpu().double()
    assert not dsh[~vis].any() and not dsh[:, n:].any()
    dsh = dsh[vis]
    cl = st["clamped"].cpu()[vis]
    clamped = torch.stack([(cl & 1) != 0, (cl & 2) != 0, (cl & 4) != 0], 1)
    assert not dsh.permute(0, 2, 1)[clamped].any()
    basis = sh_basis64(sh_dirs64(g["means3D"].cpu()[vis], rs.campos.cpu()), D)
    want = basis[:, :, None] * (dsh[:, 0, :] / SH_C0)[:, None, :]
    row_scale = want.abs().amax(dim=(1, 2), keepdim=True).clamp_min(1e-30)
    err = ((dsh[:, :n] - want) / row_scale).abs().max().item()
    assert err <= 2e-6, err
    assert int((dsh[:, 0].abs() > 0).sum()) > 1000
    # the view-direction term and the geometry: the whole dL/dmeans3D against the oracle's backward
    A = {k: v.cpu().numpy() for k, v in g.items()}
    kw = dict(shs=A["shs"], scales=A["scales"], rots=A["rotations"])
    f = cpu.forward(rs, A["means3D"], A["opacities"], **kw)
    assert np.array_equal(f["pre"]["radii"], radii.cpu().numpy())
    b = cpu.backward(rs, f, A["means3D"], cot.cpu().numpy(), **kw)
    for k, mine in (("means3D", gr["means3D"]), ("sh", gr["shs"])):
        ref = b[k].astype(np.float64)
        e = np.abs(mine.cpu().numpy().astype(np.float64) - ref).max() / max(np.abs(ref).max(), 1e-30)
        assert e <= 2e-3, (k, e)


@pytest.mark.parametrize("mode", ("dense", "sparse_rows", "dense_side_stream"))
@pytest.mark.parametrize("M", (1, 4, 9, 16))
def test_unrendered_gradient_rows_through_the_abi(cuda_device, M, mode):
    """fb200_backward into gradient buffers pre-filled with NaN.  Dense contract: every unrendered row is written with
    zeros -- whole runs of 32 (coalesced fill), the partial runs and the 23-row tail.  sparse_rows=1: unrendered rows are
    not touched.  dense_side_stream: debug bit 32 (what `rasterizer.ZERO_OVERLAP` sets) moves the fill of the whole runs
    to a side stream for P >= 4096."""
    dev = cuda_device
    D = math.isqrt(M) - 1
    rs, g = _scene(M, D, dev)
    R = fb.forward_with_state(rs, g["means3D"], g["opacities"], shs=g["shs"], scales=g["scales"],
                              rotations=g["rotations"])["num_rendered"]
    prm, inp, ws, color, radii, st, keep = _one_phase(rs, g, P, W, H, D, R + 17, dev)
    assert st[_lib.ST_NUM_RENDERED] == R and st[_lib.ST_OVERFLOW] == 0
    _check_unrendered_pattern(radii)
    nan = float("nan")
    outs = dict(means2D=torch.full((P, 3), nan, device=dev), opacities=torch.full((P, 1), nan, device=dev),
                means3D=torch.full((P, 3), nan, device=dev), shs=torch.full((P, M, 3), nan, device=dev),
                scales=torch.full((P, 3), nan, device=dev), rotations=torch.full((P, 4), nan, device=dev))
    grads = Grads(d_dL_dmeans2D=_p(outs["means2D"]), d_dL_dcolors=None, d_dL_dopacity=_p(outs["opacities"]),
                  d_dL_dmeans3D=_p(outs["means3D"]), d_dL_dcov3D=None, d_dL_dsh=_p(outs["shs"]),
                  d_dL_dscales=_p(outs["scales"]), d_dL_drotations=_p(outs["rotations"]),
                  sparse_rows=1 if mode == "sparse_rows" else 0)
    if mode == "dense_side_stream":
        prm.debug = 32
    cot = _cot(dev, 6)
    L = _lib.lib()
    _lib.check(L.fb200_backward(C.byref(prm), C.byref(inp), C.byref(ws), _p(radii), _p(cot), C.byref(grads),
                                C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
    torch.cuda.synchronize(dev)
    dead = radii <= 0
    _, r_ref, ref = _grads(rs, g, cot)
    assert torch.equal(r_ref, radii)
    for k, t in outs.items():
        rows = t.reshape(P, -1)
        if mode == "sparse_rows":
            assert torch.isnan(rows[dead]).all(), k
        else:
            assert not rows[dead].any() and not torch.isnan(rows[dead]).any(), k
        assert torch.isfinite(rows[~dead]).all(), k
        assert rel_err_stats(rows[~dead], ref[k].reshape(P, -1)[~dead])[0] <= 1e-3, k


@pytest.mark.parametrize("M,D", ((4, 2), (9, 3)))
def test_plain_degree_beyond_the_row_is_refused(cuda_device, M, D):
    rs, g = _scene(M, D, cuda_device)
    before = _lib.kernel_launches()
    with pytest.raises(_lib.Fb200Error, match="sh_degree / sh_coeffs inconsistent"):
        fb.GaussianRasterizer(rs)(means3D=g["means3D"], means2D=None, opacities=g["opacities"], shs=g["shs"],
                                  scales=g["scales"], rotations=g["rotations"])
    assert _lib.kernel_launches() == before


# ---- frosting: fused attribute kernels and frosting mode -------------------------------------------------------------
def _frosting(R, Pn, dev, seed=13, W_=200, H_=120, faces=500):
    cam = scenes.make_camera(W_, H_, device=dev)
    params, mesh = scenes.frosting_layer(Pn, cam, seed, n_faces_target=faces, device=dev, view_distance=4.5,
                                         sh_coeffs=R + 1)
    return cam, params, mesh


@pytest.mark.parametrize("density", (1.0, 0.6, 0.3))
@pytest.mark.parametrize("Pn", (3001, 4096 + 17))
@pytest.mark.parametrize("R", (0, 3, 8, 15))
def test_fused_attribute_kernels_at_every_rest_width(cuda_device, R, Pn, density):
    """fb200_frosting_attributes(_backward) against the float64 torch statement of Frosting's properties.  Mask
    densities 0.6 / 0.3 put most warps on the staged / unstaged rest-row path; rows 64..95 are all masked (the warp's
    coalesced zero fill), rows 96..127 all live."""
    dev = cuda_device
    _, params, mesh = _frosting(R, Pn, dev, seed=13 + R)
    live = torch.ones(Pn, dtype=torch.bool)
    if density < 1.0:
        live = torch.rand(Pn, generator=torch.Generator().manual_seed(Pn + R)) < density
        live[64:96] = False
        live[96:128] = True
    mask = None if density == 1.0 else live.to(dev)
    p32 = {k: v.detach().clone().requires_grad_(True) for k, v in params.items()}
    m32 = dict(mesh, inner=mesh["inner"].clone().requires_grad_(True), outer=mesh["outer"].clone().requires_grad_(True))
    out = fb.frosting_attributes_fused(p32, m32, mask)
    p64 = {k: v.detach().double().requires_grad_(True) for k, v in params.items()}
    m64 = dict(mesh, inner=mesh["inner"].double().requires_grad_(True), outer=mesh["outer"].double().requires_grad_(True))
    ref = scenes.frosting_attributes(p64, m64)
    lv = live.to(dev)
    for k, v in out.items():
        assert v.shape == ref[k].shape, k
        r = ref[k].detach()[lv]
        assert (v[lv].double() - r).abs().max().item() <= 1e-6 * max(1.0, r.abs().max().item()), k
    gen = torch.Generator().manual_seed(R * 7 + Pn)
    cot = {k: torch.randn(v.shape, generator=gen).to(dev) for k, v in out.items()}
    sum((out[k] * cot[k]).sum() for k in out).backward()
    rows = lv.double().view(-1, 1)
    sum((ref[k] * cot[k].double() * rows.view(-1, *([1] * (ref[k].dim() - 1)))).sum() for k in ref).backward()
    for k in PARAM_KEYS:
        mine, want = p32[k].grad, p64[k].grad
        assert mine.shape == want.shape, k
        assert torch.isfinite(mine).all(), k
        assert not mine[~lv].any(), k
        if want.numel():
            assert (mine.double() - want).abs().max().item() <= 2e-5 * want.abs().max().item(), k
    for k in ("inner", "outer"):
        want = m64[k].grad
        assert (m32[k].grad.double() - want).abs().max().item() <= 2e-5 * want.abs().max().item(), k


def _frosting_geometry(params, mesh, rs):
    """Frosting mode's preprocess state (radii, depth, packed records, clamp bits) from the geometry phase alone."""
    fp, keep, dev = _params_block(*(params[k] for k in PARAM_KEYS), mesh["inner"], mesh["outer"], mesh["cells"],
                                  mesh["faces"], None)
    _, radii, call, _ = fbr._launch_forward(None, None, None, None, None, None, None, rs, None, geometry_only=True,
                                            frosting=(fp, keep, dev))
    Pn, Wn, Hn = call.prm.P, call.prm.image_width, call.prm.image_height
    lay = _lib.Layout()
    _lib.check(_lib.lib().fb200_get_layout(Pn, Wn, Hn, 0, C.byref(lay)))

    def view(off, nbytes, dtype):
        base = (-call.geom.data_ptr()) % 128
        return call.geom[base + off: base + off + nbytes].view(dtype)
    return dict(radii=radii.cpu().numpy(), depth=view(lay.geom_depth, Pn * 4, torch.float32).cpu().numpy(),
                rec=view(lay.geom_rec, Pn * 48, torch.float32).view(Pn, 12).cpu().numpy(),
                clamped=view(lay.geom_clamped, Pn, torch.uint8).cpu().numpy())


@pytest.mark.parametrize("R,D", FROSTING_SH)
def test_frosting_mode_preprocess_is_bit_exact_with_the_oracle(cuda_device, R, D):
    """Frosting mode builds the attributes inside preprocess with the same device functions as the fused attribute
    kernel, so its packed records equal the C oracle's preprocess of that kernel's outputs bit for bit."""
    dev = cuda_device
    cam, params, mesh = _frosting(R, 3001, dev, seed=11 + R)
    rs = scenes.settings_for(cam, D, device=dev)
    st = _frosting_geometry(params, mesh, rs)
    with torch.no_grad():
        a = fb.frosting_attributes_fused(params, mesh)
    A = {k: v.cpu().numpy() for k, v in a.items()}
    pre = cpu.preprocess(cpu.Camera(rs), A["means3D"], A["opacities"], shs=A["shs"], scales=A["scales"],
                         rots=A["rotations"])
    assert np.array_equal(st["radii"], pre["radii"])
    vis = st["radii"] > 0
    assert 200 < vis.sum() < 3001
    rec = st["rec"][vis]
    assert np.array_equal(st["depth"][vis].view(np.int32), _bits(pre["depths"][vis]))
    assert np.array_equal(rec[:, 0:2].view(np.int32), _bits(pre["xy"][vis]))
    assert np.array_equal(rec[:, 2:6].view(np.int32), _bits(pre["conic_opacity"][vis]))
    assert np.array_equal(rec[:, 6:9].view(np.int32), _bits(pre["rgb"][vis]))
    cl = st["clamped"][vis]
    assert np.array_equal(np.stack([cl & 1, (cl >> 1) & 1, (cl >> 2) & 1], 1), pre["clamped"][vis])


@pytest.mark.parametrize("R,D", [(R, D) for (R, D) in FROSTING_SH if (D + 1) ** 2 < R + 1])
def test_frosting_mode_never_reads_rest_coefficients_past_the_degree(cuda_device, R, D):
    """SH warm-up: the rest coefficients past (D + 1)^2 - 1 set to NaN change nothing in the image, get exact-zero
    gradients, and no gradient is NaN."""
    dev = cuda_device
    cam, params, mesh = _frosting(R, 4096 + 17, dev, seed=17 + R, W_=241, H_=133)
    rs = scenes.settings_for(cam, D, device=dev)
    n = (D + 1) ** 2
    poisoned = dict(params, sh_rest=params["sh_rest"].clone())
    poisoned["sh_rest"][:, n - 1:] = float("nan")
    cot = torch.randn(3, 133, 241, generator=torch.Generator().manual_seed(9)).to(dev)
    res = []
    for src in (params, poisoned):
        p = {k: v.detach().clone().requires_grad_(True) for k, v in src.items()}
        color, radii = fb.frosting_render(p, mesh, rs)
        (color * cot).sum().backward()
        res.append((color, radii, p))
    (c0, r0, p0), (c1, r1, p1) = res
    assert torch.equal(r0, r1) and 200 < int((r0 > 0).sum()) < 4096
    assert torch.equal(c0.view(torch.int32), c1.view(torch.int32))
    for k in PARAM_KEYS:
        assert torch.isfinite(p1[k].grad).all(), k
        assert rel_err_stats(p1[k].grad, p0[k].grad)[0] <= 1e-3, k
    assert not p1["sh_rest"].grad[:, n - 1:].any() and not p0["sh_rest"].grad[:, n - 1:].any()
    assert float(p1["sh_dc"].grad.abs().max()) > 0


@pytest.mark.parametrize("R,D", ((8, 3), (16, 3)))
def test_frosting_mode_refuses_inconsistent_layouts(cuda_device, R, D):
    dev = cuda_device
    cam, params, mesh = _frosting(R, 3001, dev)
    rs = scenes.settings_for(cam, D, device=dev)
    before = _lib.kernel_launches()
    with pytest.raises(_lib.Fb200Error, match="sh_degree / sh_coeffs inconsistent" if R <= 15 else r"sh_rest <= 15"):
        fb.frosting_render(params, mesh, rs)
    assert _lib.kernel_launches() == before
