"""Pins the C oracle (oracle/raster_oracle.c) to the UNMODIFIED reference, whose outputs for these inputs are recorded in
tests/golden/ref_outputs.npz (tests/golden/make_ref_golden.py), and the CUDA mesh prepass to its C restatement."""
import numpy as np
import pytest
import torch

import frosting_b200 as fb
from frosting_b200 import scenes
from oracle import cpu
from tests.util import scene, golden_case, check_inputs, check_forward, grad_sample_index, spread

pytestmark = pytest.mark.gpu

CONFIGS = [(6000, 200, 136, 31, 3, 0.0), (4000, 96, 64, 32, 1, 1.0), (10_000, 256, 256, 1235, 0, 0.0)]
IDS = ["D3", "D1_bg1", "C1"]
FWD_FIELDS = ("radii", "depth", "means2D", "conic", "rgb", "cov3D", "touched", "num_rendered", "point_list", "keys",
              "ranges", "n_contrib")
GRADS = ("means3D", "means2D", "sh", "opacities", "scales", "rotations", "colors", "cov3D")
COLOR_SAMPLE = 1024


def cotangent(H, W, device):
    return torch.randn(3, H, W, generator=torch.Generator().manual_seed(1)).to(device)


@pytest.mark.parametrize("cfg", CONFIGS, ids=IDS)
def test_c_oracle_matches_compiled_reference(cfg, cuda_device):
    P, W, H, seed, D, bg = cfg
    cam, g, rs = scene(P, W, H, seed, D, cuda_device, bg)
    cot = cotangent(H, W, cuda_device)
    case = golden_case("oracle_" + IDS[CONFIGS.index(cfg)])
    check_inputs(case, *(g[k] for k in ("means3D", "opacities", "shs", "scales", "rotations")), cot)
    A = {k: v.cpu().numpy() for k, v in g.items()}
    o = cpu.forward(rs, A["means3D"], A["opacities"], shs=A["shs"], scales=A["scales"], rots=A["rotations"])
    vis = o["pre"]["radii"] > 0
    pre = o["pre"]
    # integer-determining stage and binning: bit-exact on the CPU as well
    check_forward(case, dict(
        radii=pre["radii"], depth=pre["depths"][vis].view(np.int32), means2D=pre["xy"][vis].view(np.int32),
        conic=pre["conic_opacity"][vis].view(np.int32), rgb=pre["rgb"][vis].view(np.int32),
        cov3D=pre["cov3D"][vis].view(np.int32), touched=pre["tiles_touched"][vis],
        num_rendered=o["binned"]["num_rendered"], point_list=o["binned"]["point_list"], keys=o["binned"]["keys"],
        ranges=o["binned"]["ranges"]))
    # blend: host expf differs from libdevice's by ~2 ulp, so allow a handful of threshold flips.  The reference's
    # per-pixel counts are stood in for by ours, which must equal them bit for bit.
    st = fb.forward_with_state(rs, g["means3D"], g["opacities"], shs=g["shs"], scales=g["scales"], rotations=g["rotations"])
    check_forward(case, {"n_contrib": st["n_contrib"]})
    nc_ref = st["n_contrib"].cpu().numpy()
    assert (o["n_contrib"].astype(np.int32) != nc_ref).mean() < 1e-3
    err = np.abs(o["color"].reshape(-1)[spread(o["color"].size, COLOR_SAMPLE)] - case["color"])
    assert np.quantile(err, 0.999) <= 1e-5 and err.max() <= 5e-3
    # backward (oracle accumulates in fp64, the reference with unordered float atomics)
    ob = cpu.backward(rs, o, A["means3D"], cot.cpu().numpy(), shs=A["shs"], scales=A["scales"], rots=A["rotations"])
    radii = torch.from_numpy(pre["radii"])
    for k in GRADS:
        a = torch.from_numpy(ob[k])
        mine = a.reshape(-1)[grad_sample_index(a, radii)].double().numpy()
        scale = max(float(case[k + ".stats"][0]), 1e-30)
        assert np.abs(mine - case[k + ".sample"]).max() / scale <= 2e-3, (k, np.abs(mine - case[k + ".sample"]).max() / scale)
        assert abs(np.abs(ob[k]).max() - scale) <= 2e-3 * scale, (k, np.abs(ob[k]).max(), scale)


def test_mesh_prepass_cuda_matches_c_restatement(cuda_device):
    """CUDA triangle raster vs oracle_mesh_raster: same pix_to_face, same visible set, incl. near-plane clipping,
    huge and sub-pixel triangles.  (No nvdiffrast oracle exists here: parity unpinned, DESIGN.md section 4.)"""
    dev = cuda_device
    W, H = 320, 200
    for case in ("sphere_far", "sphere_inside", "big_tris"):
        if case == "sphere_far":
            verts, faces, _ = scenes.uv_sphere(40, 64)
            cam = scenes.ring_cameras(5, W, H, radius=10.0)[2]
        elif case == "sphere_inside":          # camera inside the shell: triangles cross the near plane
            verts, faces, _ = scenes.uv_sphere(12, 16)
            cam = scenes.make_camera(W, H, scenes.look_at_w2c((0.0, 0.0, 5.0), (1.0, 0.3, 9.0)))
        else:
            g = torch.Generator().manual_seed(3)
            verts = torch.randn(60, 3, generator=g) * 3 + torch.tensor([0.0, 0.0, 7.0])
            faces = torch.randint(0, 60, (40, 3), generator=g, dtype=torch.int32)
            cam = scenes.make_camera(W, H)
        p2f_c, fv_c = cpu.mesh_raster(verts.numpy(), faces.numpy(), cam.full_proj_transform.numpy(), H, W, True)
        p2f, fv, _ = fb.rasterize_mesh(verts.to(dev), faces.to(dev), cam.full_proj_transform.to(dev), H, W,
                                       mark_last_on_bg=True)
        diff = (p2f.cpu().numpy() != p2f_c).mean()
        assert diff == 0.0, (case, diff)
        # the work-list path (default) and the every-class-over-all-faces path are the same rasteriser
        p2f_all, fv_all, _ = fb.rasterize_mesh(verts.to(dev), faces.to(dev), cam.full_proj_transform.to(dev), H, W,
                                               mark_last_on_bg=True, work_lists=False)
        assert torch.equal(p2f_all, p2f) and torch.equal(fv_all, fv), case
        assert np.array_equal(fv.cpu().numpy(), fv_c), case
        assert (p2f_c >= 0).any(), case
    # MeshRasterizer surface (frosting_utils/mesh_rasterization.py:109-172): shapes, -1 background, +1 convention
    verts, faces, _ = scenes.uv_sphere(20, 24)
    cam = scenes.ring_cameras(3, W, H, radius=10.0)[1]
    mr = fb.MeshRasterizer(cameras=[cam])
    p = mr((verts.to(dev), faces.to(dev)), return_only_pix_to_face=True)
    assert p.shape == (1, H, W, 1) and int(p.min()) == -1
    fr = mr((verts.to(dev), faces.to(dev)))
    assert fr.bary_coords.shape == (1, H, W, 1, 3) and fr.zbuf.shape == (1, H, W, 1)
    hit = fr.pix_to_face[0, ..., 0] >= 0
    b = fr.bary_coords[0, :, :, 0][hit]
    assert torch.allclose(b.sum(-1), torch.ones_like(b[:, 0]), atol=1e-4) and float(b.min()) > -1e-3
    raw = fb.nvdiff_rasterization(cam, H, W, verts=verts.to(dev), faces=faces.to(dev), return_indices_only=True)
    assert torch.equal(raw[0] - 1, p[0, ..., 0])
    # gaussian mask == _index_mask[_point_cell_indices] ++ ones (frosting_model.py:1564-1576), incl. the -1 quirk
    F = faces.shape[0]
    face_idx = p.unique()                                 # contains -1 when there is background
    index_mask = torch.zeros(F, dtype=torch.bool, device=dev)
    index_mask[face_idx.long()] = True                    # -1 marks the LAST face, as in the reference
    cells = torch.randint(0, F, (5000,), device=dev)
    expect = torch.cat([index_mask[cells], torch.ones(7, dtype=torch.bool, device=dev)])
    _, fv2, _ = fb.rasterize_mesh(verts.to(dev), faces.to(dev), cam.full_proj_transform.to(dev), H, W, mark_last_on_bg=True)
    got = fb.gaussian_render_mask(fv2, cells, 5007)
    assert torch.equal(got.bool(), expect)
