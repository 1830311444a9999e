"""CPU suite: the C oracle against golden vectors produced by the UNMODIFIED reference on a B200
(tests/golden/make_golden.py).  The reference ships no fixtures of its own (SURVEY.md section 4), so these
vectors -- plus tests/test_oracle_vs_ref_gpu.py on the GPU box -- are what pins the oracle."""
import glob
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import cpu

GOLD = sorted(p for p in glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.npz"))
              if not os.path.basename(p).startswith(("loss_", "adam", "frosting_", "ref_outputs")))


def _settings(z):
    return SimpleNamespace(image_width=int(z["W"]), image_height=int(z["H"]), tanfovx=float(z["tanfovx"]),
                           tanfovy=float(z["tanfovy"]), viewmatrix=torch.from_numpy(z["viewmatrix"]),
                           projmatrix=torch.from_numpy(z["projmatrix"]), campos=torch.from_numpy(z["campos"]),
                           bg=torch.full((3,), float(z["bg"])), sh_degree=int(z["D"]), scale_modifier=1.0)


def test_golden_fixtures_present():
    assert len(GOLD) >= 3, "golden vectors missing: run tests/golden/make_golden.py on the GPU box"


@pytest.mark.parametrize("path", GOLD, ids=lambda p: os.path.basename(p)[:-4])
def test_oracle_reproduces_reference_golden_vectors(path):
    z = np.load(path)
    rs = _settings(z)
    kw = dict(scales=z["scales"], rots=z["rotations"])
    if "shs" in z.files:
        kw["shs"] = z["shs"]
    else:
        kw["colors_precomp"] = z["colors_precomp"]
    o = cpu.forward(rs, z["means3D"], z["opacities"], **kw)
    vis = z["radii"] > 0
    # integer-determining stage: bit-exact
    assert np.array_equal(o["pre"]["radii"], z["radii"])
    assert np.array_equal(o["pre"]["depths"][vis].view(np.int32), z["depths"][vis].view(np.int32))
    assert np.array_equal(o["pre"]["xy"][vis].view(np.int32), z["means2D"][vis].view(np.int32))
    assert np.array_equal(o["pre"]["conic_opacity"][vis].view(np.int32), z["conic_opacity"][vis].view(np.int32))
    if "shs" in z.files:
        assert np.array_equal(o["pre"]["rgb"][vis].view(np.int32), z["rgb"][vis].view(np.int32))
    assert np.array_equal(o["pre"]["tiles_touched"][vis].astype(np.int32), z["tiles_touched"][vis])
    assert o["binned"]["num_rendered"] == int(z["num_rendered"])
    assert np.array_equal(o["binned"]["point_list"].astype(np.int32), z["point_list"])
    assert np.array_equal(o["binned"]["ranges"].astype(np.int32), z["ranges"])
    # blend (libm expf vs libdevice expf: ~2 ulp, a handful of threshold flips allowed)
    assert (o["n_contrib"].astype(np.int32) != z["n_contrib"]).mean() < 2e-3
    err = np.abs(o["color"] - z["color"])
    assert np.quantile(err, 0.999) <= 1e-5 and err.max() <= 5e-3, (np.quantile(err, 0.999), err.max())
    tol_T = np.abs(o["final_T"] - z["final_T"])
    assert np.quantile(tol_T, 0.999) <= 1e-5
    # backward
    b = cpu.backward(rs, o, z["means3D"], z["cot"], **kw)
    names = ["means3D", "means2D", "opacities", "scales", "rotations", "colors", "cov3D"] + (["sh"] if "shs" in z.files else [])
    for k in names:
        a, r = b[k].astype(np.float64).ravel(), z["g_" + k].astype(np.float64).ravel()
        scale = max(np.abs(r).max(), 1e-30)
        assert np.abs(a - r).max() / scale <= 2e-3, (k, np.abs(a - r).max() / scale)


def test_oracle_gradients_against_finite_differences():
    """Coarse independent check of the oracle's backward maths (signs, chain structure): central differences of
    the oracle's own forward.  The renderer is truncated at the 3-sigma tile rect and at alpha < 1/255, and the
    analytic gradient (the reference's, backward.cu) ignores those boundary terms, so agreement is ~5-15 %, not
    tight; the tight pin is the golden-vector test above."""
    rng = np.random.RandomState(0)
    P, W, H = 5, 160, 160
    from frosting_b200 import scenes
    cam = scenes.make_camera(W, H)
    rs = scenes.settings_for(cam, 1)
    means = np.stack([rng.uniform(-0.5, 0.5, P), rng.uniform(-0.5, 0.5, P), rng.uniform(2.0, 3.0, P)], 1).astype(np.float32)
    scales = rng.uniform(0.12, 0.25, (P, 3)).astype(np.float32)
    q = rng.randn(P, 4).astype(np.float32); rots = q / np.linalg.norm(q, axis=1, keepdims=True)
    opac = rng.uniform(0.3, 0.8, (P, 1)).astype(np.float32)
    shs = (rng.randn(P, 4, 3) * 0.3).astype(np.float32); shs[:, 0] += 1.0
    yy, xx = np.meshgrid(np.linspace(-1, 1, H), np.linspace(-1, 1, W), indexing="ij")
    cot = np.stack([xx, yy, 0.5 + 0.5 * xx * yy]).astype(np.float32)       # smooth cotangent

    def loss(m=means, s=scales, r=rots, o=opac, c=shs):
        f = cpu.forward(rs, m, o, shs=c, scales=s, rots=r)
        return float((f["color"].astype(np.float64) * cot).sum()), f

    _, f0 = loss()
    g = cpu.backward(rs, f0, means, cot, shs=shs, scales=scales, rots=rots)
    checks = [("means3D", means, "m"), ("scales", scales, "s"), ("rotations", rots, "r"), ("opacities", opac, "o"), ("sh", shs, "c")]
    for name, arr, key in checks:
        flat = arr.reshape(-1)
        for idx in rng.choice(flat.size, size=min(8, flat.size), replace=False):
            h = 2e-3 * max(1.0, abs(float(flat[idx])))
            ap, am = arr.copy(), arr.copy()
            ap.reshape(-1)[idx] += h; am.reshape(-1)[idx] -= h
            fd = (loss(**{key: ap})[0] - loss(**{key: am})[0]) / (float(ap.reshape(-1)[idx]) - float(am.reshape(-1)[idx]))
            an = float(g[name].reshape(-1)[idx])
            assert abs(fd - an) <= 0.25 * max(abs(an), abs(fd), 0.2 * np.abs(g[name]).max()), (name, idx, fd, an)


def test_oracle_binning_is_stable_and_ranges_partition():
    rng = np.random.RandomState(1)
    from frosting_b200 import scenes
    cam = scenes.make_camera(96, 64)
    g = scenes.random_gaussians(800, cam, 9)
    g["means3D"][:, 2] = torch.tensor([3.0, 4.0]).repeat(400)        # massive depth ties
    rs = scenes.settings_for(cam, 0)
    A = {k: v.numpy() for k, v in g.items()}
    o = cpu.forward(rs, A["means3D"], A["opacities"], shs=A["shs"], scales=A["scales"], rots=A["rotations"])
    keys, pl, rg = o["binned"]["keys"], o["binned"]["point_list"], o["binned"]["ranges"]
    R = o["binned"]["num_rendered"]
    assert np.all(np.diff(keys.astype(np.uint64)) >= 0)
    # stable: equal keys keep ascending Gaussian index (emission order)
    same = keys[1:] == keys[:-1]
    assert np.all(pl[1:][same] > pl[:-1][same])
    covered = np.zeros(R, bool)
    for t, (a, b) in enumerate(rg):
        if b > a:
            assert np.all((keys[a:b] >> np.uint64(32)) == t)
            covered[a:b] = True
    assert covered.all()
    assert np.array_equal(cpu.mark_visible(rs, A["means3D"]), A["means3D"][:, 2] > 0.2)


def _frosting_golden():
    import os
    import numpy as np
    import torch
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "frosting_attrs.npz"))
    params = {k[len("param_"):]: torch.from_numpy(z[k]) for k in z.files if k.startswith("param_")}
    mesh = {k[len("mesh_"):]: torch.from_numpy(z[k]) for k in z.files if k.startswith("mesh_")}
    return z, params, mesh


def test_frosting_attribute_restatement_is_pinned_to_the_reference_properties():
    """`scenes.frosting_attributes` -- the oracle of the fused attribute kernels and of bench.py's reference arm -- against
    vectors produced by EXECUTING the reference's own property source (frosting_model.py:643-799, cut out with ast by
    tests/golden/make_frosting_attr_golden.py): outputs and autograd gradients."""
    import numpy as np
    import torch
    from frosting_b200 import scenes
    z, params, mesh = _frosting_golden()
    leaf = {k: v.clone().requires_grad_(True) for k, v in params.items()}
    m = dict(mesh)
    m["inner"] = mesh["inner"].clone().requires_grad_(True)
    m["outer"] = mesh["outer"].clone().requires_grad_(True)
    out = scenes.frosting_attributes(leaf, m)
    for k, v in out.items():
        np.testing.assert_allclose(v.detach().numpy(), z[f"out_{k}"], rtol=1e-6, atol=1e-7, err_msg=k)
    sum((out[k] * torch.from_numpy(z[f"cot_{k}"])).sum() for k in out).backward()
    for k, v in leaf.items():
        ref = z[f"grad_{k}"]
        np.testing.assert_allclose(v.grad.numpy(), ref, rtol=2e-5, atol=2e-6 * np.abs(ref).max(), err_msg=k)
    # inner = base - t n, outer = base + t n  =>  d/d(base) = d/d(inner) + d/d(outer)
    both = (m["inner"].grad + m["outer"].grad).numpy()
    np.testing.assert_allclose(both, z["grad_base_verts"], rtol=2e-5, atol=2e-6 * np.abs(z["grad_base_verts"]).max())
