"""GPU parity: frosting_b200 (through its C ABI) against the UNMODIFIED reference rasterizer, whose outputs for these
inputs are recorded in tests/golden/ref_outputs.npz (tests/golden/make_ref_golden.py; SURVEY.md section 8c).
Integer / index work bit-exact, forward colour <= 1e-4 abs, gradients <= 1e-3 relative (tests/util.py::rel_err_stats)."""
import pytest
import torch

import frosting_b200 as fb
from frosting_b200 import rasterizer as fbr
from oracle import cpu
from tests.util import scene, rel_err_stats, golden_case, check_inputs, check_forward, check_grad, ours_forward_fields

pytestmark = pytest.mark.gpu

CONFIGS = [
    # P, W, H, seed, sh_degree, bg
    (10_000, 256, 256, 1235, 0, 0.0),      # BASELINE config 1 shape
    (60_000, 400, 304, 7, 3, 1.0),         # ragged: 304 = 19*16, 400 = 25*16
    (200_000, 803, 597, 11, 2, 0.0),       # W, H not multiples of 16
    (500_000, 800, 800, 1236, 3, 0.0),     # BASELINE config 2
]
KEYS = ("means3D", "opacities", "shs", "scales", "rotations")
FWD_FIELDS = ("num_rendered", "radii", "depth", "touched", "means2D", "conic", "rgb", "clamped", "ranges", "point_list",
              "key_depth", "key_index", "n_contrib", "final_T", "color")
LIST_FIELDS = ("num_rendered", "point_list", "n_contrib", "color")


def _id(c):
    return f"P{c[0]}_{c[1]}x{c[2]}_D{c[4]}"


def _fields(st, names):
    f = ours_forward_fields(st)
    return {k: f[k] for k in names}


def cotangent(H, W, device):
    return torch.randn(3, H, W, generator=torch.Generator().manual_seed(99)).to(device)


@pytest.mark.parametrize("cfg", CONFIGS, ids=_id)
def test_forward_bit_exact_vs_reference(cfg, cuda_device):
    P, W, H, seed, D, bg = cfg
    cam, g, rs = scene(P, W, H, seed, D, cuda_device, bg)
    case = golden_case("parity_fwd_" + _id(cfg))
    check_inputs(case, *(g[k] for k in KEYS))
    st = fb.forward_with_state(rs, g["means3D"], g["opacities"], shs=g["shs"], scales=g["scales"],
                               rotations=g["rotations"])
    # per-Gaussian integers and integer-determining floats, binning (ranges, sorted order, keys), per-pixel integer
    # state: bit-exact; colour within 1e-4 abs.  Reference key = tile<<32 | depth_bits; ours = depth_bits<<32 | idx.
    check_forward(case, _fields(st, FWD_FIELDS))


@pytest.mark.parametrize("cfg", CONFIGS[:3], ids=_id)
def test_backward_vs_reference(cfg, cuda_device):
    P, W, H, seed, D, bg = cfg
    cam, g, rs = scene(P, W, H, seed, D, cuda_device, bg)
    cot = cotangent(H, W, cuda_device)
    case = golden_case("parity_bwd_" + _id(cfg))
    check_inputs(case, *(g[k] for k in KEYS), cot)

    leaves = {k: g[k].clone().requires_grad_(True) for k in KEYS}
    means2D = torch.zeros(P, 3, device=cuda_device, requires_grad=True)
    color, radii = fb.GaussianRasterizer(rs)(
        means3D=leaves["means3D"], means2D=means2D, opacities=leaves["opacities"], shs=leaves["shs"],
        scales=leaves["scales"], rotations=leaves["rotations"])
    (color * cot).sum().backward()
    check_forward(case, {"radii": radii})
    mine = dict(means3D=leaves["means3D"].grad, means2D=means2D.grad, sh=leaves["shs"].grad,
                opacities=leaves["opacities"].grad, scales=leaves["scales"].grad, rotations=leaves["rotations"].grad)
    for k, v in mine.items():
        assert v is not None and v.shape == (means2D.shape if k == "means2D" else g["shs" if k == "sh" else k].shape), k
        check_grad(case, k, v, radii, tag=_id(cfg))
    assert torch.equal(means2D.grad[:, 2], torch.zeros_like(means2D.grad[:, 2]))


@pytest.mark.parametrize("cfg", CONFIGS[1:3], ids=lambda c: f"P{c[0]}_{c[1]}x{c[2]}_D{c[4]}")
def test_subtile_culling_is_output_neutral(cfg, cuda_device):
    """Culled pairs contribute nothing by construction, so outputs must be BIT-identical with culling off."""
    P, W, H, seed, D, bg = cfg
    cam, g, rs = scene(P, W, H, seed, D, cuda_device, bg)
    kw = dict(shs=g["shs"], scales=g["scales"], rotations=g["rotations"])
    a = fb.forward_with_state(rs, g["means3D"], g["opacities"], **kw)
    fbr.NO_CULL = True
    try:
        b = fb.forward_with_state(rs, g["means3D"], g["opacities"], **kw)
    finally:
        fbr.NO_CULL = False
    assert torch.equal(a["n_contrib"], b["n_contrib"])
    assert torch.equal(a["color"].view(torch.int32), b["color"].view(torch.int32))
    assert torch.equal(a["final_T"].view(torch.int32), b["final_T"].view(torch.int32))


def precomp_inputs(device):
    """Inputs of the colors_precomp + cov3D_precomp case.  The covariances are the C oracle's preprocess output, which is
    bit-exact with the reference's geometry buffer (test_oracle_vs_ref_gpu.py), so both sides see the covariance the
    reference derives from these scales / rotations; culled rows get a small isotropic one."""
    P, W, H = 50_000, 320, 240
    cam, g, rs = scene(P, W, H, 5, 0, device, 0.5)
    gen = torch.Generator().manual_seed(3)
    colors = torch.rand(P, 3, generator=gen).to(device)
    A = {k: g[k].cpu().numpy() for k in ("means3D", "opacities", "scales", "rotations")}
    pre = cpu.preprocess(cpu.Camera(rs), A["means3D"], A["opacities"], colors_precomp=colors.cpu().numpy(),
                         scales=A["scales"], rots=A["rotations"])
    cov = torch.from_numpy(pre["cov3D"]).to(device)
    cov[torch.from_numpy(pre["radii"] <= 0).to(device)] = \
        0.01 * torch.eye(3, device=device)[[0, 0, 0, 1, 1, 2], [0, 1, 2, 1, 2, 2]]
    cot = torch.randn(3, H, W, generator=gen).to(device)
    return rs, g, colors, cov, cot


def test_precomputed_colour_and_covariance_path(cuda_device):
    """colors_precomp + cov3D_precomp branch (forward.cu:204-215,243-249; depth/normal passes of
    sugar_model.py:2364-2375 use colors_precomp)."""
    rs, g, colors, cov, cot = precomp_inputs(cuda_device)
    P = colors.shape[0]
    case = golden_case("parity_precomp")
    check_inputs(case, g["means3D"], g["opacities"], colors, cov, cot)
    st = fb.forward_with_state(rs, g["means3D"], g["opacities"], colors_precomp=colors, cov3D_precomp=cov)
    check_forward(case, _fields(st, ("radii", "point_list", "color")))
    m3 = g["means3D"].clone().requires_grad_(True)
    col = colors.clone().requires_grad_(True)
    cv = cov.clone().requires_grad_(True)
    op = g["opacities"].clone().requires_grad_(True)
    m2 = torch.zeros(P, 3, device=cuda_device, requires_grad=True)
    color, radii = fb.GaussianRasterizer(rs)(means3D=m3, means2D=m2, opacities=op, colors_precomp=col, cov3D_precomp=cv)
    (color * cot).sum().backward()
    for name, mine in (("means3D", m3.grad), ("colors", col.grad), ("cov3D", cv.grad), ("opacities", op.grad),
                       ("means2D", m2.grad)):
        check_grad(case, name, mine, radii, frac_bar=5e-3, tag="precomp")


def test_visibility_mask_equals_boolean_gather(cuda_device):
    """In-kernel occlusion mask == the reference's boolean-gather of every attribute
    (frosting_model.py:1578-1586): same image, gradients scattered back to the kept rows."""
    P, W, H = 80_000, 400, 300
    cam, g, rs = scene(P, W, H, 21, 3, cuda_device)
    gen = torch.Generator().manual_seed(4)
    mask = (torch.rand(P, generator=gen) < 0.6).to(cuda_device)
    cot = torch.randn(3, H, W, generator=gen).to(cuda_device)
    r = fb.GaussianRasterizer(rs)

    def run(masked_in_kernel):
        leaves = {k: g[k].clone().requires_grad_(True) for k in ("means3D", "opacities", "shs", "scales", "rotations")}
        if masked_in_kernel:
            m2 = torch.zeros(P, 3, device=cuda_device, requires_grad=True)
            color, radii = r(means3D=leaves["means3D"], means2D=m2, opacities=leaves["opacities"], shs=leaves["shs"],
                             scales=leaves["scales"], rotations=leaves["rotations"], visibility_mask=mask)
        else:
            m2 = torch.zeros(int(mask.sum()), 3, device=cuda_device, requires_grad=True)
            color, radii = r(means3D=leaves["means3D"][mask], means2D=m2, opacities=leaves["opacities"][mask],
                             shs=leaves["shs"][mask], scales=leaves["scales"][mask], rotations=leaves["rotations"][mask])
        (color * cot).sum().backward()
        return color.detach(), radii, {k: v.grad for k, v in leaves.items()}

    c1, r1, g1 = run(True)
    c2, r2, g2 = run(False)
    assert torch.equal(c1.view(torch.int32), c2.view(torch.int32))
    assert torch.equal(r1[mask], r2) and int(r1[~mask].abs().sum()) == 0
    for k in g1:
        m, frac = rel_err_stats(g1[k], g2[k])
        assert m <= 1e-3 and frac <= 1e-3, (k, m, frac)     # atomic-order noise between two runs (tail seen: 1.7e-4)
        assert float(g1[k][~mask].abs().sum()) == 0.0


def test_edge_cases(cuda_device):
    dev = cuda_device
    cam, g, rs = scene(2_000, 100, 60, 2, 1, dev, 0.25)
    r = fb.GaussianRasterizer(rs)
    # P = 0
    z = torch.zeros(0, 3, device=dev)
    color, radii = r(means3D=z, means2D=z, opacities=torch.zeros(0, 1, device=dev), shs=torch.zeros(0, 16, 3, device=dev),
                     scales=z, rotations=torch.zeros(0, 4, device=dev))
    assert color.shape == (3, 60, 100) and torch.allclose(color, torch.full_like(color, 0.25)) and radii.numel() == 0
    # everything behind the camera
    m = g["means3D"].clone(); m[:, 2] = -1.0
    color, radii = r(means3D=m, means2D=torch.zeros_like(m), opacities=g["opacities"], shs=g["shs"], scales=g["scales"],
                     rotations=g["rotations"])
    assert int(radii.abs().sum()) == 0 and torch.allclose(color, torch.full_like(color, 0.25))
    # argument validation, same messages as DGR/diff_gaussian_rasterization/__init__.py:191-195
    with pytest.raises(Exception, match="excatly one of either SHs or precomputed colors"):
        r(means3D=m, means2D=m, opacities=g["opacities"], scales=g["scales"], rotations=g["rotations"])
    with pytest.raises(Exception, match="exactly one of either scale/rotation pair"):
        r(means3D=m, means2D=m, opacities=g["opacities"], shs=g["shs"])
    # markVisible == near-plane test
    vis = r.markVisible(g["means3D"])
    assert vis.dtype == torch.bool and torch.equal(vis, g["means3D"][:, 2] > 0.2)
    # a single huge Gaussian covering every tile (exercises long rects, single-instance tiles)
    rs, one = edge_one(dev)
    st = fb.forward_with_state(rs, one["means3D"], one["opacities"], shs=one["shs"], scales=one["scales"],
                               rotations=one["rotations"])
    T = ((100 + 15) // 16) * ((60 + 15) // 16)
    assert st["num_rendered"] == T and int(st["radii"][0]) > 0
    check_forward(golden_case("parity_edge_one"), {"color": st["color"]})


def edge_one(device):
    cam, g, rs = scene(2_000, 100, 60, 2, 1, device, 0.25)
    one = dict(means3D=torch.tensor([[0.0, 0.0, 3.0]], device=device), opacities=torch.tensor([[0.9]], device=device),
               scales=torch.full((1, 3), 5.0, device=device), rotations=torch.tensor([[1.0, 0, 0, 0]], device=device),
               shs=torch.ones(1, 16, 3, device=device))
    return rs, one


def long_tile_scenes(device):
    from frosting_b200 import scenes
    cam = scenes.make_camera(64, 48, device=device)
    rs = scenes.settings_for(cam, 1, device=device)
    for P in (3_000, 9_000, 60_000):
        g = scenes.random_gaussians(P, cam, 77, device=device, large_frac=0.0, near_frac=0.0)
        g["scales"] = g["scales"] * 3.0
        g["means3D"][: P // 60, :2] *= 0.02          # pile extra splats on the centre tiles
        yield P, rs, g


def test_long_tile_lists_all_sort_classes(cuda_device):
    """Force per-tile lists through the small (<= 2048, static smem), medium (<= 8192, 160 KB dynamic smem) and
    global-memory sort classes (binning.cu)."""
    covered = set()
    for P, rs, g in long_tile_scenes(cuda_device):
        case = golden_case(f"parity_long_{P}")
        check_inputs(case, *(g[k] for k in KEYS))
        st = fb.forward_with_state(rs, g["means3D"], g["opacities"], shs=g["shs"], scales=g["scales"], rotations=g["rotations"])
        counts = st["tile_count"]
        print(f"P={P}: tile list lengths min {int(counts.min())} max {int(counts.max())}")
        if bool(((counts > 1) & (counts <= 2048)).any()): covered.add("small")
        if bool(((counts > 2048) & (counts <= 8192)).any()): covered.add("medium")
        if bool((counts > 8192).any()): covered.add("global")
        check_forward(case, _fields(st, LIST_FIELDS))
    assert covered == {"small", "medium", "global"}, covered


def depth_tie_scene(device):
    from frosting_b200 import scenes
    P, W, H = 30_000, 160, 128
    cam = scenes.make_camera(W, H, device=device)
    g = scenes.random_gaussians(P, cam, 5, device=device, large_frac=0.0, near_frac=0.0)
    g["means3D"][:, 2] = torch.tensor([3.0, 4.0, 5.0, 4.0], device=device).repeat(P // 4)   # only 3 distinct depths
    return P, scenes.settings_for(cam, 0, device=device), g


def test_equal_depth_ties_follow_gaussian_index(cuda_device):
    """Exact depth ties: the reference's stable radix sort keeps ascending Gaussian index
    (rasterizer_impl.cu:98-108 emission order); our per-tile sort must reproduce it."""
    P, rs, g = depth_tie_scene(cuda_device)
    case = golden_case("parity_ties")
    check_inputs(case, *(g[k] for k in KEYS))
    st = fb.forward_with_state(rs, g["means3D"], g["opacities"], shs=g["shs"], scales=g["scales"], rotations=g["rotations"])
    check_forward(case, _fields(st, LIST_FIELDS))


def test_fused_frosting_attributes_match_torch_chain(cuda_device):
    """Row a20: one kernel vs Frosting's softmax/gather/sum/sigmoid/exp/normalize/cat chain
    (frosting_scene/frosting_model.py:713-799, restated in scenes.frosting_attributes): values 1e-6, gradients 1e-5
    relative to scale, incl. the scatter-added shell-vertex gradients; masked rows get zero gradient."""
    dev = cuda_device
    from frosting_b200 import scenes
    cam = scenes.make_camera(200, 120, device=dev)
    params, mesh = scenes.frosting_layer(30_000, cam, 11, n_faces_target=5000, device=dev)
    gen = torch.Generator().manual_seed(5)
    cots = {k: torch.randn(s, generator=gen).to(dev) for k, s in
            dict(means3D=(30_000, 3), opacities=(30_000, 1), scales=(30_000, 3), rotations=(30_000, 4), shs=(30_000, 16, 3)).items()}

    def run(fn, mask):
        p = {k: v.clone().requires_grad_(True) for k, v in params.items()}
        m = dict(mesh); m["inner"] = mesh["inner"].clone().requires_grad_(True); m["outer"] = mesh["outer"].clone().requires_grad_(True)
        out = fn(p, m) if mask is None else fn(p, m, mask)
        w = 1.0 if mask is None else mask.float()
        loss = sum(((out[k] * cots[k]).reshape(30_000, -1).sum(1) * w).sum() for k in cots)
        loss.backward()
        grads = {k: v.grad for k, v in p.items()}
        grads["inner"], grads["outer"] = m["inner"].grad, m["outer"].grad
        return {k: v.detach() for k, v in out.items()}, grads

    ref_out, ref_g = run(scenes.frosting_attributes, None)
    out, g = run(fb.frosting_attributes_fused, None)
    for k in ref_out:
        assert out[k].shape == ref_out[k].shape
        assert (out[k] - ref_out[k]).abs().max().item() <= 1e-6 * max(1.0, ref_out[k].abs().max().item()), k
    for k in ref_g:
        scale = ref_g[k].abs().max().item()
        assert (g[k] - ref_g[k]).abs().max().item() <= 2e-5 * scale, (k, (g[k] - ref_g[k]).abs().max().item() / scale)
    # masked variant: kept rows identical, dropped rows contribute nothing
    mask = torch.rand(30_000, generator=gen).to(dev) < 0.4
    out_m, g_m = run(fb.frosting_attributes_fused, mask)

    def ref_masked(p, m):
        return scenes.frosting_attributes(p, m)
    ro, rg = run(lambda p, m, mk: scenes.frosting_attributes(p, m), mask)
    for k in ro:
        assert (out_m[k][mask] - ro[k][mask]).abs().max().item() <= 1e-6 * max(1.0, ro[k].abs().max().item()), k
    for k in rg:
        scale = rg[k].abs().max().item()
        assert (g_m[k] - rg[k]).abs().max().item() <= 2e-5 * scale, (k, "masked")
    # end to end: fused attributes + in-kernel mask feed the rasterizer exactly like the torch chain + gathers
    rs = scenes.settings_for(cam, 3, device=dev)
    a1 = fb.frosting_attributes_fused(params, mesh, mask)
    a2 = scenes.frosting_attributes(params, mesh)
    r = fb.GaussianRasterizer(rs)
    z = torch.zeros(30_000, 3, device=dev)
    c1, _ = r(means3D=a1["means3D"], means2D=z, opacities=a1["opacities"], shs=a1["shs"], scales=a1["scales"],
              rotations=a1["rotations"], visibility_mask=mask)
    c2, _ = r(means3D=a2["means3D"][mask], means2D=z[mask], opacities=a2["opacities"][mask], shs=a2["shs"][mask],
              scales=a2["scales"][mask], rotations=a2["rotations"][mask])
    # the two attribute paths agree to ~1 ulp, which is enough to flip an alpha < 1/255 or tile-rect decision
    # for a handful of pixel/Gaussian pairs (each worth up to ~4e-3): compare statistically
    d = (c1 - c2).abs()
    assert (d > 1e-4).float().mean().item() < 1e-3 and d.max().item() < 2e-2


def test_backward_twice_over_one_forward(cuda_device):
    """The accumulators are cleared by the forward for the FIRST backward only (fb200_workspace.acc_zeroed_by_forward);
    a second backward over the same graph must clear them itself and give the same gradients."""
    P, W, H = 20_000, 256, 160
    cam, g, rs = scene(P, W, H, 9, 2, cuda_device, 0.0)
    leaves = {k: g[k].clone().requires_grad_(True) for k in ("means3D", "opacities", "shs", "scales", "rotations")}
    m2 = torch.zeros(P, 3, device=cuda_device, requires_grad=True)
    color, _ = fb.GaussianRasterizer(rs)(means3D=leaves["means3D"], means2D=m2, opacities=leaves["opacities"],
                                         shs=leaves["shs"], scales=leaves["scales"], rotations=leaves["rotations"])
    cot = torch.randn(3, H, W, generator=torch.Generator().manual_seed(1)).to(cuda_device)
    loss = (color * cot).sum()
    loss.backward(retain_graph=True)
    first = {k: v.grad.clone() for k, v in leaves.items()}
    for v in leaves.values():
        v.grad = None
    loss.backward()
    for k, v in leaves.items():
        m, frac = rel_err_stats(v.grad, first[k])
        assert m <= 1e-3 and frac <= 1e-3, (k, m, frac)          # equal up to the order of the float atomics
