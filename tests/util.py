"""Shared helpers for the parity tests."""
import hashlib
import os

import numpy as np
import torch

from frosting_b200 import scenes

# The reference rasterizer's outputs for the parity tests' inputs, recorded by tests/golden/make_ref_golden.py.
# Bit-exact arrays are stored as digests, float arrays as a fixed sample plus their full-array scale.
REF_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_outputs.npz")
COLOR_SAMPLE = 512
GRAD_SAMPLE = 256
FLOAT_FIELDS = ("color",)
_golden = None


def scene(P, W, H, seed, sh_degree, device, bg=0.0):
    cam = scenes.make_camera(W, H, device=device)
    g = scenes.random_gaussians(P, cam, seed, device=device)
    rs = scenes.settings_for(cam, sh_degree, bg=torch.full((3,), float(bg)), device=device)
    return cam, g, rs


# ---- float64 statement of the SH colour (computeColorFromSH) ------------------------------------------------------
SH_C0 = 0.28209479177387814
SH_C1 = 0.4886025119029199
SH_C2 = (1.0925484305920792, -1.0925484305920792, 0.31539156525252005, -1.0925484305920792, 0.5462742152960396)
SH_C3 = (-0.5900435899266435, 2.890611442640554, -0.4570457994644658, 0.3731763325901154, -0.4570457994644658,
         1.445305721320277, -0.5900435899266435)


def sh_layouts():
    """Every (coefficients per row M, degree D) the plain path accepts: M in {1, 4, 9, 16}, (D + 1)^2 <= M."""
    return [(M, D) for M in (1, 4, 9, 16) for D in range(4) if (D + 1) ** 2 <= M]


def sh_dirs64(means, campos):
    """Unit view directions (means - campos) / |means - campos| in float64 (differentiable w.r.t. means)."""
    d = torch.as_tensor(means).double() - torch.as_tensor(campos).double().reshape(1, 3)
    return d / d.norm(dim=1, keepdim=True)


def sh_basis64(dirs, D):
    """[N, (D+1)^2] real SH basis values at unit directions `dirs` [N, 3], float64, in the coefficient order and sign
    convention of computeColorFromSH."""
    x, y, z = dirs[:, 0], dirs[:, 1], dirs[:, 2]
    b = [torch.full_like(x, SH_C0)]
    if D > 0:
        b += [-SH_C1 * y, SH_C1 * z, -SH_C1 * x]
    if D > 1:
        xx, yy, zz = x * x, y * y, z * z
        b += [SH_C2[0] * x * y, SH_C2[1] * y * z, SH_C2[2] * (2 * zz - xx - yy), SH_C2[3] * x * z, SH_C2[4] * (xx - yy)]
    if D > 2:
        b += [SH_C3[0] * y * (3 * xx - yy), SH_C3[1] * x * y * z, SH_C3[2] * y * (4 * zz - xx - yy),
              SH_C3[3] * z * (2 * zz - 3 * xx - 3 * yy), SH_C3[4] * x * (4 * zz - xx - yy), SH_C3[5] * z * (xx - yy),
              SH_C3[6] * x * (xx - 3 * yy)]
    return torch.stack(b, 1)


def sh_color64(shs, dirs, D):
    """computeColorFromSH in float64: (colour before the clamp = sum_k b_k(dir) sh_k + 0.5 [N, 3], clamp bits [N, 3]).
    Only the first (D+1)^2 coefficients of each row are read; the clamped colour is raw.clamp_min(0)."""
    n = (D + 1) ** 2
    raw = (sh_basis64(dirs, D)[:, :, None] * torch.as_tensor(shs)[:, :n].double()).sum(1) + 0.5
    return raw, raw < 0


def rel_err_stats(a, b):
    """Gradient tolerance used throughout: error relative to the tensor's scale, plus the fraction of
    significant elements whose own relative error exceeds 1e-3."""
    a, b = a.double().flatten(), b.double().flatten()
    if b.numel() == 0:                  # e.g. the SH rest gradient of a degree-0 model: [P, 0, 3]
        return 0.0, 0.0
    scale = b.abs().max().clamp_min(1e-30)
    diff = (a - b).abs()
    max_rel_to_scale = (diff.max() / scale).item()
    sig = b.abs() > 1e-4 * scale
    if sig.any():
        el = diff[sig] / b.abs()[sig]
        frac_bad = (el > 1e-3).double().mean().item()
    else:
        frac_bad = 0.0
    return max_rel_to_scale, frac_bad


# ---- recorded reference outputs ------------------------------------------------------------------------------------
def digest(t):
    """Digest of an integer array (float arrays are passed as their int32 bit views), independent of the dtype."""
    a = (t.detach().to(torch.int64).contiguous().cpu().numpy() if torch.is_tensor(t)
         else np.ascontiguousarray(t, dtype=np.int64))
    return hashlib.sha256(repr(a.shape).encode() + a.tobytes()).hexdigest()[:24]


def inputs_digest(*tensors):
    return digest(torch.cat([t.detach().float().reshape(-1).cpu().view(torch.int32) for t in tensors]))


def spread(n, k):
    """Up to k distinct indices spread evenly over range(n) (golden-ratio sequence), identical on every machine."""
    return np.unique((np.arange(min(n, k), dtype=np.float64) * 0.6180339887498949 % 1.0 * n).astype(np.int64))


def grad_sample_index(g, radii):
    """Flat indices of a fixed sample of gradient elements, taken from the rows of visible Gaussians."""
    rows = torch.nonzero(radii > 0).squeeze(1).cpu().numpy()
    per = g[0].numel() if g.shape[0] else 1
    s = spread(rows.size * per, GRAD_SAMPLE)
    return torch.from_numpy(rows[s // per] * per + s % per)


def _flat_sample(t, idx):
    return t.detach().reshape(-1)[idx.to(t.device)].float().cpu()


def record_forward(f):
    """Reference forward fields -> record: a digest per integer field, a sample + channel means of the colour."""
    rec = {}
    for k, v in f.items():
        if k == "num_rendered":
            rec[k] = np.int64(v)
        elif k in FLOAT_FIELDS:
            rec[k] = _flat_sample(v, torch.from_numpy(spread(v.numel(), COLOR_SAMPLE))).numpy()
            rec[k + ".mean"] = v.detach().reshape(v.shape[0], -1).double().mean(1).cpu().numpy()
        else:
            rec[k] = np.str_(digest(v))
    return rec


def record_grad(g, radii, g2=None):
    """Reference gradient -> record: full-tensor scale, a fixed sample, and (given a second reference backward
    over the same forward) the reference's own fraction of elements off by > 1e-3 relative."""
    scale = g.detach().abs().max().item() if g.numel() else 0.0
    frac0 = rel_err_stats(g2, g)[1] if g2 is not None else float("nan")
    return {"stats": np.array([scale, frac0]), "sample": _flat_sample(g, grad_sample_index(g, radii)).numpy()}


def golden_case(name):
    global _golden
    if _golden is None:
        with np.load(REF_GOLDEN, allow_pickle=False) as z:
            _golden = {k: z[k] for k in z.files}
    pre = name + "/"
    case = {k[len(pre):]: v for k, v in _golden.items() if k.startswith(pre)}
    assert case, f"no recorded reference outputs for {name} in {REF_GOLDEN}"
    return case


def check_inputs(case, *tensors):
    assert str(case["inputs"]) == inputs_digest(*tensors), \
        "the inputs differ from those the reference outputs were recorded for (tests/golden/make_ref_golden.py)"


def check_forward(case, mine, color_tol=1e-4):
    """Our forward fields (reference layout) against the recorded reference fields of `case`."""
    for k, v in mine.items():
        if k == "num_rendered":
            assert int(v) == int(case[k]), (k, int(v), int(case[k]))
        elif k in FLOAT_FIELDS:
            ref = torch.from_numpy(case[k])
            err = (_flat_sample(v, torch.from_numpy(spread(v.numel(), COLOR_SAMPLE))) - ref).abs().max().item()
            assert err <= color_tol, f"forward {k} max abs err {err} (sampled)"
            means = v.detach().reshape(v.shape[0], -1).double().mean(1).cpu().numpy()
            assert np.abs(means - case[k + ".mean"]).max() <= color_tol, f"forward {k} channel means"
        else:
            assert digest(v) == str(case[k]), f"{k} differs from the reference's (bit-exact)"


def check_grad(case, key, g, radii, max_rel=1e-3, frac_bar=None, tag=""):
    """Max error relative to the reference's full-tensor scale and fraction of significant elements off by > 1e-3,
    both over the recorded sample.  frac_bar None: max(2e-3, 3 x the reference's own atomic-order noise)."""
    scale, frac0 = (float(x) for x in case[key + ".stats"])    # full-tensor scale, reference self-noise
    scale = max(scale, 1e-30)
    ref = torch.from_numpy(case[key + ".sample"]).double()
    mine = _flat_sample(g, grad_sample_index(g, radii)).double()
    diff = (mine - ref).abs()
    m = diff.max().item() / scale if diff.numel() else 0.0
    sig = ref.abs() > 1e-4 * scale
    frac = (diff[sig] / ref.abs()[sig] > 1e-3).double().mean().item() if sig.any() else 0.0
    if frac_bar is None:
        frac_bar = max(2e-3, 3 * frac0)
    mine_scale = g.detach().abs().max().item() if g.numel() else 0.0
    print(f"[{tag}] {key}: max err/scale {m:.3e}, frac rel>1e-3 {frac:.3e} (sampled), scale {mine_scale:.4e} vs {scale:.4e}")
    assert m <= max_rel, f"{tag} {key}: max err relative to scale {m}"
    assert frac <= frac_bar, f"{tag} {key}: {frac} of significant sampled elements differ by >1e-3 rel"
    assert abs(mine_scale - scale) <= max_rel * scale, f"{tag} {key}: scale {mine_scale} vs the reference's {scale}"


def ours_forward_fields(st, rows=None, index_map=None):
    """Our forward state (forward_with_state) in the reference's layout.  rows: our rows present in the reference's
    call (boolean-gathered inputs), index_map: our Gaussian index -> reference row."""
    rows = slice(None) if rows is None else rows
    radii = st["radii"][rows]
    vis = radii > 0
    rect = st["rect"][rows]
    touched = ((rect[:, 1] & 0xffff) - (rect[:, 0] & 0xffff)) * (((rect[:, 1] >> 16) & 0xffff) - ((rect[:, 0] >> 16) & 0xffff))
    rec = st["rec"][rows]
    cl = st["clamped"][rows]
    pl = st["point_list"] if index_map is None else index_map[st["point_list"].long()].int()
    return dict(num_rendered=st["num_rendered"], radii=radii,
                depth=st["depth"][rows][vis].view(torch.int32), touched=touched[vis],
                means2D=rec[vis][:, 0:2].contiguous().view(torch.int32),
                conic=rec[vis][:, 2:6].contiguous().view(torch.int32),
                rgb=rec[vis][:, 6:9].contiguous().view(torch.int32),
                clamped=torch.stack([cl & 1, (cl >> 1) & 1, (cl >> 2) & 1], 1)[vis],
                ranges=st["ranges"], point_list=pl, key_depth=st["keys"] >> 32, key_index=st["keys"] & 0xffffffff,
                n_contrib=st["n_contrib"], final_T=st["final_T"].view(torch.int32), color=st["color"])
