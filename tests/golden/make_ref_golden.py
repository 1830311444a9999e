"""Records the UNMODIFIED reference rasterizer's outputs for the GPU parity tests into tests/golden/ref_outputs.npz.

    python tests/golden/make_ref_golden.py [OUT_DIR]       (on a B200, with oracle/_ref built by oracle/build_ref.py)

Every case runs the reference on exactly the inputs its test builds (the same helpers and seeds) and stores, per case,
a digest of those inputs, a digest of every array the test compares bit-exactly, and a fixed sample of every float
array (colour images and the eight gradients) with its full-array scale and the reference's own atomic-order noise.
The tests then compare our outputs with these records, so they need neither the reference nor its build."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from frosting_b200 import camera_batch as cbm   # noqa: E402
from frosting_b200 import scenes                 # noqa: E402
import frosting_b200 as fb                       # noqa: E402
from oracle import cpu, refdgr                   # noqa: E402
from tests import util                           # noqa: E402
from tests import test_bench_configs_gpu as tbc  # noqa: E402
from tests import test_c_abi_gpu as tca          # noqa: E402
from tests import test_extra_channels_gpu as tex  # noqa: E402
from tests import test_oracle_vs_ref_gpu as tov  # noqa: E402
from tests import test_parity_gpu as tpg         # noqa: E402

KEYS = ("means3D", "opacities", "shs", "scales", "rotations")
GRADS = ("means3D", "means2D", "sh", "opacities", "scales", "rotations")


def ref_fields(ref, P, H, W):
    """The reference's forward buffers in the field names of tests/util.py::ours_forward_fields."""
    R = ref["num_rendered"]
    gv, bv, iv = refdgr.geom_views(ref["geom"], P), refdgr.binning_views(ref["binning"], R), refdgr.img_views(ref["img"], H, W)
    vis = ref["radii"] > 0
    return dict(num_rendered=R, radii=ref["radii"], depth=gv["depths"][vis].view(torch.int32),
                touched=gv["tiles_touched"][vis], means2D=gv["means2D"][vis].view(torch.int32),
                conic=gv["conic_opacity"][vis].view(torch.int32), rgb=gv["rgb"][vis].view(torch.int32),
                clamped=gv["clamped"][vis], ranges=iv["ranges"], point_list=bv["point_list"],
                key_depth=bv["point_list_keys"] & 0xffffffff, key_index=bv["point_list"],
                n_contrib=iv["n_contrib"], final_T=iv["accum_alpha"].view(torch.int32), color=ref["color"],
                cov3D=gv["cov3D"][vis].view(torch.int32), keys=bv["point_list_keys"])


def pick(d, *keys):
    return {k: d[k] for k in keys}


class Recorder:
    def __init__(self):
        self.out = {}

    def put(self, case, rec):
        for k, v in rec.items():
            self.out[f"{case}/{k}"] = v
        print(case, flush=True)

    def grads(self, case, rb, rb2, radii, keys=GRADS):
        for k in keys:
            for f, v in util.record_grad(rb[k], radii, None if rb2 is None else rb2[k]).items():
                self.out[f"{case}/{k}.{f}"] = v


def parity(rec, dev):
    ids = lambda c: f"P{c[0]}_{c[1]}x{c[2]}_D{c[4]}"
    for cfg in tpg.CONFIGS:
        P, W, H, seed, D, bg = cfg
        cam, g, rs = util.scene(P, W, H, seed, D, dev, bg)
        ref = refdgr.forward(rs, g["means3D"], g["opacities"], shs=g["shs"], scales=g["scales"], rotations=g["rotations"])
        f = util.record_forward(pick(ref_fields(ref, P, H, W), *tpg.FWD_FIELDS))
        f["inputs"] = np.str_(util.inputs_digest(*(g[k] for k in KEYS)))
        rec.put("parity_fwd_" + ids(cfg), f)
    for cfg in tpg.CONFIGS[:3]:
        P, W, H, seed, D, bg = cfg
        cam, g, rs = util.scene(P, W, H, seed, D, dev, bg)
        cot = tpg.cotangent(H, W, dev)
        kw = dict(shs=g["shs"], scales=g["scales"], rotations=g["rotations"])
        ref = refdgr.forward(rs, g["means3D"], g["opacities"], **kw)
        rb = refdgr.backward(rs, ref, g["means3D"], cot, **kw)
        rb2 = refdgr.backward(rs, ref, g["means3D"], cot, **kw)
        case = "parity_bwd_" + ids(cfg)
        rec.put(case, {"inputs": np.str_(util.inputs_digest(*(g[k] for k in KEYS), cot)),
                       "radii": np.str_(util.digest(ref["radii"]))})
        rec.grads(case, rb, rb2, ref["radii"])

    inp = tpg.precomp_inputs(dev)
    rs, g, colors, cov, cot = inp
    ref = refdgr.forward(rs, g["means3D"], g["opacities"], colors_precomp=colors, cov3D_precomp=cov)
    rb = refdgr.backward(rs, ref, g["means3D"], cot, colors_precomp=colors, cov3D_precomp=cov)
    f = util.record_forward(pick(ref_fields(ref, g["means3D"].shape[0], rs.image_height, rs.image_width),
                                 "radii", "point_list", "color"))
    f["inputs"] = np.str_(util.inputs_digest(g["means3D"], g["opacities"], colors, cov, cot))
    rec.put("parity_precomp", f)
    rec.grads("parity_precomp", rb, None, ref["radii"], ("means3D", "colors", "cov3D", "opacities", "means2D"))

    rs, one = tpg.edge_one(dev)
    ref = refdgr.forward(rs, one["means3D"], one["opacities"], shs=one["shs"], scales=one["scales"], rotations=one["rotations"])
    rec.put("parity_edge_one", util.record_forward({"color": ref["color"]}))

    for P, rs, g in tpg.long_tile_scenes(dev):
        ref = refdgr.forward(rs, g["means3D"], g["opacities"], shs=g["shs"], scales=g["scales"], rotations=g["rotations"])
        f = util.record_forward(pick(ref_fields(ref, P, rs.image_height, rs.image_width), *tpg.LIST_FIELDS))
        f["inputs"] = np.str_(util.inputs_digest(*(g[k] for k in KEYS)))
        rec.put(f"parity_long_{P}", f)

    P, rs, g = tpg.depth_tie_scene(dev)
    ref = refdgr.forward(rs, g["means3D"], g["opacities"], shs=g["shs"], scales=g["scales"], rotations=g["rotations"])
    f = util.record_forward(pick(ref_fields(ref, P, rs.image_height, rs.image_width), *tpg.LIST_FIELDS))
    f["inputs"] = np.str_(util.inputs_digest(*(g[k] for k in KEYS)))
    rec.put("parity_ties", f)


def bench_configs(rec, dev):
    for cam_index in tbc.C3_CAMS:
        wl = cbm.build_workload("c3", dev)
        cbm.visible_faces(wl)
        P, W, H, D = wl["P"], wl["W"], wl["H"], wl["D"]
        rs = scenes.settings_for(wl["cams"][cam_index], D, device=dev)
        a = wl["attrs"]
        keep = fb.gaussian_render_mask(wl["face_visible"][cam_index], wl["mesh"]["cells"], P).bool()
        g = {k: a[k][keep].contiguous() for k in KEYS}
        ref = refdgr.forward(rs, g["means3D"], g["opacities"], shs=g["shs"], scales=g["scales"], rotations=g["rotations"])
        cot = wl["cot_host"][cam_index].to(dev)
        f = util.record_forward(pick(ref_fields(ref, g["means3D"].shape[0], H, W), *tbc.FWD_FIELDS))
        f["inputs"] = np.str_(util.inputs_digest(*(g[k] for k in KEYS), cot))
        rb = refdgr.backward(rs, ref, g["means3D"], cot, shs=g["shs"], scales=g["scales"], rotations=g["rotations"])
        rb2 = refdgr.backward(rs, ref, g["means3D"], cot, shs=g["shs"], scales=g["scales"], rotations=g["rotations"])
        case = f"bench_c3_cam{cam_index}"
        rec.put(case, f)
        rec.grads(case, rb, rb2, ref["radii"])
        del wl, g, ref, rb, rb2
        torch.cuda.empty_cache()
    for name in ("c5", "c2"):
        wl = cbm.build_workload(name, dev, cams_per_gpu=1)
        P, W, H, D = wl["P"], wl["W"], wl["H"], wl["D"]
        rs = scenes.settings_for(wl["cams"][0], D, device=dev)
        a = wl["attrs"]
        kw = dict(shs=a["shs"], scales=a["scales"], rotations=a["rotations"])
        ref = refdgr.forward(rs, a["means3D"], a["opacities"], **kw)
        cot = wl["cot_host"][0].to(dev)
        f = util.record_forward(pick(ref_fields(ref, P, H, W), *tbc.FWD_FIELDS))
        f["inputs"] = np.str_(util.inputs_digest(*(a[k] for k in KEYS), cot))
        rb = refdgr.backward(rs, ref, a["means3D"], cot, **kw)
        rb2 = refdgr.backward(rs, ref, a["means3D"], cot, **kw)
        rec.put(f"bench_{name}", f)
        rec.grads(f"bench_{name}", rb, rb2, ref["radii"])
        del wl, a, ref, rb, rb2
        torch.cuda.empty_cache()
    for c in range(tbc.SWEEP_CHUNKS):
        rs, means, op, col, scales, q = tbc.sweep_chunk(c, dev)
        W, H, n = rs.image_width, rs.image_height, means.shape[0]
        ref = refdgr.forward(rs, means, op, colors_precomp=col, scales=scales, rotations=q)
        gv = refdgr.geom_views(ref["geom"], n)
        vis = ref["radii"] > 0
        m2, rad = gv["means2D"][vis], ref["radii"][vis].float()
        gx, gy = (W + 15) // 16, (H + 15) // 16
        rec.put(f"sweep_{c}", util.record_forward(dict(
            num_rendered=ref["num_rendered"], radii=ref["radii"], depth=gv["depths"][vis].view(torch.int32),
            touched=gv["tiles_touched"][vis],
            rect_minx=((m2[:, 0] - rad) / 16).int().clamp(0, gx), rect_miny=((m2[:, 1] - rad) / 16).int().clamp(0, gy))))
        del ref, gv, means, op, col, scales, q
        torch.cuda.empty_cache()


def c_abi(rec, dev):
    P, rs, g = tca.many_tiles_scene(dev)
    ref = refdgr.forward(rs, g["means3D"], g["opacities"], shs=g["shs"], scales=g["scales"], rotations=g["rotations"])
    f = util.record_forward(pick(ref_fields(ref, P, rs.image_height, rs.image_width), "num_rendered", "radii",
                                 "point_list", "n_contrib", "color"))
    f["inputs"] = np.str_(util.inputs_digest(*(g[k] for k in KEYS)))
    rec.put("cabi_many_tiles", f)


def extra_channels(rec, dev):
    for E, bg_e in tex.PARAMS:
        rs, g, feats, cot_c, cot_e = tex.extra_inputs(E, dev)
        P, H, W = feats.shape[0], rs.image_height, rs.image_width
        kw = dict(scales=g["scales"], rotations=g["rotations"])
        ref1 = refdgr.forward(rs, g["means3D"], g["opacities"], shs=g["shs"], **kw)
        f3 = torch.zeros(P, 3, device=dev); f3[:, :E] = feats
        rs2 = rs._replace(bg=torch.full((3,), bg_e, device=dev))
        ref2 = refdgr.forward(rs2, g["means3D"], g["opacities"], colors_precomp=f3, **kw)
        cot2 = torch.zeros(3, H, W, device=dev); cot2[:E] = cot_e
        rb1 = refdgr.backward(rs, ref1, g["means3D"], cot_c, shs=g["shs"], **kw)
        rb2 = refdgr.backward(rs2, ref2, g["means3D"], cot2, colors_precomp=f3, **kw)
        case = f"extra_E{E}_bg{bg_e:g}"
        f = util.record_forward({"radii": ref1["radii"], "color": ref2["color"][:E]})
        f["inputs"] = np.str_(util.inputs_digest(*(g[k] for k in KEYS), feats, cot_c, cot_e))
        rec.put(case, f)
        want = {k: rb1[k] + rb2[k] for k in ("means3D", "means2D", "opacities", "scales", "rotations")}
        want["sh"], want["features"] = rb1["sh"], rb2["colors"][:, :E]
        rec.grads(case, want, None, ref1["radii"], tuple(want))


def oracle_vs_ref(rec, dev):
    for cfg, name in zip(tov.CONFIGS, tov.IDS):
        P, W, H, seed, D, bg = cfg
        cam, g, rs = util.scene(P, W, H, seed, D, dev, bg)
        ref = refdgr.forward(rs, g["means3D"], g["opacities"], shs=g["shs"], scales=g["scales"], rotations=g["rotations"])
        cot = tov.cotangent(H, W, dev)
        rb = refdgr.backward(rs, ref, g["means3D"], cot, shs=g["shs"], scales=g["scales"], rotations=g["rotations"])
        f = util.record_forward(pick(ref_fields(ref, P, H, W), *tov.FWD_FIELDS))
        f["color"] = ref["color"].reshape(-1)[torch.from_numpy(util.spread(ref["color"].numel(), tov.COLOR_SAMPLE)).to(dev)].cpu().numpy()
        f["inputs"] = np.str_(util.inputs_digest(*(g[k] for k in KEYS), cot))
        case = f"oracle_{name}"
        rec.put(case, f)
        rec.grads(case, rb, None, ref["radii"], tov.GRADS)


def main(out_dir):
    dev = torch.device("cuda:0")
    refdgr.module()
    cpu.build()
    rec = Recorder()
    for part in (parity, c_abi, extra_channels, oracle_vs_ref, bench_configs):
        part(rec, dev)
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, "ref_outputs.npz")
    np.savez_compressed(path, **rec.out)
    print(path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden"))
