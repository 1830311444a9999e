#!/usr/bin/env python
"""bench.py -- forward+backward frames/sec of the render path on BASELINE.json's headline config.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c3|c2|c5] [--quick]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (config C3 of BASELINE.json): 2 M frosting-layer Gaussians bound to the prism cells of a ~1 M-face
UV-sphere shell (frosting_b200/scenes.py), occlusion culling ON, 1920x1080, SH degree 3, ring of cameras of radius 6
(SURVEY.md 8d), synthetic data, random-init parameters.  A "step" is one frame: occlusion mask -> rasterizer forward
-> scalar loss (color * G).sum() -> backward to means3D / SH / opacity / scale / rotation (+ the means2D sink), for one
camera; every rank owns 8 cameras of the ring (config C4's sharding: camera batch split across GPUs, Gaussians
replicated, the only collective is the NCCL all-reduce of the scalar loss) and cycles through them, so per-GPU work
is fixed as N grows ("weak" scaling).  `value` = frames all ranks finished / max-over-ranks time.  The frame loop is
frosting_b200.camera_batch.CameraBatch (package API); this file only times it.

--impl reference runs the UNMODIFIED reference rasterizer compiled from /root/reference into oracle/_ref
(oracle/build_ref.py) through its own entry points, with Frosting's boolean-gather masking
(frosting_scene/frosting_model.py:1564-1586) in torch, on the same scene, cameras and loss.  The reference has no CPU
implementation of this path (SURVEY.md 8c); its own CUDA code is the stock code path.  That process never maps
libfrosting_b200.so: the visible-face sets (the prepass the reference gets from nvdiffrast, absent here) are computed by
a CHILD process before anything is timed and handed over in a file.

Sub-blocks of the JSON line (N = 1 only, each with the shipped kernels): `dropin` (Frosting's boolean gathers in torch
+ our rasterizer, no API extension), `c2`, `c5` (BASELINE configs 2 and 5, with their own roofline), `c3_ring10`
(round 1's camera distance), `prepass_ms` (the occlusion prepass at 1 M faces / 1080p), `frosting_step`,
`frosting_train_step`, `dp_train_step` (+ `dp_check`).

Timing: CUDA events around exactly K steps after W warm-up steps, barrier + synchronize on both sides, max over
ranks.

--dump-outputs DIR writes, right after the timed steps, what the last timed step handed its caller as DIR/<name>.npy
(float32): the image, and radii and every gradient at a fixed seeded sample of Gaussian rows (DUMP_ROWS, the same on
every run).  Scene, cameras and cotangents are seeded, so two builds run with the same arguments can be compared
output for output.  Inputs are larger than L2 (472 MB of attributes are read per frame, 126 MB L2), no flush needed.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from frosting_b200 import camera_batch as cb   # noqa: E402  (imports no native code)

METRIC = "fwd+bwd frames/sec @2M Gaussians 1080p"
UNIT = "frames/s"
DP_LEG_TIMEOUT_S = 240
DUMP_ROWS = 65536
DUMP_MAX_BYTES = 64 << 20
RING_RADIUS = float(os.environ.get("FB200_RING_RADIUS", str(cb.RING_RADIUS)))


def log(*a):
    print(*a, file=sys.stderr, flush=True)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        rows = [l.split(", ") for (t, l) in self.lines if t0 - 0.05 <= t <= t1 + 0.25]
        if not rows:
            rows = [l.split(", ") for (_, l) in self.lines[-3:]]
        sm, reasons, mx = [], set(), None
        for r in rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        if not sm:
            return None
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ---- the reference arm -----------------------------------------------------------------------------------------------
def visible_faces_in_child(name, rank, world, ring_radius, local_rank):
    """The reference arm must not map libfrosting_b200.so: a child process runs the CUDA prepass (the stand-in for
    nvdiffrast, SURVEY.md 8d) for this rank's cameras and leaves the visible-face sets in a file."""
    fd, path = tempfile.mkstemp(suffix=".pt", prefix="fb200_vis_")
    os.close(fd)
    code = ("import sys, torch; sys.path.insert(0, %r); from frosting_b200 import camera_batch as cb; "
            "dev = torch.device('cuda', %d); torch.cuda.set_device(dev); "
            "wl = cb.build_workload(%r, dev, %d, %d, ring_radius=%r); "
            "torch.save([v.cpu() for v in cb.visible_faces(wl)], %r)"
            % (ROOT, local_rank, name, rank, world, ring_radius, path))
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    subprocess.run([sys.executable, "-c", code], check=True, stdout=subprocess.DEVNULL, env=env)
    vis = torch.load(path)
    os.unlink(path)
    return vis


class ReferenceBatch:
    """The reference arm's frames: the reference's own chain, nothing of this repo's native code.
    mode "raster": attributes -> boolean gathers (frosting_model.py:1564-1586) -> reference rasterizer -> loss -> backward
    mode "frosting": torch property ops (frosting_model.py:713-799, restated in scenes.frosting_attributes) first;
    loss "l1_dssim": the reference's torch loss (frosting_utils/loss_utils.py:17-63, restated in loss.torch_reference)."""

    def __init__(self, wl, device, mode="raster", loss="cot"):
        from oracle import refdgr
        from frosting_b200 import scenes
        refdgr.module()
        self.refdgr, self.scenes, self.wl, self.device = refdgr, scenes, wl, device
        self.mode, self.loss_mode = mode, loss
        if mode == "raster":
            self.leaves = {k: v.clone().requires_grad_(True) for k, v in wl["attrs"].items()}
        else:
            self.params = {k: v.clone().requires_grad_(True) for k, v in wl["params"].items()}
        self.cells = wl["mesh"]["cells"] if wl["mesh"] is not None else None
        self.gt = None

    def settings(self, cam):
        return self.scenes.settings_for(cam, self.wl["D"], device=self.device)

    def frame(self, i, rs, cot):
        if self.mode == "raster":
            a = self.leaves
            for v in a.values():
                v.grad = None
        else:
            for v in self.params.values():
                v.grad = None
            a = self.scenes.frosting_attributes(self.params, self.wl["mesh"])
        m3, op, sh, sc, ro = (a[k] for k in ("means3D", "opacities", "shs", "scales", "rotations"))
        if self.wl["face_visible"] is not None:
            render_mask = self.wl["face_visible"][i].bool()[self.cells]
            m3, op, sh, sc, ro = m3[render_mask], op[render_mask], sh[render_mask], sc[render_mask], ro[render_mask]
        means2D = torch.zeros_like(m3, requires_grad=True)
        color, radii = self.refdgr.RefRasterize.apply(m3, means2D, sh, op, sc, ro, rs)
        self.last = dict(color=color, radii=radii, means2D=means2D)
        if self.loss_mode == "l1_dssim":
            from frosting_b200.loss import torch_reference     # restates frosting_utils/loss_utils.py:17-63 verbatim
            loss = torch_reference(color, self.gt[i], 0.2)
        else:
            loss = (color * cot).sum()
        loss.backward()
        return loss.detach()


class OursDPTrain(cb.CameraBatch):
    """One data-parallel TRAINING iteration (row f3): every rank renders its camera from the shared parameters
    (fused attributes -> mask -> rasterizer -> fused L1 + D-SSIM -> backward writing into the gradient slab), then ONE
    kernel per rank reduces its shard of all ranks' gradients over NVLink peer memory, applies Adam (the reference's
    groups / learning rates, frosting_optimizer.py:74-101) and stores the new parameters into every rank's slab."""
    handles_collective = True

    def __init__(self, wl, device):
        import frosting_b200 as fb
        opt = fb.FrostingAdam.for_frosting(wl["params"])
        super().__init__(wl, device, mode="frosting", mask="lookup", loss="l1_dssim", optimizer=opt)

    def frame(self, i, rs, cot):
        loss = super().frame(i, rs, cot).reshape(1).clone()
        self.opt.update_learning_rate()
        self.opt.step(loss=loss)            # the loss all-reduce doubles as the pre-step rendezvous
        return loss


class ReferenceDPTrain(ReferenceBatch):
    """What a torch user gets from the reference today: its render chain, NCCL all-reduce of every .grad (averaged),
    torch.optim.Adam(lr=0.0, eps=1e-15) over the same groups (frosting_optimizer.py:74-101,116-118)."""
    handles_collective = True

    def __init__(self, wl, device):
        super().__init__(wl, device, mode="frosting", loss="l1_dssim")
        from frosting_b200.optim import OptimizationParams
        o = OptimizationParams()
        lr = {"bary_logits": o.position_bary_coords_lr_init, "sh_dc": o.feature_lr, "sh_rest": o.feature_lr / 20.0,
              "opacity_logits": o.opacity_lr, "log_scales": o.scaling_lr, "quats": o.rotation_lr}
        self.opt = torch.optim.Adam([{"params": [self.params[k]], "lr": lr[k], "name": k} for k in lr], lr=0.0, eps=1e-15)
        self.world = dist.get_world_size() if dist.is_initialized() else 1

    def frame(self, i, rs, cot):
        loss = super().frame(i, rs, cot).reshape(1).clone()
        if self.world > 1:
            dist.all_reduce(loss)
            for v in self.params.values():
                dist.all_reduce(v.grad)
                v.grad.div_(self.world)
        self.opt.step()
        return loss


# ---- timing ----------------------------------------------------------------------------------------------------------
def timed_loop(step, wl, device, steps, warmup, world, e2e, count_launches=False):
    """Returns seconds for exactly `steps` steps (max over ranks)."""
    cams = wl["cams"]
    n = len(cams)
    copy_stream = torch.cuda.Stream(device)
    cur = torch.cuda.current_stream(device)
    if not e2e:
        rs_dev = [step.settings(c) for c in cams]
        cot_dev = [c.to(device) for c in wl["cot_host"]]
    own_collective = getattr(step, "handles_collective", False)

    def fetch(i):
        """H2D of step inputs from pinned host memory on the copy stream (double-buffered)."""
        cam = cams[i % n]
        with torch.cuda.stream(copy_stream):
            cot = wl["cot_host"][i % n].to(device, non_blocking=True)
            cd = wl["cam_host"][i % n].to(device, non_blocking=True)   # camera record H2D
            rs = step.settings(cam)._replace(viewmatrix=cd[0:16].view(4, 4), projmatrix=cd[16:32].view(4, 4),
                                             campos=cd[32:35], bg=cd[35:38])
            ev = torch.cuda.Event(); ev.record(copy_stream)
        return rs, cot, ev

    loss_pin = [torch.zeros(1, pin_memory=True) for _ in range(2)] if e2e else None

    def run(k_steps, offset):
        losses = []
        # the path's only collective: every frame's scalar loss is summed over the ranks by its own asynchronous NCCL
        # all-reduce; the compute stream never waits for it, the results are collected before the timed region ends
        reducer = cb.LossReducer() if (world > 1 and not own_collective) else None
        pending = None                      # (pinned slot, event) of the previous step's loss read-back
        nxt = fetch(offset) if e2e else None
        for k in range(k_steps):
            i = (offset + k) % n
            if e2e:
                rs, cot, ev = nxt
                cur.wait_event(ev)
                cot.record_stream(cur)
                rs.viewmatrix.record_stream(cur)
                if k + 1 < k_steps:
                    nxt = fetch(offset + k + 1)
            else:
                rs, cot = rs_dev[i], cot_dev[i]
            loss = step.frame(i, rs, cot)
            if reducer is not None:
                reducer.add(loss)
            if e2e:
                # D2H read of the step's result, every step: async copy into pinned memory, consumed one step later so
                # the read-back of step k overlaps step k+1 instead of draining the GPU (losses lag by one step, as an
                # asynchronous logger would see them); the last one is collected before the timed region ends
                if pending is not None:
                    pending[1].synchronize()
                    losses.append(float(pending[0][0]))
                slot = loss_pin[k & 1]
                slot.copy_(loss.reshape(1), non_blocking=True)
                ev = torch.cuda.Event(); ev.record(cur)
                pending = (slot, ev)
        if e2e and pending is not None:
            pending[1].synchronize()
            losses.append(float(pending[0][0]))
        if reducer is not None:
            reducer.collect()
        return losses

    if not getattr(step, "primed", False):
        # untimed priming pass over every camera of this rank (each has its own visible set, hence its own
        # tensor sizes): the caching allocator and the capacity hints settle before the W warm-up steps
        run(2 * n, 0)
        step.primed = True
    run(warmup, 0)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(device)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = 0
    if count_launches:
        from frosting_b200 import _lib
        l0 = _lib.kernel_launches()
    t0 = time.time()
    a.record()
    run(steps, warmup)
    b.record()
    torch.cuda.synchronize(device)
    if count_launches:
        timed_loop.launches = _lib.kernel_launches() - l0
    if world > 1:
        dist.barrier()
    t1 = time.time()
    secs = a.elapsed_time(b) / 1e3
    if world > 1:
        t = torch.tensor([secs], device=device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        secs = float(t.item())
    return secs, t0, t1


def stage_profile(step, wl, device, steps):
    """Average device time of each kernel stage (CUDA events on the launching stream, inside the library)."""
    from frosting_b200 import _lib
    import frosting_b200 as fb
    cams = wl["cams"]
    rs_dev = [step.settings(c) for c in cams]
    cot_dev = [c.to(device) for c in wl["cot_host"]]
    _lib.profile_enable(True)
    acc = {k: 0.0 for k in _lib.STAGES}
    Rs, Vs = [], []
    try:
        for k in range(steps):
            i = k % len(cams)
            step.frame(i, rs_dev[i], cot_dev[i])
            torch.cuda.synchronize(device)
            for kk, v in _lib.profile_read().items():
                acc[kk] += v
            Rs.append(int(fb.rasterizer.last_num_rendered(device)))
            Vs.append(int((step.last["radii"] > 0).sum()))
    finally:
        _lib.profile_enable(False)
    return {k: v / steps for k, v in acc.items()}, sum(Rs) / len(Rs), sum(Vs) / len(Vs)


def rooflines(prof, R_avg, W, H, workload):
    """SURVEY.md 8d: algorithmic bytes of the blend kernels / their live CUDA-event time vs the measured HBM peak."""
    peaks = {"hbm_gbs": 6650.0, "src": "fallback (B200_PROFILING.md)"}
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk):
        peaks = {"hbm_gbs": float(json.load(open(pk))["hbm_gbs"]), "src": "measured"}
    T = ((W + 15) // 16) * ((H + 15) // 16)
    Npx = H * W
    b_fwd = 40 * R_avg + 20 * Npx + 8 * T + 12
    b_bwd = 76 * R_avg + 20 * Npx + 8 * T + 12
    traffic = {}
    tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tp):
        traffic = json.load(open(tp)).get(workload, {})

    def roof(bytes_, ms, key):
        ach = bytes_ / (ms * 1e-3) / 1e9
        return {"bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": ach / peaks["hbm_gbs"], "traffic": traffic.get(key), "kernel": key,
                "kernel_ms": ms, "algorithmic_bytes": bytes_, "peak_source": peaks["src"],
                "instances_R": R_avg}
    return (roof(b_bwd, prof["render_bwd"], traffic.get("bwd_kernel_name", "render_bwd_t16_kernel")),
            roof(b_fwd, prof["render_fwd"], traffic.get("fwd_kernel_name", "render_fwd_pair_kernel")))


def cpu_baseline(wl, step, sample_cam=0):
    """One full frame (fwd+bwd) of the same workload on the host through the C oracle (1 thread)."""
    from oracle import cpu
    import numpy as np
    cam = wl["cams"][sample_cam]
    rs = step.settings(cam)
    A = {k: v.detach().cpu().numpy() for k, v in wl["attrs"].items()}
    vis = None
    if wl["face_visible"] is not None:
        vis = wl["face_visible"][sample_cam].bool()[wl["mesh"]["cells"]].cpu().numpy().astype(np.uint8)
    cot = wl["cot_host"][sample_cam].numpy()
    t = time.perf_counter()
    f = cpu.forward(rs, A["means3D"], A["opacities"], shs=A["shs"], scales=A["scales"], rots=A["rotations"],
                    visibility=vis)
    cpu.backward(rs, f, A["means3D"], cot, shs=A["shs"], scales=A["scales"], rots=A["rotations"])
    dt = time.perf_counter() - t
    return dict(value=1.0 / dt, unit=UNIT, cores=1, kind="port",
                sample=f"1 full frame (fwd+bwd) of the same workload, camera {sample_cam}, oracle/raster_oracle.c, "
                       f"single thread, {dt:.1f} s"), f["binned"]["num_rendered"]


def dp_oracle_check(device, world, rank):
    """Driver-visible correctness of the data-parallel step (row f3): a small synthetic slab goes through the SAME kernel
    and transport for 3 steps on all ranks with per-rank gradients; every rank's parameters must be bit-identical and
    must match the numpy restatement of torch.optim.Adam over the rank-ordered gradient sum (oracle/adam.py::dp_step --
    the oracle used as the checker, never as the thing measured)."""
    import numpy as np
    from frosting_b200 import optim
    from oracle import adam as adam_oracle
    shapes = {"a": (1001, 6), "b": (1001, 1, 3), "c": (1001, 15, 3), "d": (1001, 1), "e": (333,), "f": (1001, 4)}
    lrs = {"a": 0.005, "b": 0.0025, "c": 0.000125, "d": 0.05, "e": 0.005, "f": 0.001}

    def grads(t, r, k, n):
        rng = np.random.default_rng(100000 * t + 100 * r + k)
        g = rng.standard_normal(n).astype(np.float32) * (10.0 ** rng.integers(-6, 1, n)).astype(np.float32)
        g[rng.random(n) < 0.3] = 0.0
        return g
    rng = np.random.default_rng(3)
    init = {n: rng.standard_normal(sh).astype(np.float32) for n, sh in shapes.items()}
    opt = optim.FrostingAdam({n: torch.from_numpy(x).to(device) for n, x in init.items()}, lrs)
    for t in range(1, 4):
        for k, n in enumerate(shapes):
            opt.grads[n].copy_(torch.from_numpy(grads(t, rank, k, init[n].size)).view(shapes[n]))
        opt.step()
    torch.cuda.synchronize(device)
    mine = torch.cat([opt.params[n].detach().reshape(-1) for n in shapes])
    if world > 1:
        every = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(every, mine)
    else:
        every = [mine]
    identical = all(bool(torch.equal(e.view(torch.int32), every[0].view(torch.int32))) for e in every)
    err = 0.0
    for k, n in enumerate(shapes):
        p, m, v = init[n].reshape(-1).copy(), np.zeros(init[n].size, np.float32), np.zeros(init[n].size, np.float32)
        for t in range(1, 4):
            p, m, v = adam_oracle.dp_step(p, [grads(t, r, k, init[n].size) for r in range(world)], m, v, lrs[n], t,
                                          1.0 / world)
        got = opt.params[n].detach().cpu().numpy().reshape(-1)
        err = max(err, float(np.max(np.abs(got - p) / (5e-7 + 3e-6 * np.abs(p)))))
    out = {"world": world, "transport": opt.slabs.transport, "replicas_bit_identical": identical,
           "max_err_vs_oracle_in_tolerances": err, "pass": bool(identical and err <= 1.0),
           "note": "3 steps of the reduce+Adam+publish kernel on a synthetic slab vs oracle/adam.py (rtol 3e-6, atol 5e-7)"}
    opt.close()
    return out


def dump_outputs(step, out_dir, P):
    """The last frame's image, and its radii and gradients at DUMP_ROWS fixed rows, as float32 .npy files."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    rows = torch.randperm(P, generator=torch.Generator().manual_seed(0))[:min(P, DUMP_ROWS)].sort().values
    arrays = {"color": step.last["color"]}
    tensors = dict(getattr(step, "leaves", None) or step.params)
    if step.last.get("means2D") is not None:
        tensors["means2D"] = step.last["means2D"]
    per_row = {"radii": step.last["radii"], **{"grad_" + k: v.grad for k, v in tensors.items() if v.grad is not None}}
    for k, v in per_row.items():
        # a gathered call (boolean-masked inputs) returns fewer rows than the scene has: sample only rows it has
        arrays[k] = v[rows[rows < v.shape[0]].to(v.device)]
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed {DUMP_MAX_BYTES}")
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)
    log(f"[bench] wrote {len(arrays)} arrays ({total / 2**20:.1f} MB) to {out_dir}")


def make_step(impl, wl, device, **kw):
    if impl == "ours":
        return cb.CameraBatch(wl, device, **kw)
    kw.pop("mask", None)
    return ReferenceBatch(wl, device, **kw)


def load_workload(name, device, rank, world, impl, local_rank, ring_radius):
    wl = cb.build_workload(name, device, rank, world, ring_radius=ring_radius)
    if wl["mesh"] is not None:
        if impl == "ours":
            cb.visible_faces(wl)
        else:
            wl["face_visible"] = [v.to(device) for v in visible_faces_in_child(name, rank, world, ring_radius, local_rank)]
    return wl


def side_config(name, impl, device, steps, warmup, local_rank, ring_radius=RING_RADIUS):
    """A secondary BASELINE config on one GPU: value (+ stage times and rooflines for our arm)."""
    wl = load_workload(name, device, 0, 1, impl, local_rank, ring_radius)
    step = make_step(impl, wl, device)
    secs, _, _ = timed_loop(step, wl, device, steps, warmup, 1, e2e=False)
    out = {"value": steps / secs, "unit": UNIT, "ms_per_step": 1e3 * secs / steps, "steps": steps,
           "workload": cb.WORKLOAD_TEXT[name] + (f", ring radius {ring_radius:g}" if wl["kind"] == "frosting" else "")}
    if impl == "ours":
        prof, R_avg, V_avg = stage_profile(step, wl, device, min(steps, 8))
        out["roofline"], out["roofline_fwd"] = rooflines(prof, R_avg, wl["W"], wl["H"], name)
        out["stage_ms"] = prof
        out["scene"] = {"P": wl["P"], "V": V_avg, "R": R_avg, "R_over_P": R_avg / wl["P"]}
    del step, wl
    torch.cuda.empty_cache()
    return out


def prepass_ms(wl, device, reps=10):
    """The occlusion prepass alone (row a19): ~1 M faces rasterised at 1080p + the Gaussian mask, per frame, as
    Frosting's inference path runs it (frosting_model.py:1524-1539)."""
    import frosting_b200 as fb
    cam = wl["cams"][0]
    m = wl["mesh"]

    def once():
        _, fv, _ = fb.rasterize_mesh(m["verts"], m["faces"], cam.full_proj_transform, cam.image_height, cam.image_width,
                                     mark_last_on_bg=True)
        return fb.gaussian_render_mask(fv.to(torch.uint8), m["cells"], wl["P"])
    for _ in range(3):
        once()
    torch.cuda.synchronize(device)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        once()
    b.record()
    torch.cuda.synchronize(device)
    return {"value": a.elapsed_time(b) / reps, "unit": "ms", "faces": int(m["faces"].shape[0]),
            "image": f"{cam.image_width}x{cam.image_height}",
            "note": "mesh raster (z-buffer atomics + resolve + visible-face marks) + face_visible[cell] mask, per frame"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(cb.WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="developer runs: headline + stage profile only")
    ap.add_argument("--with-dp", action="store_true", help="with --quick: also run the data-parallel training leg")
    ap.add_argument("--frame", default="raster", choices=["raster", "frosting"],
                    help="developer runs: time the frame from Frosting's parameters (frosting_render) as the main loop")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's outputs to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    # stdout carries exactly ONE JSON line: route fd 1 to stderr for the whole run (NCCL / C libraries print their
    # banners there) and write the result to the saved descriptor at the end
    sys.stdout.flush()
    result_fd = os.dup(1)
    os.dup2(2, 1)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=device)
    if args.gpus != world and rank == 0:
        log(f"[bench] --gpus {args.gpus} but WORLD_SIZE={world}: using WORLD_SIZE")
    ours = args.impl == "ours"

    if not ours:
        from oracle import refdgr
        if not refdgr.available():
            if rank == 0:
                os.write(result_fd, (json.dumps({"impl": "reference", "unavailable":
                                                 "oracle/_ref/ref_dgr_C.so not built (needs /root/reference)"}) + "\n").encode())
            return

    wl = load_workload(args.workload, device, rank, world, args.impl, local_rank, RING_RADIUS)
    step = make_step(args.impl, wl, device, mode=args.frame) if args.frame != "raster" else make_step(args.impl, wl, device)
    log(f"[bench] rank {rank}: workload {args.workload} built in {wl['gen_s']:.1f}s, impl={args.impl}")

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    secs, t0, t1 = timed_loop(step, wl, device, args.steps, args.warmup, world, e2e=False, count_launches=ours)
    clocks = sampler.stop(t0, t1) if sampler else None
    launches_timed = timed_loop.launches if ours else 0   # kernels of libfrosting_b200.so launched inside the timed region
    if args.dump_outputs and rank == 0:
        dump_outputs(step, args.dump_outputs, wl["P"])
    value = world * args.steps / secs

    e2e_value = None
    if not args.quick:
        secs_e2e, _, _ = timed_loop(step, wl, device, args.steps, args.warmup, world, e2e=True)
        e2e_value = world * args.steps / secs_e2e
    H, W, P = wl["H"], wl["W"], wl["P"]
    h2d = 3 * H * W * 4 + (16 + 16 + 3 + 3) * 4
    d2h = 4
    ring_txt = f", ring radius {RING_RADIUS:g}" if wl["kind"] == "frosting" else ""

    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * secs / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {
            "workload": cb.WORKLOAD_TEXT[args.workload] + ring_txt,
            "gaussians": P, "image": f"{W}x{H}", "sh_degree": wl["D"], "cameras_per_gpu": cb.CAMS_PER_GPU,
            "parallelism": f"camera-batch x{world} (Gaussians replicated, asynchronous NCCL all-reduce of the frames' "
                           "scalar losses, 8 frames per collective)",
            "frame": "occlusion culling (visible-face lookup inside preprocess) + rasterizer forward + (color*G).sum() + "
                     "backward to all attributes",
            "l2": "inputs larger than L2: ~236 B x P of attributes read per frame, no flush needed",
        },
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "note": "per step: cotangent image + camera record copied from pinned host memory on a copy "
                        "stream, loss copied back to pinned memory every step (read one step later); model parameters "
                        "stay resident as in the reference"},
        "gpu_launches": launches_timed,
    }
    if clocks:
        out["clocks"] = clocks
    if not ours:
        out["impl"] = "reference"
        out["cpu_baseline"] = {"value": value, "unit": UNIT, "cores": 0, "kind": "reference",
                               "sample": "the reference's own CUDA rasterizer (oracle/_ref, built from /root/reference) "
                                         "on the GPU: the reference has no CPU implementation of this path"}
        out["reference_notes"] = ("visible-face sets come from a child process (this process maps no repo library); "
                                  "frosting_step / frosting_train_step / dp_train_step use this repo's torch RESTATEMENTS of "
                                  "the reference's property chain and loss (scenes.frosting_attributes, loss.torch_reference)")
    else:
        try:
            prof, R_avg, V_avg = stage_profile(step, wl, device, min(args.steps, 16))
            out["roofline"], out["roofline_fwd"] = rooflines(prof, R_avg, W, H, args.workload)
            out["stage_ms"] = prof
            out["scene"] = {"P": P, "V": V_avg, "R": R_avg, "R_over_P": R_avg / P}
        except Exception as ex:   # measurement must not take the headline down with it
            out["roofline_error"] = repr(ex)
        if rank == 0 and world == 1 and not args.no_cpu_baseline and not args.quick:
            try:
                out["cpu_baseline"], _ = cpu_baseline(wl, step)
            except Exception as ex:
                out["cpu_baseline_error"] = repr(ex)

    side_steps = max(10, min(args.steps, 40))
    gts = None
    if wl.get("params") is not None and not args.quick:
        if ours:
            dstep = cb.CameraBatch(wl, device, mode="raster", mask="gather")
            secs_g, _, _ = timed_loop(dstep, wl, device, args.steps, args.warmup, world, e2e=False)
            out["dropin"] = {"value": world * args.steps / secs_g, "unit": UNIT,
                             "note": "plain drop-in: Frosting's boolean gathers in torch (frosting_model.py:1578-1586) + our "
                                     "rasterizer, no visibility_mask extension"}
            del dstep
        fstep = make_step(args.impl, wl, device, mode="frosting")
        secs_f, _, _ = timed_loop(fstep, wl, device, args.steps, args.warmup, world, e2e=False)
        out["frosting_step"] = {"value": world * args.steps / secs_f, "unit": UNIT,
                                "note": "secondary: the same frame starting from Frosting's learnable parameters "
                                        "(attribute construction, row a20, inside the step)"}
        # ... and with the trainers' real loss, 0.8 L1 + 0.2 (1 - SSIM) against a ground-truth image (refine.py:407-409)
        gtg = torch.Generator().manual_seed(99 + rank)
        gts = [torch.rand(3, H, W, generator=gtg).to(device) for _ in wl["cams"]]
        fstep = make_step(args.impl, wl, device, mode="frosting", loss="l1_dssim")
        fstep.gt = gts
        secs_t, _, _ = timed_loop(fstep, wl, device, args.steps, args.warmup, world, e2e=False)
        out["frosting_train_step"] = {"value": world * args.steps / secs_t, "unit": UNIT,
                                      "note": "secondary: parameters -> attributes -> mask -> rasterizer -> 0.8 L1 + 0.2 (1-SSIM) "
                                              "-> backward (ours: fused loss kernel, row f2; reference: its torch loss)"}
        del fstep
        if ours and world == 1:
            try:
                out["prepass_ms"] = prepass_ms(wl, device)
            except Exception as ex:
                out["prepass_error"] = repr(ex)

    # ---- the data-parallel TRAINING iteration (row f3).  It is the only leg that maps memory across ranks; it runs under
    # a watchdog, so a stuck rendezvous cannot take the line down
    if wl.get("params") is not None and (not args.quick or args.with_dp):
        if gts is None:
            gtg = torch.Generator().manual_seed(99 + rank)
            gts = [torch.rand(3, H, W, generator=gtg).to(device) for _ in wl["cams"]]
        lock, finished = threading.Lock(), [False]

        def bail():
            with lock:
                if finished[0]:
                    return
                out["dp_train_step_error"] = f"timeout: leg abandoned after {DP_LEG_TIMEOUT_S} s"
                if rank == 0:
                    os.write(result_fd, (json.dumps(out) + "\n").encode())
                os._exit(0)

        timer = threading.Timer(DP_LEG_TIMEOUT_S, bail)
        timer.daemon = True
        timer.start()
        try:
            dstep = OursDPTrain(wl, device) if ours else ReferenceDPTrain(wl, device)
            dstep.gt = gts
            secs_d, _, _ = timed_loop(dstep, wl, device, args.steps, args.warmup, world, e2e=False)
            out["dp_train_step"] = {
                "value": world * args.steps / secs_d, "unit": UNIT,
                "note": "secondary: one camera per rank per iteration, loss as above, then gradient mean over the ranks + Adam "
                        "with the reference's groups (ours: ONE peer-memory reduce+Adam+publish kernel per rank, row f3; "
                        "reference: NCCL all-reduce of each .grad + torch.optim.Adam)"}
            if ours:
                out["dp_train_step"]["transport"] = dstep.opt.slabs.transport
                try:
                    chk = dstep.opt.replica_check()
                except Exception as ex:
                    chk = {"error": repr(ex)}
                dstep.opt.close()
                try:
                    chk.update(dp_oracle_check(device, world, rank))
                except Exception as ex:
                    chk["oracle_check_error"] = repr(ex)
                out["dp_check"] = chk
            del dstep
        except Exception as ex:
            out["dp_train_step_error"] = repr(ex)
        with lock:
            finished[0] = True
        timer.cancel()

    # ---- the other BASELINE configs, one GPU, shipped kernels (they are parity-test cases first: tests/test_bench_configs_gpu.py)
    if world == 1 and args.workload == "c3" and not args.quick:
        del step
        wl.clear()
        torch.cuda.empty_cache()
        for name, rr in (("c2", RING_RADIUS), ("c5", RING_RADIUS), ("c3_ring10", 10.0)):
            try:
                out[name] = side_config("c3" if name == "c3_ring10" else name, args.impl, device, side_steps,
                                        max(3, args.warmup // 2), local_rank, ring_radius=rr)
            except Exception as ex:
                out[name + "_error"] = repr(ex)

    if rank == 0:
        os.write(result_fd, (json.dumps(out) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
