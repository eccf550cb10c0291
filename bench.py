#!/usr/bin/env python
"""bench.py -- headline benchmark of the rasterizer hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

metric   Mpixels/s, forward + backward, pixels = B x image_size^2 output pixels
workload BASELINE.json headline / SURVEY.md 8(d): B = 64 independent 5000-face meshes per GPU (seeded UV-spheres,
         neural_renderer_b200/synthetic.py), image 256 x 256, anti_aliasing off, textures [B,F,4,4,4,3] ~ U(0,1),
         `rasterize(faces, textures)` forward + backward with a dense N(0,1) upstream gradient (RGB path:
         grad wrt faces and textures).  N > 1: one process per GPU, every rank renders its own 64 meshes (batch
         sharding, no data-path collective) -> "scaling": "weak"; value = all ranks' pixels / max-over-ranks time.
step     one forward + backward pass over one batch.

One JSON line on rank 0.  Besides the base contract it carries
  e2e            the same metric through the public API from pinned HOST buffers: every step copies its own inputs
                 (sub-batch by sub-batch, the copy of sub-batch k+1 overlapping the kernels of sub-batch k INSIDE the
                 step) and reads loss + grad_faces back; `e2e.sequential` = copy -> compute -> read-back with no overlap,
                 `e2e.pipelined` = whole-batch double buffering across steps,
  kernels_ms_per_step  average device time per kernel of one step (CUDA events on the launching stream, separate pass),
  roofline       the dominant kernel against the measured HBM peak, with THAT kernel's own algorithmic bytes,
  roofline_fwd / roofline_bwd   pass-level: forward rasterize (the north-star's >= 70 % target) / whole backward,
  roofline_kernels  every kernel: its algorithmic bytes / its time,
  roofline_issue  issue-slot roofline of the dominant kernel (warp instructions from the committed ncu capture /
                 (SMs x 4 schedulers x SM clock x kernel time)) -- the edge scan is issue / shared-memory bound,
  modes          forward-only and fwd+bwd for silhouette / RGB / depth at the headline shape (SURVEY.md 8(d)),
  configs        BASELINE.json configs[0..2] (teapot silhouette 64^2, teapot RGB 256^2 batch 8, 70k faces 512^2 batch 32),
  shared_mesh    BASELINE.json configs[4] per-GPU share (1 M faces, 1024^2, 8 viewpoints per GPU) with the NCCL
                 sum-all-reduce of the shared vertex / texture gradients -- at every N, the path that communicates,
  cpu_baseline   the CPU oracle (oracle/nr_oracle.c, a port -- the reference ships no CPU path) on a bounded sample,
  reference_gpu  the reference's own CuPy kernels re-hosted (oracle/_ref) on the same GPU, same inputs.
`--impl reference` runs the reference's own implementation of the path: its unmodified CUDA kernel strings
re-hosted without CuPy (oracle/refhost.py + oracle/_ref/*.so) on the GPU -- the reference has no CPU path; if those
binaries are missing, the CPU oracle port is timed instead (and the line says so).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOAD = dict(batch_per_gpu=64, num_faces=5000, image_size=256, texture_size=4, anti_aliasing=False,
                near=0.1, far=100, eps=1e-4, background=(0.0, 0.0, 0.0))
N_SUB = 8        # sub-batches of the end-to-end step
NUM_SMS = 148

from neural_renderer_b200.distributed import shard_range  # noqa: E402,F401  (re-exported for the tests)

_JSON_OUT = None


def emit(obj):
    """the one JSON line of the run, on the process' original stdout"""
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    out.write(json.dumps(obj) + "\n")
    out.flush()


def algorithmic_bytes(B, F, S, ts):
    """SURVEY.md 8(d): compulsory traffic of the RGB passes (inputs once, outputs + saved maps once)."""
    P, T = B * S * S, ts ** 3
    fwd = 36 * B * F + 12 * T * B * F + 32 * P
    bwd = 72 * B * F + 12 * T * B * F + 40 * P
    return fwd, bwd


def mode_bytes(mode, B, F, S, ts):
    """SURVEY.md 8(d) per output mode: (forward, backward)."""
    P, T = B * S * S, ts ** 3
    if mode == "silhouette":
        return 36 * B * F + 8 * P, 72 * B * F + 12 * P
    if mode == "depth":
        # depth backward: faces r/w, depth, fim, weight map, upstream gradient (the survey lists no formula)
        return 36 * B * F + 20 * P, 72 * B * F + 24 * P
    return 36 * B * F + 12 * T * B * F + 32 * P, 72 * B * F + 12 * T * B * F + 40 * P


def kernel_bytes(B, F, S, ts):
    """What each kernel of the RGB step must move at least (its own inputs once, its own outputs once)."""
    P, T = B * S * S, ts ** 3
    return {
        # faces in, boxes out: only rasters with more than 2048 strips per axis still launch it (otherwise the counting
        # pass of k_strip_bin computes the boxes itself)
        "k_face_bbox": 36 * B * F + 8 * B * F + B * ((F + 31) // 32) * 8,
        # forward: z-buffer fill; faces in + one 8-byte z-buffer reduction per pixel (records: L2); z-buffer in + textures
        # in + every output map out (the pass-level figure is SURVEY.md's 36*B*F + 12*T*B*F + 32*P, see roofline_fwd)
        "memset_zbuf": 8 * P,
        "k_raster_faces": 36 * B * F + 8 * P,
        "k_resolve": 8 * P + 12 * T * B * F + 32 * P,
        # zero-fill of grad_faces (the zero-fill of grad_textures is a side job of k_edge_scan's CTAs, below)
        "memset_grads": 36 * B * F,
        # K6: grad_rgb 12 + fim 4 + weight_map 12 + depth_map 4 per pixel in, grad_textures out (reductions)
        "k_texture_grad": 32 * P + 12 * T * B * F,
        # K5: faces in, grad_faces out, rgb 12 + grad_rgb 12 + fim 4 per pixel in; plus grad_textures zero-filled once
        "k_edge_scan": 72 * B * F + 28 * P + 12 * T * B * F,
        # strip binning, two launches: (count) faces in, boxes out; (fill) boxes in, lists out (<= 8 entries per face and
        # axis; sparse) -- per launch: the average of the two
        "k_strip_bin": (36 * B * F + 8 * B * F + 8 * B * F) // 2,
        "k_strip_scan": 0,
    }


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Polls SM clock / throttle reasons through NVML while the benchmark runs."""

    def __init__(self, index):
        self.samples = []
        self.ok = False
        self._stop = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # pragma: no cover
            self.err = repr(e)
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                clk = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                self.samples.append((time.perf_counter(), clk, reasons))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.ok:
            self.t.start()

    def stop(self):
        self._stop.set()
        if self.ok:
            self.t.join(1.0)

    def summary(self, t0, t1):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        nv = self.nv
        inside = [s for s in self.samples if t0 <= s[0] <= t1]
        window = "timed_region"
        if len(inside) < 3:  # region shorter than a few polls: fall back to everything sampled under load
            inside = self.samples
            window = "whole_run"
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        seen = set()
        for _, _, r in inside:
            for bit, nm in names.items():
                if r & bit:
                    seen.add(nm)
        return {"sm_mhz": float(np.median([s[1] for s in inside])), "sm_max_mhz": float(self.sm_max),
                "reasons": sorted(seen), "samples": len(inside), "window": window}


def make_inputs(B, rank):
    from neural_renderer_b200 import synthetic
    w = WORKLOAD
    faces = synthetic.sphere_faces(B, w["num_faces"], seed=1234 + 1000 * rank)
    tex = synthetic.random_textures(B, w["num_faces"], w["texture_size"], seed=4321 + rank)
    gen = torch.Generator().manual_seed(99 + rank)
    grad = torch.randn((B, 3, w["image_size"], w["image_size"]), generator=gen)
    return torch.from_numpy(faces), torch.from_numpy(tex), grad


# ------------------------------------------------------------------------------------------------ step functions
def ours_step(faces, tex, grad, keep=None):
    """`keep`: a dict that receives the rendered image (for --dump-outputs)"""
    import neural_renderer_b200 as nr
    w = WORKLOAD
    faces.grad = None
    tex.grad = None
    img = nr.rasterize(faces, tex, w["image_size"], w["anti_aliasing"], w["near"], w["far"], w["eps"], w["background"])
    img.backward(grad)  # upstream gradient dL/dI = grad, i.e. L = sum(I * grad)
    with torch.no_grad():
        loss = (img * grad).sum()
    if keep is not None:
        keep["image"] = img.detach()
    return loss


DUMP_BYTES = 64 * 10 ** 6
NPY_HEADER = 128  # bytes np.save puts before the data of a 1- to 4-dimensional float32 array


def dump_outputs(out_dir, image, grad_faces, grad_textures):
    """--dump-outputs: what one headline step hands its caller, as float32 .npy files, at most DUMP_BYTES in all.
    In that order, each of the image, grad_faces and grad_textures is written whole as <name>.npy when it fits what
    is left of the budget, else as <name>_sample.npy: the elements of the flattened tensor at a fixed, seeded set of
    indices, as many as fit.  Returns {file name: shape}."""
    os.makedirs(out_dir, exist_ok=True)
    shapes, written = {}, 0
    for name, t in (("image", image), ("grad_faces", grad_faces), ("grad_textures", grad_textures)):
        room = (DUMP_BYTES - written - NPY_HEADER) // 4
        if room <= 0:
            break
        if t.numel() > room:
            flat = t.reshape(-1)
            idx = np.sort(np.random.default_rng(0).choice(flat.numel(), room, replace=False))
            t, name = flat[torch.from_numpy(idx).to(flat.device)], name + "_sample"
        path = os.path.join(out_dir, name + ".npy")
        a = t.detach().float().cpu().numpy()
        np.save(path, a)
        written += os.path.getsize(path)
        shapes[name + ".npy"] = list(a.shape)
    assert written <= DUMP_BYTES, written
    return shapes


def ref_gpu_step(faces, tex, grad):
    import refhost
    w = WORKLOAD
    res = refhost.rasterize_rgbad(faces, tex, w["image_size"], w["anti_aliasing"], w["near"], w["far"], w["eps"],
                                  w["background"], True, False, False)
    gf, gt = res.backward(grad, None, None)  # same upstream gradient as the other arm
    loss = (res["rgb"] * grad).sum()
    return loss, gf, gt


def oracle_cpu_step(faces_np, tex_np, grad_np):
    import nr_oracle as o
    w = WORKLOAD
    res = o.rasterize_rgbad(faces_np, tex_np, w["image_size"], w["anti_aliasing"], w["near"], w["far"], w["eps"],
                            w["background"], True, False, False)
    loss = float((res["rgb"] * grad_np).sum())
    gf, gt = res.backward(grad_np, None, None)
    return loss, gf, gt


class InputPipeline:
    """Whole-batch double buffering ACROSS steps (`e2e.pipelined`): the copy of step i+1's inputs (pinned host memory,
    its own stream) overlaps the kernels of step i.  Every step still pays for the copy of one full set of inputs
    inside the timed region."""

    def __init__(self, dev, host_tensors):
        self.host = [t.pin_memory() for t in host_tensors]
        self.bufs = [[torch.empty(t.shape, dtype=t.dtype, device=dev) for t in host_tensors] for _ in range(2)]
        self.copy_stream = torch.cuda.Stream(dev)
        self.ready = [torch.cuda.Event() for _ in range(2)]  # copy into the slot has finished
        self.free = [torch.cuda.Event() for _ in range(2)]   # the step that used the slot has finished
        self.i = 0
        self._issue(0)

    def _issue(self, slot):
        with torch.cuda.stream(self.copy_stream):
            self.copy_stream.wait_event(self.free[slot])
            for d, h in zip(self.bufs[slot], self.host):
                d.copy_(h, non_blocking=True)
            self.ready[slot].record(self.copy_stream)

    def acquire(self):
        slot = self.i & 1
        torch.cuda.current_stream().wait_event(self.ready[slot])
        self._issue(slot ^ 1)  # start moving the next step's inputs
        return slot, self.bufs[slot]

    def release(self, slot):
        self.free[slot].record(torch.cuda.current_stream())
        self.i += 1


class SubBatchStep:
    """The end-to-end step (`e2e.value`).  One step = the whole batch, processed as N_SUB sub-batches: the host ->
    device copy of sub-batch k+1 (copy stream) overlaps the forward + backward kernels of sub-batch k (compute
    stream), and each sub-batch's grad_faces goes back to the host as soon as it exists.  Nothing crosses a step
    boundary: the first copy of a step waits for the previous step's last kernel, so every step copies ITS OWN inputs
    inside the timed region.  Sub-batches are independent rasterizer calls, exactly like the batch shards of the
    multi-GPU run (batch items are independent; rasterize.py:389's batch-0 texture-depth quirk is call-local there
    too).  `run_sub(f, t, g) -> (loss, grad_faces)` is the arm's own forward + backward."""

    def __init__(self, dev, faces_h, tex_h, grad, run_sub, n_sub=N_SUB):
        self.dev = dev
        B = faces_h.shape[0]
        self.cuts = [(B * k // n_sub, B * (k + 1) // n_sub) for k in range(n_sub)]
        self.faces_p, self.tex_p = faces_h.pin_memory(), tex_h.pin_memory()
        self.f_dev = torch.empty(faces_h.shape, dtype=faces_h.dtype, device=dev)
        self.t_dev = torch.empty(tex_h.shape, dtype=tex_h.dtype, device=dev)
        self.grad = grad
        self.gf_host = torch.empty_like(faces_h).pin_memory()
        self.loss_host = torch.zeros((n_sub,), dtype=torch.float32).pin_memory()
        self.copy_stream = torch.cuda.Stream(dev)
        self.ready = [torch.cuda.Event() for _ in self.cuts]
        self.step_done = torch.cuda.Event()
        self.step_done.record(torch.cuda.current_stream(dev))
        self.run_sub = run_sub
        self.h2d = faces_h.numel() * 4 + tex_h.numel() * 4
        self.d2h = faces_h.numel() * 4 + 4 * n_sub

    def __call__(self):
        main = torch.cuda.current_stream(self.dev)
        with torch.cuda.stream(self.copy_stream):
            self.copy_stream.wait_event(self.step_done)  # the previous step no longer reads the staging buffers
            for k, (lo, hi) in enumerate(self.cuts):
                self.f_dev[lo:hi].copy_(self.faces_p[lo:hi], non_blocking=True)
                self.t_dev[lo:hi].copy_(self.tex_p[lo:hi], non_blocking=True)
                self.ready[k].record(self.copy_stream)
        for k, (lo, hi) in enumerate(self.cuts):
            main.wait_event(self.ready[k])
            loss, gf = self.run_sub(self.f_dev[lo:hi], self.t_dev[lo:hi], self.grad[lo:hi])
            self.loss_host[k:k + 1].copy_(loss.detach().reshape(1), non_blocking=True)
            self.gf_host[lo:hi].copy_(gf, non_blocking=True)
        self.step_done.record(main)


def _ours_sub(f, t, g):
    f = f.detach().requires_grad_(True)
    t = t.detach().requires_grad_(True)
    loss = ours_step(f, t, g)
    return loss, f.grad


def _ref_sub(f, t, g):
    loss, gf, _ = ref_gpu_step(f, t, g)
    return loss, gf


def timed_loop(step, steps, warmup, barrier):
    """W warm-up steps, then exactly K steps bracketed by barrier + synchronize, timed with CUDA events on the
    current stream."""
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    barrier()
    return e0.elapsed_time(e1), t0, t1


def median_ms(fn, n=10, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts))


# ------------------------------------------------------------------------------------- shared mesh (configs[4])
def shared_mesh_measure(args, world, rank, dev, barrier, distributed):
    """BASELINE.json configs[4] per-GPU share: ONE shared mesh rendered from many viewpoints, viewpoints sharded over
    the ranks, vertex / texture gradients summed across ranks with NCCL (the only collective this path has).  The
    geometry goes in as vertices + indices (no [V,F,3,3] tensor), the textures as one shared set (NR_TEX_SHARED), and
    the texture all-reduce starts between the two halves of the rasterizer's backward (overlap_texture_allreduce) so
    that it runs underneath the edge scan.  Returns a dict (identical on every rank up to the max-reduction)."""
    import neural_renderer_b200 as nr
    from neural_renderer_b200 import synthetic
    from neural_renderer_b200.distributed import allreduce_shared_grads, overlap_texture_allreduce
    import torch.distributed as dist
    F, S, ts, V = args.shared_faces, args.shared_image, 2, args.views_per_gpu
    v_np, f_np = synthetic.sphere_mesh(F)
    vertices = torch.from_numpy((v_np * 0.55).astype(np.float32)).to(dev).requires_grad_(True)   # shared parameters
    textures = torch.rand((F, ts, ts, ts, 3), generator=torch.Generator().manual_seed(7)).to(dev).requires_grad_(True)
    faces_idx = torch.from_numpy(f_np).to(dev)
    lo, hi = shard_range(world * V, rank, world)
    az = torch.arange(lo, hi, dtype=torch.float32) * (360.0 / (world * V))
    eyes = nr.get_points_from_angles(torch.full_like(az, 2.732), torch.full_like(az, 30.0), az).to(dev)
    renderer = nr.Renderer()
    renderer.image_size, renderer.anti_aliasing, renderer.fill_back = S, False, False
    renderer.eye = eyes
    renderer.reference_exact = False  # viewpoint shards: every view samples with its own depths (rasterize.py:389 would
    #                                   tie the result to which viewpoint happens to be item 0 of a rank's shard)
    grad = torch.randn((V, 3, S, S), generator=torch.Generator().manual_seed(99 + rank)).to(dev)
    steps, warmup = max(3, min(args.steps, 5)), 3

    def make_step(overlap, fused):
        renderer.fused = fused

        def step():
            vertices.grad = None
            textures.grad = None
            vv, ff = vertices[None].expand(V, -1, -1), faces_idx[None].expand(V, -1, -1)
            if fused:
                tt = textures[None]                                  # one shared set, sampled in place
            else:
                tt = textures[None].expand(V, -1, -1, -1, -1, -1)    # round-1 formulation: materialised per view
            if overlap:
                with overlap_texture_allreduce():
                    (renderer.render(vv, ff, tt) * grad).sum().backward()
                allreduce_shared_grads([vertices])
            else:
                (renderer.render(vv, ff, tt) * grad).sum().backward()
                allreduce_shared_grads([vertices, textures])
        return step

    def run(step):
        ms, _, _ = timed_loop(step, steps, warmup, barrier)
        if distributed:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps

    ms_overlap = run(make_step(True, True))
    ms_serial = run(make_step(False, True))
    ms_unfused = run(make_step(False, False))   # faces [V,F,3,3] + per-view texture copies: the round-1 path
    renderer.fused = True
    # the collective alone (same buffers), for the bus bandwidth
    ar_ms, bus = None, None
    nbytes = (vertices.numel() + textures.numel()) * 4
    if distributed:
        vertices.grad = torch.zeros_like(vertices)
        textures.grad = torch.zeros_like(textures)

        def ar():
            allreduce_shared_grads([vertices, textures])
        ar_ms = run(ar)
        bus = 2.0 * (world - 1) / world * nbytes / (ar_ms * 1e-3) / 1e9
    value = world * V * S * S / (ms_overlap * 1e-3) / 1e6
    return {
        "workload": "configs[4] share: Renderer.render fwd+bwd, ONE shared %d-face mesh, %dx%d, ts=%d, %d viewpoints/GPU; "
                    "indexed geometry (no [V,F,3,3] tensor), shared texture set, sum all-reduce of vertex (%.1f MB) and "
                    "texture (%.1f MB) gradients" % (F, S, S, ts, V, vertices.numel() * 4 / 1e6, textures.numel() * 4 / 1e6),
        "n_gpus": world, "steps": steps, "value": round(value, 2), "unit": "Mpixels/s",
        "ms_per_step": round(ms_overlap, 4),
        "ms_per_step_allreduce_after_backward": round(ms_serial, 4),
        "ms_per_step_round1_formulation": round(ms_unfused, 4),
        "allreduce_ms": None if ar_ms is None else round(ar_ms, 4),
        "allreduce_bytes": nbytes,
        "allreduce_bus_gbs": None if bus is None else round(bus, 1),
        "collective": ("nccl all_reduce(sum): textures launched between the two halves of the rasterizer backward "
                       "(overlaps the edge scan), vertices after it") if distributed else "none (1 rank)",
        "timing": "CUDA events on the compute stream, max over ranks",
    }


# --------------------------------------------------------------------- per-mode / per-config side measurements
def modes_measure(dev, peak):
    import neural_renderer_b200 as nr
    w = WORKLOAD
    B, F, S, ts = w["batch_per_gpu"], w["num_faces"], w["image_size"], w["texture_size"]
    faces_h, tex_h, _ = make_inputs(B, 0)
    fa = faces_h.to(dev).requires_grad_(True)
    ta = tex_h.to(dev).requires_grad_(True)
    gen = torch.Generator().manual_seed(99)
    g3 = torch.randn((B, 3, S, S), generator=gen).to(dev)
    g1 = torch.randn((B, S, S), generator=gen).to(dev)
    calls = {"silhouette": (lambda: nr.rasterize_silhouettes(fa, S, False), g1),
             "rgb": (lambda: nr.rasterize(fa, ta, S, False), g3),
             "depth": (lambda: nr.rasterize_depth(fa, S, False), g1)}
    rows = []
    for mode, (fwd, g) in calls.items():
        def fb():
            fa.grad = None
            ta.grad = None
            fwd().backward(g)

        def f_only():
            with torch.no_grad():
                fwd()
        t_f, t_fb = median_ms(f_only), median_ms(fb)
        bf, bb = mode_bytes(mode, B, F, S, ts)
        rows.append({"mode": mode, "fwd_ms": round(t_f, 4), "fwd_bwd_ms": round(t_fb, 4),
                     "fwd_mpixels_per_s": round(B * S * S / t_f / 1e3, 1), "fwd_bwd_mpixels_per_s": round(B * S * S / t_fb / 1e3, 1),
                     "fwd_algorithmic_mb": round(bf / 1e6, 1), "fwd_hbm_frac": round(bf / (t_f * 1e-3) / 1e9 / peak, 4),
                     "bwd_algorithmic_mb": round(bb / 1e6, 1),
                     "fwd_bwd_hbm_frac": round((bf + bb) / (t_fb * 1e-3) / 1e9 / peak, 4)})
    return {"shape": "headline: B=%d, F=%d, %dx%d, ts=%d, anti-aliasing off" % (B, F, S, S, ts),
            "timing": "whole API calls (torch allocation + every kernel of the pass), CUDA events, median of 10",
            "rows": rows}


def configs_measure(dev):
    """BASELINE.json configs[0..2] through the public API (ours only; parity for each is in tests/test_gpu_configs.py)."""
    import neural_renderer_b200 as nr
    from neural_renderer_b200 import synthetic
    out = []
    d = np.load(os.path.join(ROOT, "tests", "golden", "teapot.npz"))

    def teapot(B):
        v = torch.from_numpy(np.stack([d["vertices"]] * B)).to(dev).requires_grad_(True)
        f = torch.from_numpy(np.stack([d["faces"]] * B)).to(dev)
        return v, f
    # configs[0]: teapot silhouette 64x64 (anti-aliased), batch 1, through Renderer
    v, f = teapot(1)
    r = nr.Renderer()
    r.image_size = 64
    g = torch.randn((1, 64, 64), device=dev)

    def c0():
        v.grad = None
        r.render_silhouettes(v, f).backward(g)

    def c0f():
        with torch.no_grad():
            r.render_silhouettes(v, f)
    out.append({"config": "configs[0]: teapot silhouette 64x64 (anti-aliased), batch 1, Renderer.render_silhouettes",
                "fwd_ms": round(median_ms(c0f), 4), "fwd_bwd_ms": round(median_ms(c0), 4)})
    # configs[1]: teapot RGB + texture 256x256 batch 8, fwd + bwd, Renderer defaults (fill_back, anti-aliasing, lighting)
    v8, f8 = teapot(8)
    t8 = torch.rand((8, f8.shape[1], 4, 4, 4, 3), device=dev).requires_grad_(True)
    r8 = nr.Renderer()
    g8 = torch.randn((8, 3, 256, 256), device=dev)

    def c1():
        v8.grad = None
        t8.grad = None
        r8.render(v8, f8, t8).backward(g8)

    def c1f():
        with torch.no_grad():
            r8.render(v8, f8, t8)
    t1 = median_ms(c1)
    out.append({"config": "configs[1]: teapot RGB 256x256 (anti-aliased, fill_back, lighting), batch 8, Renderer.render",
                "fwd_ms": round(median_ms(c1f), 4), "fwd_bwd_ms": round(t1, 4),
                "fwd_bwd_mpixels_per_s": round(8 * 256 * 256 / t1 / 1e3, 1)})
    del v8, f8, t8, g8
    # configs[2]: ~70k faces, depth + RGB, 512x512, batch 32 (synthetic 70k-face spheres, ts = 2)
    B, F, S, ts = 32, 70000, 512, 2
    fa = torch.from_numpy(synthetic.sphere_faces(B, F)).to(dev).requires_grad_(True)
    ta = torch.from_numpy(synthetic.random_textures(B, F, ts)).to(dev).requires_grad_(True)
    g3 = torch.randn((B, 3, S, S), device=dev)
    g1 = torch.randn((B, S, S), device=dev)

    def fwd3():
        return nr.rasterize_rgbad(fa, ta, S, False, 0.1, 100, 1e-4, [0, 0, 0], True, False, True)

    def c2():
        fa.grad = None
        ta.grad = None
        o = fwd3()
        torch.autograd.backward([o["rgb"], o["depth"]], [g3, g1])

    def c2f():
        with torch.no_grad():
            fwd3()
    t2 = median_ms(c2, n=5)
    out.append({"config": "configs[2]: 70k-face spheres, depth + RGB, 512x512, batch 32, ts 2",
                "fwd_ms": round(median_ms(c2f, n=5), 4), "fwd_bwd_ms": round(t2, 4),
                "fwd_bwd_mpixels_per_s": round(B * S * S / t2 / 1e3, 1)})
    del fa, ta, g3, g1
    torch.cuda.empty_cache()
    return out


def bind_near_gpu(local_rank):
    """Run this process on the CPUs next to its GPU (NVML's ideal affinity) BEFORE any pinned host buffer is allocated:
    pinned pages are placed on the NUMA node of the thread that first touches them, and a host -> device copy from the
    far socket of a two-socket box runs at 3/4 of the PCIe rate (the end-to-end figures swung 675 .. 845 Mpixels/s with
    the box).  Host-side placement only; both arms do it.  Returns what was done, for the JSON line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = None
        try:
            uuid = str(torch.cuda.get_device_properties(local_rank).uuid)
            h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        before = len(os.sched_getaffinity(0))
        pynvml.nvmlDeviceSetCpuAffinity(h)
        return {"cpu_affinity": "nvmlDeviceSetCpuAffinity", "cpus_before": before, "cpus": len(os.sched_getaffinity(0))}
    except Exception as e:  # pragma: no cover
        return {"cpu_affinity": "unchanged", "why": repr(e)[:120]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-sample", type=int, default=64, help="batch items of the workload timed on the CPU oracle")
    ap.add_argument("--no-side-measurements", action="store_true",
                    help="skip kernels / rooflines / modes / configs / cpu_baseline / reference_gpu")
    ap.add_argument("--no-shared-mesh", action="store_true", help="skip the configs[4] shared-mesh measurement")
    ap.add_argument("--workload", default="headline", choices=["headline", "shared_mesh"])
    ap.add_argument("--shared-faces", type=int, default=1000000)
    ap.add_argument("--shared-image", type=int, default=1024)
    ap.add_argument("--views-per-gpu", type=int, default=8)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the image, grad_faces and a fixed sample of grad_textures of the "
                         "last headline step to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload != "headline"):
        ap.error("--dump-outputs writes the outputs of the headline workload of --impl ours")
    args.warmup = max(args.warmup, 3)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    distributed = world > 1
    # stdout carries exactly ONE JSON line: whatever libraries write to file descriptor 1 meanwhile (NCCL prints its
    # version banner there) is diverted to stderr; the line itself goes to the saved descriptor at the very end
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    host_placement = bind_near_gpu(local_rank) if torch.cuda.is_available() else {"cpu_affinity": "unchanged"}
    w = WORKLOAD
    B, F, S, ts = w["batch_per_gpu"], w["num_faces"], w["image_size"], w["texture_size"]
    sys.path.insert(0, os.path.join(ROOT, "oracle"))

    if args.impl == "reference":
        return reference_arm(args, world, rank, local_rank, host_placement)

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA GPU: this package has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if distributed:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
        barrier = lambda: dist.barrier(device_ids=[local_rank])  # noqa: E731
    else:
        barrier = lambda: None  # noqa: E731

    from neural_renderer_b200 import _lib
    lib = _lib.load()  # fails loudly when libnr_b200.so is missing

    if args.workload == "shared_mesh":  # stand-alone form of the shared-mesh measurement
        sm = shared_mesh_measure(args, world, rank, dev, barrier, distributed)
        if rank == 0:
            emit(dict({"metric": "Mpixels/s fwd+bwd, shared mesh, viewpoint-sharded", "higher_is_better": True,
                       "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                       "impl": "ours", "warmup": 3, "config": {"workload": sm["workload"]}}, **sm))
        if distributed:
            dist.destroy_process_group()
        return

    faces_h, tex_h, grad_h = make_inputs(B, rank)
    faces = faces_h.to(dev).requires_grad_(True)
    tex = tex_h.to(dev).requires_grad_(True)
    grad = grad_h.to(dev)

    sampler = ClockSampler(local_rank)
    sampler.start()

    def reduce_max(ms):
        if distributed:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    # ---- headline: device-resident inputs
    last = {} if args.dump_outputs else None

    def step():
        ours_step(faces, tex, grad, keep=last)

    ms, t0, t1 = timed_loop(step, args.steps, args.warmup, barrier)
    ms = reduce_max(ms)
    pixels = world * B * S * S
    value = pixels * args.steps / (ms * 1e-3) / 1e6
    clocks = sampler.summary(t0, t1)
    sampler.stop()  # the poller thread takes the GIL every 2 ms: keep it out of the launch-bound measurements below
    dumped = None
    if args.dump_outputs and rank == 0:
        dumped = dump_outputs(args.dump_outputs, last["image"], faces.grad, tex.grad)
    last = None

    # count our kernel launches of one step through the library's own accounting
    import neural_renderer_b200 as nr
    faces.grad = None
    tex.grad = None
    img = nr.rasterize(faces, tex, S, False, w["near"], w["far"], w["eps"], w["background"])
    n_fwd = lib.nr_b200_last_launch_count()
    (img * grad).sum().backward()
    n_bwd = lib.nr_b200_last_launch_count()
    launches_per_step = n_fwd + n_bwd
    del img

    # ---- end to end: host (pinned) inputs in, loss + vertex gradients out, copies inside the timed region
    sub = SubBatchStep(dev, faces_h, tex_h, grad, _ours_sub)
    e2e_ms, _, _ = timed_loop(sub, args.steps, args.warmup, barrier)
    e2e_ms = reduce_max(e2e_ms)
    e2e_value = pixels * args.steps / (e2e_ms * 1e-3) / 1e6

    #      beside it: strictly sequential (copy everything, compute, read back) ...
    faces_p, tex_p = sub.faces_p, sub.tex_p
    gf_host = sub.gf_host
    loss_host = torch.empty((), dtype=torch.float32).pin_memory()

    def e2e_seq_step():
        f = faces_p.to(dev, non_blocking=True).requires_grad_(True)
        t = tex_p.to(dev, non_blocking=True).requires_grad_(True)
        loss = ours_step(f, t, grad)
        loss_host.copy_(loss.detach(), non_blocking=True)
        gf_host.copy_(f.grad, non_blocking=True)

    seq_ms, _, _ = timed_loop(e2e_seq_step, args.steps, args.warmup, barrier)
    seq_ms = reduce_max(seq_ms)
    seq_value = pixels * args.steps / (seq_ms * 1e-3) / 1e6

    #      ... and whole-batch double buffering across steps
    pipe = InputPipeline(dev, [faces_h, tex_h])

    def e2e_pipelined_step():
        slot, (f_buf, t_buf) = pipe.acquire()
        f = f_buf.detach().requires_grad_(True)
        t = t_buf.detach().requires_grad_(True)
        loss = ours_step(f, t, grad)
        loss_host.copy_(loss.detach(), non_blocking=True)
        gf_host.copy_(f.grad, non_blocking=True)
        pipe.release(slot)

    pipe_ms, _, _ = timed_loop(e2e_pipelined_step, args.steps, args.warmup, barrier)
    pipe_ms = reduce_max(pipe_ms)
    pipe_value = pixels * args.steps / (pipe_ms * 1e-3) / 1e6
    del pipe

    out = {
        "metric": "Mpixels/s fwd+bwd @ 256x256, 5k faces, batch 64", "value": round(value, 2), "unit": "Mpixels/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 4),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "impl": "ours",
        "config": {"workload": "headline: rasterize() fwd+bwd RGB, B=%d/GPU x F=%d faces, %dx%d, ts=%d, "
                               "anti_aliasing off (BASELINE.json metric; configs[3] batch-sharded shape per GPU)"
                               % (B, F, S, S, ts),
                   "global_batch": world * B, "num_faces": F, "image_size": S, "texture_size": ts,
                   "parallelism": "batch-sharded x%d (no data-path collective)" % world,
                   "l2": "no explicit flush: per-step working set (textures 245.8 MB + grad_textures 245.8 MB + "
                         "maps 134 MB) exceeds the 126 MB L2",
                   "upstream_grad": "dense N(0,1), seed 99"},
        "clocks": clocks,
        "e2e": {"value": round(e2e_value, 2), "unit": "Mpixels/s", "ms_per_step": round(e2e_ms / args.steps, 4),
                "h2d_bytes_per_step": sub.h2d, "d2h_bytes_per_step": sub.d2h,
                "what": "per step: pinned host faces+textures -> device in %d sub-batches, the copy of sub-batch k+1 "
                        "overlapping rasterize fwd+bwd of sub-batch k inside the step; loss + grad_faces of every "
                        "sub-batch -> host; no overlap across step boundaries" % N_SUB,
                "sequential": {"value": round(seq_value, 2), "unit": "Mpixels/s", "ms_per_step": round(seq_ms / args.steps, 4),
                               "what": "copy the whole batch, then compute, then read back (no overlap at all)"},
                "pipelined": {"value": round(pipe_value, 2), "unit": "Mpixels/s", "ms_per_step": round(pipe_ms / args.steps, 4),
                              "what": "whole-batch double buffering: the copy of the NEXT step's inputs overlaps this "
                                      "step's kernels (one full copy per step inside the timed region)"}},
        "host": host_placement,
        "gpu_launches": launches_per_step * args.steps,
        "gpu_launches_per_step": launches_per_step,
    }
    if dumped:
        out["dump_outputs"] = {"dir": args.dump_outputs, "files": dumped}
    del sub

    # ---- side measurements (rank 0, N = 1, outside the headline region)
    if rank == 0 and not args.no_side_measurements:
        peak, peak_src = measured_peaks()
        fwd_bytes, bwd_bytes = algorithmic_bytes(B, F, S, ts)
        kb = kernel_bytes(B, F, S, ts)
        lib.nr_b200_set_profiling(1)
        _lib.read_profile()
        nprof = max(5, min(args.steps, 20))
        for _ in range(nprof):
            ours_step(faces, tex, grad)
        torch.cuda.synchronize()
        prof = _lib.read_profile()
        lib.nr_b200_set_profiling(0)
        per, count = {}, {}
        for name, v in prof:
            per[name] = per.get(name, 0.0) + v
            count[name] = count.get(name, 0) + 1
        # a name can appear twice per step (k_face_bbox runs in both passes): per-step totals
        kern = {k: round(v / nprof, 5) for k, v in per.items()}
        launches = {k: count[k] // nprof for k in count}
        out["kernels_ms_per_step"] = kern
        fwd_names = ("memset_zbuf", "k_raster_faces", "k_raster_big", "k_resolve")
        fwd_ms = sum(kern.get(k, 0.0) for k in fwd_names)
        bwd_ms = sum(v for k, v in kern.items()) - fwd_ms

        counts = {}
        try:  # per-launch counters of the committed ncu --set full capture of THIS build at THIS shape (profiles/)
            with open(os.path.join(ROOT, "profiles", "ncu_counts.json")) as f:
                counts = json.load(f)
        except Exception:
            pass

        def roof(bytes_, ms_):
            ach = bytes_ / (ms_ * 1e-3) / 1e9 if ms_ > 0 else 0.0
            return {"bound": "hbm", "achieved": round(ach, 1), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 4),
                    "traffic": None, "peak_source": peak_src, "algorithmic_bytes": bytes_, "ms": round(ms_, 5)}

        def with_ncu(r, kernel):
            c = counts.get("kernels", {}).get(kernel)
            if c and c.get("dram_bytes") is not None:
                r["traffic_ncu_capture"] = {"bytes_per_launch": c["dram_bytes"], "source": counts.get("source"),
                                            "note": "from the committed ncu capture, not measured in this run"}
            return r

        rk = {}
        for k, v in kern.items():
            n = max(launches.get(k, 1), 1)
            if kb.get(k):
                rk[k] = with_ncu(dict(roof(kb[k], v / n), launches_per_step=n), k)
        out["roofline_kernels"] = rk
        dom = max(kern, key=lambda k: kern[k]) if kern else None
        if dom and dom in rk:
            out["roofline"] = dict(rk[dom], kernel=dom,
                                   note="the dominant kernel's OWN algorithmic bytes / its duration (CUDA events)")
        out["roofline_fwd"] = dict(roof(fwd_bytes, fwd_ms), kernels=" + ".join(fwd_names),
                                   note="forward rasterize pass, 391.5 MB algorithmic (SURVEY.md 8(d))")
        out["roofline_bwd"] = dict(roof(bwd_bytes, bwd_ms),
                                   kernels="memset_grads + k_strip_bin x2 + k_edge_scan (+ zero-fill of grad_textures) + k_texture_grad",
                                   note="whole backward pass, 436.6 MB algorithmic (SURVEY.md 8(d))")
        out["roofline_step"] = roof(fwd_bytes + bwd_bytes, ms / args.steps)
        # issue-slot roofline of the kernels the HBM roof does not describe (warp instructions from the ncu capture)
        sm_hz = (clocks.get("sm_mhz") or 1965.0) * 1e6
        issue = {}
        for k in ("k_edge_scan", "k_resolve", "k_raster_faces"):
            c = counts.get("kernels", {}).get(k)
            if c and c.get("warp_instructions") and kern.get(k):
                peak_ips = NUM_SMS * 4 * sm_hz
                ach = c["warp_instructions"] / (kern[k] * 1e-3)
                issue[k] = {"bound": "issue", "warp_instructions": c["warp_instructions"],
                            "achieved": round(ach / 1e9, 1), "peak": round(peak_ips / 1e9, 1), "unit": "G warp-inst/s",
                            "frac": round(ach / peak_ips, 4),
                            "l1_lsu_wavefront_pct_ncu": c.get("l1_lsu_wavefront_pct"),
                            "source": counts.get("source"),
                            "note": "instruction count from the committed ncu capture of this build; time from this run"}
        if issue:
            out["roofline_issue"] = issue

        if world == 1:
            try:
                out["modes"] = modes_measure(dev, peak)
            except Exception as e:  # pragma: no cover
                out["modes"] = {"unavailable": repr(e)[:200]}
            try:
                out["configs"] = configs_measure(dev)
            except Exception as e:  # pragma: no cover
                out["configs"] = {"unavailable": repr(e)[:200]}

        # reference's own kernels on this GPU (the reported baseline of BASELINE.md section 2); N = 1 only
        try:
            if world > 1:
                raise RuntimeError("reported at N=1 only")
            import refhost
            if refhost.available(S, F, ts, w["near"], w["far"], w["eps"], 1, 0, 0):
                fr, tr = faces.detach(), tex.detach()
                rsteps = max(3, args.steps // 4)
                rms, _, _ = timed_loop(lambda: ref_gpu_step(fr, tr, grad), rsteps, 3, lambda: None)
                out["reference_gpu"] = {"value": round(B * S * S * rsteps / (rms * 1e-3) / 1e6, 2),
                                        "unit": "Mpixels/s", "ms_per_step": round(rms / rsteps, 3), "steps": rsteps,
                                        "what": "reference CuPy kernel strings re-hosted (oracle/_ref), same inputs, 1 GPU"}
            else:
                out["reference_gpu"] = {"unavailable": "oracle/_ref binaries for the headline shape not built"}
        except Exception as e:  # pragma: no cover
            out["reference_gpu"] = {"unavailable": repr(e)[:200]}

        # CPU oracle (port) on a bounded sample of the same workload; N = 1 only (torchrun pins OMP threads to 1)
        try:
            if world > 1:
                raise RuntimeError("reported at N=1 only")
            import nr_oracle as o
            nb = max(1, min(B, args.cpu_sample))
            fn, tn, gn = faces_h[:nb].numpy(), tex_h[:nb].numpy(), grad_h[:nb].numpy()
            tc0 = time.perf_counter()
            oracle_cpu_step(fn, tn, gn)
            tc = time.perf_counter() - tc0
            out["cpu_baseline"] = {"value": round(nb * S * S / tc / 1e6, 4), "unit": "Mpixels/s",
                                   "cores": o.num_threads(), "kind": "port",
                                   "sample": "%d of the %d batch items, fwd+bwd, %.1f s" % (nb, B, tc)}
        except Exception as e:  # pragma: no cover
            out["cpu_baseline"] = {"unavailable": repr(e)[:200]}

    # ---- the path that communicates (every rank takes part), after the headline so that it cannot disturb it
    del faces, tex, grad
    torch.cuda.empty_cache()
    if not args.no_shared_mesh:
        try:
            sm = shared_mesh_measure(args, world, rank, dev, barrier, distributed)
            out["shared_mesh"] = sm
        except Exception as e:  # pragma: no cover
            out["shared_mesh"] = {"unavailable": repr(e)[:300]}

    sampler.stop()
    if rank == 0:
        emit(out)
    if distributed:
        dist.destroy_process_group()


def reference_arm(args, world, rank, local_rank, host_placement=None):
    """The reference's own implementation of the path, same workload / metric (rank 0 only)."""
    if rank != 0:
        return
    w = WORKLOAD
    B, F, S, ts = w["batch_per_gpu"], w["num_faces"], w["image_size"], w["texture_size"]
    faces_h, tex_h, grad_h = make_inputs(B, 0)
    base = {"metric": "Mpixels/s fwd+bwd @ 256x256, 5k faces, batch 64", "unit": "Mpixels/s", "n_gpus": 1,
            "steps": args.steps, "warmup": args.warmup, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference", "host": host_placement}
    use_gpu = False
    if torch.cuda.is_available():
        import refhost
        use_gpu = refhost.available(S, F, ts, w["near"], w["far"], w["eps"], 1, 0, 0)
    if use_gpu:
        torch.cuda.set_device(local_rank)
        dev = torch.device("cuda", local_rank)
        faces, tex, grad = faces_h.to(dev), tex_h.to(dev), grad_h.to(dev)
        sampler = ClockSampler(local_rank)
        sampler.start()
        ms, t0, t1 = timed_loop(lambda: ref_gpu_step(faces, tex, grad), args.steps, args.warmup, lambda: None)
        value = B * S * S * args.steps / (ms * 1e-3) / 1e6
        # end to end, the same three ways as the other arm
        sub = SubBatchStep(dev, faces_h, tex_h, grad, _ref_sub)
        e2e_ms, _, _ = timed_loop(sub, args.steps, args.warmup, lambda: None)
        e2e_value = B * S * S * args.steps / (e2e_ms * 1e-3) / 1e6
        faces_p, tex_p, gf_host = sub.faces_p, sub.tex_p, sub.gf_host
        loss_host = torch.empty((), dtype=torch.float32).pin_memory()

        def e2e_seq_step():
            f = faces_p.to(dev, non_blocking=True)
            t = tex_p.to(dev, non_blocking=True)
            loss, gf, _ = ref_gpu_step(f, t, grad)
            loss_host.copy_(loss, non_blocking=True)
            gf_host.copy_(gf, non_blocking=True)

        seq_ms, _, _ = timed_loop(e2e_seq_step, args.steps, args.warmup, lambda: None)
        seq_value = B * S * S * args.steps / (seq_ms * 1e-3) / 1e6
        pipe = InputPipeline(dev, [faces_h, tex_h])  # same double-buffered staging as the other arm

        def e2e_pipelined_step():
            slot, (f, t) = pipe.acquire()
            loss, gf, _ = ref_gpu_step(f, t, grad)
            loss_host.copy_(loss, non_blocking=True)
            gf_host.copy_(gf, non_blocking=True)
            pipe.release(slot)

        pipe_ms, _, _ = timed_loop(e2e_pipelined_step, args.steps, args.warmup, lambda: None)
        pipe_value = B * S * S * args.steps / (pipe_ms * 1e-3) / 1e6
        clocks = sampler.summary(t0, t1)
        sampler.stop()
        best_name, best_value, best_ms = max(
            (("sub-batched (copy of sub-batch k+1 under the kernels of sub-batch k)", e2e_value, e2e_ms),
             ("sequential (copy, compute, read back)", seq_value, seq_ms),
             ("pipelined (whole-batch double buffering: the copy of the next step's inputs under this step's kernels)",
              pipe_value, pipe_ms)), key=lambda t: t[1])
        base.update({
            "value": round(value, 2), "ms_per_step": round(ms / args.steps, 4), "clocks": clocks,
            "config": {"workload": "headline: reference kernels (K1,K2,K4,K5,K6 of rasterize.py, unmodified strings "
                                   "re-hosted without CuPy) fwd+bwd RGB, B=%d x F=%d, %dx%d, ts=%d" % (B, F, S, S, ts),
                       "device": "cuda (the reference ships no CPU implementation: rasterize.py:893-897)",
                       "global_batch": B, "num_faces": F, "image_size": S, "texture_size": ts},
            "cpu_baseline": {"value": round(value, 2), "unit": "Mpixels/s", "cores": 0, "kind": "reference",
                             "sample": "full workload on the GPU: the reference has no CPU path, its own CUDA kernels "
                                       "are the baseline (oracle/_ref)"},
            # The reference's K5 runs one thread per face (rasterize.py:527): a sub-batch of 8 items leaves most of the GPU
            # idle, so the sub-batch overlap that helps the other arm HURTS this one.  The arm is credited with the
            # fastest of its three end-to-end variants (each copies a full set of inputs per step inside the timed region).
            "e2e": {"value": round(best_value, 2), "unit": "Mpixels/s", "ms_per_step": round(best_ms / args.steps, 4),
                    "h2d_bytes_per_step": sub.h2d, "d2h_bytes_per_step": sub.d2h,
                    "what": "fastest end-to-end variant of this arm: " + best_name,
                    "sub_batched": {"value": round(e2e_value, 2), "unit": "Mpixels/s", "ms_per_step": round(e2e_ms / args.steps, 4),
                                    "what": "same %d-sub-batch overlapped step as the other arm" % N_SUB},
                    "sequential": {"value": round(seq_value, 2), "unit": "Mpixels/s", "ms_per_step": round(seq_ms / args.steps, 4)},
                    "pipelined": {"value": round(pipe_value, 2), "unit": "Mpixels/s",
                                  "ms_per_step": round(pipe_ms / args.steps, 4)}},
            "gpu_launches": 0,
        })
    else:
        import nr_oracle as o
        nb = max(1, min(B, args.cpu_sample))
        fn, tn, gn = faces_h[:nb].numpy(), tex_h[:nb].numpy(), grad_h[:nb].numpy()
        for _ in range(min(args.warmup, 1)):
            oracle_cpu_step(fn[:1], tn[:1], gn[:1])
        t0 = time.perf_counter()
        steps = max(1, min(args.steps, 3))
        for _ in range(steps):
            oracle_cpu_step(fn, tn, gn)
        dt = (time.perf_counter() - t0) / steps
        value = nb * S * S / dt / 1e6
        base.update({
            "value": round(value, 4), "steps": steps, "ms_per_step": round(dt * 1e3, 2),
            "config": {"workload": "headline sample on the CPU oracle port (oracle/_ref binaries absent)",
                       "global_batch": nb, "num_faces": F, "image_size": S, "texture_size": ts},
            "cpu_baseline": {"value": round(value, 4), "unit": "Mpixels/s", "cores": o.num_threads(), "kind": "port",
                             "sample": "%d of %d batch items per step" % (nb, B)},
            "e2e": {"value": round(value, 4), "unit": "Mpixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        })
    emit(base)


if __name__ == "__main__":
    main()
