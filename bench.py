#!/usr/bin/env python
"""bench.py -- forward+backward rendered images/s through the drop-in SoftRenderer (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config C2|C3|C5] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" = one pass of the hot path over one batch of synthetic input (SURVEY.md §8d, config C2 by
default: 642-vertex / 1280-face CUB-like mesh, 256x256 render (512x512 raster), batch 16 per GPU,
T2 = 36 surface textures):
    verts = mean_shape + delta_v[b];  images = SoftRenderer(256, 'softmax')(verts, faces, cams, tex)
    loss  = 2.5 * neg_iou_loss(alpha, mask) + 3.0 * texture_loss_masks(rgb, img, mask, alpha)
    loss.backward()  -> d/d mean_shape [V,3], d/d texture [F,T2,3];  N>1: one all-reduce of the flat
    [V*3 + F*T2*3] gradient (our one-shot peer-memory kernel inside the step's CUDA graph; NCCL fallback).
(--config C3 adds, per BASELINE.json config 3: per-image textures sampled from a texture flow, texture-dt,
texture-cycle on the hard renderer's visibility (the reference drops that render's image, loss_utils.py:327-329) and
chamfer correspondence; C5 is the 5120-face 1024x1024 sweep point.)
Rank 0 prints ONE JSON line.  `value` = images/s with inputs resident in HBM; `e2e` = the same step
with that step's inputs copied from pinned host memory and the loss read back, inside the timed
region.  `roofline` = the dominant kernel (raster forward or backward, whichever is slower): algorithmic
bytes / CUDA-event time of that kernel alone (events recorded by the C ABI around the launch), against
MEASURED_PEAKS.json; `roofline.other_kernels` = the same for the other raster kernel and each loss kernel.
`cpu_baseline` / `--impl reference` = the reference's own rasteriser code compiled for the host
(oracle/_ref, "reference") or our CPU restatement (oracle B, "port") on a bounded sample.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    # name: subdiv, image_size, batch per GPU, tex_res, losses ("st": silhouette + texture; "full": + texture-flow sampler,
    # distance-transform loss, texture-cycle loss (hard render) and chamfer correspondence -- BASELINE.json config 3)
    "C2": dict(subdiv=3, image_size=256, batch=16, tex_res=6, losses="st",
               desc="CUB-like 642v/1280f mesh, 256x256 render, batch 16/GPU, silhouette+texture loss"),
    "C3": dict(subdiv=3, image_size=512, batch=32, tex_res=6, losses="full",
               desc="CUB-like 642v/1280f mesh, 512x512 render, batch 32/GPU, silhouette+texture loss on textures sampled "
                    "from a texture flow + texture-dt + texture-cycle (hard renderer visibility) + chamfer correspondence"),
    "C5": dict(subdiv=4, image_size=1024, batch=8, tex_res=6, losses="st",
               desc="2562v/5120f mesh, 1024x1024 render, batch 8/GPU, silhouette+texture loss"),
}
NUM_SETS = 8  # rotating input sets so the step inputs exceed the 126 MB L2


def alg_bytes_per_image(image_size, F, T2):
    """SURVEY.md §8(d): compulsory fp32 traffic per rendered image at the soft_rasterize contract."""
    fwd = F * (44 + 12 * T2) + 48 * image_size * image_size
    bwd = 16 * image_size * image_size + F * (72 + 24 * T2)
    return fwd, bwd


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


# ------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 6:
                continue
            try:
                sm.append(float(p[0]))
                mx = float(p[1])
            except ValueError:
                continue
            for n, v in zip(names, p[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline (CPU; the ONLY place bench.py touches oracle/)
# ------------------------------------------------------------------------------------------------
def cpu_workload(cfg, batch, seed=0):
    import numpy as np
    from umr_b200 import synth
    rng = np.random.default_rng(seed)
    v, f = synth.icosphere(cfg["subdiv"])
    verts = synth.bird_like(v, rng, batch)
    cams = synth.cameras(rng, batch)
    fv = synth.raster_space_faces(verts, f, cams)
    tex = rng.uniform(0, 1, size=(batch, f.shape[0], cfg["tex_res"] ** 2, 3)).astype(np.float32)
    g = rng.normal(size=(batch, 4, cfg["image_size"], cfg["image_size"])).astype(np.float32)
    return fv, tex, g


def cpu_reference_step(cfg, fv, tex, g, impl, nthreads):
    """One fwd+bwd of the rasteriser core (prep + forward + 2x2 pool + backward) on the host."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import softras
    img, fwd, rc = softras.render(fv, tex, cfg["image_size"], anti_aliasing=True, impl=impl, nthreads=nthreads,
                                  aggr_func_rgb="softmax", sigma_val=1e-5, dist_eps=1e-10, gamma_val=1e-4)
    softras.render_backward(fwd, rc, g, anti_aliasing=True, impl=impl, nthreads=nthreads)
    return img


def cpu_arm(cfg, steps, warmup, budget_s=None):
    """Times the reference CPU path; returns (images_per_s, ms_per_step, info)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import softras
    impl, kind = ("A", "reference") if softras.have_oracle_a() else ("B", "port")
    # threads actually usable by this process (affinity mask and cgroup quota), not os.cpu_count(): on a shared box
    # the latter oversubscribes OpenMP and made the round-1 CPU arm swing 5.7x between boxes (VERDICT r1 #10)
    cores = softras.host_threads(cap=256)
    os.environ.setdefault("OMP_PROC_BIND", "close")
    sub = 2  # bounded sample: a 2-image sub-batch of the workload per step
    fv, tex, g = cpu_workload(cfg, sub)
    for _ in range(max(warmup, 1)):
        cpu_reference_step(cfg, fv, tex, g, impl, cores)
    t0 = time.perf_counter()
    done = 0
    for _ in range(steps):
        cpu_reference_step(cfg, fv, tex, g, impl, cores)
        done += 1
        if budget_s is not None and time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    ips = done * sub / dt
    info = {"value": ips, "unit": "images/s", "cores": cores, "kind": kind, "host_cpu_count": os.cpu_count(),
            "sample": "%d step(s) x %d-image sub-batch of %s, rasteriser core fwd+bwd (prep+forward+2x2 pool+"
                      "backward), OpenMP over the threads this process may use (affinity + cgroup quota)" % (done, sub, cfg["name"])}
    return ips, dt / done * 1e3, info


# ------------------------------------------------------------------------------------------------
# GPU workload
# ------------------------------------------------------------------------------------------------
class Workload:
    def __init__(self, cfg, device, rank, seed=0):
        import numpy as np
        import torch
        from umr_b200 import synth
        from umr_b200.nnutils import smr
        self.cfg, self.device = cfg, device
        B, IS, R = cfg["batch"], cfg["image_size"], cfg["tex_res"]
        v, f = synth.icosphere(cfg["subdiv"])
        self.V, self.F, self.T2 = v.shape[0], f.shape[0], R * R
        prng = np.random.default_rng(seed)            # shared parameters: identical on every rank
        base = synth.bird_like(v, prng, 1, noise=0.0)[0]
        self.mean_shape = torch.from_numpy(base).to(device).requires_grad_(True)
        self.texture = torch.from_numpy(prng.uniform(0, 1, size=(self.F, self.T2, 3)).astype(np.float32)
                                        ).to(device).requires_grad_(True)
        self.faces = torch.from_numpy(f.astype(np.int64)).to(device)[None].repeat(B, 1, 1)
        self.renderer = smr.SoftRenderer(IS, "softmax").to(device)
        self.renderer.ambient_light_only()  # like MultiTextureLoss (loss_utils.py:286)
        self.hard = smr.SoftRenderer(IS, "hard").to(device)
        self.full = cfg.get("losses") == "full"
        hard = self.hard
        rng = np.random.default_rng(1000 + rank)      # per-rank data shard
        self.host, self.dev = [], []
        for _ in range(NUM_SETS):
            delta = rng.normal(0, 0.02, size=(B, self.V, 3)).astype(np.float32)
            cams = synth.cameras(rng, B)
            imgs = synth.smooth_images(rng, B, IS)
            # GT mask = hard-render alpha > 0.5 of the same mesh under a perturbed camera (§8d)
            cams_gt = cams.copy()
            cams_gt[:, 0] *= rng.uniform(0.9, 1.1, size=B).astype(np.float32)
            cams_gt[:, 1:3] += rng.uniform(-0.05, 0.05, size=(B, 2)).astype(np.float32)
            with torch.no_grad():
                vv = self.mean_shape.detach()[None] + torch.from_numpy(delta).to(device)
                a, _, _ = hard(vv, self.faces, torch.from_numpy(cams_gt).to(device))
                masks = (a[:, 3] > 0.5).float().cpu()
            h = [torch.from_numpy(delta).pin_memory(), torch.from_numpy(cams).pin_memory(),
                 torch.from_numpy(imgs).pin_memory(), masks.pin_memory()]
            if self.full:  # §8d: texture flow, barrier distance transform of the GT mask, 2-D part points
                flow = synth.texture_flow(rng, B, self.F, R)
                dts = np.stack([synth.dt_barrier(m) for m in masks.numpy()])[:, None].astype(np.float32)
                pts = synth.part_points(rng, B)
                h += [torch.from_numpy(flow).pin_memory(), torch.from_numpy(dts).pin_memory()]
                h += [torch.from_numpy(p).pin_memory() for p in pts]
            self.host.append(h)
            self.dev.append([t.to(device) for t in h])
        self.h2d_bytes = sum(t.numel() * t.element_size() for t in self.host[0])
        from umr_b200.dist import FlatGradAllReduce
        shared = [self.mean_shape] if self.full else [self.mean_shape, self.texture]
        self.reducer = FlatGradAllReduce(shared, average=True, backend=os.environ.get("UMR_ALLREDUCE", "auto"))
        self.reduce_in_graph = self.reducer.backend in ("p2p", "none")
        if self.full:
            from umr_b200.nnutils import loss_utils
            self.flow = torch.zeros(B, self.F, R, R, 2, device=device, requires_grad=True)  # per-image texture flow (leaf)
            self.tex_cycle = loss_utils.TexCycle()
            self.corr = loss_utils.CorrLossChamfer(None, IS, part_vertices=[
                torch.from_numpy(p) for p in synth.part_vertex_sets(np.random.default_rng(7), self.V)])
        self.stage = [torch.empty_like(t, device=device) for t in self.host[0]]
        self.stage2 = None

    def step(self, inputs, world, reduce=True):
        import torch
        from umr_b200.nnutils import geom_utils, loss_utils
        delta, cams, imgs, masks = inputs[:4]
        self.reducer.zero_grads()         # .grad of the shared parameters are views of ONE flat buffer (no pack/unpack)
        verts = self.mean_shape[None] + delta
        if not self.full:
            tex = self.texture[None]      # [1,F,T2,3]: batch-shared texture parameter (no repeat(B) copies)
        else:
            # per-image textures sampled from the texture flow (geom_utils.py:41-59; train_s2.py:236-242)
            flow_in, dts = inputs[4], inputs[5]
            self.flow.grad = None
            with torch.no_grad():
                self.flow.copy_(flow_in)
            tex = geom_utils.sample_textures(self.flow, imgs).view(delta.shape[0], self.F, self.T2, 3)
        images, _, _ = self.renderer(verts, self.faces, cams, tex)
        # 2.5 * neg_iou_loss(alpha, masks) + 3.0 * texture_loss_masks(rgb, imgs, masks, alpha) (train_s2.py:49-59 weights),
        # fused: one reduction forward, one kernel backward (tests/test_losses_gpu.py checks it against the composition)
        loss = loss_utils.mask_texture_loss(images, imgs, masks, 2.5, 3.0)
        if self.full:
            # + 3.0 * texture_dt_loss + 1.0 * TexCycle (visibility from the HARD render, loss_utils.py:327-329)
            #   + 10.0 * CorrLossChamfer on the mean shape (train_s2.py:49-59 weights, :297-316)
            loss = loss + 3.0 * loss_utils.texture_dt_loss(self.flow, dts)
            p2f, visible = self.hard.visible_faces(verts.detach(), self.faces, cams)   # as MultiTextureLoss does (image dropped)
            cyc, _ = self.tex_cycle(self.flow, p2f, None, visible=visible)
            head, belly, neck, back = inputs[6:10]
            ms = self.mean_shape[None].expand(delta.shape[0], -1, -1)
            corr, _ = self.corr(head, belly, back, neck, ms, cams)   # (argument order as train_s2.py:311 passes them)
            loss = loss + 1.0 * cyc + 10.0 * corr
        loss.backward()
        # N>1: ONE all-reduce of the flat shared-parameter gradient (SURVEY.md §8e).  Our p2p kernel is a plain kernel and
        # lives inside the captured graph; an NCCL fallback is issued after the replay (finish()).
        if reduce or self.reduce_in_graph:
            self.reducer.reduce()
        # what a caller of the step receives: the loss, the rendered images and the gradients of the trained tensors.
        # Detached: a returned tensor that kept this step's autograd graph alive would break the next graph capture.
        out = {"loss": loss.detach(), "images": images.detach(), "grad_mean_shape": self.mean_shape.grad}
        if self.full:
            out["grad_texture_flow"] = self.flow.grad
        else:
            out["grad_texture"] = self.texture.grad
        return out

    def finish(self):
        """The part of a step that stays outside the CUDA graph: only the NCCL fallback of the all-reduce."""
        if not self.reduce_in_graph:
            self.reducer.reduce()

    def step_resident(self, i, world):
        return self.step(self.dev[i % NUM_SETS], world)

    def step_e2e(self, i, world):
        """Eager e2e step, same prefetch pipeline as gstep_e2e (H2D of step i+1 under the compute of step i)."""
        import torch
        if self.stage2 is None:
            self._init_e2e_pipeline()
        cur = torch.cuda.current_stream()
        if self._e2e_next is None:
            self._prefetch(i, cur)
        k = i % 2
        cur.wait_event(self._copied[k])
        out = self.step(self.stage2[k], world)
        self._consumed[k].record(cur)
        self._prefetch(i + 1, cur)
        float(out["loss"].item())                    # D2H read of the step's result
        return out

    def _init_e2e_pipeline(self):
        import torch
        self.stage2 = [self.stage, [torch.empty_like(t) for t in self.stage]]
        self._copy_stream = torch.cuda.Stream()
        self._copied = [torch.cuda.Event(), torch.cuda.Event()]
        self._consumed = [torch.cuda.Event(), torch.cuda.Event()]
        for e in self._consumed:
            e.record(torch.cuda.current_stream())
        self._e2e_next = None

    # ---- CUDA-graph variants: the same step(), captured once per static input buffer set ----------
    def capture(self, world):
        from umr_b200.graph import GraphedStep
        self.g_res = []
        pool = None
        for i in range(NUM_SETS):
            g = GraphedStep(lambda i=i: self.step(self.dev[i], world, reduce=False), warmup=2 if i == 0 else 1, pool=pool)
            pool = g.pool()
            self.g_res.append(g)
        if self.stage2 is None:
            self._init_e2e_pipeline()
        self.g_e2e2 = [GraphedStep(lambda k=k: self.step(self.stage2[k], world, reduce=False), warmup=1, pool=pool)
                       for k in (0, 1)]

    def gstep_resident(self, i, world):
        out = self.g_res[i % NUM_SETS]()
        self.finish()
        return out

    def gstep_e2e(self, i, world):
        """e2e step with the H2D copy of step i+1 overlapped with the compute of step i: two static staging
        buffer sets (one captured graph each), a copy stream, and events in both directions.  Every step's
        inputs still come from pinned host memory and every step's loss is still read back, all inside the
        timed region -- this is what a prefetching data loader does."""
        import torch
        cur = torch.cuda.current_stream()
        if self._e2e_next is None:                       # first step of a run: nothing prefetched yet
            self._prefetch(i, cur)
        k = i % 2
        cur.wait_event(self._copied[k])                  # inputs of step i have landed in stage set k
        out = self.g_e2e2[k]()
        self._consumed[k].record(cur)                    # stage set k may be overwritten after this point
        self.finish()
        self._prefetch(i + 1, cur)                       # H2D of step i+1 runs under the compute of step i
        float(out["loss"].item())                        # D2H read of the step's result (syncs this stream)
        return out

    def _prefetch(self, i, cur):
        import torch
        k = i % 2
        h = self.host[i % NUM_SETS]
        with torch.cuda.stream(self._copy_stream):
            self._copy_stream.wait_event(self._consumed[k])
            for s, t in zip(self.stage2[k], h):
                s.copy_(t, non_blocking=True)
            self._copied[k].record(self._copy_stream)
        self._e2e_next = i

    def reset_e2e(self):
        self._e2e_next = None


def _graph_time_ms(fn, iters=20):
    """Device time of one call of fn(): `iters` calls captured in ONE CUDA graph (no host launch gaps), replayed and
    timed with CUDA events on the launching stream."""
    import torch
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, capture_error_mode="thread_local"):
        for _ in range(iters):
            fn()
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def other_kernel_rooflines(cfg, F, T2, peak, device, face_ids=None):
    """Achieved HBM GB/s of every loss kernel at this config's sizes: algorithmic bytes (SURVEY.md §8d per-unit figures x
    units per launch, listed per entry) / device time of the launch(es), measured live with CUDA events."""
    import torch
    from umr_b200 import ops
    from umr_b200.nnutils import chamfer_python
    B, IS = cfg["batch"], cfg["image_size"]
    R = int(round(T2 ** 0.5))
    g = torch.Generator(device=device).manual_seed(3)
    rnd = lambda *sh: torch.rand(*sh, device=device, generator=g)
    imgs, rgba = rnd(B, 3, IS, IS), rnd(B, 4, IS, IS)
    masks = (rnd(B, IS, IS) > 0.5).float()
    flow = (rnd(B, F, R, R, 2) * 1.8 - 0.9)
    dts = rnd(B, 1, IS, IS)
    out = []

    def add(name, fn, nbytes, what):
        try:
            ms = _graph_time_ms(fn)
            gbs = nbytes / (ms * 1e-3) / 1e9
            out.append({"kernel": name, "kernel_ms": ms, "alg_bytes_per_launch": int(nbytes), "achieved": gbs,
                        "frac": gbs / peak if peak else None, "bytes": what})
        except Exception as ex:  # never let a side measurement break the headline
            out.append({"kernel": name, "error": repr(ex)})

    N = F * T2
    fl = flow.reshape(B, N, 2)
    add("k_sample_fwd<3> (sample_textures)", lambda: ops.BilinearSampleFunction.apply(imgs, fl),
        B * (N * (8 + 12) + 12 * IS * IS), "B*(F*T2*(8+12) + 12*is^2)")
    # backward kernels are timed through the C ABI directly (autograd inside a capture is not capture-safe everywhere)
    import ctypes
    from umr_b200 import _lib
    lib = _lib.load()
    vp = lambda t: ctypes.c_void_p(t.data_ptr())
    stream = lambda: ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    go, gfl = rnd(B, N, 3), torch.empty(B, N, 2, device=device)
    add("k_sample_bwd<3>", lambda: _lib.check(lib.umr_bilinear_sample_backward(vp(imgs), vp(fl), vp(go), vp(gfl), None, B, 3, IS, IS,
                                                                               N, stream()), "sample_bwd"),
        B * N * (12 + 8 + 8), "B*F*T2*(12+8+8)")
    add("k_sample_fwd<1> (texture_dt_loss)", lambda: ops.BilinearSampleFunction.apply(dts, fl),
        B * (N * (8 + 4) + 4 * IS * IS), "B*(F*T2*(8+4) + 4*is^2)")
    add("k_losshead_partial+finalize (IoU + masked L1)", lambda: ops.mask_texture_loss(rgba, imgs, masks, 2.5, 3.0),
        B * IS * IS * (16 + 12 + 4), "B*is^2*(16+12+4)")
    stats, per_img, lossv = torch.empty(B, 3, device=device), torch.empty(B, 2, device=device), torch.empty(1, device=device)
    _lib.check(lib.umr_loss_head_forward(vp(rgba), vp(imgs), vp(masks), vp(stats), vp(per_img), vp(lossv), B, IS * IS, 2.5, 3.0,
                                         stream()), "loss_head_forward")
    gl, grgba = torch.ones(1, device=device), torch.empty_like(rgba)
    add("k_losshead_bwd", lambda: _lib.check(lib.umr_loss_head_backward(vp(rgba), vp(imgs), vp(masks), vp(stats), vp(gl), vp(grgba),
                                                                       B, IS * IS, 2.5, 3.0, stream()), "loss_head_backward"),
        B * IS * IS * (16 + 12 + 4 + 16), "B*is^2*(16+12+4 read + 16 written)")
    add("k_iou_partial+finalize (neg_iou_loss)", lambda: ops.neg_iou_per_image(rgba[:, 3], masks), B * IS * IS * 8, "B*is^2*(4+4)")
    # face-id plane of a real hard render (piecewise constant, as the kernel meets it in MultiTextureLoss)
    ids = face_ids if face_ids is not None else torch.full((B, 4 * IS * IS), -1.0, device=device)
    p2f = rnd(B, F, 2)
    add("k_visible+k_texcycle_fwd (TexCycle)", lambda: ops.tex_cycle(flow.reshape(B, F, T2, 2), p2f, ids),
        B * (4 * IS * IS * 4 + F * T2 * 8), "B*(S^2*4 + F*T2*8)")
    for nm, (cb, n, m) in (("train 128x[40 x 10]", (128, 40, 10)), ("train 128x[80 x 30]", (128, 80, 30)),
                           ("eval 1x[20000 x 642] (test_kp.py:180)", (1, 20000, 642))):
        a, b = rnd(cb, n, 2) - 0.5, rnd(cb, m, 2) - 0.5
        add("k_chamfer_nn<2> x2 (distChamfer, %s)" % nm, lambda a=a, b=b: chamfer_python.distChamfer(a, b),
            cb * (n + m) * (8 + 4 + 4), "B*(N+M)*(8+4+4)")
    return out


def reference_gpu_leg(cfg, ours_fwd_ms, ours_bwd_ms):
    """The reference's OWN CUDA kernels rebuilt for sm_100a (baseline/_ref, built by baseline/build_ref_gpu.py in the
    build container; absent -> None) timed on the same GPU at this config: the GPU "kernel to beat" (SURVEY.md §8d)."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    try:
        import ref_gpu_compare as rc
    except Exception:
        return None
    mod = rc.load("soft_rasterize_ref")
    if mod is None:
        return None
    B, IS = cfg["batch"], cfg["image_size"]
    S = 2 * IS
    fv, tex = rc.scene(B, cfg["tex_res"], seed=0, subdiv=cfg["subdiv"])
    ghi = torch.randn(B, 4, S, S, device="cuda")
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    tf = tb = 0.0
    n = 3
    for it in range(n + 1):
        ev[0].record()
        colors, _, aggr, finfo = rc.ref_forward(mod, fv, tex, S, 1)
        ev[1].record()
        rc.ref_backward(mod, fv, tex, colors, finfo, aggr, ghi, S, 1)
        ev[2].record()
        torch.cuda.synchronize()
        if it:  # first pass = warm-up
            tf += ev[0].elapsed_time(ev[1])
            tb += ev[1].elapsed_time(ev[2])
    tf, tb = tf / n, tb / n
    return {"what": "reference soft_rasterize CUDA kernels (external/SoftRas, rebuilt for sm_100a, default nvcc flags) incl. "
                    "the host-side buffer fills of functional/soft_rasterize.py:47-62 done on the device, same mesh/batch",
            "fwd_ms": tf, "bwd_ms": tb, "images_per_s": B / ((tf + tb) * 1e-3),
            "ours_raster_kernels_ms": [ours_fwd_ms, ours_bwd_ms],
            "speedup_raster_kernels": (tf + tb) / (ours_fwd_ms + ours_bwd_ms) if ours_fwd_ms + ours_bwd_ms > 0 else None}


DUMP_MAX_VALUES = 4 << 20  # per array: at most 4 arrays x 16 MB of float32 in one dump


def write_outputs(path, outputs):
    """Writes each output as <path>/<name>.npy (float32).  An array of more than DUMP_MAX_VALUES values is replaced by
    the values at DUMP_MAX_VALUES positions of its flattened form, drawn with a fixed seed, in ascending order, so
    two runs with the same arguments write the same positions.  Returns {name: {"shape", "stored"}}."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    info = {}
    for name, a in outputs.items():
        stored = a
        if a.size > DUMP_MAX_VALUES:
            idx = np.sort(np.random.default_rng(0).choice(a.size, DUMP_MAX_VALUES, replace=False))
            stored = a.ravel()[idx]
        np.save(os.path.join(path, name + ".npy"), stored.astype(np.float32))
        info[name] = {"shape": list(a.shape), "stored": "all" if stored is a else "%d sampled values" % stored.size}
    return info


def run_gpu(args, cfg):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        import datetime
        # a rank that dies must fail the job quickly instead of leaving the others in a collective
        dist.init_process_group("nccl", device_id=device, timeout=datetime.timedelta(seconds=180))
    from umr_b200 import _lib, raster
    lib = _lib.load()
    torch.manual_seed(0)
    wl = Workload(cfg, device, rank)
    K, W = args.steps, max(args.warmup, 3)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, profile=False):
        for i in range(W):
            fn(i, world)
        barrier()
        sampler = ClockSampler(local) if rank == 0 else None
        if sampler:
            sampler.start()
        l0 = lib.umr_launch_count()
        sink = [] if profile else None
        raster.set_profile_sink(sink)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(K):
            out = fn(W + i, world)
        e1.record()
        barrier()
        raster.set_profile_sink(None)
        ms = e0.elapsed_time(e1)
        launches = lib.umr_launch_count() - l0
        clocks = sampler.stop() if sampler else None
        if dist is not None:
            t = torch.tensor([ms], device=device, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, launches, clocks, sink, out

    # The captured graph holds everything of the step EXCEPT the NCCL all-reduce (capturing the collective
    # hung at N=8 in testing); the collective and the scatter back into .grad are issued after each replay.
    use_graph = not args.no_graph
    # eager pass: also records the raster kernels' own durations through the C-ABI event hooks
    ms_eager, launches, clocks_eager, sink, last = timed(wl.step_resident, profile=True)
    kern = raster.collect_profile(sink)  # {"fwd": [ms...], "bwd": [ms...]}
    if use_graph:
        wl.capture(world)
        ms_res, _, clocks, _, last = timed(wl.gstep_resident)
    else:
        ms_res, clocks = ms_eager, clocks_eager
    # the outputs of the last step of the pass `value` is measured on, copied before the next pass overwrites them
    outputs = {k: v.detach().float().cpu().numpy() for k, v in last.items()} if args.dump_outputs else None
    wl.reset_e2e()
    ms_e2e, _, clocks_e2e, _, _ = timed(wl.gstep_e2e if use_graph else wl.step_e2e)

    B = cfg["batch"]
    total_images = B * world * K
    value = total_images / (ms_res * 1e-3)
    e2e = total_images / (ms_e2e * 1e-3)
    fwd_b, bwd_b = alg_bytes_per_image(cfg["image_size"], wl.F, wl.T2)
    peak, peak_src = measured_peak_gbs()
    bwd_ms = sum(kern["bwd"]) / max(len(kern["bwd"]), 1)
    fwd_ms = sum(kern["fwd"]) / max(len(kern["fwd"]), 1)
    achieved = (bwd_b * B) / (bwd_ms * 1e-3) / 1e9 if bwd_ms > 0 else 0.0
    fwd_achieved = (fwd_b * B) / (fwd_ms * 1e-3) / 1e9 if fwd_ms > 0 else 0.0

    tj = {}
    try:  # dram bytes per launch from the committed `ncu --set full` captures (profiles/traffic.json)
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f).get(cfg["name"], {})
    except Exception:
        tj = {}
    rast = [{"kernel": "k_raster_fwd3<softmax> (forward: binned per-pixel raster + pair-record emission)", "kernel_ms": fwd_ms,
             "alg_bytes_per_launch": fwd_b * B, "achieved": fwd_achieved, "frac": fwd_achieved / peak if peak else None,
             "traffic": tj.get("k_raster_fwd3")},
            {"kernel": "k_raster_bwd2<softmax,texgrad> (+ k_raster_bwd_pairs_list fallback; streamed backward)",
             "kernel_ms": bwd_ms, "alg_bytes_per_launch": bwd_b * B, "achieved": achieved,
             "frac": achieved / peak if peak else None, "traffic": tj.get("k_raster_bwd2")}]
    rast.sort(key=lambda r: -r["kernel_ms"])
    dom = rast[0]
    others = rast[1:]
    if rank == 0 and world == 1 and not args.no_other_kernels:
        with torch.no_grad():
            d0 = wl.dev[0]
            _, _, aggr = wl.hard(wl.mean_shape.detach()[None] + d0[0], wl.faces, d0[1])
        others += other_kernel_rooflines(cfg, wl.F, wl.T2, peak, device, aggr[:, 1].reshape(B, -1).contiguous())
    out = {
        "metric": "render fwd+bwd images/sec @256x256 1280-face mesh" if cfg["name"] == "C2"
        else "render fwd+bwd images/sec (%s)" % cfg["name"],
        "value": value, "unit": "images/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_res / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "%s: %s" % (cfg["name"], cfg["desc"]), "global_batch": B * world,
                   "image_size": cfg["image_size"], "raster_size": 2 * cfg["image_size"], "faces": wl.F,
                   "vertices": wl.V, "texture_res": cfg["tex_res"], "parallelism": "dp%d" % world,
                   "l2": "inputs rotate over %d pre-generated batches (> 126 MB L2 together with the per-step "
                         "buffers)" % NUM_SETS,
                   "cuda_graph": use_graph, "eager_ms_per_step": ms_eager / K,
                   "allreduce": {"none": "single process", "p2p": "own one-shot kernel over NVLink peer memory "
                                 "(umr_p2p_allreduce), inside the captured graph", "nccl": "ncclAllReduce(AVG) issued after "
                                 "each graph replay"}.get(wl.reducer.backend, wl.reducer.backend)},
        "e2e": {"value": e2e, "unit": "images/s", "h2d_bytes_per_step": wl.h2d_bytes, "d2h_bytes_per_step": 4,
                "ms_per_step": ms_e2e / K,
                "pipeline": "H2D of step i+1 (copy stream, pinned memory) overlaps the graph replay of step i; "
                            "loss.item() every step" if use_graph else
                            "H2D of step i+1 (copy stream, pinned memory) overlaps the eager step i; loss.item() every step"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": {"bound": "hbm", "kernel": dom["kernel"], "achieved": dom["achieved"], "peak": peak, "unit": "GB/s",
                     "frac": dom["frac"], "traffic": dom["traffic"], "peak_source": peak_src, "kernel_ms": dom["kernel_ms"],
                     "timing": "CUDA events recorded by the C ABI around the kernel launch, %d eager steps of the same "
                               "workload inside this run" % K,
                     "alg_bytes_per_launch": dom["alg_bytes_per_launch"],
                     "whole_step": {"alg_bytes": (fwd_b + bwd_b) * B, "achieved": (fwd_b + bwd_b) * B / (ms_res / K * 1e-3) / 1e9,
                                    "frac": (fwd_b + bwd_b) * B / (ms_res / K * 1e-3) / 1e9 / peak if peak else None},
                     "other_kernels": others},
    }
    if rank == 0 and outputs is not None:
        out["dump_outputs"] = write_outputs(args.dump_outputs, outputs)
    if rank == 0 and world == 1 and not args.no_reference_gpu:
        try:
            out["reference_gpu"] = reference_gpu_leg(cfg, fwd_ms, bwd_ms)
        except Exception as ex:
            out["reference_gpu"] = {"error": repr(ex)}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            _, _, info = cpu_arm(cfg, steps=64, warmup=1, budget_s=12.0)
            out["cpu_baseline"] = info
        except Exception as ex:  # the oracle is test infrastructure; never let it break the GPU number
            out["cpu_baseline"] = {"value": None, "error": repr(ex)}
    if rank == 0:
        print(json.dumps(out))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def run_reference(args, cfg):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return  # the CPU arm runs on rank 0 only; other ranks exit 0 without work
    ips, ms, info = cpu_arm(cfg, steps=args.steps, warmup=max(args.warmup, 1))
    fwd_b, bwd_b = alg_bytes_per_image(cfg["image_size"], 20 * 4 ** cfg["subdiv"], cfg["tex_res"] ** 2)
    out = {"impl": "reference",
           "metric": "render fwd+bwd images/sec @256x256 1280-face mesh" if cfg["name"] == "C2"
           else "render fwd+bwd images/sec (%s)" % cfg["name"],
           "value": ips, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 1),
           "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
           "data": "synthetic",
           "config": {"workload": "%s: %s" % (cfg["name"], cfg["desc"]), "note": "CPU arm: each step is a bounded "
                      "2-image sample of the workload (the reference has no CPU path of its own; this is its "
                      "rasteriser code compiled for the host, or our restatement when that is unavailable)"},
           "cpu_baseline": info,
           "e2e": {"value": ips, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 400; 8 with --impl reference)")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C2", choices=sorted(CONFIGS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-kernels", action="store_true", help="skip the loss-kernel roofline lines")
    ap.add_argument("--no-reference-gpu", action="store_true", help="skip timing baseline/_ref (the reference's CUDA kernels)")
    ap.add_argument("--no-graph", action="store_true", help="time the eager step instead of its CUDA-graph replay")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the loss, images and gradients of the last timed step "
                    "as DIR/<name>.npy (float32; arrays above %d values as a fixed seeded sample)" % DUMP_MAX_VALUES)
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 8 if args.impl == "reference" else 400  # each CPU step of the reference arm takes ~1 s
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU path only")
    cfg = dict(CONFIGS[args.config], name=args.config)
    if args.impl == "reference":
        run_reference(args, cfg)
    else:
        run_gpu(args, cfg)


if __name__ == "__main__":
    main()
