#!/usr/bin/env python
"""Benchmark of the perturbed shading hot path (BASELINE.json metric:
"perturbed shader fwd+bwd pixel·face·samples/sec; % HBM roofline; 1/2/4/8 GPU").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--fragments rasterised|realistic|dense] [--impl reference]
                    [--dump-outputs DIR]

A step is one fused forward + one fused backward of the shader over one batch of fragments at BASELINE config 2 per GPU
(8 views, 256x256, K=50, nb_samples=64; weak scaling: every rank shades its own 8 views, the only collective on the path
is the all-reduce of the three scalar gradients).  The headline fragment set is an ACTUAL rasterisation (SURVEY.md §8d:
"valid count per covered pixel from a real rasterisation if available"): the 1280-face icosphere of the reference's
experiments seen by 8 orbiting cameras, 35 valid entries per covered pixel.  The SURVEY's synthetic sets (realistic = mean 4
valid entries, dense = all 50), every other BASELINE config, both shardings, the Philox4x32-7 and per-sample-noise modes,
the SoftRas pair, the Phong shader, the whole renderer, the reference on this GPU and peak memory are in `also`.
Prints ONE JSON line (rank 0).  See DESIGN.md §Measurement for every field.
"""

from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time
import types

import torch

# the benchmark writes nothing into the source tree (which may be read-only), bytecode caches included
sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "perturbed shader fwd+bwd pixel·face·samples/sec"
UNIT = "pixel·face·samples/s"
SIGMA, GAMMA, ALPHA, EPS = 1e-3, 1e-2, 1.0, 1e-10  # experiments/eval.py:69 defaults (SURVEY.md §8d)
BACKGROUND = (1.0, 1.0, 1.0)
DUMP_BYTES = 60_000_000  # --dump-outputs writes at most this much (under 64 MB with the .npy headers)

# BASELINE.json configs (per-GPU shapes; SURVEY.md §8 table).  Config 3 is 64 poses sharded by batch over 8 GPUs: 8 per GPU.
CONFIGS = {
    1: dict(N=1, HW=64, K=50, S=16, name="config 1: 1 view x 64x64, K=50, nb_samples=16"),
    2: dict(N=8, HW=256, K=50, S=64, name="config 2: 8 views x 256x256, K=50, nb_samples=64"),
    3: dict(N=8, HW=512, K=100, S=256, name="config 3 per-GPU share: 8 of 64 poses x 512x512, K=100, nb_samples=256"),
    4: dict(N=1, HW=128, K=50, S=4096, name="config 4: 1 view x 128x128, K=50, nb_samples=4096"),
    5: dict(N=16, HW=1024, K=50, S=32, name="config 5: 16 views x 1024x1024, K=50, nb_samples=32"),
}

_REAL_STDOUT = None


def quiet_stdout():
    """stdout must carry exactly ONE JSON line.  Libraries write banners to the C-level stdout (NCCL prints its
    version there whatever NCCL_DEBUG_FILE says), so file descriptor 1 is pointed at stderr for the whole run and the
    JSON line goes to a private duplicate of the original stdout."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--fragments", default="rasterised", choices=["rasterised", "realistic", "dense"])
    ap.add_argument("--views", type=int, default=CONFIGS[2]["N"])
    ap.add_argument("--image-size", type=int, default=CONFIGS[2]["HW"])
    ap.add_argument("--faces-per-pixel", type=int, default=CONFIGS[2]["K"])
    ap.add_argument("--nb-samples", type=int, default=CONFIGS[2]["S"])
    ap.add_argument("--no-also", action="store_true", help="headline only")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-renderer-legs", action="store_true", help="skip the Phong / renderer legs of `also`")
    ap.add_argument("--no-config-legs", action="store_true", help="skip BASELINE configs 1, 3, 4, 5 in `also`")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (float32; a fixed sample of pixels "
                         "when the whole would exceed 60 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def measured_traffic(kernel, kind, N, HW, K, S):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` (main + fallback pass) from the committed
    ncu --set full capture of THIS workload (profiles/traffic.json, written from the .ncu-rep by
    profiles/ncu_summary.py); None when this workload was not captured."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(p))[f"{kind}:{N}x{HW}x{K}x{S}"][kernel]
    except Exception:
        return None


def measured_issue(kind, N, HW, K, S):
    """Issue-slot utilisation (smsp__issue_active, % of peak) and ncu duration of every kernel of the step from the same
    committed capture: the number that says how close the kernels are to the resource that actually binds them."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(p))[f"{kind}:{N}x{HW}x{K}x{S}"]["kernels"]
    except Exception:
        return None


def alg_bytes(P, K):
    """SURVEY.md §8d, API-faithful: fwd reads pix_to_face 8 + zbuf 4 + dists 4 + colors 12 per pixel·face and writes RGBA
    16 per pixel; bwd re-reads the same 28, writes grad_dists 4 + grad_zbuf 4 + grad_colors 12 and reads grad_image 16 per
    pixel."""
    PF = P * K
    return 28 * PF + 16 * P, 48 * PF + 16 * P


def min_bytes(P, K, V):
    """Bytes the kernels cannot avoid on fragments with V valid entries (padding is never read beyond the pix_to_face
    scan): fwd = scan 8 PF + 20 per valid entry + image; bwd = the scan (8 PF; the tile blob replaces it on sparse tiles)
    + 28 per valid entry + the zero-fill of the three gradient tensors (20 PF, mandatory writes) + grad_image."""
    PF = P * K
    return 8 * PF + 20 * V + 16 * P, 8 * PF + 28 * V + 20 * PF + 16 * P


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons (NVML) while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self._halt = index, [], set(), None, threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._halt.wait(0.002)

    def finish(self):
        self._halt.set()
        if self.is_alive():
            self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------------------------------------------------
# fragment sets
# ------------------------------------------------------------------------------------------------
def rasterised_fragments(args, dev, rank=0):
    """Fragments of an ACTUAL rasterisation at the benchmark shapes: the 1280-face icosphere (sphere_642.obj of
    experiments/eval.py:289) seen by N orbiting cameras (dist 2.7, fov 60), blur_radius = log(1/1e-4 - 1) * sigma
    (eval.py:137), produced by pert_rasterize_fwd; texels = per-face colours gathered through pix_to_face."""
    import math
    import pertrenderer_b200 as pb
    N, HW, K = args.views, args.image_size, args.faces_per_pixel
    verts, faces = pb.synthetic_mesh(1280, device=dev)
    R, T = pb.look_at_view_transform(dist=2.7, elev=30.0, azim=torch.linspace(0, 315, N) + 7.0 * rank, device=dev)
    cam = pb.OpenGLPerspectiveCameras(R=R, T=T, device=dev)
    rast = pb.MeshRasterizer(cam, pb.RasterizationSettings(image_size=HW, blur_radius=math.log(1.0 / 1e-4 - 1.0) * SIGMA,
                                                           faces_per_pixel=K))
    with torch.no_grad():
        fr = rast(pb.TriMeshes(verts, faces).extend(N))
    fc = torch.rand((N * faces.shape[0], 3), device=dev, generator=torch.Generator(device=dev).manual_seed(7))
    col = pb.FaceTexels(fc).materialize(fr.pix_to_face)
    return fr, col.contiguous()


def make_fragments(kind, N, HW, K, S, dev, rank=0):
    from pertrenderer_b200 import synthetic_fragments
    if kind == "rasterised":
        fr, col = rasterised_fragments(types.SimpleNamespace(views=N, image_size=HW, faces_per_pixel=K, nb_samples=S), dev, rank)
        return fr, col
    return synthetic_fragments(N, HW, HW, K, kind=kind, sigma=SIGMA, seed=rank, device=dev)


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline
# ------------------------------------------------------------------------------------------------
def _reference_step(device, side, K, S, kind):
    """One forward+backward of the reference's RandomSimpleShader(GaussianRast, GaussianAgg) on a side x side pixel crop of
    the workload.  Uses the UNMODIFIED reference from oracle/_ref when it was installed (oracle/build_ref.py), else the
    oracle port.  Returns (callable, kind-string)."""
    from oracle import ref_loader as R
    from pertrenderer_b200 import synthetic_fragments
    # the reference's cost depends on tensor SIZES only (dense ops over (S,N,H,W,K)), so the synthetic set of the same shape
    # stands for every fragment set, and pixels are independent: units/s of the crop extrapolates to the whole job
    fr, col = synthetic_fragments(1, side, side, K, kind="realistic" if kind == "rasterised" else kind, sigma=SIGMA, seed=0,
                                  device="cpu")
    G = torch.randn((1, side, side, 4), generator=torch.Generator().manual_seed(1)).to(device)
    p2f, zbuf, dists, col = (t.to(device) for t in (fr.pix_to_face, fr.zbuf, fr.dists, col))
    mods = R.load()
    if mods is not None:
        rr, sr, sa = mods
        shader = rr.RandomSimpleShader(device=device, cameras=R.Cameras(torch.ones(1, device=device), 100.0 * torch.ones(1, device=device)),
                                       smoothrast=sr.GaussianRast(nb_samples=S, sigma=SIGMA),
                                       smoothagg=sa.GaussianAgg(nb_samples=S, gamma=GAMMA, alpha=ALPHA),
                                       blend_params=R.Blend(1e-4, 1e-4, BACKGROUND))

        def one():
            d, z, c = (t.detach().clone().requires_grad_(True) for t in (dists, zbuf, col))
            img = shader(R.Fragments(p2f, z, None, d), R.Texels(c))
            (img * G).sum().backward()
            return img
        return one, "reference"
    from oracle import pert_oracle as O

    def one_port():
        U, V = O.draw_noise((1, side, side, K), S, S)  # the reference draws its noise inside forward
        st, _ = O.shade_fwd_bwd(p2f, zbuf, dists, col, BACKGROUND, 1.0, 100.0, SIGMA, GAMMA, ALPHA, EPS, U, V, G)
        return st.image
    return one_port, "port"


def cpu_reference_run(args, steps, warmup, budget_s=25.0):
    """Times the reference's CPU implementation of the path on a bounded pixel crop of the same workload, with every host
    thread torch can use."""
    K, S = args.faces_per_pixel, args.nb_samples
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    side = 96  # 9216 pixels: ~0.4 GB per (S,N,H,W,K) temporary at K=50, S=64; the reference keeps ~10 alive
    one, kind = _reference_step("cpu", side, K, S, args.fragments)
    units = side * side * K * S
    t_start = time.perf_counter()
    for _ in range(warmup):
        one()
        if time.perf_counter() - t_start > budget_s / 2:
            break
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        one()
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_start > budget_s and len(times) >= 2:
            break
    t = sum(times) / len(times)
    what = "unmodified randomras from oracle/_ref" if kind == "reference" else "oracle port of randomras (oracle/pert_oracle.py)"
    return {"value": units / t, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": f"1 x {side}x{side} pixel crop, K={K}, S={S}: RandomSimpleShader(GaussianRast, GaussianAgg) fwd+bwd incl. "
                      f"its noise draws, {what}, mean of {len(times)} runs, torch CPU {torch.get_num_threads()} threads",
            "ms_per_step": t * 1e3, "steps_run": len(times), "side": side}


def reference_cuda_run(args, dev):
    """The reference's own ATen op chain on THIS GPU (the "before" number SURVEY §0.1 / §8d names): one view of the
    workload (the reference keeps ~40 B per pixel·face·sample alive, so the whole batch does not fit its memory model)."""
    K, S = args.faces_per_pixel, args.nb_samples
    side = min(args.image_size, 256)
    one, kind = _reference_step(dev, side, K, S, args.fragments)
    for _ in range(2):
        one()
    torch.cuda.synchronize(dev)
    torch.cuda.reset_peak_memory_stats(dev)
    base = torch.cuda.memory_allocated(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 5
    e0.record()
    for _ in range(n):
        one()
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / n
    units = side * side * K * S
    return {"kind": kind + " (torch CUDA ops on this GPU)", "value": units / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms,
            "sample": f"1 x {side}x{side} pixels, K={K}, S={S}, fwd+bwd incl. noise draws, mean of {n}",
            "peak_memory_bytes": int(torch.cuda.max_memory_allocated(dev) - base),
            "peak_memory_bytes_per_unit": (torch.cuda.max_memory_allocated(dev) - base) / units}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cb = cpu_reference_run(args, max(args.steps, 2), max(args.warmup, 1), budget_s=120.0)
    side = cb["side"]
    line = {
        "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": cb["steps_run"], "warmup": args.warmup, "ms_per_step": cb["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {**workload_config(args, 1),
                   "timed_sample": f"each step = 1 x {side}x{side} pixel crop of that workload ({side * side} of "
                                   f"{args.views * args.image_size ** 2} pixels; pixels are independent, units/s extrapolates); "
                                   "ms_per_step is the time of that crop"},
        "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def workload_config(args, world):
    inputs_gb = args.views * args.image_size ** 2 * args.faces_per_pixel * 28 / 1e9
    return {
        "workload": f"BASELINE config 2 per GPU: {args.views} views x {args.image_size}x{args.image_size}, "
                    f"K={args.faces_per_pixel}, nb_samples={args.nb_samples}, RandomSimpleShader "
                    "(GaussianRast+GaussianAgg) fwd+bwd",
        "fragments": args.fragments,
        "fragments_note": {"rasterised": "pert_rasterize_fwd of the 1280-face icosphere, 8 orbiting cameras, blur radius "
                                         "log(1/1e-4-1)*sigma: 48% coverage, 35 valid entries per covered pixel",
                           "realistic": "SURVEY 8d synthetic: 60% coverage, geometric valid count (mean 4)",
                           "dense": "SURVEY 8d synthetic: all 50 entries valid, dists uniform in the blur band"}[args.fragments],
        "views_per_gpu": args.views, "global_views": args.views * world,
        "image_size": args.image_size, "faces_per_pixel": args.faces_per_pixel, "nb_samples": args.nb_samples,
        "sigma": SIGMA, "gamma": GAMMA, "alpha": ALPHA, "flags": 0, "parallelism": f"batch-shard x{world}",
        "timing": "one device-timed window of the requested steps, bracketed by barrier + synchronize, max over ranks",
        "l2": f"inputs ({inputs_gb:.2f} GB per step) exceed the 126 MB L2; no explicit flush",
    }


def dump_outputs(dirname, outputs):
    """Writes what one step hands its caller, (image, grad_dists, grad_zbuf, grad_colors, grad_scalars), as
    <dirname>/<name>.npy in float32, so that two builds run with the same arguments can be compared entry by entry.  The
    per-pixel arrays are flattened to (pixels, ...); when together they exceed DUMP_BYTES, every one of them keeps the same
    fixed sample of pixels (seed 0, ascending pixel order)."""
    import numpy as np
    image = outputs[0]
    P = image.shape[0] * image.shape[1] * image.shape[2]
    per_pixel = {name: t.reshape((P,) + t.shape[3:])
                 for name, t in zip(("image", "grad_dists", "grad_zbuf", "grad_colors"), outputs[:4])}
    n = min(P, DUMP_BYTES // sum(4 * t[0].numel() for t in per_pixel.values()))
    pix = torch.randperm(P, generator=torch.Generator().manual_seed(0))[:n].sort().values.to(image.device)
    os.makedirs(dirname, exist_ok=True)
    for name, t in per_pixel.items():
        np.save(os.path.join(dirname, name + ".npy"), t[pix].float().cpu().numpy())
    np.save(os.path.join(dirname, "grad_scalars.npy"), outputs[4].float().cpu().numpy())


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
def device_timed(cfg, kind, dev, steps, warmup, world, rank, sampler=None, flags=0, face=False, soft=False,
                 fragments=None, dump_dir=None):
    """Inputs resident in HBM; K timed steps of pert_shade_fwd + pert_shade_bwd through the C ABI.  With `dump_dir`,
    rank 0 writes what the last timed step returned there (dump_outputs)."""
    import torch.distributed as dist
    from pertrenderer_b200 import ops
    N, HW, K, S = cfg["N"], cfg["HW"], cfg["K"], cfg["S"]
    fr, col = fragments if fragments is not None else make_fragments(kind, N, HW, K, S, dev, rank)
    G = torch.randn((N, HW, HW, 4), device=dev, generator=torch.Generator(device=dev).manual_seed(1 + rank))
    P = N * HW * HW
    V = int((fr.pix_to_face >= 0).sum().item())
    torch.manual_seed(1234 + rank)
    F = 1280  # faces of data/objs/sphere/sphere_642.obj (SURVEY.md §8d)
    table = None
    if face:  # texels gathered through pix_to_face inside the kernels: no (N,H,W,K,3) tensor at all
        table = torch.rand((F, 3), device=dev, generator=torch.Generator(device=dev).manual_seed(7))
        col = None
        p2f = fr.pix_to_face.clamp(max=F - 1)
    else:
        p2f = fr.pix_to_face

    def problem():
        return ops.ShadeProblem(pix_to_face=p2f, zbuf=fr.zbuf, dists=fr.dists, colors=col, face_colors=table, znear=1.0,
                                zfar=100.0, background=BACKGROUND, sigma=SIGMA, gamma=GAMMA, alpha=ALPHA, eps=EPS,
                                S_rast=S, S_agg=S, seed_rast=ops.draw_seed(), seed_agg=ops.draw_seed(),
                                pixel_offset=rank * P, flags=flags)

    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
    comm = torch.cuda.Stream(device=dev) if world > 1 else None

    def step(e=None):
        pr = problem()
        if e is not None:
            e[0].record()
        if soft:  # SoftRast + SoftAgg (deterministic): the shaders' default operator pair
            image = ops.soft_shade_forward(pr)
        else:
            image, saved = ops.shade_forward(pr)
        if e is not None:
            e[1].record()
        gd, gz, gc, scal = ops.soft_shade_backward(pr, G) if soft else ops.shade_backward(pr, saved, G)
        if e is not None:
            e[2].record()
        if world > 1:
            # the only collective of batch sharding: d/d(sigma, gamma, alpha), 3 floats.  Nothing on the GPU waits for
            # it (the caller reads the scalar gradients on the host after the step, eval.py:386-392), so it runs on
            # its own stream behind backward and overlaps the next step's forward; the timed region ends only after
            # the last all-reduce (main stream waits for the side stream before the closing event).
            done = torch.cuda.Event()
            done.record()
            comm.wait_event(done)
            with torch.cuda.stream(comm):
                scal.record_stream(comm)
                dist.all_reduce(scal)
        return image, gd, gz, gc, scal

    for _ in range(warmup):
        step()
    torch.cuda.synchronize(dev)
    torch.cuda.reset_peak_memory_stats(dev)
    mem_base = torch.cuda.memory_allocated(dev)
    if sampler is not None:
        sampler.start()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for i in range(steps):
        if i == steps - 1:
            outputs = step(ev[i])
        else:
            step(ev[i])
    if world > 1:
        torch.cuda.current_stream(dev).wait_stream(comm)
    t1.record()
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    total_ms = t0.elapsed_time(t1)
    if world > 1:
        t = torch.tensor([total_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = t.item()
    peak_mem = int(torch.cuda.max_memory_allocated(dev) - mem_base)
    if dump_dir is not None and rank == 0:
        dump_outputs(dump_dir, outputs)
    del outputs
    fwd_ms = sum(e[0].elapsed_time(e[1]) for e in ev) / steps
    bwd_ms = sum(e[1].elapsed_time(e[2]) for e in ev) / steps
    units = P * K * S
    fb, bb = alg_bytes(P, K)
    fmin, bmin = min_bytes(P, K, V)
    if face:  # SURVEY.md §8d, inlined gather variant: 40 PF + 32 P + 24 F over forward + backward
        fb, bb = 16 * P * K + 16 * P + 12 * F, 24 * P * K + 16 * P + 12 * F
        fmin, bmin = 8 * P * K + 8 * V + 16 * P + 12 * F, 8 * P * K + 16 * V + 8 * P * K + 16 * P + 12 * F
    peak, peak_src = peaks()
    dom = "pert_shade_bwd" if bwd_ms >= fwd_ms else "pert_shade_fwd"
    dom_ms, dom_bytes = (bwd_ms, bb) if bwd_ms >= fwd_ms else (fwd_ms, fb)
    traffic = None if (face or soft or flags) else measured_traffic(dom, kind, N, HW, K, S)
    roof = {"bound": "hbm", "kernel": dom, "achieved": dom_bytes / dom_ms / 1e6, "peak": peak, "unit": "GB/s",
            "frac": dom_bytes / dom_ms / 1e6 / peak, "traffic": traffic, "peak_source": peak_src,
            "issue_slots": None if (face or soft or flags) else measured_issue(kind, N, HW, K, S),
            "algorithmic_bytes_per_launch": dom_bytes, "kernel_ms": dom_ms,
            "fwd": {"ms": fwd_ms, "alg_bytes": fb, "gbs": fb / fwd_ms / 1e6, "frac": fb / fwd_ms / 1e6 / peak},
            "bwd": {"ms": bwd_ms, "alg_bytes": bb, "gbs": bb / bwd_ms / 1e6, "frac": bb / bwd_ms / 1e6 / peak},
            "fwd_bwd_frac": (fb + bb) / (fwd_ms + bwd_ms) / 1e6 / peak,
            # against the bytes the kernels cannot avoid on THIS fragment set (padding is never read beyond the scan)
            "min_bytes": {"fwd": fmin, "bwd": bmin, "fwd_bwd_frac": (fmin + bmin) / (fwd_ms + bwd_ms) / 1e6 / peak,
                          "valid_entries": V, "valid_fraction": V / (P * K)}}
    return {"value": units * world * steps / (total_ms * 1e-3), "ms_per_step": total_ms / steps, "roofline": roof,
            "peak_memory_bytes": peak_mem,
            # kernels of libpertshade.so per step: forward main + fallback pass (two launches: coverage samples,
            # aggregation + blend), backward main + fallback pass, scalar-gradient finalize
            "launches": 6 * steps}


def leg(res, **extra):
    out = {"value": res["value"], "unit": UNIT, "ms_per_step": res["ms_per_step"], "roofline": res["roofline"]}
    out.update(extra)
    return out


def config_legs(dev, rank, steps):
    """BASELINE configs 1, 3 (per-GPU share), 4, 5 at one GPU, device-timed like the headline."""
    out = {}
    plan = [(1, "rasterised"), (1, "realistic"), (3, "rasterised"), (3, "realistic"), (4, "rasterised"), (5, "realistic")]
    for c, kind in plan:
        cfg = CONFIGS[c]
        n = max(3, min(steps, 10)) if c in (1, 4) else 3
        try:
            r = device_timed(cfg, kind, dev, n, 3, 1, rank)
            out[f"config{c}_{kind}"] = leg(r, config=cfg["name"], fragments=kind, steps=n,
                                           peak_memory_bytes=r["peak_memory_bytes"])
        except Exception as e:  # a leg must never take the headline down
            out[f"config{c}_{kind}"] = {"error": repr(e)[:200]}
        torch.cuda.empty_cache()
    return out


def graph_leg(dev, kind="rasterised", steps=50):
    """BASELINE config 1 (1 x 64^2, K=50, S=16: launch-bound, 2.4 us at the roofline) with forward + backward captured in ONE
    CUDA graph (ops.GraphedShadeStep: device-side seeds stepped by a pert_seed_advance node), against the same step
    launched eagerly."""
    from pertrenderer_b200 import ops
    cfg = CONFIGS[1]
    N, HW, K, S = cfg["N"], cfg["HW"], cfg["K"], cfg["S"]
    fr, col = make_fragments(kind, N, HW, K, S, dev, 0)
    G = torch.randn((N, HW, HW, 4), device=dev, generator=torch.Generator(device=dev).manual_seed(1))
    step = ops.GraphedShadeStep(fr.pix_to_face, fr.zbuf.contiguous(), fr.dists.contiguous(), col, G, sigma=SIGMA, gamma=GAMMA,
                                alpha=ALPHA, eps=EPS, S_rast=S, S_agg=S, background=BACKGROUND)
    for _ in range(5):
        step.replay()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step.replay()
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / steps
    eager = device_timed(cfg, kind, dev, steps, 5, 1, 0, fragments=(fr, col))
    units = N * HW * HW * K * S
    return {"config": cfg["name"], "fragments": kind, "ms_per_step_graph": ms, "ms_per_step_eager": eager["ms_per_step"],
            "value": units / (ms * 1e-3), "unit": UNIT, "launches_per_step": 9,
            "note": "one graph replay = seed advance + memsets + forward (main + two-launch fallback pass) + backward (main + fallback "
                    "pass) + scalar finalize"}


def explicit_noise_leg(dev, kind, steps=5):
    """SURVEY section 8d: "explicit-noise mode where HBM really binds".  BASELINE config 2 with both noise tensors
    materialised in HBM, U (S,N,H,W,K) and V (S,N,H,W,K+1) -- the reference's own data flow, the parity path of the kernels
    (bit-comparable with the oracle) -- against the survey's byte count for this mode: the Philox-mode bytes plus
    4 S (PF + P K1) per pass."""
    from pertrenderer_b200 import ops
    cfg = CONFIGS[2]
    N, HW, K, S = cfg["N"], cfg["HW"], cfg["K"], cfg["S"]
    fr, col = make_fragments(kind, N, HW, K, S, dev, 0)
    G = torch.randn((N, HW, HW, 4), device=dev, generator=torch.Generator(device=dev).manual_seed(1))
    gen = torch.Generator(device=dev).manual_seed(5)
    U = torch.randn((S, N, HW, HW, K), device=dev, generator=gen)
    V = torch.randn((S, N, HW, HW, K + 1), device=dev, generator=gen)
    pr = ops.ShadeProblem(pix_to_face=fr.pix_to_face, zbuf=fr.zbuf, dists=fr.dists, colors=col, znear=1.0, zfar=100.0,
                          background=BACKGROUND, sigma=SIGMA, gamma=GAMMA, alpha=ALPHA, eps=EPS, S_rast=S, S_agg=S,
                          noise_rast=U, noise_agg=V)
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
    for i in range(-2, steps):
        if i >= 0:
            ev[i][0].record()
        image, saved = ops.shade_forward(pr)
        if i >= 0:
            ev[i][1].record()
        ops.shade_backward(pr, saved, G)
        if i >= 0:
            ev[i][2].record()
    torch.cuda.synchronize(dev)
    fwd = sorted(e[0].elapsed_time(e[1]) for e in ev)[steps // 2]
    bwd = sorted(e[1].elapsed_time(e[2]) for e in ev)[steps // 2]
    P = N * HW * HW
    PF = P * K
    noise = 4 * S * (PF + P * (K + 1))
    fb, bb = 28 * PF + 16 * P + noise, 48 * PF + 16 * P + noise
    peak, peak_src = peaks()
    del U, V
    torch.cuda.empty_cache()
    return {"config": cfg["name"], "fragments": kind, "ms_per_step": fwd + bwd, "value": PF * S / ((fwd + bwd) * 1e-3), "unit": UNIT,
            "fwd": {"ms": fwd, "alg_bytes": fb, "frac": fb / fwd / 1e6 / peak}, "bwd": {"ms": bwd, "alg_bytes": bb, "frac": bb / bwd / 1e6 / peak},
            "fwd_bwd_frac": (fb + bb) / (fwd + bwd) / 1e6 / peak, "noise_bytes_per_pass": noise, "peak": peak, "peak_source": peak_src,
            "note": "explicit noise tensors in HBM (13.5 GB): the exact-noise parity mode of the kernels (phase-split generic "
                    "instantiation), not the production path; backward reads V only (the coverage sums are saved by forward), "
                    "the byte count follows SURVEY 8d and charges U to it as well"}


def pose_iteration_leg(dev, niter=100):
    """One pose-optimisation trial of examples/pose_optimisation.py (eval.py:320-409: cube, 128x128, K=50, S=16, 100 Adam
    iterations through MeshRenderer(MeshRasterizer, RandomPhongShader(GaussianRast, GaussianAgg))): wall-clock ms per
    iteration of the eager loop and of the loop with one CUDA graph per iteration (capture included)."""
    import math
    import runpy
    import time
    import pertrenderer_b200 as pb
    ex = runpy.run_path(os.path.join(ROOT, "examples", "pose_optimisation.py"), run_name="pose_example")
    d = str(dev)
    verts, faces, colors = ex["cube_mesh"](d)
    mesh = pb.TriMeshes(verts, faces, face_colors=colors)
    R, T = pb.look_at_view_transform(dist=6.7, elev=30.0, azim=120.0, device=d)
    cameras = pb.OpenGLPerspectiveCameras(R=R, T=T, fov=60, device=d)
    lights = pb.PointLights(location=[[0.0, 2.0, -2.0]], device=d)
    hard = ex["make_renderer"]("hard", cameras, lights, 1e-4, 1e-4, 1, 128, d)
    R_true = ex["so3_exp"](torch.tensor([0.3, -0.5, 0.2], device=d))
    with torch.no_grad():
        target = hard(mesh.update_padded(verts @ R_true))[..., :3]
    axis = torch.tensor([0.6, 0.0, 0.8], device=d)
    w0 = ex["so3_log"](R_true @ ex["so3_exp"](math.radians(30.0) * axis))
    out = {"workload": "cube (12 faces), 128x128, K=50, S=16, 30 degrees off, %d Adam iterations, lr 5e-2" % niter}
    for name, fn in (("eager", lambda r: ex["optimize_pose"](mesh, verts, r, target, w0, niter, 5e-2, False)),
                     ("graph", lambda r: ex["optimize_pose_graphed"](mesh, verts, r, target, w0, niter, 5e-2))):
        fn(ex["make_renderer"]("gaussian", cameras, lights, SIGMA, GAMMA, 16, 128, d))  # warm-up trial
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        w = fn(ex["make_renderer"]("gaussian", cameras, lights, SIGMA, GAMMA, 16, 128, d))
        torch.cuda.synchronize(dev)
        out["ms_per_iteration_" + name] = 1e3 * (time.perf_counter() - t0) / niter
        out["final_angle_deg_" + name] = ex["angle_deg"](ex["so3_exp"](w), R_true)
    out["note"] = ("wall clock around a whole trial; graph = 3 eager iterations + capture + replays, every iteration (render + "
                   "loss + backward + best-pose bookkeeping + gradient guard + Adam) one CUDA graph with device-side seeds")
    return out


def sample_sharded_leg(dev, world, rank, steps):
    """BASELINE config 4 (1 x 128^2, K=50, S=4096) with the noise samples split over the ranks
    (dist.smooth_rgb_blend_sample_sharded: three all-reduces over NCCL), against the unsharded job on every rank:
    with sync_seeds the sharded job reproduces the single-GPU sample path, so the difference is rounding only."""
    import torch.distributed as dist
    import pertrenderer_b200 as pb
    from pertrenderer_b200 import _cabi, ops
    from pertrenderer_b200 import dist as pdist
    cfg = CONFIGS[4]
    N, HW, K, S = cfg["N"], cfg["HW"], cfg["K"], cfg["S"]
    fr, col = make_fragments("rasterised", N, HW, K, S, dev, 0)  # replicated inputs: the same on every rank
    G = torch.randn((N, HW, HW, 4), device=dev, generator=torch.Generator(device=dev).manual_seed(1))
    rastop, aggop = pb.GaussianRast(nb_samples=S, sigma=SIGMA), pb.GaussianAgg(nb_samples=S, gamma=GAMMA, alpha=ALPHA)
    blend = pb.BlendParams(background_color=BACKGROUND)

    def run(sharded, seed, sync=False):
        torch.manual_seed(seed)
        d, z, c = (t.detach().clone().requires_grad_(True) for t in (fr.dists, fr.zbuf, col))
        f = pb.Fragments(fr.pix_to_face, z, None, d)
        if sharded:
            img = pdist.smooth_rgb_blend_sample_sharded(c, f, rastop, aggop, blend, sync_seeds=sync)
        else:
            img = pb.smooth_rgb_blend(c, f, rastop, aggop, blend)
        (img * G).sum().backward()
        return img.detach(), d.grad, z.grad, c.grad

    # correctness: per-sample flags make the sharded and the unsharded job draw the same sample path
    with ops.kernel_flags(_cabi.F_PER_SAMPLE_NOISE):
        a = run(True, 99, sync=True)
        b = run(False, 99)

    def rel(x, y):
        return ((x - y).abs().max() / y.abs().max().clamp(min=1e-30)).item()
    err = {"image_max_abs": (a[0] - b[0]).abs().max().item(), "grad_dists_rel": rel(a[1], b[1]),
           "grad_zbuf_rel": rel(a[2], b[2]), "grad_colors_rel": rel(a[3], b[3])}
    t = torch.tensor([max(err.values())], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    err["max_over_ranks"] = t.item()

    def timed(sharded):
        for i in range(3):
            run(sharded, i)
        dist.barrier()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            run(sharded, 10 + i)
        e1.record()
        torch.cuda.synchronize(dev)
        dist.barrier()
        ms = torch.tensor([e0.elapsed_time(e1) / steps], device=dev)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()
    ms_sharded, ms_single = timed(True), timed(False)
    units = N * HW * HW * K * S
    # the same job with every rank's phases and the three all-reduces captured in one CUDA graph per rank
    graph = {}
    try:
        d, z, c = fr.dists.contiguous(), fr.zbuf.contiguous(), col
        step = pdist.GraphedSampleShardedStep(fr.pix_to_face, z, d, c, G, sigma=SIGMA, gamma=GAMMA, alpha=ALPHA, eps=EPS,
                                              S_rast=S, S_agg=S, background=BACKGROUND)
        for _ in range(3):
            step.replay()
        dist.barrier()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(4 * steps):
            step.replay()
        e1.record()
        torch.cuda.synchronize(dev)
        dist.barrier()
        ms = torch.tensor([e0.elapsed_time(e1) / (4 * steps)], device=dev)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        img = step.image.clone()
        dist.broadcast(img, src=0)
        graph = {"ms_per_step_graph": ms.item(), "speedup_graph": ms_single / ms.item(),
                 "ranks_agree": bool(torch.equal(img, step.image)), "value_graph": units / (ms.item() * 1e-3)}
        step.close()  # the graph holds NCCL kernels: release it before the process group goes away
    except Exception as e:
        graph = {"graph_error": repr(e)[:300]}
    return {"config": cfg["name"], "fragments": "rasterised", "world": world, **graph,
            "note": "public API + autograd (smooth_rgb_blend_sample_sharded vs smooth_rgb_blend), default noise flags for "
                    "the timing, PERT_F_PER_SAMPLE_NOISE + synchronised seeds for the comparison",
            "ms_per_step_sharded": ms_sharded, "ms_per_step_one_gpu": ms_single, "speedup": ms_single / ms_sharded,
            "value": units / (ms_sharded * 1e-3), "unit": UNIT, "error_vs_unsharded": err}


def phong_timed(args, kind, dev, steps, warmup, rank):
    """RandomPhongShader step (random_rasterizer.py:60-130), inputs resident: pert_phong_fwd -> pert_shade_fwd ->
    pert_shade_bwd -> pert_phong_bwd through the C ABI.  Per-face colours (gathered in the Phong kernel), sphere
    mesh of 1280 faces, one point light; gradients to the face tables (vertices, normals) and bary_coords."""
    import pertrenderer_b200 as pb
    from pertrenderer_b200 import ops, shading
    N, HW, K, S = args.views, args.image_size, args.faces_per_pixel, args.nb_samples
    F = 1280
    fr, _ = pb.synthetic_fragments(N, HW, HW, K, kind=kind, sigma=SIGMA, n_faces=F, seed=rank, device=dev)
    verts, faces = pb.synthetic_mesh(F, device=dev)
    F = faces.shape[0]
    p2f = fr.pix_to_face.clamp(max=F - 1)
    bary = pb.synthetic_bary(p2f, seed=rank)
    mesh = pb.TriMeshes(verts, faces)
    fv, fn = verts[faces].contiguous(), mesh.verts_normals_packed()[faces].contiguous()
    fc = torch.rand((F, 3), device=dev, generator=torch.Generator(device=dev).manual_seed(7))
    lighting = shading.pack_lighting(pb.PointLights(location=[[0.0, 2.0, -2.0]], device=dev), pb.Materials(device=dev),
                                     pb.ViewCameras(R=torch.eye(3)[None], T=[[0.0, 0.0, 6.7]], device=dev), N, dev)
    G = torch.randn((N, HW, HW, 4), device=dev, generator=torch.Generator(device=dev).manual_seed(1 + rank))
    P = N * HW * HW
    V = int((p2f >= 0).sum().item())
    torch.manual_seed(4321 + rank)
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(5)] for _ in range(steps)]

    def step(i=None):
        rec = (lambda j: ev[i][j].record()) if i is not None else (lambda j: None)
        rec(0)
        colors = shading.phong_forward(p2f, bary, fv, fn, None, fc, lighting, sparse=True)
        rec(1)
        pr = ops.ShadeProblem(pix_to_face=p2f, zbuf=fr.zbuf, dists=fr.dists, colors=colors, znear=1.0, zfar=100.0,
                              background=BACKGROUND, sigma=SIGMA, gamma=GAMMA, alpha=ALPHA, eps=EPS, S_rast=S, S_agg=S,
                              seed_rast=ops.draw_seed(), seed_agg=ops.draw_seed(), pixel_offset=rank * P)
        image, saved = ops.shade_forward(pr)
        rec(2)
        gd, gz, gc, scal = ops.shade_backward(pr, saved, G)
        rec(3)
        out = shading.phong_backward(p2f, bary, fv, fn, None, fc, lighting, gc, need_texels=False, sparse=True)
        rec(4)
        return out

    for _ in range(warmup):
        step()
    torch.cuda.synchronize(dev)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for i in range(steps):
        step(i)
    t1.record()
    torch.cuda.synchronize(dev)
    total_ms = t0.elapsed_time(t1)
    seg = [sum(e[j].elapsed_time(e[j + 1]) for e in ev) / steps for j in range(4)]
    peak, peak_src = peaks()
    PF = P * K
    # Bytes the sparse Phong pass must move: the pix_to_face scan (8 per entry) + per VALID entry bary 12 and colours 12
    # (fwd: written; bwd: grad_colors read) + the zero-fill of grad_bary (12 per entry, done by torch inside the timed
    # region) + the face tables.  The API-faithful figure (dense colours / grad tensors, 32 PF and 44 PF) counts bytes the
    # sparse mode never touches, so it is reported as a byte count only, not as a roofline fraction.
    pf_b, pb_b = 8 * PF + 24 * V + 84 * F, 8 * PF + 24 * V + 12 * PF + 156 * F
    return {"fragments": kind,
            "note": "RandomPhongShader: pert_phong_fwd -> pert_shade_fwd -> pert_shade_bwd -> pert_phong_bwd; per-face "
                    "colours, 1280-face sphere, one point light; gradients to face vertices / normals and bary_coords; "
                    "sparse mode (padded entries of colors are neither written nor read; grad_bary is zero-filled by "
                    "torch inside the timed region); fractions are against the bytes the sparse pass must move",
            "value": P * K * S * steps / (total_ms * 1e-3), "unit": UNIT, "ms_per_step": total_ms / steps,
            "phong_fwd": {"ms": seg[0], "min_bytes": pf_b, "gbs": pf_b / seg[0] / 1e6, "frac": pf_b / seg[0] / 1e6 / peak,
                          "api_faithful_bytes": 32 * PF + 84 * F},
            "shade_fwd_ms": seg[1], "shade_bwd_ms": seg[2],
            "phong_bwd": {"ms": seg[3], "min_bytes": pb_b, "gbs": pb_b / seg[3] / 1e6, "frac": pb_b / seg[3] / 1e6 / peak,
                          "api_faithful_bytes": 44 * PF + 156 * F},
            "peak": peak, "peak_source": peak_src, "launches_per_step": 8}


def renderer_timed(args, dev, steps, warmup, rank):
    """The whole renderer of experiments/eval.py:165-177 through the public API: MeshRenderer(MeshRasterizer,
    RandomPhongShader(GaussianRast, GaussianAgg)) forward + autograd backward to the mesh vertices, 1280-face icosphere,
    N orbiting cameras, config-2 shapes.  Segments timed with CUDA events: rasterise / shade forward / everything
    backward."""
    import math
    import pertrenderer_b200 as pb
    N, HW, K, S = args.views, args.image_size, args.faces_per_pixel, args.nb_samples
    verts, faces = pb.synthetic_mesh(1280, device=dev)
    R, T = pb.look_at_view_transform(dist=2.7, elev=30.0, azim=torch.linspace(0, 315, N) + 7.0 * rank, device=dev)
    cam = pb.OpenGLPerspectiveCameras(R=R, T=T, device=dev)
    blur = math.log(1.0 / 1e-4 - 1.0) * SIGMA
    rast = pb.MeshRasterizer(cam, pb.RasterizationSettings(image_size=HW, blur_radius=blur, faces_per_pixel=K))
    shader = pb.RandomPhongShader(device=dev, cameras=cam, lights=pb.PointLights(location=[[0.0, 2.0, -2.0]], device=dev),
                                  blend_params=pb.BlendParams(background_color=BACKGROUND),
                                  smoothrast=pb.GaussianRast(nb_samples=S, sigma=SIGMA),
                                  smoothagg=pb.GaussianAgg(nb_samples=S, gamma=GAMMA, alpha=ALPHA))
    fc = torch.rand((faces.shape[0], 3), device=dev, generator=torch.Generator(device=dev).manual_seed(7))
    mesh = pb.TriMeshes(verts, faces, face_colors=fc).extend(N)
    G = torch.randn((N, HW, HW, 4), device=dev, generator=torch.Generator(device=dev).manual_seed(1 + rank))
    v = mesh.verts_padded().clone().requires_grad_(True)
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(steps)]
    stats = {}

    def step(i=None):
        rec = (lambda j: ev[i][j].record()) if i is not None else (lambda j: None)
        v.grad = None
        m = mesh.update_padded(v)
        rec(0)
        frag = rast(m)
        rec(1)
        img = shader(frag, m)
        rec(2)
        (img * G).sum().backward()
        rec(3)
        if i is None and not stats:
            valid = frag.pix_to_face >= 0
            stats["coverage"] = valid.any(-1).float().mean().item()
            stats["valid_per_covered_pixel"] = valid.sum(-1)[valid.any(-1)].float().mean().item()

    for _ in range(warmup):
        step()
    torch.cuda.synchronize(dev)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for i in range(steps):
        step(i)
    t1.record()
    torch.cuda.synchronize(dev)
    total_ms = t0.elapsed_time(t1)
    seg = [sum(e[j].elapsed_time(e[j + 1]) for e in ev) / steps for j in range(3)]
    P = N * HW * HW
    return {"note": "MeshRenderer(MeshRasterizer, RandomPhongShader(GaussianRast, GaussianAgg)), public API + autograd to the "
                    "mesh vertices; 1280-face icosphere, blur_radius = log(1/1e-4-1)*sigma; includes the host reads of the "
                    "scalar gradients (sigma, gamma, alpha are CPU leaves)",
            "value": P * K * S * steps / (total_ms * 1e-3), "unit": UNIT, "ms_per_step": total_ms / steps,
            "rasterize_ms": seg[0], "shade_fwd_ms": seg[1], "backward_ms": seg[2], **stats}


def e2e_timed(args, kind, dev, steps, warmup, world, rank):
    """End to end through the public API (RandomSimpleShader + autograd) with HOST buffers: every
    step copies that step's Fragments and texels from pinned host memory (double-buffered on a copy
    stream, so the copy of step i+1 overlaps the kernels of step i) and reads the image, the loss
    and the scalar gradients back to the host."""
    import pertrenderer_b200 as pb
    N, HW, K, S = args.views, args.image_size, args.faces_per_pixel, args.nb_samples
    fr, col = make_fragments(kind, N, HW, K, S, dev, rank)
    host = [t.cpu().pin_memory() for t in (fr.pix_to_face, fr.zbuf, fr.dists, col)]
    G = torch.randn((N, HW, HW, 4), device=dev, generator=torch.Generator(device=dev).manual_seed(1 + rank))
    del fr, col
    bufs = [[torch.empty_like(h, device=dev) for h in host] for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    copy_stream = torch.cuda.Stream(device=dev)
    img_host = torch.empty((N, HW, HW, 4), dtype=torch.float32).pin_memory()
    shader = pb.RandomSimpleShader(device=dev, cameras=pb.DepthCameras(n=N, device=dev),
                                   smoothrast=pb.GaussianRast(nb_samples=S, sigma=SIGMA),
                                   smoothagg=pb.GaussianAgg(nb_samples=S, gamma=GAMMA, alpha=ALPHA),
                                   blend_params=pb.BlendParams(background_color=BACKGROUND))
    h2d = sum(h.numel() * h.element_size() for h in host)
    d2h = img_host.numel() * 4 + 4 + 12
    main = torch.cuda.current_stream(dev)

    def upload(slot):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[slot])
            for b, h in zip(bufs[slot], host):
                b.copy_(h, non_blocking=True)
            ready[slot].record(copy_stream)

    def step(i, last):
        slot = i & 1
        if not last:
            upload((i + 1) & 1)
        main.wait_event(ready[slot])
        p2f, z, d, c = bufs[slot]
        z, d, c = (t.detach().requires_grad_(True) for t in (z, d, c))  # fresh leaves sharing the buffers
        img = shader(pb.Fragments(p2f, z, None, d), pb.TexelMeshes(c))
        loss = (img * G).sum()
        loss.backward()
        consumed[slot].record(main)
        img_host.copy_(img.detach(), non_blocking=True)
        s, g, a = shader.get_smoothing()
        out = (loss.item(), s.grad.item(), g.grad.item(), a.grad.item())  # device -> host reads (sync)
        for t in (s, g, a):
            t.grad = None
        return out

    for e in consumed:
        e.record(main)
    total = warmup + steps
    upload(0)
    for i in range(warmup):
        step(i, False)
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(warmup, total):
        step(i, i == total - 1)
    e1.record()
    torch.cuda.synchronize(dev)
    wall_ms = (time.perf_counter() - t0) * 1e3
    ms = max(e0.elapsed_time(e1), wall_ms)
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    units = N * HW * HW * K * S
    return {"value": units * world * steps / (ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
            "d2h_bytes_per_step": d2h, "ms_per_step": ms / steps,
            "note": "public API (RandomSimpleShader+autograd), pinned host inputs, double-buffered H2D on a copy stream; "
                    "bound by the host->device copy of the dense (N,H,W,K) Fragments the reference's API takes"}


def run_b200_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the perturbed shading path has no CPU fallback")
    from pertrenderer_b200 import _cabi
    _cabi.load()  # fail loudly if the sm_100a library is missing
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # stdout carries exactly one JSON line
        dist.init_process_group("nccl", device_id=dev)
    cfg = dict(N=args.views, HW=args.image_size, K=args.faces_per_pixel, S=args.nb_samples)
    sampler = ClockSampler(local) if rank == 0 else None
    main = device_timed(cfg, args.fragments, dev, args.steps, args.warmup, world, rank, sampler, dump_dir=args.dump_outputs)
    clocks = sampler.finish() if sampler is not None else None
    also = None
    if not args.no_also:
        n2, n4 = max(3, args.steps // 2), max(3, args.steps // 4)
        also = {}
        for kind in ("rasterised", "realistic", "dense"):
            if kind != args.fragments:
                o = device_timed(cfg, kind, dev, n4 if kind == "dense" else n2, 3, world, rank)
                also["fragments_" + kind] = leg(o, fragments=kind)
        p7 = device_timed(cfg, args.fragments, dev, n2, 3, world, rank, flags=_cabi.F_PHILOX7)
        also["philox7"] = leg(p7, fragments=args.fragments, flags="PERT_F_PHILOX7",
                              note="Philox4x32-7 (the Crush-resistant minimum of Salmon et al.) instead of Philox4x32-10: "
                                   "another noise stream of the same law")
        ps = device_timed(cfg, args.fragments, dev, n4, 3, world, rank, flags=_cabi.F_PER_SAMPLE_NOISE)
        also["per_sample_noise"] = leg(ps, fragments=args.fragments, flags="PERT_F_PER_SAMPLE_NOISE",
                                       note="every coverage sample drawn one by one and backward regenerating every V_sj of "
                                            "every logit: the reference's sample path (pert_noise_fill's tensor), bit for "
                                            "bit; the default draws coverage flips from their binomial law and "
                                            "never-winning logits' score noise once per logit")
        if world > 1:
            c3 = device_timed(CONFIGS[3], "realistic", dev, 3, 3, world, rank)
            also["config3_batch_sharded"] = leg(c3, config=CONFIGS[3]["name"], fragments="realistic",
                                                global_poses=CONFIGS[3]["N"] * world)
            try:
                also["sample_sharded"] = sample_sharded_leg(dev, world, rank, 5)
            except Exception as e:
                also["sample_sharded"] = {"error": repr(e)[:300]}
        else:
            fc = device_timed(cfg, "realistic", dev, n2, 3, world, rank, face=True)
            sf = device_timed(cfg, "realistic", dev, n2, 3, world, rank, soft=True)
            also["softras_pair"] = leg(sf, fragments="realistic",
                                       note="SoftRast + SoftAgg (the shaders' DEFAULT operators, deterministic) through the "
                                            "fused soft kernels; same algorithmic bytes; 'units' counts nb_samples like the "
                                            "headline although this pair draws no samples")
            also["face_colour_gather"] = leg(fc, fragments="realistic",
                                             note="texel colours gathered through pix_to_face inside the kernels (per-face "
                                                  "colour table of 1280 faces), gradient scattered by atomics; algorithmic "
                                                  "bytes 40 PF + 32 P + 24 F")
            if not args.no_config_legs:
                also["configs"] = config_legs(dev, rank, args.steps)
                try:
                    also["config1_cuda_graph"] = graph_leg(dev)
                except Exception as e:
                    also["config1_cuda_graph"] = {"error": repr(e)[:300]}
            if not args.no_renderer_legs:
                also["random_phong_shader"] = phong_timed(args, "realistic", dev, n2, 3, rank)
                also["renderer"] = renderer_timed(args, dev, n4, 3, rank)
                try:
                    also["explicit_noise"] = explicit_noise_leg(dev, args.fragments)
                except Exception as e:
                    also["explicit_noise"] = {"error": repr(e)[:300]}
                try:
                    also["pose_optimisation"] = pose_iteration_leg(dev)
                except Exception as e:
                    also["pose_optimisation"] = {"error": repr(e)[:300]}
            try:
                also["reference_torch_cuda"] = reference_cuda_run(args, dev)
            except Exception as e:
                also["reference_torch_cuda"] = {"error": repr(e)[:300]}
            torch.cuda.empty_cache()
    e2e = None
    if not args.no_e2e:
        e2e = e2e_timed(args, args.fragments, dev, args.steps, args.warmup, world, rank)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cb = cpu_reference_run(args, 3, 1, budget_s=25.0)
        cpu = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    line = {
        "metric": METRIC, "value": main["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args, world),
        "clocks": clocks, "e2e": e2e, "gpu_launches": main["launches"], "roofline": main["roofline"],
        "cpu_baseline": cpu, "peak_memory_bytes": main["peak_memory_bytes"], "also": also,
    }
    emit(line)


def main():
    args = parse_args()
    quiet_stdout()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_b200_arm(args)


if __name__ == "__main__":
    main()
