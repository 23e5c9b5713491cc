"""Coarse bins of the rasteriser for large meshes: the synchronising two-pass binning (pert_rasterize_bin, its total read
back to size the lists, as rasterize_meshes did before the bounded bins) against the bounded bins
(pert_rasterize_bin_bounded, lists sized C * F from shapes alone, PERT_RAST_BIN_WIDE), each followed by the forward.

Shapes: 1 x 128^2 (eval-like), 8 x 256^2 and BASELINE config 5's 16 x 1024^2, all K = 50 and eval.py's blur at sigma =
1e-3, the icosphere of 20480 faces (100000 faces for config 5) seen by orbiting cameras.  Per shape and path:
  device ms  median over the timed calls of CUDA events around one call (bins + forward)
  wall ms    host wall time per call of an eager loop of `steps` calls, the device synchronised once at the end
  host ms    host time per call to enqueue that loop (before the final synchronise): what the CPU is busy with
  list MiB   bin arrays allocated (count, offset, cursor, face lists)
  entries    total list entries, and the bound C * F of the bounded layout
  wide       faces in the wide lists
The fragments of the two paths are compared bit for bit, and the path an eager rasterize_meshes selects is listed.  Then the pose iteration of examples/pose_optimisation.py at
128^2 on the 20480-face mesh (Gaussian pair, 16 samples, K = 50), eager (the example's loop) and as one CUDA graph per
iteration, ms per iteration over `--pose-iters` iterations after three warm-up iterations.

    python tools/time_raster_bins.py [--steps 50] [--pose-iters 100] [--out FILE] [--lib LIBPATH]

--lib measures another build of libpertshade.so, e.g. one compiled with -DPERT_RASTER_BIN_CAP=4 or 16 (the NVCC_FLAGS of
pertrenderer_b200/build.py plus that define), to compare values of C.
"""
import argparse
import math
import os
import runpy
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pertrenderer_b200 as pb  # noqa: E402
from pertrenderer_b200 import _cabi  # noqa: E402
from pertrenderer_b200 import rasterizer  # noqa: E402
from pertrenderer_b200.rasterizer import _raster_struct  # noqa: E402

SIGMA = 1e-3
BLUR = math.log(1.0 / 1e-4 - 1.0) * SIGMA
SHAPES = [("eval-like 1x128^2", 1, 128, 20480), ("8x256^2", 8, 256, 20480), ("config 5 16x1024^2", 16, 1024, 100000)]
K = 50
MiB = 1024.0 * 1024.0


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = f"nvidia-smi unavailable: {e!r}"
    return torch.cuda.get_device_name(0), q


def scene(N, HW, n_faces, dev):
    verts, faces = pb.synthetic_mesh(n_faces, device=dev)
    R, T = pb.look_at_view_transform(dist=2.7, elev=30.0, azim=torch.linspace(0, 315, N), device=dev)
    ndc = pb.FoVPerspectiveCameras(R=R, T=T, device=dev).transform_points_ndc(verts)
    fv = ndc[:, faces].reshape(-1, 3, 3).contiguous()
    fs = torch.arange(N + 1, device=dev, dtype=torch.int64) * faces.shape[0]
    return fv, fs


class Path:
    """One rasterisation (bins + forward) into preallocated outputs; `info` holds the bin statistics of the last call."""

    def __init__(self, bounded, fv, fs, N, HW, dev, out):
        self.bounded, self.fv, self.fs, self.N, self.HW, self.dev, self.out = bounded, fv, fs, N, HW, dev, out
        self.info = None

    def __call__(self):
        lib, dev, N = _cabi.load(), self.dev, self.N
        st = _cabi.stream_ptr(dev)
        rs = _raster_struct(self.fv, self.fs, N, self.HW, self.HW, K, BLUR, False)
        if self.bounded:
            fill, capacity = _cabi.raster_bin_fns()
            nb = int(lib.pert_rasterize_num_bins(rs)) + N
        else:
            fill = lib.pert_rasterize_bin
            nb = int(lib.pert_rasterize_num_bins(rs))
        count = torch.zeros((nb,), dtype=torch.int32, device=dev)
        _cabi.check(fill(rs, _cabi.ptr(count), None, None, None, st), "bin count")
        ends = torch.cumsum(count, 0, dtype=torch.int64)
        offset = (ends - count).contiguous()
        n_lists = int(capacity(rs)) if self.bounded else int(ends[-1].item())  # the read-back the bounded bins remove
        lists = torch.empty((max(n_lists, 1),), dtype=torch.int64, device=dev)
        cursor = torch.zeros((nb,), dtype=torch.int32, device=dev)
        _cabi.check(fill(rs, _cabi.ptr(count), _cabi.ptr(offset), _cabi.ptr(cursor), _cabi.ptr(lists), st), "bin fill")
        rs.bin_count, rs.bin_offset, rs.bin_faces = count.data_ptr(), offset.data_ptr(), lists.data_ptr()
        if self.bounded:
            rs.flags |= _cabi.RAST_BIN_WIDE
        _cabi.check(lib.pert_rasterize_fwd(rs, *(_cabi.ptr(t) for t in self.out), st), "pert_rasterize_fwd")
        self.info = (count, nb, lists.numel())


def time_path(path, steps):
    for _ in range(3):
        path()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in ev:
        a.record()
        path()
        b.record()
    torch.cuda.synchronize()
    dev_ms = statistics.median(a.elapsed_time(b) for a, b in ev)
    t0 = time.perf_counter()
    for _ in range(steps):
        path()
    t1 = time.perf_counter()
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    return dev_ms, (t2 - t0) * 1e3 / steps, (t1 - t0) * 1e3 / steps


def bin_stats(path, N):
    count, nb, n_lists = path.info
    total = int(count.long().sum())
    wide = int(count[nb - N:].long().sum()) if path.bounded else 0
    mib = (n_lists * 8 + nb * (4 + 8 + 4)) / MiB
    return total, wide, mib


def pose_times(iters, dev):
    ex = runpy.run_path(os.path.join(ROOT, "examples", "pose_optimisation.py"), run_name="pose_example")
    torch.manual_seed(0)
    verts, faces = pb.synthetic_mesh(20480, device=dev)
    colors = torch.rand((faces.shape[0], 3), device=dev, generator=torch.Generator(device=dev).manual_seed(5))
    mesh = pb.TriMeshes(verts, faces, face_colors=colors)
    R, T = pb.look_at_view_transform(dist=2.7, elev=30.0, azim=120.0, device=dev)
    cameras = pb.OpenGLPerspectiveCameras(R=R, T=T, fov=60, device=dev)
    lights = pb.PointLights(location=[[0.0, 2.0, -2.0]], device=dev)
    hard = ex["make_renderer"]("hard", cameras, lights, 1e-4, 1e-4, 1, 128, dev)
    w_true = torch.tensor([0.3, -0.5, 0.2], device=dev)
    R_true = ex["so3_exp"](w_true)
    with torch.no_grad():
        target = hard(mesh.update_padded(verts @ R_true))[..., :3]
    w0 = ex["so3_log"](R_true @ ex["so3_exp"](math.radians(15.0) * torch.tensor([0.6, 0.0, 0.8], device=dev)))
    out = {}
    for mode in ("eager", "graph", "eager", "graph"):
        renderer = ex["make_renderer"]("gaussian", cameras, lights, SIGMA, 1e-2, 16, 128, dev)
        if mode == "eager":
            ex["optimize_pose"](mesh, verts, renderer, target, w0, 3, 5e-2, False)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            w = ex["optimize_pose"](mesh, verts, renderer, target, w0, iters, 5e-2, False)
            torch.cuda.synchronize()
            ms = (time.perf_counter() - t0) * 1e3 / iters
        else:
            # warm-up + capture, then the same with `iters` more replays: the difference is the replays alone
            renderer2 = ex["make_renderer"]("gaussian", cameras, lights, SIGMA, 1e-2, 16, 128, dev)
            renderer0 = ex["make_renderer"]("gaussian", cameras, lights, SIGMA, 1e-2, 16, 128, dev)
            ex["optimize_pose_graphed"](mesh, verts, renderer0, target, w0, 4, 5e-2)  # one-time costs
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ex["optimize_pose_graphed"](mesh, verts, renderer, target, w0, 4, 5e-2)
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            w = ex["optimize_pose_graphed"](mesh, verts, renderer2, target, w0, 4 + iters, 5e-2)
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            ms = ((t2 - t1) - (t1 - t0)) * 1e3 / iters
        assert torch.isfinite(w).all()
        out.setdefault(mode, []).append(ms)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--pose-iters", type=int, default=100)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_raster_bins.txt"))
    ap.add_argument("--lib", default=None, help="another build of libpertshade.so to measure")
    args = ap.parse_args()
    if args.lib:
        _cabi.LIB_PATH = os.path.abspath(args.lib)
    dev = torch.device("cuda", 0)
    name, smi = card()
    fill, capacity = _cabi.raster_bin_fns()
    probe = _cabi.PertRaster()
    probe.num_faces = 1
    C = int(capacity(probe))
    lines = [f"# tools/time_raster_bins.py --steps {args.steps} --pose-iters {args.pose_iters}"
             + (f" --lib {os.path.basename(args.lib)}" if args.lib else ""),
             f"# card: {name}; nvidia-smi name, power limit: {smi}",
             f"# C = {C} tile entries per face (bounded bins); K = {K}, blur = {BLUR:.6g}",
             f"# {'shape':<20s} {'path':<8s} {'device ms':>9s} {'wall ms':>8s} {'host ms':>8s} {'list MiB':>9s} "
             f"{'entries':>10s} {'bound C*F':>10s} {'wide':>7s}"]
    print("\n".join(lines), flush=True)
    for label, N, HW, n_faces in SHAPES:
        fv, fs = scene(N, HW, n_faces, dev)
        F = fv.shape[0]
        outs = [(torch.empty((N, HW, HW, K), dtype=torch.int64, device=dev), torch.empty((N, HW, HW, K), device=dev),
                 torch.empty((N, HW, HW, K, 3), device=dev), torch.empty((N, HW, HW, K), device=dev)) for _ in range(2)]
        res = {}
        for bounded in (False, True, False, True):  # alternated: two rounds
            p = Path(bounded, fv, fs, N, HW, dev, outs[bounded])
            res.setdefault(bounded, []).append((time_path(p, args.steps), p))
        for a, b in zip(*outs):
            x, y = (a.view(torch.int32), b.view(torch.int32)) if a.dtype == torch.float32 else (a, b)
            assert torch.equal(x, y), f"{label}: the bounded bins changed the fragments"
        rs = _raster_struct(fv, fs, N, HW, HW, K, BLUR, False)
        pick = "bounded" if rasterizer._bounded_bins_pay(rs, capacity, HW, HW, BLUR) else "sync"
        lines.append(f"  {label:<20s} an eager rasterize_meshes takes: {pick}; a captured one: bounded")
        for bounded in (False, True):
            runs = res[bounded]
            dev_ms = min(r[0][0] for r in runs)
            wall = min(r[0][1] for r in runs)
            host = min(r[0][2] for r in runs)
            total, wide, mib = bin_stats(runs[-1][1], N)
            line = (f"  {label:<20s} {'bounded' if bounded else 'sync':<8s} {dev_ms:9.3f} {wall:8.3f} {host:8.3f} {mib:9.2f} "
                    f"{total:10d} {C * F if bounded else '-':>10} {wide if bounded else '-':>7}")
            lines.append(line)
            print(line, flush=True)
        del res, outs
        torch.cuda.empty_cache()
    lines.append("# fragments of the two paths bit-identical at every shape")
    pose = pose_times(args.pose_iters, dev)
    for mode, v in pose.items():
        line = f"  pose iteration 128^2, 20480 faces, {mode:<5s}: {min(v):.3f} ms (runs: {', '.join(f'{x:.3f}' for x in v)})"
        lines.append(line)
        print(line, flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "a") as f:
        f.write("\n".join(lines) + "\n\n")


if __name__ == "__main__":
    main()
