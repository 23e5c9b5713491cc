"""Texture-atlas Phong at BASELINE config 2 (8 x 256^2, K = 50): the atlas looked up inside the Phong kernels
(pert_phong_atlas_fwd/bwd) against AtlasTexels.materialize followed by Phong on the dense texel tensor.

Fragments of a real rasterisation: bench.py's 1280-face icosphere seen by 8 orbiting cameras through MeshRasterizer, the
atlas (1280, R, R, 3) repeated per view as TriMeshes does.  One step = phong_shading forward (sparse, as RandomPhongShader
calls it with a fused pair) + backward from a fixed colour gradient, the atlas requiring grad; "+mesh" also differentiates
the vertex positions.  Device time = CUDA events around each step, median over the timed steps, the two paths alternated;
peak = torch.cuda.max_memory_allocated during one step above what was allocated before it (inputs); held = allocated after
forward above the same baseline (what autograd keeps for backward, the colours included).

    python tools/time_atlas.py [--steps 10] [--out FILE]
"""
import argparse
import os
import statistics
import subprocess
import sys
import types

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import pertrenderer_b200 as pb  # noqa: E402

N, HW, K = 8, 256, 50
MiB = 1024.0 * 1024.0


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = f"nvidia-smi unavailable: {e!r}"
    return name, q


def setup(dev):
    fr, _ = bench.rasterised_fragments(types.SimpleNamespace(views=N, image_size=HW, faces_per_pixel=K), dev)
    verts, faces = pb.synthetic_mesh(1280, device=dev)
    Rm, T = pb.look_at_view_transform(dist=2.7, elev=30.0, azim=torch.linspace(0, 315, N), device=dev)
    cams = pb.ViewCameras(R=Rm, T=T, device=dev)
    lights, mats = pb.PointLights(location=[[0.0, 2.0, -2.0]], device=dev), pb.Materials(device=dev)
    g = torch.randn(fr.pix_to_face.shape + (3,), device=dev, generator=torch.Generator(device=dev).manual_seed(1))
    g = g * (fr.pix_to_face >= 0)[..., None]
    return fr, verts, faces, cams, lights, mats, g


def make_step(path, fr, verts, faces, cams, lights, mats, g, atlas1, mesh_grad):
    def step():
        a = atlas1.detach().requires_grad_(True)
        v = verts.detach().requires_grad_(mesh_grad)
        mesh = pb.TriMeshes(v, faces).extend(N) if not mesh_grad else pb.TriMeshes(v.expand(N, -1, -1), faces)
        atlas = a.repeat(N, 1, 1, 1)
        if path == "kernel":
            texels = pb.AtlasTexels(atlas)
        else:
            texels = pb.AtlasTexels(atlas).materialize(fr.pix_to_face, fr.bary_coords)
        col = pb.phong_shading(mesh, fr, lights, cams, mats, texels, sparse=True)
        held = torch.cuda.memory_allocated()
        col.backward(g)
        return held, a.grad
    return step


def measure(steps, out):
    dev = torch.device("cuda", 0)
    name, smi = card()
    lines = [f"# tools/time_atlas.py --steps {steps}",
             "# BASELINE config 2 (8 x 256^2, K = 50), rasterised fragments (bench.py's 1280-face icosphere, 8 views); "
             "phong_shading forward (sparse) + backward, atlas requiring grad; device ms = median of CUDA-event step times, "
             "paths alternated; peak / held = max_memory_allocated during one step / allocated after forward, above the inputs",
             f"# card: {name}; nvidia-smi name, power limit: {smi}"]
    fr, verts, faces, cams, lights, mats, g = setup(dev)
    print("# fragments ready", flush=True)
    valid = (fr.pix_to_face >= 0).sum().item()
    lines.append(f"# valid entries {valid} of {fr.pix_to_face.numel()} ({valid / fr.pix_to_face.numel():.3f})")
    for R in (4, 8):
        atlas1 = torch.rand((faces.shape[0], R, R, 3), device=dev, generator=torch.Generator(device=dev).manual_seed(R))
        for mesh_grad in (False, True):
            steps_by = {p: make_step(p, fr, verts, faces, cams, lights, mats, g, atlas1, mesh_grad) for p in ("kernel", "materialize")}
            grads = {}
            for p, fn in steps_by.items():  # warm-up, and the gradients of both paths
                for _ in range(3):
                    grads[p] = fn()[1]
            print(f"# R={R} mesh_grad={mesh_grad}: warmed up", flush=True)
            diff = ((grads["kernel"] - grads["materialize"]).abs().max() / grads["materialize"].abs().max()).item()
            mem = {}
            for p, fn in steps_by.items():
                torch.cuda.synchronize()
                base = torch.cuda.memory_allocated()
                torch.cuda.reset_peak_memory_stats()
                held, _ = fn()
                torch.cuda.synchronize()
                mem[p] = ((torch.cuda.max_memory_allocated() - base) / MiB, (held - base) / MiB)
            times = {p: [] for p in steps_by}
            for _ in range(steps):
                for p, fn in steps_by.items():
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    fn()
                    e1.record()
                    e1.synchronize()
                    times[p].append(e0.elapsed_time(e1))
            tag = f"R={R} {'+mesh' if mesh_grad else 'atlas'}"
            print(f"# {tag}: timed", flush=True)
            for p in steps_by:
                lines.append(f"{tag:12s} {p:12s} {statistics.median(times[p]):8.3f} ms  peak {mem[p][0]:9.1f} MiB  "
                             f"held {mem[p][1]:9.1f} MiB")
            k, m = statistics.median(times["kernel"]), statistics.median(times["materialize"])
            lines.append(f"{tag:12s} kernel / materialize time {k / m:.3f}; peak saved {mem['materialize'][0] - mem['kernel'][0]:.1f} "
                         f"MiB, held saved {mem['materialize'][1] - mem['kernel'][1]:.1f} MiB; grad_atlas rel diff {diff:.1e}")
    text = "\n".join(lines)
    print(text)
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("tools/time_atlas.py measures on a CUDA device; none is visible")
    measure(a.steps, a.out)
