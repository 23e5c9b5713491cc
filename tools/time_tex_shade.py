"""Textures sampled inside the fused shading kernels at BASELINE config 2 (8 x 256^2, K = 50, Gaussian pair): the texel
computed where the kernels blend it (pert_shade_tex_fwd / _bwd / _render) against today's path, which materialises the
(N,H,W,K,3) colours with the texture-only Phong kernel, feeds them to pert_shade_fwd / _bwd / _render, and scatters the
colour gradient back into the table with the texture-only Phong backward.

Fragments of a real rasterisation: bench.py's 1280-face icosphere seen by 8 orbiting cameras through MeshRasterizer with
experiments/eval.py's blur.  Textures of the repeated mesh: corner colours (F,3,3), one 256 x 256 UV map, a 4 x 4 atlas.
Device ms = median over the timed steps of CUDA events around forward, backward and the forward-only render, the two paths
alternated in the same process; peak = torch.cuda.max_memory_allocated during forward + backward above what was allocated
before (the inputs).  Both paths keep grad_dists / grad_zbuf alive to the end of backward, as autograd does (they wait for
the rasteriser's backward), and both compute grad_bary, except the in-kernel atlas: its texel is piecewise constant in bary,
so its bary gradient is zero and nothing is allocated for it (the materialising path writes a zero tensor).

    python tools/time_tex_shade.py [--steps 20] [--out FILE]
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
from pertrenderer_b200 import ops, shading  # noqa: E402

N, HW, K, S = 8, 256, 50, 16
MiB = 1024.0 * 1024.0


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = f"nvidia-smi unavailable: {e!r}"
    return name, q


def textures(F, dev):
    g = torch.Generator(device=dev).manual_seed(3)
    return dict(vert=(torch.rand(F, 3, 3, device=dev, generator=g), None),
                uv=(torch.rand(1, 256, 256, 3, device=dev, generator=g), torch.rand(F, 3, 2, device=dev, generator=g)),
                atlas=(torch.rand(F, 4, 4, 3, device=dev, generator=g), None))


def src_of(kind, table, face_uvs):
    return dict(vert_colors=table) if kind == "vert" else dict(uv=(table, face_uvs)) if kind == "uv" else dict(atlas=table)


def make_paths(fr, kind, table, face_uvs, G):
    common = dict(pix_to_face=fr.pix_to_face, zbuf=fr.zbuf, dists=fr.dists, znear=1.0, zfar=100.0, background=(1.0, 1.0, 1.0),
                  sigma=1e-4, gamma=1e-4, alpha=1.0, eps=1e-10, S_rast=S, S_agg=S, seed_rast=1, seed_agg=2)
    p2f, bary = fr.pix_to_face, fr.bary_coords
    src = src_of(kind, table, face_uvs)

    def old_fwd():
        colors = shading.phong_forward(p2f, bary, None, None, None, None, None, sparse=True, unlit=True, **src)
        pr = ops.ShadeProblem(colors=colors, **common)
        return (pr,) + ops.shade_forward(pr)

    def old_bwd(st):  # grad_dists / grad_zbuf stay alive through the Phong backward, as under autograd
        pr, _, saved = st
        gd, gz, gc, _ = ops.shade_backward(pr, saved, G)
        return shading.phong_backward(p2f, bary, None, None, None, None, None, gc, need_verts=False, need_normals=False,
                                      sparse=True, unlit=True, **src)[:2], gd, gz

    def old_render():
        colors = shading.phong_forward(p2f, bary, None, None, None, None, None, sparse=True, unlit=True, **src)
        return ops.shade_render(ops.ShadeProblem(colors=colors, **common))

    tex = ops.ShadeTexture(kind=kind, bary=bary, table=table, face_uvs=face_uvs)

    def new_fwd():
        pr = ops.ShadeProblem(colors=None, texture=tex, **common)
        return (pr,) + ops.shade_forward(pr)

    def new_bwd(st):
        pr, _, saved = st
        gd, gz, g, _ = ops.shade_backward(pr, saved, G, need_bary=kind != "atlas")
        return g, gd, gz

    def new_render():
        return ops.shade_render(ops.ShadeProblem(colors=None, texture=tex, **common))

    return {"materialise": (old_fwd, old_bwd, old_render), "in-kernel": (new_fwd, new_bwd, new_render)}


def timed(fn, *args):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn(*args)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1), out


def measure(steps, out):
    dev = torch.device("cuda", 0)
    name, smi = card()
    lines = [f"# tools/time_tex_shade.py --steps {steps}",
             "# BASELINE config 2 (8 x 256^2, K = 50, S = 16), Gaussian pair, rasterised fragments (bench.py's 1280-face "
             "icosphere, 8 views, eval.py's blur); device ms = median of CUDA-event times, paths alternated; peak = "
             "max_memory_allocated during forward + backward above the inputs; both paths hold grad_dists / grad_zbuf to the end "
             "of backward, as under autograd",
             f"# card: {name}; nvidia-smi name, power limit: {smi}"]
    fr, _ = bench.rasterised_fragments(types.SimpleNamespace(views=N, image_size=HW, faces_per_pixel=K), dev)
    fr = pb.Fragments(fr.pix_to_face, fr.zbuf, fr.bary_coords.contiguous(), fr.dists)
    F = int(fr.pix_to_face.max().item()) + 1
    valid = (fr.pix_to_face >= 0).sum().item()
    lines.append(f"# valid entries {valid} of {fr.pix_to_face.numel()} ({valid / fr.pix_to_face.numel():.3f}); "
                 f"colour tensor {N * HW * HW * K * 12 / MiB:.1f} MiB")
    G = torch.randn((N, HW, HW, 4), device=dev, generator=torch.Generator(device=dev).manual_seed(1))
    for kind, (table, face_uvs) in textures(F, dev).items():
        paths = make_paths(fr, kind, table, face_uvs, G)
        res = {}
        for p, (fwd, bwd, render) in paths.items():  # warm-up, and the results of both paths
            for _ in range(2):
                st = fwd()
                res[p] = (st[1], bwd(st), render())
        img_eq = torch.equal(res["in-kernel"][0], res["materialise"][0])
        rnd_eq = torch.equal(res["in-kernel"][2], res["materialise"][2])
        gt_n, gt_o = res["in-kernel"][1][0][0], res["materialise"][1][0][0]
        gdiff = ((gt_n - gt_o).abs().max() / gt_o.abs().max()).item()
        del res
        peak = {}
        for p, (fwd, bwd, _) in paths.items():
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            r = bwd(fwd())
            torch.cuda.synchronize()
            peak[p] = (torch.cuda.max_memory_allocated() - base) / MiB
            del r
        times = {p: ([], [], []) for p in paths}
        for _ in range(steps):
            for p, (fwd, bwd, render) in paths.items():
                tf, st = timed(fwd)
                tb, _ = timed(bwd, st)
                tr, _ = timed(render)
                del st
                for lst, t in zip(times[p], (tf, tb, tr)):
                    lst.append(t)
        print(f"# {kind}: timed", flush=True)
        med = {p: [statistics.median(x) for x in times[p]] for p in paths}
        for p in paths:
            f, b, r = med[p]
            lines.append(f"{kind:6s} {p:12s} forward {f:7.3f} ms  backward {b:7.3f} ms  render {r:7.3f} ms  peak {peak[p]:8.1f} MiB")
        n, o = med["in-kernel"], med["materialise"]
        lines.append(f"{kind:6s} in-kernel / materialise: forward {n[0] / o[0]:.3f}, backward {n[1] / o[1]:.3f}, render "
                     f"{n[2] / o[2]:.3f}; peak saved {peak['materialise'] - peak['in-kernel']:.1f} MiB; image equal {img_eq}, "
                     f"render equal {rnd_eq}; grad_table rel diff {gdiff:.1e}")
    text = "\n".join(lines)
    print(text)
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("tools/time_tex_shade.py measures on a CUDA device; none is visible")
    measure(a.steps, a.out)
