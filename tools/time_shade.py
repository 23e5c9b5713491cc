"""Device-timed fused forward / backward at BASELINE config 2 (or --cfg N,HW,K,S) on the named fragment sets.
    python tools/time_shade.py [realistic dense rasterised] [--flags F] [--steps n] [--cfg 8,256,50,64]
    python tools/time_shade.py [kinds] --noise cauchy     the Cauchy pair (ArctanRast + CauchyAgg) through the public
        autograd interface, fused kernels against the operator-by-operator composition: forward ms, backward ms and
        peak memory (torch.cuda.max_memory_allocated) of each
    python tools/time_shade.py [kinds] --noise wovr       the same for the pair without control variates
        (GaussianRast_wovr + GaussianAgg_wovr)
    python tools/time_shade.py [kinds] --render [--s-agg 64,4096,65536]   forward-only render (ops.shade_render) against
        the training forward (ops.shade_forward), alternating, same seeds: device time of each, peak memory above the
        inputs of one call of each, and whether the images are equal"""
import argparse
import os
import sys
import types

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from pertrenderer_b200 import ops, synthetic_fragments  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("kinds", nargs="*", default=["realistic", "dense", "rasterised"])
ap.add_argument("--flags", type=int, default=0)
ap.add_argument("--steps", type=int, default=10)
ap.add_argument("--cfg", default="8,256,50,64")
ap.add_argument("--tag", default="")
ap.add_argument("--lib", default=None, help="alternate libpertshade.so (A/B runs of two builds in one GPU call)")
ap.add_argument("--noise", default="gaussian", choices=["gaussian", "cauchy", "wovr"])
ap.add_argument("--render", action="store_true")
ap.add_argument("--s-agg", default="64,4096,65536", help="aggregation sample counts of --render")
a = ap.parse_args()
if a.lib:
    from pertrenderer_b200 import _cabi
    _cabi.LIB_PATH = os.path.abspath(a.lib)
N, HW, K, S = (int(v) for v in a.cfg.split(","))
dev = torch.device("cuda:0")
peak = bench.peaks()[0]


def time_pair(kind, fr, col, G):
    """Fused (smooth_rgb_blend) and composition arm of the --noise pair, same inputs, median of a.steps steps each."""
    import pertrenderer_b200 as pb
    from pertrenderer_b200.random_rasterizer import _composed_rgb_blend
    rast_cls, agg_cls = (pb.ArctanRast, pb.CauchyAgg) if a.noise == "cauchy" else (pb.GaussianRast_wovr, pb.GaussianAgg_wovr)
    for name, fn in (("fused", pb.smooth_rgb_blend), ("composition", _composed_rgb_blend)):
        rast, agg = rast_cls(nb_samples=S, sigma=1e-3), agg_cls(nb_samples=S, gamma=1e-2, alpha=1.0)
        d, z, c = fr.dists.clone().requires_grad_(True), fr.zbuf.clone().requires_grad_(True), col.clone().requires_grad_(True)
        frag = pb.Fragments(fr.pix_to_face, z, None, d)
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(a.steps)]
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        for i in range(-3, a.steps):
            if i >= 0:
                ev[i][0].record()
            img = fn(c, frag, rast, agg, pb.BlendParams())
            if i >= 0:
                ev[i][1].record()
            (img * G).sum().backward()
            if i >= 0:
                ev[i][2].record()
            d.grad = z.grad = c.grad = None
            del img
        torch.cuda.synchronize()
        f = sorted(e[0].elapsed_time(e[1]) for e in ev)[len(ev) // 2]
        b = sorted(e[1].elapsed_time(e[2]) for e in ev)[len(ev) // 2]
        mem = (torch.cuda.max_memory_allocated() - base) / 2 ** 20
        print(f"{a.tag} {a.noise} {kind:10s} {name:11s} fwd {f:.4f} ms  bwd {b:.4f} ms  fwd+bwd {f + b:.4f} ms  "
              f"peak +{mem:.0f} MiB over the inputs", flush=True)


def peak_above_inputs(fn):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    out = fn()
    torch.cuda.synchronize()
    return (torch.cuda.max_memory_allocated() - base) / 2 ** 20, out


def time_render(kind, fr, col):
    """Training forward and forward-only render of the same problems, alternating step by step (config S = S_rast)."""
    for S_agg in (int(v) for v in a.s_agg.split(",")):
        steps = a.steps if S_agg <= 4096 else max(3, a.steps // 3)

        def problem(i):
            return ops.ShadeProblem(pix_to_face=fr.pix_to_face, zbuf=fr.zbuf, dists=fr.dists, colors=col, znear=1.0,
                                    zfar=100.0, background=(1.0, 1.0, 1.0), sigma=1e-3, gamma=1e-2, alpha=1.0, eps=1e-10,
                                    S_rast=S, S_agg=S_agg, seed_rast=100 + i, seed_agg=200 + i, flags=a.flags)
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(steps)]
        same = True
        for i in range(-2, steps):
            pr = problem(i)
            if i >= 0:
                ev[i][0].record()
            image, saved = ops.shade_forward(pr)
            if i >= 0:
                ev[i][1].record()
            del saved
            if i >= 0:
                ev[i][2].record()
            rendered = ops.shade_render(pr)
            if i >= 0:
                ev[i][3].record()
            same = same and torch.equal(image, rendered)
            del image, rendered
        torch.cuda.synchronize()
        t_fwd = sorted(e[0].elapsed_time(e[1]) for e in ev)[steps // 2]
        t_ren = sorted(e[2].elapsed_time(e[3]) for e in ev)[steps // 2]
        m_fwd, _ = peak_above_inputs(lambda: ops.shade_forward(problem(0)))
        m_ren, _ = peak_above_inputs(lambda: ops.shade_render(problem(0)))
        print(f"{a.tag} render {kind:10s} S_rast {S} S_agg {S_agg:6d}  training fwd {t_fwd:9.4f} ms  +{m_fwd:8.1f} MiB   "
              f"render {t_ren:9.4f} ms  +{m_ren:6.1f} MiB   speed-up {t_fwd / t_ren:5.2f}x   same image {same}", flush=True)


if a.render:
    import subprocess
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    print(f"# {torch.cuda.get_device_name(dev)}; nvidia-smi name, power limit: {q.stdout.strip() or 'unavailable'}", flush=True)

for kind in a.kinds:
    if kind == "rasterised":
        fr, col = bench.rasterised_fragments(types.SimpleNamespace(views=N, image_size=HW, faces_per_pixel=K, nb_samples=S), dev)
    else:
        fr, col = synthetic_fragments(N, HW, HW, K, kind=kind, sigma=1e-3, seed=0, device=dev)
    if a.render:
        time_render(kind, fr, col)
        continue
    G = torch.randn((N, HW, HW, 4), device=dev, generator=torch.Generator(device=dev).manual_seed(1))
    if a.noise != "gaussian":
        time_pair(kind, fr, col, G)
        continue
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(a.steps)]
    for i in range(-3, a.steps):
        pr = ops.ShadeProblem(pix_to_face=fr.pix_to_face, zbuf=fr.zbuf, dists=fr.dists, colors=col, znear=1.0, zfar=100.0,
                              background=(1.0, 1.0, 1.0), sigma=1e-3, gamma=1e-2, alpha=1.0, eps=1e-10, S_rast=S, S_agg=S,
                              seed_rast=100 + i, seed_agg=200 + i, flags=a.flags)
        if i >= 0:
            ev[i][0].record()
        image, saved = ops.shade_forward(pr)
        if i >= 0:
            ev[i][1].record()
        out = ops.shade_backward(pr, saved, G)
        if i >= 0:
            ev[i][2].record()
    torch.cuda.synchronize()
    f = sorted(e[0].elapsed_time(e[1]) for e in ev)[len(ev) // 2]
    b = sorted(e[1].elapsed_time(e[2]) for e in ev)[len(ev) // 2]
    P = N * HW * HW
    fb, bb = bench.alg_bytes(P, K)
    print(f"{a.tag} {kind:10s} fwd {f:.4f} ms ({fb / f / 1e6 / peak:.3f})  bwd {b:.4f} ms ({bb / b / 1e6 / peak:.3f})  "
          f"fwd+bwd {f + b:.4f} ms ({(fb + bb) / (f + b) / 1e6 / peak:.3f})  img {float(image.sum()):.1f}", flush=True)
