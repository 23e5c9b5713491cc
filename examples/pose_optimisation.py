#!/usr/bin/env python
"""Pose optimisation through the perturbed renderer: the experiment of experiments/eval.py (init_target :196-288,
init_renderers :124-194, optimize_pose :320-409, benchmark :576-661) on pertrenderer_b200 alone (no pytorch3d).

    python examples/pose_optimisation.py [--noise gaussian softras] [--trials 10] [--imsize 128] [--init 30]
                                          [--niter 100] [--nb-samples 16] [--adapt | --graph]

A Rubik-style cube (8 vertices, 12 faces, one colour per side: data/objs/rubiks/cube2.obj + its six-strip UV map) is
rendered at a random rotation with the hard operators (blur_radius 0, one face per pixel); the rotation is then
recovered from a start `--init` degrees away by Adam on the rotation vector, the image rendered by
MeshRenderer(MeshRasterizer(K=50, blur_radius = log(1/1e-4-1) sigma), RandomPhongShader(<noise pair>)).
Reports the final angle errors, the share of trials solved below 5 / 10 / 20 degrees, and iterations per second.
"""

from __future__ import annotations

import argparse
import math
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
import pertrenderer_b200 as pb  # noqa: E402


def cube_mesh(device):
    """Unit cube [-1,1]^3: 8 vertices, 12 faces (outward winding), one colour per side."""
    v = torch.tensor([[-1, -1, -1], [1, -1, -1], [1, 1, -1], [-1, 1, -1], [-1, -1, 1], [1, -1, 1], [1, 1, 1], [-1, 1, 1]],
                     dtype=torch.float32, device=device)
    f = torch.tensor([[0, 2, 1], [0, 3, 2], [4, 5, 6], [4, 6, 7], [0, 1, 5], [0, 5, 4], [2, 3, 7], [2, 7, 6], [1, 2, 6], [1, 6, 5],
                      [0, 4, 7], [0, 7, 3]], dtype=torch.int64, device=device)
    side = torch.tensor([[0.9, 0.1, 0.1], [0.1, 0.7, 0.1], [0.1, 0.2, 0.9], [0.9, 0.9, 0.1], [0.9, 0.5, 0.1], [0.9, 0.9, 0.9]],
                        device=device)
    return v, f, side.repeat_interleave(2, dim=0)


_HAT = {}


def so3_exp(w):
    """Rodrigues' formula (pytorch3d.transforms.so3_exponential_map, eval.py:341) for one rotation vector.  The hat
    matrix is one product with a constant (9,3) tensor: a dozen small launches instead of sixty."""
    hat = _HAT.get(w.device)
    if hat is None:
        e = torch.zeros(3, 3, 3)
        e[0, 1, 2] = e[1, 2, 0] = e[2, 0, 1] = -1.0  # K[i][j] = -eps_ijk k_k
        e[0, 2, 1] = e[1, 0, 2] = e[2, 1, 0] = 1.0
        hat = _HAT[w.device] = (e.reshape(9, 3).to(w.device), torch.eye(3, device=w.device))
    th = w.norm().clamp_min(1e-8)
    K = (hat[0] @ (w / th)).reshape(3, 3)
    return hat[1] + torch.sin(th) * K + (1 - torch.cos(th)) * (K @ K)


def so3_log(R):
    ang = torch.acos(((R.trace() - 1) / 2).clamp(-1, 1))
    ax = torch.stack((R[2, 1] - R[1, 2], R[0, 2] - R[2, 0], R[1, 0] - R[0, 1]))
    return ax / (2 * torch.sin(ang)).clamp_min(1e-8) * ang


def angle_deg(Ra, Rb):
    return math.degrees(math.acos(max(-1.0, min(1.0, ((Ra.T @ Rb).trace().item() - 1.0) / 2.0))))


def random_rotation(gen, device):
    q = torch.randn(4, generator=gen)
    q = (q / q.norm()).to(device)
    a, b, c, d = q
    return torch.stack((torch.stack((a * a + b * b - c * c - d * d, 2 * (b * c - a * d), 2 * (b * d + a * c))),
                        torch.stack((2 * (b * c + a * d), a * a - b * b + c * c - d * d, 2 * (c * d - a * b))),
                        torch.stack((2 * (b * d - a * c), 2 * (c * d + a * b), a * a - b * b - c * c + d * d))))


def make_renderer(noise, cameras, lights, sigma, gamma, nb_samples, imsize, device, K=50):
    pairs = {
        "gaussian": lambda: (pb.GaussianRast(nb_samples=nb_samples, sigma=sigma), pb.GaussianAgg(nb_samples=nb_samples, gamma=gamma, alpha=1.0)),
        "gaussian_wovr": lambda: (pb.GaussianRast_wovr(nb_samples=nb_samples, sigma=sigma),
                                  pb.GaussianAgg_wovr(nb_samples=nb_samples, gamma=gamma, alpha=1.0)),
        "cauchy": lambda: (pb.ArctanRast(sigma=sigma), pb.CauchyAgg(nb_samples=nb_samples, gamma=gamma, alpha=1.0)),
        "softras": lambda: (pb.SoftRast(sigma=sigma), pb.SoftAgg(gamma=gamma, alpha=1.0)),
        "hard": lambda: (pb.HardRast(), pb.HardAgg()),
    }
    rast_op, agg_op = pairs[noise]()
    hard = noise == "hard"
    settings = pb.RasterizationSettings(image_size=imsize, blur_radius=0.0 if hard else math.log(1.0 / 1e-4 - 1.0) * sigma,
                                        faces_per_pixel=1 if hard else K)
    return pb.MeshRenderer(
        rasterizer=pb.MeshRasterizer(cameras=cameras, raster_settings=settings),
        shader=pb.RandomPhongShader(device=device, cameras=cameras, lights=lights,
                                    blend_params=pb.BlendParams(sigma=sigma, gamma=gamma, background_color=(0.0, 0.0, 0.0)),
                                    smoothrast=rast_op, smoothagg=agg_op))


def optimize_pose(mesh, verts, renderer, target_rgb, w_init, niter, lr, adapt, adapt_params=(1.1, 1.5)):
    """eval.py:320-409: Adam on the rotation vector, best-loss pose returned; with `adapt`, after iteration 100 the
    smoothing is divided by (1.1, 1.5) and the sample count doubled every 50 iterations while the running gamma
    gradient is positive."""
    w = w_init.clone().requires_grad_(True)
    opt = torch.optim.Adam([w], lr=lr, fused=True)  # one kernel per step
    best, best_w = float("inf"), w.detach().clone()
    v_gamma = 0.0
    for i in range(niter):
        opt.zero_grad()
        img = renderer(mesh.update_padded(verts @ so3_exp(w)))
        loss = ((img[..., :3] - target_rgb) ** 2).mean()
        loss.backward()
        if loss.item() < best:
            best, best_w = loss.item(), w.detach().clone()
        if w.grad.norm().item() > 1000.0:  # eval.py:375-378
            w.grad = 1e-5 * torch.randn_like(w.grad)
        opt.step()
        if adapt and i > 100:
            sigma, gamma, _ = renderer.shader.get_smoothing()
            if gamma.grad is not None:
                v_gamma = 0.9 * v_gamma + 0.1 * gamma.grad.item()
                sigma.grad, gamma.grad = torch.zeros_like(sigma.grad), torch.zeros_like(gamma.grad)
            if v_gamma > 0 and (i + 1) % 50 == 0:
                s_new, g_new = max(sigma.item() / adapt_params[0], 5e-5), max(gamma.item() / adapt_params[1], 5e-4)
                renderer.rasterizer.raster_settings.blur_radius = math.log(1.0 / 1e-4 - 1.0) * s_new
                renderer.shader.update_smoothing(sigma=s_new, gamma=g_new)
                renderer.shader.update_nb_samples(nb_samples=min(2 * renderer.shader.get_nb_samples(), 128))
                lr = max(lr / 1.5, 1e-4)
                opt = torch.optim.Adam([w], lr=lr)
    return best_w


def optimize_pose_graphed(mesh, verts, renderer, target_rgb, w_init, niter, lr, warmup=3):
    """The same loop with ONE CUDA graph per iteration (render + loss + backward + best-pose bookkeeping + gradient guard
    + Adam): the eager loop issues ~250 launches per iteration for < 0.5 ms of kernels, a replay issues one.  What makes
    the capture possible: the noise seeds live on the device (ops.device_seeds + a seed_advance node per replay), the
    smoothing scalars do not ask for gradients (no 12-byte read-back in backward), Adam is `capturable`, and the
    best-loss / exploding-gradient logic of eval.py:371-378 runs on the device (torch.where) instead of through .item().
    The first `warmup` iterations run eagerly (they are ordinary iterations of the optimisation)."""
    from pertrenderer_b200 import ops
    dev = w_init.device
    for t in renderer.shader.get_smoothing():
        t.requires_grad_(False)
    w = w_init.clone().requires_grad_(True)
    opt = torch.optim.Adam([w], lr=lr, capturable=True)
    seeds = torch.tensor([ops.draw_seed(), ops.draw_seed()], dtype=torch.int64, device=dev)
    best = torch.full((), float("inf"), device=dev)
    best_w = w.detach().clone()

    def iteration():
        ops.seed_advance(seeds)
        opt.zero_grad(set_to_none=True)
        img = renderer(mesh.update_padded(verts @ so3_exp(w)))
        loss = ((img[..., :3] - target_rgb) ** 2).mean()
        loss.backward()
        better = loss.detach() < best
        best_w.copy_(torch.where(better, w.detach(), best_w))
        best.copy_(torch.where(better, loss.detach(), best))
        g = w.grad
        g.copy_(torch.where(g.norm() > 1000.0, 1e-5 * torch.randn_like(g), g))  # eval.py:375-378
        opt.step()

    with ops.device_seeds(seeds):
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(min(warmup, niter)):
                iteration()
        torch.cuda.current_stream(dev).wait_stream(side)
        if niter > warmup:
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                iteration()
            for _ in range(niter - warmup):  # the capture itself executes nothing
                graph.replay()
    return best_w.clone()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--noise", nargs="+", default=["softras", "gaussian"], choices=["gaussian", "gaussian_wovr", "cauchy", "softras"])
    ap.add_argument("--trials", type=int, default=10)
    ap.add_argument("--imsize", type=int, default=128)
    ap.add_argument("--init", type=float, default=30.0, help="initial perturbation in degrees (eval.py pert_init_intensity)")
    ap.add_argument("--niter", type=int, default=100)
    ap.add_argument("--lr", type=float, default=5e-2)
    ap.add_argument("--sigma", type=float, default=1e-3)
    ap.add_argument("--gamma", type=float, default=1e-2)
    ap.add_argument("--nb-samples", type=int, default=16)
    ap.add_argument("--adapt", action="store_true")
    ap.add_argument("--graph", action="store_true", help="one CUDA graph per iteration (not with --adapt: the smoothing is frozen in it)")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--kernel-flags", type=int, default=0, help="PERT_F_* flags for every perturbed op (4 = per-sample noise, 8192 = Philox-7)")
    args = ap.parse_args()
    if args.kernel_flags:
        from pertrenderer_b200 import ops
        ctx = ops.kernel_flags(args.kernel_flags)
        ctx.__enter__()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: the renderer has no CPU fallback")
    dev = "cuda:0"
    verts, faces, colors = cube_mesh(dev)
    mesh = pb.TriMeshes(verts, faces, face_colors=colors)
    R, T = pb.look_at_view_transform(dist=6.7, elev=30.0, azim=120.0, device=dev)  # eval.py:244-255
    cameras = pb.OpenGLPerspectiveCameras(R=R, T=T, fov=60, device=dev)
    lights = pb.PointLights(location=[[0.0, 2.0, -2.0]], device=dev)
    hard = make_renderer("hard", cameras, lights, 1e-4, 1e-4, 1, args.imsize, dev)
    gen = torch.Generator().manual_seed(args.seed)
    torch.manual_seed(args.seed)
    results = {}
    for noise in args.noise:  # warm-up: lazy module loading (forward AND backward) is not part of the timed iterations
        w = torch.zeros(3, device=dev).add_(0.1).requires_grad_(True)
        r = make_renderer(noise, cameras, lights, args.sigma, args.gamma, args.nb_samples, args.imsize, dev)
        opt = torch.optim.Adam([w], lr=1e-3, fused=True)
        for _ in range(3):
            opt.zero_grad()
            r(mesh.update_padded(verts @ so3_exp(w)))[..., :3].mean().backward()
            opt.step()
    for noise in args.noise:
        errs, inits, t_iter = [], [], []
        for _ in range(args.trials):
            R_true = random_rotation(gen, dev)
            with torch.no_grad():
                target = hard(mesh.update_padded(verts @ R_true))[..., :3]
            axis = torch.randn(3, generator=gen).to(dev)
            R_init = R_true @ so3_exp(math.radians(args.init) * axis / axis.norm())
            w0 = so3_log(R_init)
            renderer = make_renderer(noise, cameras, lights, args.sigma, args.gamma, args.nb_samples, args.imsize, dev)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            if args.graph and not args.adapt and noise in ("gaussian", "gaussian_wovr", "cauchy", "softras"):  # the fused pairs (device-side seeds)
                w = optimize_pose_graphed(mesh, verts, renderer, target, w0, args.niter, args.lr)
            else:
                w = optimize_pose(mesh, verts, renderer, target, w0, args.niter, args.lr, args.adapt)
            torch.cuda.synchronize()
            t_iter.append((time.perf_counter() - t0) / args.niter)
            inits.append(angle_deg(so3_exp(w0), R_true))
            errs.append(angle_deg(so3_exp(w), R_true))
        solved = {th: sum(e < th for e in errs) / len(errs) for th in (5, 10, 20)}
        results[noise] = dict(mean_init=sum(inits) / len(inits), mean_final=sum(errs) / len(errs), solved=solved,
                              ms_per_iteration=1e3 * sum(t_iter) / len(t_iter))
        print(f"{noise:9s} init {results[noise]['mean_init']:.1f} deg -> final {results[noise]['mean_final']:.2f} deg | "
              f"solved <5/10/20 deg: {solved[5]:.0%} / {solved[10]:.0%} / {solved[20]:.0%} | "
              f"{results[noise]['ms_per_iteration']:.2f} ms per iteration (render + backward + Adam, {args.imsize}x{args.imsize}, "
              f"K=50, S={args.nb_samples})")
    return results


if __name__ == "__main__":
    main()
