"""Parity of the fragment-producer kernels (pert_rasterize_fwd / pert_rasterize_bwd, through the C ABI) with the CPU
oracle (oracle/raster_oracle.py: pytorch3d 0.4.0's naive rasteriser restated), and the end-to-end renderer
MeshRenderer(MeshRasterizer, RandomPhongShader) of experiments/eval.py:165-177 on a small pose optimisation."""

import math

import pytest
import torch

from conftest import rel_err
from oracle import raster_oracle as RO
from raster_util import check_fragments

pytestmark = pytest.mark.gpu

DEV = "cuda"


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _faces_ndc(n_faces, n_views, seed=0, elev=20.0):
    """Packed NDC faces of a sphere seen by n_views orbiting cameras, on the CPU."""
    import pertrenderer_b200 as pb
    verts, faces = pb.synthetic_mesh(n_faces, device="cpu")
    R, T = pb.look_at_view_transform(dist=2.7, elev=elev, azim=torch.linspace(0.0, 150.0, n_views) + 10.0 * seed)
    cam = pb.FoVPerspectiveCameras(R=R, T=T)
    ndc = cam.transform_points_ndc(verts)  # (N,V,3)
    fv = ndc[:, faces].reshape(-1, 3, 3).contiguous()
    F_ = faces.shape[0]
    return fv, [i * F_ for i in range(n_views + 1)]


@pytest.mark.parametrize("cfg", [
    dict(n_faces=80, views=2, H=24, W=24, K=8, blur=1e-3),
    dict(n_faces=320, views=1, H=40, W=33, K=6, blur=5e-3),      # non-square, partial tiles
    dict(n_faces=1280, views=3, H=32, W=32, K=50, blur=9.21e-3),  # eval.py: K=50, blur = log(1/1e-4-1)*sigma
    dict(n_faces=20, views=1, H=16, W=16, K=2, blur=0.0),         # K smaller than the number of overlapping faces
    dict(n_faces=320, views=1, H=24, W=24, K=100, blur=9.21e-3),  # K > 64: K-buffer in the output rows
])
def test_rasterize_forward_matches_oracle(cfg):
    import pertrenderer_b200 as pb
    fv, start = _faces_ndc(cfg["n_faces"], cfg["views"], seed=cfg["K"])
    got = pb.rasterize_meshes(fv.to(DEV), torch.tensor(start, device=DEV), (cfg["H"], cfg["W"]), cfg["blur"], cfg["K"])
    torch.cuda.synchronize()
    ref = check_fragments(got, fv, start, cfg["H"], cfg["W"], cfg["K"], cfg["blur"])
    assert (ref[0] >= 0).float().mean() > 0.02
    z = got[1].cpu()
    valid = got[0].cpu() >= 0
    # ascending depth, padding last
    zz = torch.where(valid, z, torch.full_like(z, float("inf")))
    assert (zz[..., 1:] >= zz[..., :-1]).all()
    assert (valid[..., 1:] <= valid[..., :-1]).all()


def test_coarse_bins_give_the_same_fragments(monkeypatch):
    """Meshes of thousands of faces go through per-tile candidate lists (pert_rasterize_bin); the fragments are those of
    the walk over all faces, and of the oracle."""
    import pertrenderer_b200 as pb
    from pertrenderer_b200 import rasterizer
    fv, start = _faces_ndc(5120, 2, seed=1)
    H, W, K, blur = 40, 72, 8, 2e-3
    fs = torch.tensor(start, device=DEV)
    monkeypatch.setattr(rasterizer, "BIN_MIN_FACES", 1024)
    binned = pb.rasterize_meshes(fv.to(DEV), fs, (H, W), blur, K)
    monkeypatch.setattr(rasterizer, "BIN_MIN_FACES", 10 ** 9)
    plain = pb.rasterize_meshes(fv.to(DEV), fs, (H, W), blur, K)
    for a, b in zip(binned, plain):
        assert torch.equal(a, b)
    check_fragments(binned, fv, start, H, W, K, blur)
    # gradients flow through the binned forward as well
    fvg = fv.to(DEV).requires_grad_(True)
    monkeypatch.setattr(rasterizer, "BIN_MIN_FACES", 1024)
    out = pb.rasterize_meshes(fvg, fs, (H, W), blur, K)
    (out[1].sum() + out[3].sum()).backward()
    assert torch.isfinite(fvg.grad).all() and fvg.grad.abs().sum() > 0


def test_rasterize_backward_matches_oracle_autograd():
    import pertrenderer_b200 as pb
    H = W = 28
    K = 6
    fv, start = _faces_ndc(80, 2, seed=3)
    blur = 4e-3
    fv_c = fv.to(DEV).requires_grad_(True)
    p2f, zbuf, bary, dists = pb.rasterize_meshes(fv_c, torch.tensor(start, device=DEV), H, blur, K)
    gen = torch.Generator().manual_seed(0)
    gz, gb, gd = torch.randn(zbuf.shape, generator=gen), torch.randn(bary.shape, generator=gen), torch.randn(dists.shape, generator=gen)
    gz[torch.rand(zbuf.shape, generator=gen) < 0.3] = 0.0
    ((zbuf * gz.to(DEV)).sum() + (bary * gb.to(DEV)).sum() + (dists * gd.to(DEV)).sum()).backward()
    # oracle: autograd over the restated formulas of the SAME selection
    fv_o = fv.clone().requires_grad_(True)
    z_o, b_o, d_o = RO.fragments_from_selection(fv_o, p2f.cpu(), H, W)
    mask = p2f.cpu() >= 0
    ((z_o * gz)[mask].sum() + (b_o * gb)[mask].sum() + (d_o * gd)[mask].sum()).backward()
    assert rel_err(fv_c.grad.cpu(), fv_o.grad) <= 2e-4  # fp32 sums of thousands of terms with 1/area^2 factors
    # each kind of gradient alone
    for which in range(3):
        fv_c2 = fv.to(DEV).requires_grad_(True)
        out = pb.rasterize_meshes(fv_c2, torch.tensor(start, device=DEV), H, blur, K)
        (out[1 + which] * (gz, gb, gd)[which].to(DEV)).sum().backward()
        fv_o2 = fv.clone().requires_grad_(True)
        ref = RO.fragments_from_selection(fv_o2, p2f.cpu(), H, W)
        m = mask if which != 1 else mask[..., None].expand_as(ref[1])
        (ref[which] * (gz, gb, gd)[which])[m].sum().backward()
        assert rel_err(fv_c2.grad.cpu(), fv_o2.grad) <= 2e-4, which


def test_renderer_chain_matches_oracle_chain():
    """MeshRasterizer -> RandomPhongShader(SoftRast, SoftAgg) against the oracle chain (raster oracle -> Phong oracle ->
    blend oracle) on the same mesh and camera: same selection, same image, and the same gradient on the fragments and on
    the mesh vertices (the quantity pose optimisation differentiates, eval.py:341-369)."""
    import pertrenderer_b200 as pb
    from oracle import pert_oracle as O
    from oracle import phong_oracle as PO
    torch.manual_seed(0)
    verts, faces = pb.synthetic_mesh(80, device="cpu")
    verts = verts * torch.tensor([1.0, 0.6, 0.8])
    fc = torch.rand(faces.shape[0], 3, generator=torch.Generator().manual_seed(1))
    R, T = pb.look_at_view_transform(dist=2.7, elev=30.0, azim=120.0)
    H = W = 32
    K = 20
    sigma, gamma = 1e-2, 5e-2
    blur = math.log(1.0 / 1e-4 - 1.0) * sigma
    G = torch.randn(1, H, W, 4, generator=torch.Generator().manual_seed(2))
    # oracle chain
    v_o = verts.clone().requires_grad_(True)
    cam_o = pb.OpenGLPerspectiveCameras(R=R, T=T)
    fv_o = cam_o.transform_points_ndc(v_o)[0][faces]
    p2f = RO.rasterize(fv_o.detach(), [0, faces.shape[0]], H, W, K, blur)[0]
    z_o, b_o, d_o = RO.fragments_from_selection(fv_o, p2f, H, W)
    for t in (z_o, b_o, d_o):
        t.retain_grad()
    mesh_o = pb.TriMeshes(v_o, faces, face_colors=fc)
    col_o = PO.phong_colors_from(mesh_o, pb.Fragments(p2f, z_o, b_o, d_o), pb.PointLights(location=[[0.0, 2.0, -2.0]]), cam_o,
                                 pb.Materials(), pb.FaceTexels(fc).materialize(p2f))
    img_o, _, _, gr = O.soft_shade_fwd_bwd(p2f, z_o.detach(), d_o.detach(), col_o.detach(), torch.tensor((0.0, 0.0, 0.0)),
                                           cam_o.znear.reshape(-1, 1, 1, 1), cam_o.zfar.reshape(-1, 1, 1, 1), sigma, gamma, 1.0, 1e-10, G)
    torch.autograd.backward([col_o, z_o, d_o], [gr["colors"], gr["zbuf"], gr["dists"]])
    # CUDA chain
    v_c = verts.to(DEV).requires_grad_(True)
    cam_c = pb.OpenGLPerspectiveCameras(R=R, T=T, device=DEV)
    rast = pb.MeshRasterizer(cam_c, pb.RasterizationSettings(image_size=H, blur_radius=blur, faces_per_pixel=K))
    shader = pb.RandomPhongShader(device=DEV, cameras=cam_c, lights=pb.PointLights(location=[[0.0, 2.0, -2.0]], device=DEV),
                                  materials=pb.Materials(device=DEV), blend_params=pb.BlendParams(background_color=(0.0, 0.0, 0.0)),
                                  smoothrast=pb.SoftRast(sigma=sigma), smoothagg=pb.SoftAgg(gamma=gamma, alpha=1.0))
    mesh_c = pb.TriMeshes(v_c, faces.to(DEV), face_colors=fc.to(DEV))
    frag_c = rast(mesh_c)
    for t in (frag_c.zbuf, frag_c.bary_coords, frag_c.dists):
        t.retain_grad()
    img_c = shader(frag_c, mesh_c)
    (img_c * G.to(DEV)).sum().backward()
    same = (frag_c.pix_to_face.cpu() == p2f).all(-1)
    assert same.float().mean() > 0.995
    m = (p2f >= 0) & same[..., None]
    assert (img_c.detach().cpu() - img_o)[same].abs().max() <= 5e-6
    assert rel_err(frag_c.zbuf.grad.cpu()[m], z_o.grad[m]) <= 1e-4
    assert rel_err(frag_c.dists.grad.cpu()[m], d_o.grad[m]) <= 1e-4
    assert rel_err(frag_c.bary_coords.grad.cpu()[m], b_o.grad[m]) <= 5e-4
    if same.all():
        assert rel_err(v_c.grad.cpu(), v_o.grad) <= 1e-3


@pytest.mark.parametrize("pair", ["softras", "gaussian"])
def test_renderer_end_to_end_pose_optimisation(pair):
    """MeshRenderer(MeshRasterizer, RandomPhongShader) as eval.py:135-177 builds it: render a target at a known rotation
    with the hard operators (eval.py:272-286), start 15 degrees off, run Adam on the rotation vector (eval.py:320-409):
    the angle error must drop.  (sigma = 3e-4: with a blur band as wide as the faces, pytorch3d-style unclipped
    barycentric extrapolation makes the image discontinuous in the pose; the CPU float64 chain behaves the same.)"""
    import pertrenderer_b200 as pb
    torch.manual_seed(0)
    verts, faces = pb.synthetic_mesh(80, device=DEV)
    verts = verts * torch.tensor([1.0, 0.6, 0.8], device=DEV)  # an ellipsoid: the pose is observable
    fc = torch.rand(faces.shape[0], 3, device=DEV, generator=torch.Generator(device=DEV).manual_seed(1))
    mesh = pb.TriMeshes(verts, faces, face_colors=fc)
    R, T = pb.look_at_view_transform(dist=2.7, elev=30.0, azim=120.0, device=DEV)
    cameras = pb.OpenGLPerspectiveCameras(R=R, T=T, device=DEV)
    lights = pb.PointLights(location=[[0.0, 2.0, -2.0]], device=DEV)
    sigma, gamma = 3e-4, 1e-2

    def make(rast_op, agg_op, sg):
        settings = pb.RasterizationSettings(image_size=48, blur_radius=math.log(1.0 / 1e-4 - 1.0) * sg, faces_per_pixel=16)
        return pb.MeshRenderer(
            rasterizer=pb.MeshRasterizer(cameras=cameras, raster_settings=settings),
            shader=pb.RandomPhongShader(device=DEV, cameras=cameras, lights=lights,
                                        blend_params=pb.BlendParams(background_color=(0.0, 0.0, 0.0)),
                                        smoothrast=rast_op, smoothagg=agg_op))

    if pair == "gaussian":
        renderer = make(pb.GaussianRast(nb_samples=64, sigma=sigma), pb.GaussianAgg(nb_samples=64, gamma=gamma, alpha=1.0), sigma)
    else:
        renderer = make(pb.SoftRast(sigma=sigma), pb.SoftAgg(gamma=gamma, alpha=1.0), sigma)
    hard = make(pb.HardRast(), pb.HardAgg(), 0.0)

    def rot(w):  # Rodrigues (so3_exponential_map, eval.py:341)
        th = w.norm().clamp_min(1e-8)
        k = w / th
        Kx = torch.zeros(3, 3, device=DEV)
        Kx[0, 1], Kx[0, 2], Kx[1, 0], Kx[1, 2], Kx[2, 0], Kx[2, 1] = -k[2], k[1], k[2], -k[0], -k[1], k[0]
        return torch.eye(3, device=DEV) + torch.sin(th) * Kx + (1 - torch.cos(th)) * (Kx @ Kx)

    w_true = torch.tensor([0.3, -0.5, 0.2], device=DEV)
    with torch.no_grad():
        target = hard(mesh.update_padded(verts @ rot(w_true)))[..., :3]
    assert target.shape == (1, 48, 48, 3) and target.sum() > 10
    axis = torch.tensor([0.6, 0.0, 0.8], device=DEV)
    w = (w_true + math.radians(15.0) * axis).clone().requires_grad_(True)
    opt = torch.optim.Adam([w], lr=2e-2)

    def angle_err():
        Rrel = rot(w.detach()).T @ rot(w_true)
        return math.degrees(math.acos(max(-1.0, min(1.0, (Rrel.trace().item() - 1.0) / 2.0))))

    a0 = angle_err()
    best_loss, a_best, closest = float("inf"), a0, a0
    for _ in range(60):
        opt.zero_grad()
        img = renderer(mesh.update_padded(verts @ rot(w)))
        loss = ((img[..., :3] - target) ** 2).mean()
        loss.backward()
        assert torch.isfinite(w.grad).all()
        if loss.item() < best_loss:  # eval.py:370-372 returns the pose of the lowest loss, not the last iterate
            best_loss, a_best = loss.item(), angle_err()
        opt.step()
        closest = min(closest, angle_err())
    assert closest < 0.4 * a0 and a_best < 0.6 * a0, (pair, a0, closest, a_best)


@pytest.mark.parametrize("pair", ["softras", "gaussian"])
def test_pose_iteration_captured_in_one_cuda_graph(pair):
    """examples/pose_optimisation.py --graph: render + loss + backward + best-pose bookkeeping + Adam of eval.py:341-394 as
    ONE CUDA graph per iteration (device-side seeds: ops.device_seeds + a seed_advance node).  The angle error must drop
    as in the eager loop, and two runs of the captured loop from the same start must differ for the perturbed pair (every
    replay draws fresh noise) and agree for the deterministic one."""
    import os
    import runpy
    from conftest import ROOT
    import pertrenderer_b200 as pb
    ex = runpy.run_path(os.path.join(ROOT, "examples", "pose_optimisation.py"), run_name="pose_example")
    torch.manual_seed(0)
    verts, faces, colors = ex["cube_mesh"](DEV)
    mesh = pb.TriMeshes(verts, faces, face_colors=colors)
    R, T = pb.look_at_view_transform(dist=6.7, elev=30.0, azim=120.0, device=DEV)
    cameras = pb.OpenGLPerspectiveCameras(R=R, T=T, fov=60, device=DEV)
    lights = pb.PointLights(location=[[0.0, 2.0, -2.0]], device=DEV)
    hard = ex["make_renderer"]("hard", cameras, lights, 1e-4, 1e-4, 1, 64, DEV)
    w_true = torch.tensor([0.3, -0.5, 0.2], device=DEV)
    R_true = ex["so3_exp"](w_true)
    with torch.no_grad():
        target = hard(mesh.update_padded(verts @ R_true))[..., :3]
    axis = torch.tensor([0.6, 0.0, 0.8], device=DEV)
    w0 = ex["so3_log"](R_true @ ex["so3_exp"](math.radians(15.0) * axis))
    a0 = ex["angle_deg"](ex["so3_exp"](w0), R_true)

    def run():
        renderer = ex["make_renderer"](pair, cameras, lights, 1e-3, 1e-2, 16, 64, DEV)
        return ex["optimize_pose_graphed"](mesh, verts, renderer, target, w0, 60, 5e-2)

    w1, w2 = run(), run()
    torch.cuda.synchronize()
    assert torch.isfinite(w1).all() and torch.isfinite(w2).all()
    if pair == "gaussian":
        a1, a2 = ex["angle_deg"](ex["so3_exp"](w1), R_true), ex["angle_deg"](ex["so3_exp"](w2), R_true)
        assert min(a1, a2) < 0.9 * a0, (pair, a0, a1, a2)  # 15 -> ~12 degrees in 60 noisy iterations at 64x64
        assert not torch.equal(w1, w2)  # fresh seeds per run and per replay
    else:
        # the deterministic pair: the captured loop is the eager loop (up to the order of the rasteriser's atomic adds)
        renderer = ex["make_renderer"](pair, cameras, lights, 1e-3, 1e-2, 16, 64, DEV)
        w_eager = ex["optimize_pose"](mesh, verts, renderer, target, w0, 60, 5e-2, False)
        assert (w1 - w2).abs().max().item() < 5e-2 and (w1 - w_eager).abs().max().item() < 5e-2, (w1, w2, w_eager)


def test_pose_optimisation_example_and_readme_snippet_run(monkeypatch, capsys):
    """examples/pose_optimisation.py (eval.py's benchmark loop, incl. the adaptive smoothing schedule) and the renderer
    snippet of README.md execute as written."""
    import os
    import re
    import runpy
    import sys
    from conftest import ROOT
    monkeypatch.setattr(sys, "argv", ["pose_optimisation.py", "--noise", "gaussian", "cauchy", "--trials", "1", "--niter", "8",
                                      "--imsize", "32", "--adapt"])
    mod = runpy.run_path(os.path.join(ROOT, "examples", "pose_optimisation.py"), run_name="pose_example")
    res = mod["main"]()
    assert set(res) == {"gaussian", "cauchy"} and all(math.isfinite(r["mean_final"]) for r in res.values())
    text = open(os.path.join(ROOT, "README.md")).read()
    snippet = [b for b in re.findall(r"```python\n(.*?)```", text, flags=re.S) if "MeshRenderer" in b][0]
    ns = {}
    exec(snippet, ns)
    assert ns["image"].shape == (1, 256, 256, 4) and torch.isfinite(ns["verts"].grad).all() and ns["verts"].grad.abs().sum() > 0


def test_integration_md_raster_stub_runs():
    """The rasteriser ctypes stub of INTEGRATION.md section 2c is executable as written and reproduces rasterize_meshes."""
    import os
    import re
    import pertrenderer_b200 as pb
    from conftest import ROOT
    from pertrenderer_b200 import _cabi
    text = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    blocks = re.findall(r"```python\n(.*?)```", text, flags=re.S)
    base = [b for b in blocks if "class PerturbedShade" in b][0].replace('"libpertshade.so"', repr(_cabi.LIB_PATH))
    stub = [b for b in blocks if "class Rasterize(" in b][0]
    ns = {}
    exec(base, ns)
    exec(stub, ns)
    fv, start = _faces_ndc(80, 2, seed=2)
    fs = torch.tensor(start, device=DEV)
    a_in, b_in = fv.to(DEV).requires_grad_(True), fv.to(DEV).requires_grad_(True)
    a = ns["Rasterize"].apply(a_in, fs, 24, 3e-3, 6)
    b = pb.rasterize_meshes(b_in, fs, 24, 3e-3, 6)
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    g = torch.randn_like(a[1])
    (a[1] * g).sum().backward()
    (b[1] * g).sum().backward()
    assert rel_err(a_in.grad, b_in.grad) <= 1e-5
