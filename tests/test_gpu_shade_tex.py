"""Textures sampled inside the fused shading kernels (pert_shade_tex_fwd / _bwd / _render) against today's path, which
materialises the colours with the texture-only Phong kernel and feeds them to pert_shade_fwd / _bwd: over the three
perturbed pairs, the three texture kinds and synthetic sparse, synthetic dense and rasterised fragments (whose barycentric
coordinates are unclipped), with in-kernel and explicit noise.  The image and every gradient but the texture's are equal
bit for bit (the colours are); the table and bary gradients agree to 1e-5 (their atomic adds sum in another order).  Also:
peak memory at BASELINE config 2, a CUDA-graph capture, and the shaders end to end through the rasteriser."""

import math

import pytest
import torch

from conftest import elementwise_close

pytestmark = pytest.mark.gpu

DEV = "cuda"
RTOL = 1e-5
PAIRS = {"gaussian": 0, "cauchy": 8, "no_vr": 0x400}  # ops.F_CAUCHY, ops.F_NO_VR
KINDS = ["vert", "uv", "atlas"]


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def _table(kind, F, N, seed):
    """(table, face_uvs) of a texture of F faces: corner colours, N maps of 7 x 9 with UVs a little outside [0, 1]
    (the border rule), or a 4 x 4 atlas."""
    g = _gen(seed)
    if kind == "vert":
        return torch.rand(F, 3, 3, device=DEV, generator=g), None
    if kind == "uv":
        return torch.rand(N, 7, 9, 3, device=DEV, generator=g), torch.rand(F, 3, 2, device=DEV, generator=g) * 1.2 - 0.1
    return torch.rand(F, 4, 4, 3, device=DEV, generator=g), None


def _fragments(frag, seed):
    """(pix_to_face, zbuf, dists, bary, F) on the GPU."""
    import pertrenderer_b200 as pb
    if frag == "raster":
        sigma = 1e-3
        verts, faces = pb.synthetic_mesh(320, device=DEV)
        R, T = pb.look_at_view_transform(dist=2.7, elev=30.0, azim=torch.tensor([10.0, 70.0]), device=DEV)
        rast = pb.MeshRasterizer(pb.OpenGLPerspectiveCameras(R=R, T=T, device=DEV),
                                 pb.RasterizationSettings(image_size=32, blur_radius=math.log(1.0 / 1e-4 - 1.0) * sigma,
                                                          faces_per_pixel=20))
        fr = rast(pb.TriMeshes(verts, faces).extend(2))
        return fr.pix_to_face, fr.zbuf, fr.dists, fr.bary_coords.contiguous(), 2 * faces.shape[0]
    F = 97
    fr, _ = pb.synthetic_fragments(2, 12, 20, 24, kind="dense" if frag == "dense" else "realistic", n_faces=F, seed=seed,
                                   device=DEV, mean_valid=6.0)
    # barycentric coordinates partly outside the triangle, as the rasteriser's blur band produces them
    bary = pb.synthetic_bary(fr.pix_to_face, seed) * 1.6 - 0.2
    return fr.pix_to_face, fr.zbuf, fr.dists, bary.contiguous(), F


def _lazy_colors(kind, p2f, bary, table, face_uvs):
    """Today's path: the (N,H,W,K,3) texels of the texture-only Phong kernel (valid entries only, as the fused pairs use)."""
    from pertrenderer_b200 import shading
    src = dict(vert_colors=table) if kind == "vert" else dict(uv=(table, face_uvs)) if kind == "uv" else dict(atlas=table)
    return shading.phong_forward(p2f, bary, None, None, None, None, None, sparse=True, unlit=True, **src)


def _lazy_grads(kind, p2f, bary, table, face_uvs, grad_colors):
    from pertrenderer_b200 import shading
    src = dict(vert_colors=table) if kind == "vert" else dict(uv=(table, face_uvs)) if kind == "uv" else dict(atlas=table)
    g_tex, g_bary, _, _ = shading.phong_backward(p2f, bary, None, None, None, None, None, grad_colors, need_verts=False,
                                                 need_normals=False, sparse=True, unlit=True, **src)
    return g_tex, g_bary


def _problems(case, kind, pair, explicit, seed=3):
    from pertrenderer_b200 import ops
    p2f, zbuf, dists, bary, F = case
    N, H, W, K = p2f.shape
    table, face_uvs = _table(kind, F, N, seed)
    S = 16
    noise_r = noise_a = None
    if explicit:
        noise_r = torch.randn(S, N, H, W, K, device=DEV, generator=_gen(seed + 1))
        noise_a = torch.randn(S, N, H, W, K + 1, device=DEV, generator=_gen(seed + 2))
    common = dict(pix_to_face=p2f, zbuf=zbuf, dists=dists, znear=1.0, zfar=100.0, background=(0.2, 0.3, 0.4), sigma=1e-3,
                  gamma=1e-2, alpha=1.0, eps=1e-10, S_rast=S, S_agg=S, seed_rast=1234 + seed, seed_agg=5678 + seed,
                  flags=PAIRS[pair], noise_rast=noise_r, noise_agg=noise_a)
    colors = _lazy_colors(kind, p2f, bary, table, face_uvs)
    old = ops.ShadeProblem(colors=colors, **common)
    new = ops.ShadeProblem(colors=None, texture=ops.ShadeTexture(kind=kind, bary=bary, table=table, face_uvs=face_uvs), **common)
    return old, new


_CASES = {}


def _case(frag):
    if frag not in _CASES:
        _CASES[frag] = _fragments(frag, seed=len(_CASES) + 1)
    return _CASES[frag]


@pytest.mark.parametrize("explicit", [False, True])
@pytest.mark.parametrize("frag", ["sparse", "dense", "raster"])
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("pair", list(PAIRS))
def test_forward_backward_and_render_equal_todays_path(pair, kind, frag, explicit):
    from pertrenderer_b200 import ops
    case = _case(frag)
    p2f, bary = case[0], case[3]
    old, new = _problems(case, kind, pair, explicit)
    img_old, saved_old = ops.shade_forward(old)
    img_new, saved_new = ops.shade_forward(new)
    assert torch.equal(img_new, img_old)
    assert torch.equal(ops.shade_render(new), img_new)

    G = torch.randn(img_old.shape, device=DEV, generator=_gen(9))
    gd_o, gz_o, gc_o, sc_o = ops.shade_backward(old, saved_old, G)
    gd_n, gz_n, (gt_n, gb_n), sc_n = ops.shade_backward(new, saved_new, G, need_bary=True)
    assert torch.equal(gd_n, gd_o) and torch.equal(gz_n, gz_o) and torch.equal(sc_n, sc_o)
    gt_o, gb_o = _lazy_grads(kind, p2f, bary, new.texture.table, new.texture.face_uvs, gc_o)
    assert gt_o.abs().sum() > 0
    assert elementwise_close(gt_n, gt_o, RTOL)
    if kind == "atlas":
        assert not gb_n.any()
    else:
        assert gb_o.abs().sum() > 0
        assert elementwise_close(gb_n, gb_o, RTOL)


@pytest.mark.parametrize("need_bary", [False, True])
def test_peak_memory_at_config_2(need_bary):
    """BASELINE config 2 (8 x 256^2, K = 50): forward + backward without the (N,H,W,K,3) colour tensor and its gradient,
    2 x 315 MB, measured as the peak of each path over the same resident inputs.  Today's path keeps grad_dists / grad_zbuf
    alive through the texture-only Phong backward, as autograd does (they wait for the rasteriser's backward).  The new
    path holds backward's small workspaces (scalar partials, the (F,3,3) table gradient) at its peak, today's path holds
    them at another moment: the saving is 2 x 315 MB less those."""
    import pertrenderer_b200 as pb
    from pertrenderer_b200 import ops
    N, H, W, K = 8, 256, 256, 50
    fr, _ = pb.synthetic_fragments(N, H, W, K, kind="realistic", n_faces=1280, seed=2, device=DEV)
    bary = pb.synthetic_bary(fr.pix_to_face, 2)
    table, _ = _table("vert", 1280, N, 4)
    common = dict(pix_to_face=fr.pix_to_face, zbuf=fr.zbuf, dists=fr.dists, znear=1.0, zfar=100.0, background=(1.0, 1.0, 1.0),
                  sigma=1e-4, gamma=1e-4, alpha=1.0, eps=1e-10, S_rast=16, S_agg=16, seed_rast=1, seed_agg=2)
    G = torch.randn((N, H, W, 4), device=DEV, generator=_gen(5))

    def old():
        from pertrenderer_b200 import shading
        colors = _lazy_colors("vert", fr.pix_to_face, bary, table, None)
        pr = ops.ShadeProblem(colors=colors, **common)
        img, saved = ops.shade_forward(pr)
        gd, gz, gc, _ = ops.shade_backward(pr, saved, G)
        return img, gd, gz, shading.phong_backward(fr.pix_to_face, bary, None, None, None, None, None, gc, need_bary=need_bary,
                                                   need_verts=False, need_normals=False, sparse=True, unlit=True,
                                                   vert_colors=table)

    def new():
        pr = ops.ShadeProblem(colors=None, texture=ops.ShadeTexture(kind="vert", bary=bary, table=table), **common)
        img, saved = ops.shade_forward(pr)
        return img, ops.shade_backward(pr, saved, G, need_bary=need_bary)

    peaks = {}
    for name, fn in (("old", old), ("new", new), ("old", old), ("new", new)):
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        out = fn()
        torch.cuda.synchronize()
        peaks[name] = torch.cuda.max_memory_allocated() - base
        del out
    colour_bytes = N * H * W * K * 3 * 4
    workspaces = 3 * ops.ShadeProblem(colors=None, texture=ops.ShadeTexture(kind="vert", bary=bary, table=table),
                                      **common).num_tiles() * 16 + table.numel() * 4 + 512  # partials, table grad, scalars
    assert peaks["old"] - peaks["new"] >= 2 * colour_bytes - workspaces, peaks


@pytest.mark.parametrize("kind", KINDS)
def test_graph_capture_replays_fresh_noise(kind):
    """Forward + backward captured in one CUDA graph with device-side seeds: every replay equals an eager call with the
    same seeds (image and scalar gradients bit for bit, table gradient to 1e-5), and other seeds give another image."""
    from pertrenderer_b200 import ops
    p2f, zbuf, dists, bary, F = _case("raster")
    N = p2f.shape[0]
    table, face_uvs = _table(kind, F, N, 7)
    seed_dev = torch.zeros(2, dtype=torch.int64, device=DEV)
    pr = ops.ShadeProblem(pix_to_face=p2f, zbuf=zbuf, dists=dists, colors=None, znear=1.0, zfar=100.0, background=(1.0, 1.0, 1.0),
                          sigma=1e-3, gamma=1e-2, alpha=1.0, eps=1e-10, S_rast=16, S_agg=16, seed_rast=11, seed_agg=12,
                          seed_device=seed_dev, texture=ops.ShadeTexture(kind=kind, bary=bary, table=table, face_uvs=face_uvs))
    G = torch.randn((N,) + tuple(p2f.shape[1:3]) + (4,), device=DEV, generator=_gen(8))

    def step():
        img, saved = ops.shade_forward(pr)
        gd, gz, (gt, gb), sc = ops.shade_backward(pr, saved, G, need_bary=True)
        return img, gd, gz, sc, gt, gb

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = step()
    images = []
    for trial in range(2):
        seed_dev.copy_(torch.tensor([101 + trial, 202 + trial], dtype=torch.int64))
        graph.replay()
        got = [t.clone() for t in captured]
        eager = step()
        for c, e in zip(got[:4], eager[:4]):
            assert torch.equal(c, e)
        assert elementwise_close(got[4], eager[4], RTOL)
        assert elementwise_close(got[5], eager[5], RTOL) if kind != "atlas" else not got[5].any()
        images.append(got[0])
    assert not torch.equal(images[0], images[1])


def _count_tex_calls(monkeypatch):
    """Counts of the calls of pert_shade_tex_fwd / _bwd / _render made through the module API from now on."""
    from pertrenderer_b200 import _cabi
    real = _cabi.shade_tex_fns
    calls = dict(fwd=0, bwd=0, render=0)

    def counting(name, fn):
        def call(*args):
            calls[name] += 1
            return fn(*args)
        return call

    monkeypatch.setattr(_cabi, "shade_tex_fns",
                        lambda: tuple(counting(n, f) for n, f in zip(("fwd", "bwd", "render"), real())))
    return calls


def _shader_scene(kind, n_views):
    """(rasteriser, RandomSimpleShader with the Gaussian pair, mesh factory) of a 320-face sphere textured with ``kind``."""
    import pertrenderer_b200 as pb
    sigma, gamma = 1e-3, 1e-2
    verts, faces = pb.synthetic_mesh(320, device=DEV)
    R, T = pb.look_at_view_transform(dist=2.7, elev=30.0, azim=torch.linspace(10.0, 130.0, n_views), device=DEV)
    cam = pb.OpenGLPerspectiveCameras(R=R, T=T, device=DEV)
    rast = pb.MeshRasterizer(cam, pb.RasterizationSettings(image_size=32, blur_radius=math.log(1.0 / 1e-4 - 1.0) * sigma,
                                                           faces_per_pixel=20))
    shader = pb.RandomSimpleShader(device=DEV, cameras=cam, smoothrast=pb.GaussianRast(nb_samples=16, sigma=sigma),
                                   smoothagg=pb.GaussianAgg(nb_samples=16, gamma=gamma), blend_params=pb.BlendParams())
    g = _gen(4)
    src = dict(vert=lambda: torch.rand(verts.shape[0], 3, device=DEV, generator=g),
               uv=lambda: torch.rand(1, 16, 16, 3, device=DEV, generator=g),
               atlas=lambda: torch.rand(faces.shape[0], 4, 4, 3, device=DEV, generator=g))[kind]()
    verts_uvs = torch.rand(verts.shape[0], 2, device=DEV, generator=g)

    def mesh_of(requires_grad):
        v = verts.clone().requires_grad_(requires_grad)
        t = src.clone().requires_grad_(requires_grad)
        tex = dict(vert=dict(verts_colors=t), uv=dict(uv=(t, verts_uvs, faces)), atlas=dict(atlas=t))[kind]
        mesh = pb.TriMeshes(v, faces, **tex)
        return (mesh.extend(n_views) if n_views > 1 else mesh), v, t

    return rast, shader, mesh_of


@pytest.mark.parametrize("n_views", [1, 2])
@pytest.mark.parametrize("kind", KINDS)
def test_random_simple_shader_end_to_end(kind, n_views, monkeypatch):
    """MeshRenderer(MeshRasterizer, RandomSimpleShader) on TriMeshes(verts_colors= / uv= / atlas=) (extend(2) for two
    views) against the same shader fed the texels that sample_lazy_textures materialises from the same fragments, under the
    same torch.manual_seed: the same image, the same vertex-position and texture gradients to 1e-5.  The textured render
    goes through pert_shade_tex_fwd / _bwd (one call each), the materialised one through neither."""
    import pertrenderer_b200 as pb
    from pertrenderer_b200.random_rasterizer import _PerturbedTexShade
    from pertrenderer_b200.shading import sample_lazy_textures
    rast, shader, mesh_of = _shader_scene(kind, n_views)
    calls = _count_tex_calls(monkeypatch)

    def render(lazy):
        mesh, v, t = mesh_of(True)
        fr = rast(mesh)
        torch.manual_seed(5)
        if lazy:
            img = shader(fr, mesh)
            assert type(img.grad_fn) is _PerturbedTexShade._backward_cls
        else:
            img = shader(fr, pb.TexelMeshes(sample_lazy_textures(mesh.sample_textures(fr), fr, sparse=True)))
        (img * G).sum().backward()
        return img.detach(), v.grad, t.grad

    G = torch.randn((n_views, 32, 32, 4), device=DEV, generator=_gen(6))
    img_n, gv_n, gt_n = render(True)
    assert calls == dict(fwd=1, bwd=1, render=0)
    img_o, gv_o, gt_o = render(False)
    assert calls == dict(fwd=1, bwd=1, render=0)
    assert torch.equal(img_n, img_o)
    assert gt_o.abs().sum() > 0 and elementwise_close(gt_n, gt_o, RTOL)
    assert gv_o.abs().sum() > 0 and elementwise_close(gv_n, gv_o, RTOL)


@pytest.mark.parametrize("kind", KINDS)
def test_random_simple_shader_without_gradients_renders_in_kernel(kind, monkeypatch):
    """Under torch.no_grad and torch.inference_mode, RandomSimpleShader on a textured mesh renders with
    pert_shade_tex_render (no forward, no colour tensor) and returns the grad-mode image bit for bit."""
    rast, shader, mesh_of = _shader_scene(kind, 2)
    calls = _count_tex_calls(monkeypatch)
    mesh, _, _ = mesh_of(True)
    fr = rast(mesh)
    torch.manual_seed(7)
    img = shader(fr, mesh)
    assert img.grad_fn is not None and calls == dict(fwd=1, bwd=0, render=0)
    for ctx in (torch.no_grad, torch.inference_mode):
        with ctx():
            mesh, _, _ = mesh_of(False)
            fr = rast(mesh)
            torch.manual_seed(7)
            out = shader(fr, mesh)
        assert out.grad_fn is None
        assert torch.equal(out, img.detach())
    assert calls == dict(fwd=1, bwd=0, render=2)
