"""Texture atlases sampled inside the Phong kernels (pert_phong_atlas_fwd / _bwd) against the materialised texel tensor of
AtlasTexels.materialize: the unlit lookup bit for bit (out-of-range, NaN and infinite barycentric coordinates included),
the lit colours bit for bit against pert_phong_fwd fed the materialised texels and within 1e-5 of the CPU oracle, the
gradients against torch autograd through materialize, the shaders end to end through this project's rasteriser, and a
CUDA-graph capture."""

import pytest
import torch

from conftest import rel_err
from oracle import phong_oracle as PO
from test_atlas_cpu import _special_values
from test_gpu_phong import _frag_to, _scene, _to

pytestmark = pytest.mark.gpu

RTOL = 1e-5
DEV = "cuda"


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _odd_bary(p2f, R, seed, finite_only=False):
    """Barycentric coordinates of the valid entries: random in the triangle, and in a third of the entries pairs drawn
    from the CPU test's set (negative down to -3, above 1, exactly k/R, on the diagonal; NaN and +-inf unless
    ``finite_only``).  -1 at padding, like the rasteriser."""
    import pertrenderer_b200 as pb
    bary = pb.synthetic_bary(p2f, seed)
    v = torch.from_numpy(_special_values(R))
    if finite_only:
        v = v[torch.isfinite(v) & (v.abs() <= 3)]
    g = torch.Generator().manual_seed(seed + 11)
    pick = (torch.rand(p2f.shape, generator=g) < 0.33) & (p2f >= 0)
    n = int(pick.sum())
    w = v[torch.randint(0, v.numel(), (n, 2), generator=g)]
    diag = torch.rand(n, generator=g) < 0.2
    w[diag, 1] = 1.0 - w[diag, 0]
    bary[pick] = torch.cat([w, torch.full((n, 1), 0.25)], 1)
    return bary


@pytest.mark.parametrize("sparse", [False, True])
@pytest.mark.parametrize("N", [1, 3])
@pytest.mark.parametrize("K", [1, 50, 100])
@pytest.mark.parametrize("R", [1, 2, 3, 4, 8])
def test_unlit_lookup_equals_materialize(R, K, N, sparse):
    import pertrenderer_b200 as pb
    from pertrenderer_b200 import shading
    F, H, W = 37, 6, 7
    fr, _ = pb.synthetic_fragments(N, H, W, K, kind="realistic", n_faces=F, seed=R * K + N, device="cpu",
                                   mean_valid=4.0 if K < 50 else 20.0)
    p2f = fr.pix_to_face
    bary = _odd_bary(p2f, R, seed=R + K)
    atlas = torch.rand(F, R, R, 3, generator=torch.Generator().manual_seed(R))
    ref = pb.AtlasTexels(atlas).materialize(p2f, bary)
    out = shading.phong_forward(p2f.to(DEV), bary.to(DEV), None, None, None, None, None, sparse=sparse, unlit=True,
                                atlas=atlas.to(DEV)).cpu()
    valid = p2f >= 0
    assert torch.equal(out[valid], ref[valid])
    if not sparse:
        assert torch.equal(out, ref)


def _lit_case(light, per_batch, R, seed):
    """A CPU scene (test_gpu_phong._scene) with an atlas, finite out-of-range coordinates in a third of the entries."""
    import pertrenderer_b200 as pb
    N, H, W, K = 3, 9, 11, 7
    fr, verts, faces, lights, mats, cams, _, _ = _scene(N, H, W, K, 300, light, per_batch, seed=seed)
    fr = pb.Fragments(fr.pix_to_face, fr.zbuf, _odd_bary(fr.pix_to_face, R, seed, finite_only=True), fr.dists)
    atlas = torch.rand(faces.shape[0], R, R, 3, generator=torch.Generator().manual_seed(seed + 5))
    return fr, verts, faces, lights, mats, cams, atlas


def _device_inputs(fr, verts, faces, lights, mats, cams):
    """(pix_to_face, bary, face_verts, face_normals, lighting) on the GPU, computed ONCE: the vertex normals are summed by
    index_add, whose CUDA order is not fixed, so two calls of phong_shading differ in the last bit of their normals."""
    import pertrenderer_b200 as pb
    from pertrenderer_b200 import shading
    p2f, bary = fr.pix_to_face.to(DEV), fr.bary_coords.to(DEV)
    mesh = pb.TriMeshes(verts.to(DEV), faces.to(DEV))
    fv = mesh.verts_packed()[mesh.faces_packed()].contiguous()
    fn = mesh.verts_normals_packed()[mesh.faces_packed()].contiguous()
    lighting = shading.pack_lighting(_to(lights, DEV), _to(mats, DEV), _to(cams, DEV), p2f.shape[0], DEV).detach().clone()
    return p2f, bary, fv, fn, lighting


@pytest.mark.parametrize("sparse", [False, True])
@pytest.mark.parametrize("per_batch", [False, True])
@pytest.mark.parametrize("light", ["point", "directional"])
def test_lit_forward_equals_dense_texels_and_oracle(light, per_batch, sparse):
    import pertrenderer_b200 as pb
    from pertrenderer_b200 import shading
    fr, verts, faces, lights, mats, cams, atlas = _lit_case(light, per_batch, 4, seed=7)
    p2f, bary, fv, fn, lighting = _device_inputs(fr, verts, faces, lights, mats, cams)
    tex = pb.AtlasTexels(atlas).materialize(fr.pix_to_face, fr.bary_coords)
    got = shading.phong_forward(p2f, bary, fv, fn, None, None, lighting, sparse=sparse, atlas=atlas.to(DEV)).cpu()
    dense = shading.phong_forward(p2f, bary, fv, fn, tex.to(DEV), None, lighting, sparse=sparse).cpu()
    valid = fr.pix_to_face >= 0
    assert torch.equal(got[valid], dense[valid])
    if not sparse:
        assert torch.equal(got, dense)
    ref = PO.phong_colors_from(pb.TriMeshes(verts, faces), fr, lights, cams, mats, tex)
    assert rel_err(got[valid], ref[valid]) <= RTOL


def _grad_inputs(light, per_batch):
    """Device inputs of the gradient tests, built once and shared by both paths (see _device_inputs)."""
    fr, verts, faces, lights, mats, cams, atlas = _lit_case(light, per_batch, 4, seed=3)
    return _device_inputs(fr, verts, faces, lights, mats, cams) + (atlas.to(DEV),)


def _grads(inputs, unlit, sparse, atlas_in_kernel):
    """Colours and gradients of one Phong call (_PhongShade) on the given inputs: the atlas, bary and, lit, the face
    corners, face normals and lighting table -- through the atlas kernels, or through torch autograd over materialize and
    the dense-texel kernels.  Every input is a fresh leaf copy."""
    import pertrenderer_b200 as pb
    from pertrenderer_b200 import shading
    p2f = inputs[0]
    bary, fv, fn, lighting, a = [t.detach().clone().requires_grad_(True) for t in inputs[1:]]
    if atlas_in_kernel:
        texels, mode = a, "atlas"
    else:
        texels, mode = pb.AtlasTexels(a).materialize(p2f, bary), "texels"
    if unlit:
        col = shading._PhongShade.apply(None, None, texels, bary, p2f, None, mode, sparse, True, 0, None) if atlas_in_kernel \
            else texels
    else:
        col = shading._PhongShade.apply(fv, fn, texels, bary, p2f, lighting, mode, sparse, False, 0, None)
    g = torch.randn(col.shape, generator=torch.Generator().manual_seed(9)).to(DEV)
    g[torch.rand(col.shape[:-1], generator=torch.Generator().manual_seed(10)).to(DEV) < 0.4] = 0.0
    col.backward(g)
    out = dict(col=col.detach(), atlas=a.grad, bary=bary.grad, fv=fv.grad, fn=fn.grad, light=lighting.grad)
    return out, p2f >= 0


@pytest.mark.parametrize("sparse", [False, True])
@pytest.mark.parametrize("light,per_batch", [("point", False), ("point", True), ("directional", False), ("directional", True)])
def test_lit_backward_matches_autograd_through_materialize(light, per_batch, sparse):
    inputs = _grad_inputs(light, per_batch)
    got, valid = _grads(inputs, False, sparse, True)
    ref, _ = _grads(inputs, False, sparse, False)
    assert torch.equal(got["col"][valid], ref["col"][valid])
    assert rel_err(got["atlas"], ref["atlas"]) <= RTOL  # atomics in no fixed order on both sides
    assert torch.equal(got["bary"], ref["bary"])  # the atlas adds nothing to bary: the dense call's gradient, bit for bit
    for k in ("fv", "fn", "light"):
        assert got[k].abs().sum() > 0 and rel_err(got[k], ref[k]) <= RTOL, k


@pytest.mark.parametrize("sparse", [False, True])
def test_unlit_backward(sparse):
    inputs = _grad_inputs("point", False)
    got, valid = _grads(inputs, True, sparse, True)
    ref, _ = _grads(inputs, True, sparse, False)
    assert torch.equal(got["col"][valid], ref["col"][valid])
    assert got["atlas"].abs().sum() > 0 and rel_err(got["atlas"], ref["atlas"]) <= RTOL
    assert got["bary"] is not None and (got["bary"] == 0).all()


@pytest.mark.parametrize("unlit", [False, True])
def test_sparse_backward_leaves_padding_untouched(unlit):
    """PERT_PHONG_SPARSE: the padded entries of grad_bary are neither read nor written (pre-filled with a sentinel)."""
    from pertrenderer_b200 import _cabi, shading
    fr, verts, faces, lights, mats, cams, atlas = _lit_case("point", False, 4, seed=5)
    p2f, bary, fv, fn, lighting = _device_inputs(fr, verts, faces, lights, mats, cams)
    a = atlas.to(DEV)
    gc = torch.randn(p2f.shape + (3,), device=DEV)
    gb = torch.full(p2f.shape + (3,), 7.0, device=DEV)
    ga = torch.zeros_like(a)
    ph = shading._phong_struct(p2f, bary, None if unlit else fv, None if unlit else fn, None, None, None if unlit else lighting,
                               _cabi.PHONG_SPARSE | (_cabi.PHONG_UNLIT if unlit else 0), atlas=a)
    rc = _cabi.phong_atlas_fns()[1](ph, _cabi.ptr(a), 4, _cabi.ptr(gc), _cabi.ptr(ga), _cabi.ptr(gb), None, None, None,
                                    _cabi.stream_ptr(torch.device(DEV)))
    _cabi.check(rc, "pert_phong_atlas_bwd")
    torch.cuda.synchronize()
    pad = p2f < 0
    assert pad.any() and (gb[pad] == 7.0).all()
    assert (gb[~pad] != 7.0).all()


def _renderer_case(shader_kind, n_views, R=4):
    import math
    import pertrenderer_b200 as pb
    H, K, sigma, gamma = 32, 20, 1e-3, 1e-2
    verts, faces = pb.synthetic_mesh(320, device=DEV)
    Rm, T = pb.look_at_view_transform(dist=2.7, elev=30.0, azim=torch.linspace(10.0, 130.0, n_views), device=DEV)
    cam = pb.OpenGLPerspectiveCameras(R=Rm, T=T, device=DEV)
    rast = pb.MeshRasterizer(cam, pb.RasterizationSettings(image_size=H, blur_radius=math.log(1.0 / 1e-4 - 1.0) * sigma,
                                                           faces_per_pixel=K))
    pair = dict(gaussian=(pb.GaussianRast(nb_samples=16, sigma=sigma), pb.GaussianAgg(nb_samples=16, gamma=gamma)),
                cauchy=(pb.ArctanRast(nb_samples=16, sigma=sigma), pb.CauchyAgg(nb_samples=16, gamma=gamma)))
    kind, _, which = shader_kind.partition("-")
    if kind == "phong":
        shader = pb.RandomPhongShader(device=DEV, cameras=cam, lights=pb.PointLights(location=[[0.0, 2.0, -2.0]], device=DEV),
                                      smoothrast=pair[which][0], smoothagg=pair[which][1], blend_params=pb.BlendParams())
    elif kind == "random":
        shader = pb.RandomSimpleShader(device=DEV, cameras=cam, smoothrast=pair[which][0], smoothagg=pair[which][1],
                                       blend_params=pb.BlendParams())
    else:
        shader = pb.SimpleShader(device=DEV, blend_params=pb.BlendParams(background_color=(0.2, 0.3, 0.4)))
    atlas = torch.rand((faces.shape[0], R, R, 3), device=DEV, generator=torch.Generator(device=DEV).manual_seed(4))
    return verts, faces, rast, shader, atlas


@pytest.mark.parametrize("n_views", [1, 2])
@pytest.mark.parametrize("shader_kind", ["phong-gaussian", "phong-cauchy", "random-gaussian", "random-cauchy", "simple"])
def test_shaders_end_to_end_through_the_rasteriser(shader_kind, n_views):
    """MeshRenderer(MeshRasterizer, shader) on TriMeshes(atlas=...) (extend(2) for two views) against the same shader fed
    the materialised texels of the same fragments, under the same torch.manual_seed: the same image, and the atlas gradient
    of torch autograd through materialize."""
    import pertrenderer_b200 as pb
    verts, faces, rast, shader, atlas = _renderer_case(shader_kind, n_views)
    a = atlas.clone().requires_grad_(True)
    mesh = pb.TriMeshes(verts, faces, atlas=a)
    mesh = mesh.extend(n_views) if n_views > 1 else mesh
    # the vertex normals are summed by index_add, in no fixed order on CUDA: both renders use the same ones
    normals = mesh.verts_normals_packed()
    mesh.verts_normals_packed = lambda: normals
    torch.manual_seed(5)
    img = pb.MeshRenderer(rast, shader)(mesh)
    G = torch.randn(img.shape, device=DEV, generator=torch.Generator(device=DEV).manual_seed(6))
    (img * G).sum().backward()

    a2 = atlas.clone().requires_grad_(True)
    with torch.no_grad():
        fr = rast(mesh)
    tex = pb.AtlasTexels(a2 if n_views == 1 else a2.repeat(n_views, 1, 1, 1)).materialize(fr.pix_to_face, fr.bary_coords)
    ref_mesh = pb.TriMeshes(mesh.verts_padded() if n_views > 1 else verts, faces, texels=tex) if shader_kind.startswith("phong") \
        else pb.TexelMeshes(tex)
    ref_mesh.verts_normals_packed = lambda: normals
    torch.manual_seed(5)
    img2 = shader(fr, ref_mesh)
    (img2 * G).sum().backward()
    assert torch.equal(img.detach(), img2.detach())
    assert a.grad.abs().sum() > 0 and rel_err(a.grad, a2.grad) <= RTOL


def test_graph_capture_equals_eager():
    """Forward and backward with an atlas captured in one CUDA graph and replayed: the eager call's colours and gradients
    (the atlas atomics sum in no fixed order: 1e-5)."""
    import pertrenderer_b200 as pb
    from pertrenderer_b200 import shading
    fr, verts, faces, lights, mats, cams, atlas = _lit_case("point", True, 4, seed=8)
    p2f, bary = fr.pix_to_face.to(DEV), fr.bary_coords.to(DEV)
    mesh = pb.TriMeshes(verts.to(DEV), faces.to(DEV))
    fv = mesh.verts_packed()[mesh.faces_packed()].contiguous()
    fn = mesh.verts_normals_packed()[mesh.faces_packed()].contiguous()
    lighting = shading.pack_lighting(_to(lights, DEV), _to(mats, DEV), _to(cams, DEV), p2f.shape[0], DEV)
    a = atlas.to(DEV)
    gc = torch.randn(p2f.shape + (3,), device=DEV)

    def step():
        col = shading.phong_forward(p2f, bary, fv, fn, None, None, lighting, sparse=True, atlas=a)
        return (col,) + tuple(shading.phong_backward(p2f, bary, fv, fn, None, None, lighting, gc, sparse=True, atlas=a,
                                                     need_lighting=True))

    eager = step()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        captured = step()
    g.replay()
    torch.cuda.synchronize()
    valid = p2f >= 0
    assert torch.equal(captured[0][valid], eager[0][valid])
    assert torch.equal(captured[2], eager[2])  # grad_bary: one store per entry
    for c, e in zip(captured[1:], eager[1:]):
        assert rel_err(c, e) <= RTOL
