"""Phong lighting of the fragment entries: the ``colors`` RandomPhongShader blends.

``phong_shading`` keeps the signature of ``pytorch3d.renderer.mesh.shading.phong_shading`` as the
reference calls it (randomras/random_rasterizer.py:103-110) and runs the hand-written kernels
``pert_phong_fwd`` / ``pert_phong_bwd`` (include/pertshade.h, csrc/phong.cu).  Objects are read by
attribute only, so pytorch3d's ``Meshes`` / ``PointLights`` / ``DirectionalLights`` / ``Materials`` /
cameras and the shims of :mod:`pertrenderer_b200.structures` both work:

    meshes.verts_packed() (V,3), meshes.faces_packed() (F,3), meshes.verts_normals_packed() (V,3)
    lights.location (point) or lights.direction (directional), .ambient_color, .diffuse_color, .specular_color
    materials.ambient_color, .diffuse_color, .specular_color, .shininess
    cameras.get_camera_center() (N,3)

Gradients flow to the mesh (vertex positions and vertex normals, through torch's own indexing
``verts[faces]``), to the texels and to ``fragments.bary_coords``; and, when they require grad, to the light
location / direction, the light and material colours, the shininess and the camera centre (a second sparse
pass, only then: experiments/eval.py:411-470 and :693-725 optimise lights and cameras).
"""

from __future__ import annotations

from typing import Optional

import torch
from torch.autograd import Function

from . import _cabi
from ._cabi import PHONG_SPARSE, PHONG_STRIDE, PHONG_UNLIT, PertPhong, check, ptr, require_cuda, stream_ptr
from .structures import AtlasTexels, FaceTexels, UVTexels, VertexTexels


def _f32c(t):
    return t if (t.dtype == torch.float32 and t.is_contiguous()) else t.to(torch.float32).contiguous()


def _rows(v, n_max, device, width=3):
    """A light / material attribute as float32 (rows, width) on ``device``, rows = 1 or N."""
    t = torch.as_tensor(v, dtype=torch.float32, device=device)  # differentiable when the caller's tensor requires grad
    if t.dim() == 0:
        t = t.reshape(1, 1).expand(1, width)
    t = t.reshape(-1, width) if width > 1 else t.reshape(-1, 1)
    if t.shape[0] not in (1, n_max):
        raise ValueError(f"lighting attributes must have 1 or N={n_max} rows, got {t.shape[0]}")
    return t


_LIGHTING_CACHE = {}


def pack_lighting(lights, materials, cameras, N, device):
    """(rows, PERT_PHONG_STRIDE) float32 table of include/pertshade.h: one row per batch element, or one
    row when nothing varies over the batch.  When no source tensor requires grad the table of the same objects is reused
    (keyed by the tensors' identity and version counters): a pose-optimisation loop re-packs nothing per iteration."""
    directional = not hasattr(lights, "location")
    srcs = [lights.direction if directional else lights.location, materials.ambient_color, lights.ambient_color,
            materials.diffuse_color, lights.diffuse_color, materials.specular_color, lights.specular_color,
            materials.shininess]
    key = None
    if all(torch.is_tensor(t) and not t.requires_grad for t in srcs) and hasattr(cameras, "R") and hasattr(cameras, "T") and \
            torch.is_tensor(cameras.R) and torch.is_tensor(cameras.T) and not cameras.R.requires_grad and not cameras.T.requires_grad:
        held = srcs + [cameras.R, cameras.T]
        key = tuple((id(t), t._version) for t in held) + (N, str(device), directional)
        hit = _LIGHTING_CACHE.get(key)
        if hit is not None:
            return hit[0]
    out = _pack_lighting(lights, materials, cameras, N, device, directional)
    if key is not None:
        if len(_LIGHTING_CACHE) > 16:
            _LIGHTING_CACHE.clear()
        _LIGHTING_CACHE[key] = (out, held)  # the sources are kept alive: their ids cannot be reused while the entry exists
    return out


def _pack_lighting(lights, materials, cameras, N, device, directional):
    loc = _rows(lights.direction if directional else lights.location, N, device)
    amb = _rows(materials.ambient_color, N, device) * _rows(lights.ambient_color, N, device)
    dif = _rows(materials.diffuse_color, N, device) * _rows(lights.diffuse_color, N, device)
    spc = _rows(materials.specular_color, N, device) * _rows(lights.specular_color, N, device)
    sh = _rows(materials.shininess, N, device, width=1)
    cam = _rows(cameras.get_camera_center(), N, device)
    rows = max(t.shape[0] for t in (loc, amb, dif, spc, sh, cam))
    kind = torch.full((1, 1), 1.0 if directional else 0.0, dtype=torch.float32, device=device)
    pad = torch.zeros((1, PHONG_STRIDE - 17), dtype=torch.float32, device=device)
    # one concatenation (differentiable: the pieces keep their autograd history)
    return torch.cat([t.expand(rows, -1) for t in (loc, amb, dif, spc, sh, cam, kind, pad)], dim=1)


def _phong_struct(pix_to_face, bary, face_verts, face_normals, texels, face_colors, lighting, flags, vert_colors=None,
                  faces_per_mesh=0, uv=None, atlas=None):
    N, H, W, K = pix_to_face.shape
    ph = PertPhong()
    ph.P, ph.HW, ph.K = N * H * W, H * W, K
    ph.light_rows = 0 if lighting is None else lighting.shape[0]
    table = face_verts if face_verts is not None else (face_colors if face_colors is not None else vert_colors)
    if uv is not None:  # (maps (M,Hm,Wm,3), face_uvs (F,3,2))
        ph.uv_map, ph.face_uvs = uv[0].data_ptr(), uv[1].data_ptr()
        ph.map_count, ph.map_h, ph.map_w = uv[0].shape[0], uv[0].shape[1], uv[0].shape[2]
        table = table if table is not None else uv[1]
    if atlas is not None:  # (F,R,R,3): passed to the atlas entry points beside the struct
        table = table if table is not None else atlas
        if atlas.shape[0] != table.shape[0]:
            raise ValueError(f"the atlas has {atlas.shape[0]} faces, the mesh {table.shape[0]}")
    ph.num_faces = table.shape[0]
    ph.flags = flags
    ph.faces_per_mesh = int(faces_per_mesh)
    ph.pix_to_face, ph.bary = pix_to_face.data_ptr(), bary.data_ptr()
    ph.face_verts = None if face_verts is None else face_verts.data_ptr()
    ph.face_normals = None if face_normals is None else face_normals.data_ptr()
    ph.texels = None if texels is None else texels.data_ptr()
    ph.face_colors = None if face_colors is None else face_colors.data_ptr()
    ph.face_vert_colors = None if vert_colors is None else vert_colors.data_ptr()
    ph.lighting = None if lighting is None else lighting.data_ptr()
    return ph


def phong_forward(pix_to_face, bary, face_verts, face_normals, texels, face_colors, lighting, sparse=False,
                  vert_colors=None, unlit=False, uv=None, atlas=None):
    """Launch pert_phong_fwd (pert_phong_atlas_fwd with ``atlas``).  Returns colors (N,H,W,K,3); with ``sparse`` the
    entries with pix_to_face < 0 are left unwritten (the fused shader kernels never read them).  Exactly one texel
    source: ``texels`` (N,H,W,K,3), ``face_colors`` (F,3), ``vert_colors`` (F,3,3), ``uv`` or ``atlas`` (F,R,R,3).
    ``unlit``: colour = texel (texture sampling only; the face tables and ``lighting`` may be None)."""
    lib = _cabi.load()
    require_cuda(pix_to_face, bary, face_verts, face_normals, texels, face_colors, lighting, vert_colors, atlas)
    N, H, W, K = pix_to_face.shape
    dev = pix_to_face.device
    with torch.cuda.device(dev):
        colors = torch.empty((N, H, W, K, 3), dtype=torch.float32, device=dev)
        ph = _phong_struct(pix_to_face, bary, face_verts, face_normals, texels, face_colors, lighting,
                           (PHONG_SPARSE if sparse else 0) | (PHONG_UNLIT if unlit else 0), vert_colors, uv=uv, atlas=atlas)
        if atlas is not None:
            rc = _cabi.phong_atlas_fns()[0](ph, ptr(atlas), atlas.shape[1], ptr(colors), stream_ptr(dev))
        else:
            rc = lib.pert_phong_fwd(ph, ptr(colors), stream_ptr(dev))
    check(rc, "pert_phong_atlas_fwd" if atlas is not None else "pert_phong_fwd")
    return colors


def phong_backward(pix_to_face, bary, face_verts, face_normals, texels, face_colors, lighting, grad_colors,
                   need_texels=True, need_bary=True, need_verts=True, need_normals=True, sparse=False, vert_colors=None,
                   unlit=False, faces_per_mesh=0, need_lighting=False, uv=None, atlas=None):
    """Launch pert_phong_bwd (pert_phong_atlas_bwd with ``atlas``).  Returns (grad_texels | grad_face_colors |
    grad_atlas, grad_bary, grad_face_verts, grad_face_normals), ``None`` where not requested.  Every entry of the dense outputs is defined (they
    flow on to the caller's own tensors): with ``sparse`` the kernel skips the padded entries, whose
    gradients are the zeros the buffers are created with."""
    lib = _cabi.load()
    require_cuda(grad_colors)
    grad_colors = _f32c(grad_colors)
    N, H, W, K = pix_to_face.shape
    dev = pix_to_face.device
    with torch.cuda.device(dev):
        alloc = torch.zeros if sparse else torch.empty
        if need_texels:
            table = face_colors if face_colors is not None else (vert_colors if vert_colors is not None else
                                                                    (uv[0] if uv is not None else atlas))
            g_tex = torch.zeros_like(table) if table is not None else alloc((N, H, W, K, 3), dtype=torch.float32, device=dev)
        else:
            g_tex = None
        g_bary = alloc((N, H, W, K, 3), dtype=torch.float32, device=dev) if need_bary else None
        g_fv = torch.zeros_like(face_verts) if (need_verts and not unlit) else None
        g_fn = torch.zeros_like(face_normals) if (need_normals and not unlit) else None
        g_light = torch.zeros_like(lighting) if (need_lighting and not unlit) else None
        ph = _phong_struct(pix_to_face, bary, face_verts, face_normals, texels, face_colors, lighting,
                           (PHONG_SPARSE if sparse else 0) | (PHONG_UNLIT if unlit else 0), vert_colors, faces_per_mesh, uv=uv,
                           atlas=atlas)
        if atlas is not None:
            rc = _cabi.phong_atlas_fns()[1](ph, ptr(atlas), atlas.shape[1], ptr(grad_colors), ptr(g_tex), ptr(g_bary), ptr(g_fv),
                                            ptr(g_fn), ptr(g_light), stream_ptr(dev))
        else:
            rc = lib.pert_phong_bwd(ph, ptr(grad_colors), ptr(g_tex), ptr(g_bary), ptr(g_fv), ptr(g_fn), ptr(g_light), stream_ptr(dev))
    check(rc, "pert_phong_atlas_bwd" if atlas is not None else "pert_phong_bwd")
    if need_lighting:
        return g_tex, g_bary, g_fv, g_fn, g_light
    return g_tex, g_bary, g_fv, g_fn


class _PhongShade(Function):
    """colors = phong(face_verts, face_normals, texel source, bary); constants: pix_to_face, lighting.
    ``tex_mode``: "texels" (N,H,W,K,3), "face" (F,3), "vert" (F,3,3), "uv" (the map) or "atlas" (F,R,R,3)."""

    @staticmethod
    def forward(ctx, face_verts, face_normals, texels, bary, pix_to_face, lighting, tex_mode, sparse, unlit, faces_per_mesh=0,
                face_uvs=None):
        fv = None if unlit else _f32c(face_verts.detach())
        fn = None if unlit else _f32c(face_normals.detach())
        tx, bc = _f32c(texels.detach()), _f32c(bary.detach())
        p2f = pix_to_face.contiguous()
        src = dict(texels=tx if tex_mode == "texels" else None, face_colors=tx if tex_mode == "face" else None,
                   vert_colors=tx if tex_mode == "vert" else None,
                   uv=(tx, _f32c(face_uvs.detach())) if tex_mode == "uv" else None, atlas=tx if tex_mode == "atlas" else None)
        ctx.uv_faces = src["uv"][1] if tex_mode == "uv" else None
        lighting = None if lighting is None else _f32c(lighting.detach())
        colors = phong_forward(p2f, bc, fv, fn, lighting=lighting, sparse=sparse, unlit=unlit, **src)
        ctx.save_for_backward(*[t for t in (fv, fn, tx, bc, p2f, lighting) if t is not None])
        ctx.tex_mode, ctx.sparse, ctx.unlit, ctx.faces_per_mesh = tex_mode, sparse, unlit, faces_per_mesh
        return colors

    @staticmethod
    def backward(ctx, grad_colors):
        if ctx.unlit:
            tx, bc, p2f = ctx.saved_tensors
            fv = fn = lighting = None
        else:
            fv, fn, tx, bc, p2f, lighting = ctx.saved_tensors
        need = ctx.needs_input_grad
        src = dict(texels=tx if ctx.tex_mode == "texels" else None, face_colors=tx if ctx.tex_mode == "face" else None,
                   vert_colors=tx if ctx.tex_mode == "vert" else None, uv=(tx, ctx.uv_faces) if ctx.tex_mode == "uv" else None,
                   atlas=tx if ctx.tex_mode == "atlas" else None)
        out = phong_backward(
            p2f, bc, fv, fn, lighting=lighting, grad_colors=grad_colors, need_texels=need[2], need_bary=need[3],
            need_verts=need[0], need_normals=need[1], sparse=ctx.sparse, unlit=ctx.unlit,
            faces_per_mesh=ctx.faces_per_mesh, need_lighting=bool(need[5]) and not ctx.unlit, **src)
        g_tex, g_bary, g_fv, g_fn = out[:4]
        g_light = out[4] if len(out) > 4 else None
        return g_fv, g_fn, g_tex, g_bary, None, g_light, None, None, None, None, None


def _texel_source(texels):
    """(tensor, tex_mode) of a texel argument: a dense tensor or one of the lazy per-face sources."""
    if isinstance(texels, FaceTexels):
        return texels.face_colors, "face"
    if isinstance(texels, VertexTexels):
        return texels.face_vert_colors(), "vert"
    if isinstance(texels, UVTexels):
        return texels.maps, "uv"
    if isinstance(texels, AtlasTexels):
        return texels.atlas, "atlas"
    return texels, "texels"


def sample_lazy_textures(texels, fragments, sparse: bool = False) -> torch.Tensor:
    """Materialise lazy texels (:class:`FaceTexels`, :class:`VertexTexels`, :class:`UVTexels`, :class:`AtlasTexels`) as
    the (N,H,W,K,3) tensor ``Meshes.sample_textures`` returns (random_rasterizer.py:101,170), with the texture-only mode
    of the Phong kernel (PERT_PHONG_UNLIT); gradients flow to the colour table, map or atlas and, for vertex colours and
    UV maps, to bary_coords (an atlas texel is piecewise constant in them)."""
    tex, mode = _texel_source(texels)
    if mode == "texels":
        return tex
    pix_to_face = fragments.pix_to_face
    if pix_to_face.dtype != torch.int64:
        pix_to_face = pix_to_face.to(torch.int64)
    bary = fragments.bary_coords
    if bary is None:
        if mode in ("vert", "uv", "atlas"):
            raise ValueError("vertex colours / UV maps / atlases need fragments.bary_coords (N,H,W,K,3)")
        bary = torch.zeros(pix_to_face.shape + (3,), dtype=torch.float32, device=pix_to_face.device)
    return _PhongShade.apply(None, None, tex, bary, pix_to_face, None, mode, bool(sparse), True, 0,
                             texels.face_uvs() if mode == "uv" else None)


def phong_shading(meshes, fragments, lights, cameras, materials, texels, sparse: bool = False) -> torch.Tensor:
    """pytorch3d.renderer.mesh.shading.phong_shading, same arguments (random_rasterizer.py:103-110).

    ``texels`` (N,H,W,K,3), or lazy :class:`FaceTexels` / :class:`VertexTexels` / :class:`UVTexels` /
    :class:`AtlasTexels` (per-face colours gathered through pix_to_face, vertex colours interpolated with bary_coords,
    UV maps sampled, atlas cells looked up, all inside the kernel: the texel tensor of ``sample_textures`` is never
    materialised).  Returns colors (N,H,W,K,3)."""
    pix_to_face = fragments.pix_to_face
    if fragments.bary_coords is None:
        raise ValueError("phong_shading needs fragments.bary_coords (N,H,W,K,3)")
    require_cuda(pix_to_face, fragments.bary_coords)
    if pix_to_face.dtype != torch.int64:
        pix_to_face = pix_to_face.to(torch.int64)
    N = pix_to_face.shape[0]
    device = pix_to_face.device
    verts = meshes.verts_packed()
    faces = meshes.faces_packed()
    vertex_normals = meshes.verts_normals_packed()
    faces_verts = verts[faces]  # (F,3,3); torch's indexing scatters the gradient back to the vertices
    faces_normals = vertex_normals[faces]
    lighting = pack_lighting(lights, materials, cameras, N, device)
    tex, mode = _texel_source(texels)
    # a batch of poses of one topology (TriMeshes.extend / update_padded): image n only sees faces [n F, (n+1) F)
    n_mesh = len(meshes) if hasattr(meshes, "faces_packed_single") else 1
    fpm = faces.shape[0] // n_mesh if (n_mesh > 1 and n_mesh == N) else 0
    return _PhongShade.apply(faces_verts, faces_normals, tex, fragments.bary_coords, pix_to_face, lighting,
                             mode, bool(sparse), False, fpm, texels.face_uvs() if mode == "uv" else None)
