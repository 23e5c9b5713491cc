"""Data contracts at the drop-in boundary, and synthetic inputs of the benchmark shapes.

pytorch3d (0.4.0 in the reference's requirements.txt:7) is not installable in this image; the hot
path only touches its objects by attribute (SURVEY.md §0.2, §8b), so duck-typed shims with the
same field names are enough.  When pytorch3d is installed its own ``Fragments`` / ``BlendParams`` /
cameras / ``Meshes`` objects work unchanged.
"""

from __future__ import annotations

import math
from typing import NamedTuple, Optional, Sequence, Union

import torch


class Fragments(NamedTuple):
    """pytorch3d.renderer.mesh.rasterizer.Fragments: (N,H,W,K) each, bary_coords (N,H,W,K,3).
    pix_to_face int64 with -1 = empty; zbuf / dists float32 with -1 = empty; K sorted near -> far,
    padding last."""
    pix_to_face: torch.Tensor
    zbuf: torch.Tensor
    bary_coords: Optional[torch.Tensor]
    dists: torch.Tensor


class BlendParams(NamedTuple):
    """pytorch3d.renderer.blending.BlendParams (only background_color is read on this path,
    random_rasterizer.py:39)."""
    sigma: float = 1e-4
    gamma: float = 1e-4
    background_color: Union[torch.Tensor, Sequence[float]] = (1.0, 1.0, 1.0)


class DepthCameras:
    """Minimal stand-in for a pytorch3d camera batch: the shader only reads ``znear`` / ``zfar`` as
    1-D tensors of length N (random_rasterizer.py:172-173)."""

    def __init__(self, znear=1.0, zfar=100.0, n=1, device="cpu"):
        self.znear = torch.as_tensor(znear, dtype=torch.float32, device=device).reshape(-1)
        self.zfar = torch.as_tensor(zfar, dtype=torch.float32, device=device).reshape(-1)
        if self.znear.numel() == 1 and n > 1:
            self.znear = self.znear.expand(n).clone()
        if self.zfar.numel() == 1 and n > 1:
            self.zfar = self.zfar.expand(n).clone()

    def to(self, device):
        self.znear, self.zfar = self.znear.to(device), self.zfar.to(device)
        return self


class TexelMeshes:
    """Stand-in for ``Meshes`` on this path: ``sample_textures(fragments)`` returns a preset
    (N,H,W,K,3) texel tensor (random_rasterizer.py:170)."""

    def __init__(self, texels: torch.Tensor):
        self.texels = texels

    def sample_textures(self, fragments):
        return self.texels


class FaceTexels:
    """Lazy texels: the colour of fragment (n,h,w,k) is ``face_colors[pix_to_face[n,h,w,k]]``.
    ``smooth_rgb_blend`` gathers it inside the fused kernels (and scatters the gradient back to
    ``face_colors``), so the (N,H,W,K,3) tensor of ``Meshes.sample_textures``
    (random_rasterizer.py:170) is never materialised."""

    def __init__(self, face_colors: torch.Tensor):
        if face_colors.dim() != 2 or face_colors.shape[1] != 3:
            raise ValueError("face_colors must be (F,3)")
        self.face_colors = face_colors

    def materialize(self, pix_to_face: torch.Tensor) -> torch.Tensor:
        mask = pix_to_face >= 0
        return self.face_colors[pix_to_face.clamp(min=0)] * mask[..., None]


class VertexTexels:
    """Lazy texels of a ``TexturesVertex`` mesh (experiments/eval.py:450): the colour of fragment (n,h,w,k) is the
    barycentric interpolation of the three vertex colours of face ``pix_to_face[n,h,w,k]``.  The Phong kernel
    interpolates it in place; ``sample_lazy_textures`` materialises it for the other consumers."""

    def __init__(self, verts_colors: torch.Tensor, faces: torch.Tensor):
        if verts_colors.dim() != 2 or verts_colors.shape[1] != 3:
            raise ValueError("verts_colors must be (V,3)")
        self.verts_colors, self.faces = verts_colors, faces

    def face_vert_colors(self) -> torch.Tensor:
        return self.verts_colors[self.faces]  # (F,3,3); torch scatters the gradient back to the vertices

    def materialize(self, pix_to_face: torch.Tensor, bary: torch.Tensor) -> torch.Tensor:
        mask = pix_to_face >= 0
        return (bary[..., None] * self.face_vert_colors()[pix_to_face.clamp(min=0)]).sum(-2) * mask[..., None]


class UVTexels:
    """Lazy texels of a UV-mapped mesh (pytorch3d ``TexturesUV`` / the legacy ``Textures(verts_uvs, faces_uvs, maps)`` of
    experiments/eval.py:750-756): the colour of fragment (n,h,w,k) is the bilinear tap of ``maps`` at the barycentric
    interpolation of the three corner UVs of face ``pix_to_face[n,h,w,k]`` (grid_sample with align_corners and border
    padding on the vertically flipped map, as pytorch3d 0.4.0 does).  ``maps`` (M,Hm,Wm,3) with M = 1 or N;
    ``verts_uvs`` (Vt,2); ``faces_uvs`` (F,3) indices into it, F = the PACKED face count."""

    def __init__(self, maps: torch.Tensor, verts_uvs: torch.Tensor, faces_uvs: torch.Tensor):
        if maps.dim() == 3:
            maps = maps[None]
        if maps.dim() != 4 or maps.shape[-1] != 3:
            raise ValueError("maps must be (M,Hm,Wm,3)")
        self.maps, self.verts_uvs, self.faces_uvs = maps, verts_uvs, faces_uvs.to(torch.int64)

    def face_uvs(self) -> torch.Tensor:
        return self.verts_uvs[self.faces_uvs]  # (F,3,2)

    def materialize(self, pix_to_face: torch.Tensor, bary: torch.Tensor) -> torch.Tensor:
        """The same sampling with torch ops (TexturesUV.sample_textures restated; reference for the tests)."""
        N, H, W, K = pix_to_face.shape
        mask = pix_to_face >= 0
        uv = (bary[..., None] * self.face_uvs()[pix_to_face.clamp(min=0)]).sum(-2)  # (N,H,W,K,2)
        grid = (uv * 2.0 - 1.0).permute(0, 3, 1, 2, 4).reshape(N * K, H, W, 2)
        maps = torch.flip(self.maps, [1]).permute(0, 3, 1, 2)  # (M,3,Hm,Wm), flipped vertically
        maps = maps.expand(N, -1, -1, -1) if maps.shape[0] == 1 else maps
        maps = maps[:, None].expand(N, K, *maps.shape[1:]).reshape(N * K, *maps.shape[1:])
        tex = torch.nn.functional.grid_sample(maps, grid, mode="bilinear", padding_mode="border", align_corners=True)
        tex = tex.reshape(N, K, 3, H, W).permute(0, 3, 4, 1, 2)
        return tex * mask[..., None]


class AtlasTexels:
    """Texels of a per-face texture atlas (pytorch3d ``TexturesAtlas``, the ShapeNet models of experiments/eval.py:216-238):
    ``atlas`` (F,R,R,3) holds an R x R grid of texels per PACKED face; the colour of fragment (n,h,w,k) is the nearest
    atlas texel at its first two barycentric coordinates, with the cell reflected when the point lies above the grid's
    diagonal.  Restates ``TexturesAtlas.sample_textures`` of pytorch3d 0.4.0 (renderer/mesh/textures.py; the package is
    not installable here: parity unpinned, anchored on the known answers of tests/test_cabi_cpu.py).  A nearest lookup:
    gradients reach the atlas (index scatter, by autograd), not the barycentric coordinates.  Deliberate differences:
    a barycentric coordinate of exactly 1 indexes cell R in pytorch3d (out of range); here it is clamped to R - 1.
    The rasteriser's barycentric coordinates are unclipped (outside [0, 1] in the blur band, far outside for sliver
    faces), where pytorch3d's rule wraps negative cells or overflows the grid: here NaN counts as 0, w R is clamped to
    [-1, R] before the truncation and the (possibly reflected) cell to the grid, so every cell is in range.  Wherever
    pytorch3d's rule picks an in-range cell without wrapping, this one picks the same cell.

    On a CUDA device the Phong kernels look the cells up in place (``pert_phong_atlas_fwd/bwd``, the same rule op for
    op); :meth:`materialize` builds the (N,H,W,K,3) tensor with torch ops."""

    def __init__(self, atlas: torch.Tensor):
        if atlas.dim() != 4 or atlas.shape[1] != atlas.shape[2] or atlas.shape[3] != 3:
            raise ValueError("atlas must be (F,R,R,3)")
        self.atlas = atlas

    def materialize(self, pix_to_face: torch.Tensor, bary: torch.Tensor) -> torch.Tensor:
        R = self.atlas.shape[1]
        mask = pix_to_face >= 0
        w01 = torch.where(mask[..., None], bary[..., :2], torch.zeros_like(bary[..., :2]))
        w01 = torch.nan_to_num(w01, nan=0.0)
        w_xy = (w01 * R).clamp(-1, R).to(torch.int64).clamp(max=R - 1)
        w0, w1 = w01.unbind(-1)
        w_x, w_y = w_xy.unbind(-1)
        below = ((w0 + w1) * R - (w_x + w_y).to(w01.dtype)) <= 1.0  # each op rounded once, as in the kernel
        w_x = torch.where(below, w_x, R - 1 - w_x).clamp(0, R - 1)
        w_y = torch.where(below, w_y, R - 1 - w_y).clamp(0, R - 1)
        return self.atlas[pix_to_face.clamp(min=0), w_y, w_x] * mask[..., None].to(self.atlas.dtype)


class FaceColorMeshes:
    """Stand-in for ``Meshes`` with one colour per (packed) face: ``sample_textures`` returns lazy
    :class:`FaceTexels` instead of a texel tensor."""

    def __init__(self, face_colors: torch.Tensor):
        self.face_colors = face_colors

    def sample_textures(self, fragments):
        return FaceTexels(self.face_colors)


def _color_rows(v, device):
    return torch.as_tensor(v, dtype=torch.float32, device=device).reshape(-1, 3)


class PointLights:
    """pytorch3d.renderer.lighting.PointLights by attribute (same constructor defaults): colours and
    ``location`` are (1,3) or (N,3) tensors."""

    def __init__(self, ambient_color=((0.5, 0.5, 0.5),), diffuse_color=((0.3, 0.3, 0.3),),
                 specular_color=((0.2, 0.2, 0.2),), location=((0, 1, 0),), device="cpu"):
        self.ambient_color = _color_rows(ambient_color, device)
        self.diffuse_color = _color_rows(diffuse_color, device)
        self.specular_color = _color_rows(specular_color, device)
        self.location = _color_rows(location, device)

    def to(self, device):
        for k in ("ambient_color", "diffuse_color", "specular_color", "location"):
            setattr(self, k, getattr(self, k).to(device))
        return self


class DirectionalLights:
    """pytorch3d.renderer.lighting.DirectionalLights by attribute: ``direction`` instead of ``location``."""

    def __init__(self, ambient_color=((0.5, 0.5, 0.5),), diffuse_color=((0.3, 0.3, 0.3),),
                 specular_color=((0.2, 0.2, 0.2),), direction=((0, 1, 0),), device="cpu"):
        self.ambient_color = _color_rows(ambient_color, device)
        self.diffuse_color = _color_rows(diffuse_color, device)
        self.specular_color = _color_rows(specular_color, device)
        self.direction = _color_rows(direction, device)

    def to(self, device):
        for k in ("ambient_color", "diffuse_color", "specular_color", "direction"):
            setattr(self, k, getattr(self, k).to(device))
        return self


class Materials:
    """pytorch3d.renderer.materials.Materials by attribute (defaults: white, shininess 64)."""

    def __init__(self, ambient_color=((1, 1, 1),), diffuse_color=((1, 1, 1),), specular_color=((1, 1, 1),),
                 shininess=64, device="cpu"):
        self.ambient_color = _color_rows(ambient_color, device)
        self.diffuse_color = _color_rows(diffuse_color, device)
        self.specular_color = _color_rows(specular_color, device)
        self.shininess = torch.as_tensor(shininess, dtype=torch.float32, device=device).reshape(-1)

    def to(self, device):
        for k in ("ambient_color", "diffuse_color", "specular_color", "shininess"):
            setattr(self, k, getattr(self, k).to(device))
        return self


class ViewCameras(DepthCameras):
    """A camera batch with extrinsics: ``R`` (N,3,3), ``T`` (N,3) in pytorch3d's row-vector convention
    ``X_view = X_world R + T``, so the camera centre is ``-T R^T`` (``get_camera_center``)."""

    def __init__(self, R, T, znear=1.0, zfar=100.0, device="cpu"):
        self.R = torch.as_tensor(R, dtype=torch.float32, device=device).reshape(-1, 3, 3)
        self.T = torch.as_tensor(T, dtype=torch.float32, device=device).reshape(-1, 3)
        super().__init__(znear=znear, zfar=zfar, n=self.R.shape[0], device=device)

    def get_camera_center(self):
        return -torch.bmm(self.T[:, None, :], self.R.transpose(1, 2))[:, 0, :]

    def to(self, device):
        super().to(device)
        self.R, self.T = self.R.to(device), self.T.to(device)
        return self


class TriMeshes:
    """Stand-in for pytorch3d ``Meshes``: ONE topology ``faces`` (F,3) with vertices (V,3), or a batch of N poses of
    it, vertices (N,V,3) (``extend`` / ``update_padded`` as in eval.py:343,281-283).  The packed representation
    (``verts_packed`` (N*V,3), ``faces_packed`` (N*F,3)) is what ``pix_to_face`` indexes.  Textures: one colour per
    face (lazy :class:`FaceTexels`), one colour per vertex (lazy :class:`VertexTexels`), a UV map (lazy
    :class:`UVTexels`), a per-face atlas (:class:`AtlasTexels`, lazy on a CUDA device) or a preset texel tensor.
    ``verts_normals_packed`` follows pytorch3d's area-weighted vertex normals (cross products of the face edges
    summed onto the corners, then normalised with eps 1e-6)."""

    def __init__(self, verts, faces, face_colors=None, texels=None, verts_colors=None, uv=None, atlas=None):
        self._verts, self._faces = verts, faces.to(torch.int64)
        self.face_colors, self.texels, self.verts_colors = face_colors, texels, verts_colors
        self.uv = uv  # (maps (M,Hm,Wm,3), verts_uvs (Vt,2), faces_uvs (F,3)): a UV-mapped mesh
        self.atlas = atlas  # (F,R,R,3): a per-face texture atlas (pytorch3d TexturesAtlas)

    def __len__(self):
        return self._verts.shape[0] if self._verts.dim() == 3 else 1

    def verts_padded(self):
        return self._verts if self._verts.dim() == 3 else self._verts[None]

    def faces_packed_single(self):
        return self._faces

    def verts_packed(self):
        return self._verts.reshape(-1, 3)

    def faces_packed(self):
        n = len(self)
        if n == 1:
            return self._faces
        V = self._verts.shape[-2]
        off = torch.arange(n, device=self._faces.device, dtype=torch.int64)[:, None, None] * V
        return (self._faces[None] + off).reshape(-1, 3)

    def verts_normals_packed(self):
        v, f = self.verts_packed(), self.faces_packed()
        vf = v[f]
        # pytorch3d adds, at every corner of a face, the cross product of the two edges leaving that corner: the three
        # products are the same vector (twice the area normal), so one cross and one scatter do it
        fn = torch.cross(vf[:, 1] - vf[:, 0], vf[:, 2] - vf[:, 0], dim=1)
        n = torch.zeros_like(v).index_add(0, f.reshape(-1), fn.repeat_interleave(3, dim=0))
        return torch.nn.functional.normalize(n, eps=1e-6, dim=1)

    def sample_textures(self, fragments):
        if self.texels is not None:
            return self.texels
        n = len(self)
        if self.atlas is not None:
            # a nearest-texel lookup: lazy on a CUDA device (the Phong kernels look the cells up in place and scatter the
            # gradient into the atlas), materialised with torch indexing elsewhere
            if fragments.bary_coords is None:
                raise ValueError("atlas textures need fragments.bary_coords (N,H,W,K,3)")
            atlas = self.atlas if n == 1 else self.atlas.repeat(n, 1, 1, 1)
            if atlas.is_cuda:
                return AtlasTexels(atlas)
            return AtlasTexels(atlas).materialize(fragments.pix_to_face, fragments.bary_coords)
        if self.uv is not None:
            maps, verts_uvs, faces_uvs = self.uv
            return UVTexels(maps, verts_uvs, faces_uvs if n == 1 else faces_uvs.repeat(n, 1))
        if self.verts_colors is not None:
            vc = self.verts_colors if n == 1 else self.verts_colors.repeat(n, 1)
            return VertexTexels(vc, self.faces_packed())
        return FaceTexels(self.face_colors if n == 1 else self.face_colors.repeat(n, 1))

    def extend(self, n: int):
        """n copies of a single mesh as one batch (pytorch3d ``Meshes.extend``)."""
        if len(self) != 1:
            raise ValueError("extend() needs a single mesh")
        return TriMeshes(self.verts_padded().expand(n, -1, -1).contiguous(), self._faces, self.face_colors, self.texels,
                         self.verts_colors, self.uv, self.atlas)

    def update_padded(self, verts):
        """Same topology and textures, new vertex positions (V,3) or (N,V,3) (pytorch3d ``Meshes.update_padded``)."""
        return TriMeshes(verts, self._faces, self.face_colors, self.texels, self.verts_colors, self.uv, self.atlas)

    update_verts = update_padded


def _icosphere(level: int):
    """Unit icosphere: 20 * 4**level faces, 10 * 4**level + 2 vertices (level 3 = 1280 faces / 642 vertices, the
    sphere_642.obj of experiments/eval.py:289), outward counter-clockwise winding."""
    t = (1.0 + math.sqrt(5.0)) / 2.0
    v = torch.tensor([[-1, t, 0], [1, t, 0], [-1, -t, 0], [1, -t, 0], [0, -1, t], [0, 1, t], [0, -1, -t], [0, 1, -t],
                      [t, 0, -1], [t, 0, 1], [-t, 0, -1], [-t, 0, 1]], dtype=torch.float64)
    f = torch.tensor([[0, 11, 5], [0, 5, 1], [0, 1, 7], [0, 7, 10], [0, 10, 11], [1, 5, 9], [5, 11, 4], [11, 10, 2],
                      [10, 7, 6], [7, 1, 8], [3, 9, 4], [3, 4, 2], [3, 2, 6], [3, 6, 8], [3, 8, 9], [4, 9, 5], [2, 4, 11],
                      [6, 2, 10], [8, 6, 7], [9, 8, 1]], dtype=torch.int64)
    v = v / v.norm(dim=1, keepdim=True)
    for _ in range(level):
        e = torch.cat((f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]))  # (3F,2) directed edges
        key = torch.sort(e, dim=1).values
        uniq, inv = torch.unique(key, dim=0, return_inverse=True)
        mid = v[uniq[:, 0]] + v[uniq[:, 1]]
        mid = mid / mid.norm(dim=1, keepdim=True)
        nv = v.shape[0]
        F_ = f.shape[0]
        a, b, c = inv[:F_] + nv, inv[F_:2 * F_] + nv, inv[2 * F_:] + nv  # midpoints of edges 01, 12, 20
        f = torch.cat((torch.stack((f[:, 0], a, c), 1), torch.stack((f[:, 1], b, a), 1), torch.stack((f[:, 2], c, b), 1),
                       torch.stack((a, b, c), 1)))
        v = torch.cat((v, mid))
    return v.float(), f


def synthetic_mesh(n_faces=1280, seed=0, device="cuda"):
    """A unit-scale triangle mesh with ``n_faces`` faces for the benchmarks and tests: the icosphere of the smallest
    level with at least that many faces (20, 80, 320, 1280, ... are closed spheres; other counts keep the first
    ``n_faces`` faces of the next level: an open sphere, still without sliver triangles).
    Returns (verts (V,3), faces (F,3))."""
    level = 0
    while 20 * 4 ** level < n_faces:
        level += 1
    verts, faces = _icosphere(level)
    return verts.to(device), faces[:n_faces].contiguous().to(device)


def synthetic_bary(pix_to_face, seed=0):
    """Random barycentric coordinates (N,H,W,K,3) for the valid entries (positive, summing to 1), -1 at
    padding like pytorch3d's rasteriser."""
    g = torch.Generator(device=pix_to_face.device).manual_seed(seed + 17)
    e = -torch.log(torch.rand(pix_to_face.shape + (3,), generator=g, device=pix_to_face.device).clamp_min(1e-9))
    b = e / e.sum(dim=-1, keepdim=True)
    return torch.where((pix_to_face >= 0)[..., None], b, torch.full_like(b, -1.0)).float()


def blur_radius(sigma: float) -> float:
    """experiments/eval.py:137: log(1/1e-4 - 1) * sigma."""
    return math.log(1.0 / 1e-4 - 1.0) * sigma


def synthetic_fragments(N, H, W, K, kind="dense", sigma=1e-3, n_faces=1280, seed=0, device="cuda",
                        coverage=0.6, mean_valid=4.0, frac_edge=0.15):
    """Synthetic Fragments + texels of the benchmark shapes (SURVEY.md §8d).

    dense:     every pixel has all K faces valid, dists ~ U(-b, b), b = blur radius.
    realistic: 60 % of pixels covered, valid count per covered pixel geometric with mean 4 (capped
               at K, padding last), dists 85 % interior -U(0, 0.05) and 15 % edge band U(-b, b).
    Valid entries: pix_to_face ~ U{0..F-1}, zbuf ascending in K ~ U(5.5, 8.0), colours ~ U(0,1).
    Padded entries: pix_to_face = -1, zbuf = dists = -1, colours = 0.
    Returns (Fragments, colors (N,H,W,K,3)).
    """
    g = torch.Generator(device=device).manual_seed(seed)
    b = blur_radius(sigma)
    shape = (N, H, W, K)
    u = lambda *s: torch.rand(*s, generator=g, device=device)  # noqa: E731
    if kind == "dense":
        valid = torch.ones(shape, dtype=torch.bool, device=device)
        dists = (u(shape) * 2 - 1) * b
    elif kind == "realistic":
        covered = u((N, H, W, 1)) < coverage
        # geometric with mean m on {1,2,...}: 1 + floor(log(U)/log(1-1/m))
        q = 1.0 - 1.0 / mean_valid
        nvalid = (1 + torch.floor(torch.log(u((N, H, W, 1)).clamp_min(1e-12)) / math.log(q))).clamp(max=K)
        nvalid = torch.where(covered, nvalid, torch.zeros_like(nvalid))
        valid = torch.arange(K, device=device).view(1, 1, 1, K) < nvalid
        edge = u(shape) < frac_edge
        dists = torch.where(edge, (u(shape) * 2 - 1) * b, -0.05 * u(shape))
    else:
        raise ValueError(f"unknown fragment kind {kind!r}")
    z = 5.5 + 2.5 * u(shape)
    z = torch.where(valid, z, torch.full_like(z, float("inf"))).sort(dim=-1).values  # ascending, padding last
    zbuf = torch.where(valid, z, torch.full_like(z, -1.0))
    dists = torch.where(valid, dists, torch.full_like(dists, -1.0))
    faces = torch.randint(0, n_faces, shape, generator=g, device=device, dtype=torch.int64)
    pix_to_face = torch.where(valid, faces, torch.full_like(faces, -1))
    colors = u((N, H, W, K, 3)) * valid[..., None]
    return Fragments(pix_to_face, zbuf.float(), None, dists.float()), colors.float()
