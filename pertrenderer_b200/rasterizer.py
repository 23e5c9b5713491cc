"""Fragment producer: the rasteriser in front of the perturbed shader.

The reference builds ``MeshRenderer(rasterizer=MeshRasterizer(cameras, raster_settings), shader=Random*Shader)``
from pytorch3d (experiments/eval.py:135-141,165-177).  pytorch3d is not installable in this image, so this module
provides the same call shape on the hand-written kernels ``pert_rasterize_fwd / pert_rasterize_bwd``
(include/pertshade.h, csrc/raster.cu): ``RasterizationSettings``, ``MeshRasterizer``, ``MeshRenderer``,
``look_at_view_transform`` and a FoV perspective camera (``OpenGLPerspectiveCameras`` of pytorch3d 0.4.0), so that
the pose-optimisation loop of eval.py:320-409 runs end to end.  Camera and projection arithmetic is plain torch
(differentiable plumbing); the rasterisation and its backward are the CUDA kernels; there is no CPU fallback.
"""

from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Optional, Tuple, Union

import torch
from torch.autograd import Function

from . import _cabi
from ._cabi import RAST_CULL_BACKFACES, PertRaster, check, ptr, require_cuda, stream_ptr
from .structures import DepthCameras, Fragments


BIN_MIN_FACES = 8192  # faces per mesh from which the forward builds coarse bins (measured: 5 k faces are faster without)


@dataclass
class RasterizationSettings:
    """pytorch3d.renderer.mesh.rasterizer.RasterizationSettings (same field names and defaults).  ``bin_size`` /
    ``max_faces_per_bin`` are accepted and ignored (the kernel culls faces per pixel tile itself);
    ``perspective_correct`` and ``clip_barycentric_coords`` must stay False (the reference's setting, eval.py:140)."""
    image_size: Union[int, Tuple[int, int]] = 256
    blur_radius: float = 0.0
    faces_per_pixel: int = 1
    bin_size: Optional[int] = None
    max_faces_per_bin: Optional[int] = None
    perspective_correct: bool = False
    clip_barycentric_coords: bool = False
    cull_backfaces: bool = False


def _raster_struct(face_verts, face_start, N, H, W, K, blur_radius, cull_backfaces, face_order=None):
    rs = PertRaster()
    rs.face_order = None if face_order is None else face_order.data_ptr()
    rs.N, rs.H, rs.W, rs.K = N, H, W, K
    rs.flags = RAST_CULL_BACKFACES if cull_backfaces else 0
    rs.blur_radius = float(blur_radius)
    rs.num_faces = face_verts.shape[0]
    rs.face_verts, rs.face_start = face_verts.data_ptr(), face_start.data_ptr()
    return rs


def _bounded_bins_pay(rs, bin_capacity, H, W, blur_radius):
    """Whether the bounded bins are no slower than the synchronising ones.  Every face's box is grown by sqrt(blur_radius)
    on each side; where that margin alone spans more than C tiles, every face goes to its image's wide list and each tile
    walks all faces of its mesh: at 8 x 256^2 and 16 x 1024^2 with eval.py's blur the bounded bins are 1.15x and 1.7x
    slower, at 1 x 128^2 they are faster and keep the host free (profiles/r10_raster_bins.txt)."""
    margin = 2.0 * math.sqrt(blur_radius) * min(H, W) / 2.0  # pixels: the box's least width and height
    return (margin / 4 + 1) * (margin / 32 + 1) <= bin_capacity(rs) // rs.num_faces  # 32x4 tiles


def _build_bins(lib, rs, N, H, W, blur_radius, dev):
    """Coarse bins of a large mesh in rs.bin_*, two kernel passes around a prefix sum; returns the tensors that hold them.
    Inside a CUDA-graph capture, or where _bounded_bins_pay, the bounded bins (one candidate list per 32x4 pixel tile and
    one wide list per image, sized from the face count: nothing is read back to the host).  Elsewhere one list per tile
    holding every face whose box overlaps it, sized from a total read back from the device: a host sync."""
    bin_bounded, bin_capacity = _cabi.raster_bin_fns()
    st = stream_ptr(dev)
    bounded = torch.cuda.is_current_stream_capturing() or _bounded_bins_pay(rs, bin_capacity, H, W, blur_radius)
    fill, name = (bin_bounded, "pert_rasterize_bin_bounded") if bounded else (lib.pert_rasterize_bin, "pert_rasterize_bin")
    nb = int(lib.pert_rasterize_num_bins(rs)) + (N if bounded else 0)
    count = torch.zeros((nb,), dtype=torch.int32, device=dev)
    check(fill(rs, ptr(count), None, None, None, st), name)
    ends = torch.cumsum(count, 0, dtype=torch.int64)
    offset = (ends - count).contiguous()
    lists = torch.empty((max(int(bin_capacity(rs) if bounded else ends[-1].item()), 1),), dtype=torch.int64, device=dev)
    cursor = torch.zeros((nb,), dtype=torch.int32, device=dev)
    check(fill(rs, ptr(count), ptr(offset), ptr(cursor), ptr(lists), st), name)
    rs.bin_count, rs.bin_offset, rs.bin_faces = count.data_ptr(), offset.data_ptr(), lists.data_ptr()
    if bounded:
        rs.flags |= _cabi.RAST_BIN_WIDE
    return [count, offset, lists]


class _Rasterize(Function):
    @staticmethod
    def forward(ctx, face_verts, face_start, H, W, K, blur_radius, cull_backfaces):
        lib = _cabi.load()
        require_cuda(face_verts, face_start)
        fv = face_verts.detach()
        fv = fv if (fv.dtype == torch.float32 and fv.is_contiguous()) else fv.to(torch.float32).contiguous()
        fs = face_start.to(torch.int64).contiguous()
        N = fs.numel() - 1
        dev = fv.device
        with torch.cuda.device(dev):
            p2f = torch.empty((N, H, W, K), dtype=torch.int64, device=dev)
            zbuf = torch.empty((N, H, W, K), dtype=torch.float32, device=dev)
            bary = torch.empty((N, H, W, K, 3), dtype=torch.float32, device=dev)
            dists = torch.empty((N, H, W, K), dtype=torch.float32, device=dev)
            rs = _raster_struct(fv, fs, N, H, W, K, blur_radius, cull_backfaces)
            keep = []
            if K <= 64 and fv.shape[0] >= BIN_MIN_FACES * N:
                keep = _build_bins(lib, rs, N, H, W, blur_radius, dev)
            rc = lib.pert_rasterize_fwd(rs, ptr(p2f), ptr(zbuf), ptr(bary), ptr(dists), stream_ptr(dev))
            del keep
        check(rc, "pert_rasterize_fwd")
        ctx.save_for_backward(fv, fs, p2f)
        ctx.cfg = (N, H, W, K, blur_radius, cull_backfaces)
        ctx.mark_non_differentiable(p2f)
        return p2f, zbuf, bary, dists

    @staticmethod
    def backward(ctx, _g_p2f, g_zbuf, g_bary, g_dists):
        lib = _cabi.load()
        fv, fs, p2f = ctx.saved_tensors
        N, H, W, K, blur_radius, cull = ctx.cfg
        dev = fv.device
        c = lambda t: None if t is None else t.to(torch.float32).contiguous()  # noqa: E731
        g_zbuf, g_bary, g_dists = c(g_zbuf), c(g_bary), c(g_dists)
        with torch.cuda.device(dev):
            g_fv = torch.zeros_like(fv)
            rs = _raster_struct(fv, fs, N, H, W, K, blur_radius, cull)
            rc = lib.pert_rasterize_bwd(rs, ptr(p2f), ptr(g_zbuf), ptr(g_bary), ptr(g_dists), ptr(g_fv), stream_ptr(dev))
        check(rc, "pert_rasterize_bwd")
        return g_fv, None, None, None, None, None, None


def rasterize_meshes(face_verts, face_start, image_size, blur_radius=0.0, faces_per_pixel=8, cull_backfaces=False):
    """pytorch3d.renderer.mesh.rasterize_meshes on packed faces.  ``face_verts`` (F,3,3): NDC x, y and view depth of
    every face corner; ``face_start`` (N+1,) int64 on the device: faces of image n.  Returns
    (pix_to_face, zbuf, bary_coords, dists) as in pytorch3d; gradients of zbuf / bary_coords / dists flow to
    ``face_verts``."""
    H, W = (image_size, image_size) if isinstance(image_size, int) else tuple(image_size)
    return _Rasterize.apply(face_verts, face_start, int(H), int(W), int(faces_per_pixel), float(blur_radius), bool(cull_backfaces))


# ------------------------------------------------------------------------------------------------------------
# cameras (pytorch3d.renderer.cameras): row-vector convention X_view = X_world R + T
# ------------------------------------------------------------------------------------------------------------
def look_at_view_transform(dist=1.0, elev=0.0, azim=0.0, degrees: bool = True, device="cpu"):
    """pytorch3d.renderer.look_at_view_transform for a camera orbiting the origin (at = 0, up = +Y).
    ``dist`` / ``elev`` / ``azim`` scalars or 1-D tensors.  Returns R (N,3,3), T (N,3)."""
    d, e, a = (torch.as_tensor(t, dtype=torch.float32, device=device).reshape(-1) for t in (dist, elev, azim))
    n = max(d.numel(), e.numel(), a.numel())
    d, e, a = (t.expand(n) for t in (d, e, a))
    if degrees:
        e, a = e * (math.pi / 180.0), a * (math.pi / 180.0)
    C = torch.stack((d * torch.cos(e) * torch.sin(a), d * torch.sin(e), d * torch.cos(e) * torch.cos(a)), dim=-1)
    z_axis = torch.nn.functional.normalize(-C, dim=-1)
    up = torch.tensor([0.0, 1.0, 0.0], device=device).expand_as(C)
    x_axis = torch.nn.functional.normalize(torch.linalg.cross(up, z_axis), dim=-1)
    y_axis = torch.nn.functional.normalize(torch.linalg.cross(z_axis, x_axis), dim=-1)
    R = torch.stack((x_axis, y_axis, z_axis), dim=-1)  # columns = camera axes
    T = -torch.bmm(C[:, None, :], R)[:, 0, :]
    return R, T


class FoVPerspectiveCameras(DepthCameras):
    """pytorch3d's FoVPerspectiveCameras / OpenGLPerspectiveCameras by attribute and method: ``R`` (N,3,3), ``T``
    (N,3), ``fov`` (degrees), ``znear``, ``zfar``, aspect ratio 1; ``get_camera_center``, ``transform_points_view``
    and ``transform_points_ndc`` (x, y projected, z = view depth: what MeshRasterizer.transform hands to the
    rasteriser)."""

    def __init__(self, R=None, T=None, fov=60.0, znear=1.0, zfar=100.0, degrees: bool = True, device="cpu"):
        self.R = torch.eye(3)[None] if R is None else torch.as_tensor(R, dtype=torch.float32)
        self.T = torch.zeros(1, 3) if T is None else torch.as_tensor(T, dtype=torch.float32)
        self.R, self.T = self.R.reshape(-1, 3, 3).to(device), self.T.reshape(-1, 3).to(device)
        self.fov = float(fov) if degrees else float(fov) * 180.0 / math.pi
        super().__init__(znear=znear, zfar=zfar, n=self.R.shape[0], device=device)

    def __len__(self):
        return self.R.shape[0]

    def get_camera_center(self):
        return -torch.bmm(self.T[:, None, :], self.R.transpose(1, 2))[:, 0, :]

    def transform_points_view(self, verts):
        """verts (N,V,3) or (V,3) world -> view."""
        v = verts if verts.dim() == 3 else verts[None]
        n = max(v.shape[0], self.R.shape[0])
        return torch.bmm(v.expand(n, -1, -1), self.R.expand(n, 3, 3)) + self.T.expand(n, 3)[:, None, :]

    def transform_points_ndc(self, verts):
        view = self.transform_points_view(verts)
        s = 1.0 / math.tan(math.radians(self.fov) / 2.0)
        z = view[..., 2]
        return torch.stack((s * view[..., 0] / z, s * view[..., 1] / z, z), dim=-1)

    def to(self, device):
        super().to(device)
        self.R, self.T = self.R.to(device), self.T.to(device)
        return self


OpenGLPerspectiveCameras = FoVPerspectiveCameras  # the name eval.py:259-262 uses


class MeshRasterizer(torch.nn.Module):
    """pytorch3d.renderer.MeshRasterizer: ``forward(meshes, **kwargs) -> Fragments``.  ``meshes`` needs
    ``verts_padded()`` (N,V,3) (or (1,V,3), broadcast over the cameras) and ``faces_packed_single()`` (F,3): one
    topology, N poses — the batched pose optimisation of BASELINE configs 2-3."""

    def __init__(self, cameras=None, raster_settings=None):
        super().__init__()
        self.cameras = cameras
        self.raster_settings = raster_settings if raster_settings is not None else RasterizationSettings()

    def transform(self, meshes, **kwargs):
        cameras = kwargs.get("cameras", self.cameras)
        if cameras is None:
            raise ValueError("Cameras must be specified either at initialization or in the forward pass of MeshRasterizer")
        return cameras.transform_points_ndc(meshes.verts_padded())  # (N,V,3)

    def forward(self, meshes, **kwargs) -> Fragments:
        rs = kwargs.get("raster_settings", self.raster_settings)
        if rs.perspective_correct or rs.clip_barycentric_coords:
            raise ValueError("perspective_correct / clip_barycentric_coords are not implemented (the reference rasterises "
                             "with both off, experiments/eval.py:135-141)")
        ndc = self.transform(meshes, **kwargs)
        if ndc.shape[0] != len(meshes):
            raise ValueError(f"{ndc.shape[0]} cameras for {len(meshes)} mesh(es): extend the mesh first (meshes.extend(N))")
        N, V, _ = ndc.shape
        faces = meshes.faces_packed_single()
        F_ = faces.shape[0]
        face_verts = ndc[:, faces]  # (N,F,3,3); torch's indexing scatters the gradient back to the vertices
        face_start = torch.arange(N + 1, device=ndc.device, dtype=torch.int64) * F_
        p2f, zbuf, bary, dists = rasterize_meshes(face_verts.reshape(N * F_, 3, 3), face_start, rs.image_size, rs.blur_radius,
                                                  rs.faces_per_pixel, rs.cull_backfaces)
        return Fragments(pix_to_face=p2f, zbuf=zbuf, bary_coords=bary, dists=dists)


class MeshRenderer(torch.nn.Module):
    """pytorch3d.renderer.MeshRenderer: rasterise, then shade (eval.py:165-177)."""

    def __init__(self, rasterizer, shader):
        super().__init__()
        self.rasterizer, self.shader = rasterizer, shader

    def forward(self, meshes_world, **kwargs) -> torch.Tensor:
        fragments = self.rasterizer(meshes_world, **kwargs)
        return self.shader(fragments, meshes_world, **kwargs)
