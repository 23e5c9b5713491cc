"""CPU oracle for the fragment producer (TEST INFRASTRUCTURE ONLY).

The reference builds its Fragments with pytorch3d's ``MeshRasterizer`` (``experiments/eval.py:135-141,165-169``:
``RasterizationSettings(image_size, blur_radius=log(1/1e-4-1)*sigma, faces_per_pixel=50, perspective_correct=False)``).
This module restates, in dense torch-CPU arithmetic over every (pixel, face) pair, what that call computes.

Only ``tests/`` and the CPU legs of ``bench.py`` / ``__graft_entry__.smoke()`` may import it; the product path
(``pertrenderer_b200.rasterizer``) never routes through it.

Parity status: UNPINNED at this boundary.  The arithmetic lives in pytorch3d 0.4.0 (``requirements.txt:7``), which
is neither vendored under ``/root/reference`` nor installable here, and the reference holds no fixture for it.
Restated from the published algorithm of that release:

    renderer/mesh/rasterize_meshes.py      rasterize_meshes (naive path), pix_to_ndc
    csrc/rasterize_meshes/rasterize_meshes.cu   CheckPixelInsideFace, RasterizeMeshesNaiveCudaKernel
    csrc/utils/geometry_utils.cuh          EdgeFunctionForward, BarycentricCoordsForward, PointLineDistanceForward,
                                           PointTriangleDistanceForward  (kEpsilon = 1e-8)
    renderer/mesh/rasterizer.py            MeshRasterizer.transform (NDC x, y; view-space depth as z)
    renderer/cameras.py                    FoVPerspectiveCameras / OpenGLPerspectiveCameras projection, look_at_view_transform

Semantics kept: pixel (0,0) is the top-left corner and NDC has +X left, +Y up; a face is a candidate for a pixel
when the pixel centre lies inside it, or within sqrt(blur_radius) of its bounding box AND at squared distance
< blur_radius of the triangle; zero-area faces, faces entirely behind the camera and points with interpolated
depth < 0 are skipped, and with ``cull_backfaces`` so are faces with edge(v0, v1, v2) < 0; the K candidates of smallest depth are kept, ascending, ties in face order; barycentric
coordinates are not clipped, not perspective-corrected; ``dists`` is the signed squared distance (negative
inside); padding is -1 everywhere.  Known divergence: when MORE than K faces qualify, pytorch3d's replace-the-
farthest rule may keep a different face among equal depths.

Anchors that ARE checked (``tests/test_raster_oracle.py``): closed-form triangles (centre pixel, edge distance,
vertex distance, depth order), and finite differences of the gradients.  Gradients here come from autograd over
the restated forward formulas of the selected (pixel, face) pairs; the CUDA backward is hand-derived.
"""

from __future__ import annotations

import math

import torch

K_EPS = 1e-8


def pix_to_ndc(i, S1, S2):
    """rasterize_meshes.cu PixToNonSquareNdc: centre of pixel i along an axis of S1 pixels (other axis S2)."""
    rng = (S1 / S2) if S1 > S2 else 1.0
    return -rng + (2.0 * i + 1.0) * rng / S1


def pixel_centers(H, W, dtype=torch.float32):
    """(H,W,2) NDC coordinates (x, y) of the pixel centres; row 0 is the TOP row (y = +1 side), column 0 the
    LEFT column (x = +1 side)."""
    yi = (H - 1 - torch.arange(H, dtype=dtype))
    xi = (W - 1 - torch.arange(W, dtype=dtype))
    yf = pix_to_ndc(yi, H, W)
    xf = pix_to_ndc(xi, W, H)
    return torch.stack((xf[None, :].expand(H, W), yf[:, None].expand(H, W)), dim=-1)


def edge_function(p, v0, v1):
    """geometry_utils.cuh EdgeFunctionForward."""
    return (p[..., 0] - v0[..., 0]) * (v1[..., 1] - v0[..., 1]) - (p[..., 1] - v0[..., 1]) * (v1[..., 0] - v0[..., 0])


def barycentric(p, v0, v1, v2):
    """geometry_utils.cuh BarycentricCoordsForward (area + kEpsilon in the denominator)."""
    area = edge_function(v2, v0, v1) + K_EPS
    return torch.stack((edge_function(p, v1, v2) / area, edge_function(p, v2, v0) / area, edge_function(p, v0, v1) / area), dim=-1)


def point_line_distance(p, v0, v1):
    """geometry_utils.cuh PointLineDistanceForward: squared distance to the SEGMENT v0-v1."""
    v1v0 = v1 - v0
    l2 = (v1v0 * v1v0).sum(-1)
    t = (v1v0 * (p - v0)).sum(-1) / l2.clamp_min(K_EPS * 1e-30 + 1e-38)
    tt = t.clamp(0.0, 1.0)
    proj = v0 + tt[..., None] * v1v0
    d = ((p - proj) ** 2).sum(-1)
    d_deg = ((p - v1) ** 2).sum(-1)
    return torch.where(l2 <= K_EPS, d_deg, d)


def point_triangle_distance(p, v0, v1, v2):
    """geometry_utils.cuh PointTriangleDistanceForward: min over the three edges."""
    e01 = point_line_distance(p, v0, v1)
    e02 = point_line_distance(p, v0, v2)
    e12 = point_line_distance(p, v1, v2)
    return torch.minimum(torch.minimum(e01, e02), e12)


def _rasterize_pixels(pxy, v, f0, K, blur_radius, cull_backfaces):
    """The K-deep fragments of the pixel centres pxy (P,1,2) against the faces v (Fn,3,3), Fn >= 1."""
    Fn = v.shape[0]
    v0, v1, v2 = (v[None, :, i, :2] for i in range(3))
    z = v[None, :, :, 2]
    area = edge_function(v0, v1, v2)
    zero_area = (area <= K_EPS) & (area >= -K_EPS)
    back = (area < 0) if cull_backfaces else torch.zeros_like(zero_area)
    r = math.sqrt(blur_radius)
    xs, ys = v[None, :, :, 0], v[None, :, :, 1]
    outside = (pxy[..., 0] > xs.max(-1).values + r) | (pxy[..., 0] < xs.min(-1).values - r) | \
              (pxy[..., 1] > ys.max(-1).values + r) | (pxy[..., 1] < ys.min(-1).values - r)
    bary = barycentric(pxy, v0, v1, v2)  # (P,Fn,3)
    pz = (bary * z).sum(-1)
    dist = point_triangle_distance(pxy, v0, v1, v2)
    inside = (bary > 0).all(-1)
    ok = ~(z.max(-1).values < 0) & ~outside & ~zero_area & ~back & ~(pz < 0) & (inside | (dist < blur_radius))
    key = torch.where(ok, pz, torch.full_like(pz, float("inf")))
    order = torch.sort(key, dim=1, stable=True).indices[:, :K]  # ties keep face order
    if Fn < K:
        order = torch.cat((order, order.new_zeros(order.shape[0], K - Fn)), dim=1)
    sel_ok = torch.gather(ok, 1, order)
    if Fn < K:
        sel_ok[:, Fn:] = False
    g = lambda t: torch.gather(t, 1, order)  # noqa: E731
    p2f = torch.where(sel_ok, order + f0, torch.full_like(order, -1))
    zb = torch.where(sel_ok, g(pz), torch.full_like(g(pz), -1.0))
    sd = torch.where(inside, -dist, dist)
    ds = torch.where(sel_ok, g(sd), torch.full_like(zb, -1.0))
    bc = torch.gather(bary, 1, order[..., None].expand(-1, -1, 3))
    bc = torch.where(sel_ok[..., None], bc, torch.full_like(bc, -1.0))
    return p2f, zb, bc, ds


def rasterize(face_verts, face_start, H, W, K, blur_radius, cull_backfaces=False, chunk_pairs=1 << 21):
    """rasterize_meshes (naive).  face_verts (F,3,3): NDC x, y and view depth z of the packed faces;
    face_start (N+1,): faces [face_start[n], face_start[n+1]) belong to image n (an empty range gives an image of
    padding).  ``cull_backfaces`` drops the faces with edge(v0, v1, v2) < 0.  Pixels are evaluated in chunks of about
    ``chunk_pairs`` (pixel, face) pairs, which bounds the memory and leaves the result unchanged.
    Returns pix_to_face (N,H,W,K) int64, zbuf, bary (N,H,W,K,3), dists (N,H,W,K), padding -1."""
    fv = face_verts
    N = len(face_start) - 1
    pxy = pixel_centers(H, W, fv.dtype).reshape(-1, 1, 2)  # (HW,1,2)
    out = []
    for n in range(N):
        f0, f1 = int(face_start[n]), int(face_start[n + 1])
        v = fv[f0:f1]  # (Fn,3,3)
        if v.shape[0] == 0:
            out.append((torch.full((H, W, K), -1, dtype=torch.int64), torch.full((H, W, K), -1.0, dtype=fv.dtype),
                        torch.full((H, W, K, 3), -1.0, dtype=fv.dtype), torch.full((H, W, K), -1.0, dtype=fv.dtype)))
            continue
        step = max(1, chunk_pairs // v.shape[0])
        parts = [_rasterize_pixels(pxy[i:i + step], v, f0, K, blur_radius, cull_backfaces) for i in range(0, H * W, step)]
        p2f, zb, bc, ds = (torch.cat([p[i] for p in parts]) for i in range(4))
        out.append((p2f.reshape(H, W, K), zb.reshape(H, W, K), bc.reshape(H, W, K, 3), ds.reshape(H, W, K)))
    return tuple(torch.stack([o[i] for o in out]) for i in range(4))


def fragments_from_selection(face_verts, pix_to_face, H, W):
    """zbuf, bary, dists of the SELECTED (pixel, face) pairs as differentiable functions of face_verts: the
    quantities whose backward rasterize_meshes' autograd Function implements (RasterizeMeshesBackwardCuda)."""
    N = pix_to_face.shape[0]
    K = pix_to_face.shape[-1]
    mask = pix_to_face >= 0
    v = face_verts[pix_to_face.clamp(min=0)]  # (N,H,W,K,3,3)
    pxy = pixel_centers(H, W, face_verts.dtype).reshape(1, H, W, 1, 2).expand(N, H, W, K, 2)
    v0, v1, v2 = v[..., 0, :2], v[..., 1, :2], v[..., 2, :2]
    bary = barycentric(pxy, v0, v1, v2)
    pz = (bary * v[..., 2]).sum(-1)
    dist = point_triangle_distance(pxy, v0, v1, v2)
    inside = (bary > 0).all(-1)
    sd = torch.where(inside, -dist, dist)
    neg = torch.full_like(pz, -1.0)
    return (torch.where(mask, pz, neg), torch.where(mask[..., None], bary, torch.full_like(bary, -1.0)),
            torch.where(mask, sd, neg))


# ----------------------------------------------------------------------------------------------------------
# cameras (renderer/cameras.py): world -> view -> NDC, as MeshRasterizer.transform feeds rasterize_meshes
# ----------------------------------------------------------------------------------------------------------
def look_at_view_transform(dist, elev_deg, azim_deg):
    """renderer/cameras.py look_at_view_transform (at = origin, up = +Y).  Returns R (3,3), T (3,) in the
    row-vector convention X_view = X_world R + T."""
    e, a = math.radians(elev_deg), math.radians(azim_deg)
    C = torch.tensor([dist * math.cos(e) * math.sin(a), dist * math.sin(e), dist * math.cos(e) * math.cos(a)], dtype=torch.float64)
    z_axis = torch.nn.functional.normalize(-C, dim=0)  # at - camera_position
    up = torch.tensor([0.0, 1.0, 0.0], dtype=torch.float64)
    x_axis = torch.nn.functional.normalize(torch.linalg.cross(up, z_axis), dim=0)
    y_axis = torch.nn.functional.normalize(torch.linalg.cross(z_axis, x_axis), dim=0)
    R = torch.stack((x_axis, y_axis, z_axis), dim=1)  # columns are the camera axes: X_view = X_world R + T
    T = -(C @ R)
    return R.float(), T.float()


def project_to_ndc(verts_world, R, T, fov_deg=60.0):
    """FoVPerspectiveCameras (aspect 1): view = world R + T; x_ndc = x/(z tan(fov/2)), y likewise; MeshRasterizer
    keeps the VIEW depth as z."""
    view = verts_world @ R + T
    s = 1.0 / math.tan(math.radians(fov_deg) / 2.0)
    return torch.stack((s * view[..., 0] / view[..., 2], s * view[..., 1] / view[..., 2], view[..., 2]), dim=-1)
