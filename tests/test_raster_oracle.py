"""CPU checks of the fragment-producer row: closed-form known answers of the oracle (oracle/raster_oracle.py restates
pytorch3d 0.4.0's naive rasteriser; the reference holds no fixture at that boundary), camera shims, and argument
validation of the C ABI without a GPU."""

import ctypes
import math

import pytest
import torch

import pertrenderer_b200 as pb
from oracle import raster_oracle as RO
from pertrenderer_b200 import _cabi


def test_pixel_centres_top_left_is_plus_plus():
    c = RO.pixel_centers(4, 4)
    assert torch.allclose(c[0, 0], torch.tensor([0.75, 0.75]))   # top-left pixel: +X is left, +Y is up
    assert torch.allclose(c[3, 3], torch.tensor([-0.75, -0.75]))
    c2 = RO.pixel_centers(2, 4)  # non-square: the long axis spans [-2, 2]
    assert torch.allclose(c2[0, 0], torch.tensor([1.5, 0.5]))


def _tri(z=(2.0, 2.0, 2.0)):
    # counter-clockwise in NDC as seen with +X left: covers the centre of a 4x4 image
    return torch.tensor([[[-0.6, -0.6, z[0]], [0.6, -0.6, z[1]], [0.0, 0.7, z[2]]]])


def test_single_triangle_known_answers():
    fv = _tri(z=(1.0, 2.0, 3.0))
    H = W = 4
    p2f, zbuf, bary, dists = RO.rasterize(fv, [0, 1], H, W, 2, blur_radius=0.0)
    # pixel (row 2, col 1) has centre (+0.25, -0.25): inside
    assert p2f[0, 2, 1, 0] == 0 and p2f[0, 2, 1, 1] == -1
    b = bary[0, 2, 1, 0]
    assert abs(b.sum().item() - 1.0) < 1e-6 and (b > 0).all()
    # barycentric coordinates reproduce the pixel centre and the depth
    assert torch.allclose((b[:, None] * fv[0, :, :2]).sum(0), torch.tensor([0.25, -0.25]), atol=1e-6)
    assert abs(zbuf[0, 2, 1, 0].item() - (b * fv[0, :, 2]).sum().item()) < 1e-6
    # signed squared distance: negative inside; the closest edge is the right one, (0.6,-0.6)-(0,0.7):
    # |cross(p - a, b - a)|^2 / |b - a|^2 = 0.245^2 / 2.05 (the bottom edge is 0.35 away)
    assert abs(dists[0, 2, 1, 0].item() + 0.245 ** 2 / 2.05) < 1e-6
    # the corner pixel (0,0) at (0.75, 0.75) is outside and, without blur, not a fragment
    assert p2f[0, 0, 0, 0] == -1 and zbuf[0, 0, 0, 0] == -1 and dists[0, 0, 0, 0] == -1 and (bary[0, 0, 0, 0] == -1).all()


def test_blur_band_and_vertex_distance():
    fv = _tri()
    # pixel (3, 0): centre (0.75, -0.75); closest point of the triangle is the vertex (0.6, -0.6): d2 = 2 * 0.15^2
    d2 = 2 * 0.15 ** 2
    out_small = RO.rasterize(fv, [0, 1], 4, 4, 1, blur_radius=d2 * 0.99)
    out_big = RO.rasterize(fv, [0, 1], 4, 4, 1, blur_radius=d2 * 1.01)
    assert out_small[0][0, 3, 0, 0] == -1
    assert out_big[0][0, 3, 0, 0] == 0 and abs(out_big[3][0, 3, 0, 0].item() - d2) < 1e-6  # positive: outside


def test_depth_order_ties_and_k_truncation():
    a, b, c = _tri(z=(3.0, 3.0, 3.0)), _tri(z=(1.0, 1.0, 1.0)), _tri(z=(3.0, 3.0, 3.0))
    fv = torch.cat((a, b, c))
    p2f, zbuf, _, _ = RO.rasterize(fv, [0, 3], 4, 4, 3, 0.0)
    assert p2f[0, 2, 1].tolist() == [1, 0, 2]  # nearest first; equal depths keep face order
    assert torch.allclose(zbuf[0, 2, 1], torch.tensor([1.0, 3.0, 3.0]), atol=1e-6)
    p2f2, _, _, _ = RO.rasterize(fv, [0, 3], 4, 4, 2, 0.0)
    assert p2f2[0, 2, 1].tolist() == [1, 0]  # K nearest
    # behind the camera / zero area: skipped
    behind = _tri(z=(-1.0, -2.0, -3.0))
    flat = torch.tensor([[[0.0, 0.0, 1.0], [0.5, 0.5, 1.0], [1.0, 1.0, 1.0]]])
    p2f3, _, _, _ = RO.rasterize(torch.cat((behind, flat)), [0, 2], 4, 4, 2, 1e-2)
    assert (p2f3 == -1).all()
    # two images with their own face ranges
    p2f4, _, _, _ = RO.rasterize(fv, [0, 1, 3], 4, 4, 2, 0.0)
    assert p2f4[0, 2, 1].tolist() == [0, -1] and p2f4[1, 2, 1].tolist() == [1, 2]


def test_cull_backfaces_drops_negative_winding_only():
    tri = _tri()  # edge(v0, v1, v2) = -1.56: a back face
    assert RO.edge_function(tri[0, 0, :2], tri[0, 1, :2], tri[0, 2, :2]) < 0
    flipped = tri[:, [0, 2, 1]]
    for fv, culled in ((tri, True), (flipped, False)):
        plain = RO.rasterize(fv, [0, 1], 4, 4, 1, 0.0)
        cull = RO.rasterize(fv, [0, 1], 4, 4, 1, 0.0, cull_backfaces=True)
        assert plain[0][0, 2, 1, 0] == 0
        if culled:
            assert (cull[0] == -1).all() and (cull[1] == -1).all() and (cull[2] == -1).all() and (cull[3] == -1).all()
        else:
            for a, b in zip(plain, cull):
                assert torch.equal(a, b)


def test_empty_image_in_a_batch_is_padding():
    fv = torch.cat((_tri(z=(1.0, 1.0, 1.0)), _tri(z=(2.0, 2.0, 2.0))))
    p2f, zbuf, bary, dists = RO.rasterize(fv, [0, 1, 1, 2], 4, 4, 3, 1e-3)
    assert p2f.shape == (3, 4, 4, 3) and bary.shape == (3, 4, 4, 3, 3)
    for t in (p2f, zbuf, bary, dists):
        assert (t[1] == -1).all()
    assert p2f[0, 2, 1].tolist() == [0, -1, -1] and p2f[2, 2, 1].tolist() == [1, -1, -1]
    assert abs(zbuf[2, 2, 1, 0].item() - 2.0) < 1e-6
    empty = RO.rasterize(fv[:0], [0, 0], 4, 4, 2, 0.0)
    assert all((t == -1).all() for t in empty)


def test_pixel_chunks_do_not_change_the_result():
    torch.manual_seed(3)
    c = torch.rand(60, 1, 2) * 1.6 - 0.8
    fv = torch.cat((c + 0.3 * torch.rand(60, 3, 2) - 0.15, 1.0 + torch.rand(60, 3, 1)), dim=-1).double()
    full = RO.rasterize(fv, [0, 25, 60], 9, 13, 5, 4e-3, chunk_pairs=1 << 30)
    for pairs in (1, 37, 60 * 50):
        part = RO.rasterize(fv, [0, 25, 60], 9, 13, 5, 4e-3, chunk_pairs=pairs)
        for a, b in zip(full, part):
            assert torch.equal(a, b)
    assert (full[0] >= 0).sum() > 50 and full[1].dtype == torch.float64


def test_selected_fragment_gradients_match_finite_differences():
    torch.manual_seed(1)
    fv = (_tri(z=(1.0, 2.0, 3.0)) + 0.05 * torch.randn(1, 3, 3)).double()
    p2f, _, _, _ = RO.rasterize(fv.float(), [0, 1], 6, 6, 1, 0.05)
    assert (p2f >= 0).sum() > 6
    f = lambda v: RO.fragments_from_selection(v, p2f, 6, 6)  # noqa: E731
    assert torch.autograd.gradcheck(f, (fv.requires_grad_(),), eps=1e-6, atol=1e-5)


def test_camera_shims_match_the_oracle_restatement():
    R, T = pb.look_at_view_transform(dist=6.7, elev=30.0, azim=120.0)
    R2, T2 = RO.look_at_view_transform(6.7, 30.0, 120.0)
    assert torch.allclose(R[0], R2, atol=1e-6) and torch.allclose(T[0], T2, atol=1e-5)
    assert torch.allclose(R[0] @ R[0].T, torch.eye(3), atol=1e-6)
    cam = pb.OpenGLPerspectiveCameras(R=R, T=T, fov=60)
    assert abs(cam.get_camera_center().norm().item() - 6.7) < 1e-4
    origin = cam.transform_points_ndc(torch.zeros(1, 3))
    assert torch.allclose(origin[0, 0], torch.tensor([0.0, 0.0, 6.7]), atol=1e-4)  # looks at the origin, depth = dist
    v = torch.randn(5, 3)
    assert torch.allclose(cam.transform_points_ndc(v)[0], RO.project_to_ndc(v, R2, T2), atol=1e-5)
    # a point one unit above the origin lands on the +Y side, tan(30 deg) scaling
    up = cam.transform_points_ndc(torch.tensor([[0.0, 1.0, 0.0]]))[0, 0]
    assert up[1] > 0
    m = pb.TriMeshes(torch.randn(7, 3), torch.tensor([[0, 1, 2], [3, 4, 5]])).extend(3)
    assert m.verts_packed().shape == (21, 3) and m.faces_packed()[2].tolist() == [7, 8, 9] and len(m) == 3


def test_raster_struct_layout_and_validation_without_gpu():
    assert ctypes.sizeof(_cabi.PertRaster) == 88
    assert _cabi.PertRaster.face_verts.offset == 40
    lib = _cabi.load()
    rs = _cabi.PertRaster()
    assert lib.pert_rasterize_fwd(None, None, None, None, None, None) == -1
    rs.N, rs.H, rs.W, rs.K, rs.num_faces = 1, 8, 8, 0, 4
    assert lib.pert_rasterize_fwd(rs, None, None, None, None, None) == -2
    rs.K = 2000
    assert lib.pert_rasterize_fwd(rs, None, None, None, None, None) == -3
    rs.K = 4
    rs.blur_radius = -1.0
    assert lib.pert_rasterize_fwd(rs, None, None, None, None, None) == -7
    rs.blur_radius = 0.0
    assert lib.pert_rasterize_fwd(rs, None, None, None, None, None) == -1
    assert lib.pert_rasterize_bwd(rs, None, None, None, None, None, None) == -1
    with pytest.raises(RuntimeError, match="CUDA"):
        pb.rasterize_meshes(torch.rand(4, 3, 3), torch.tensor([0, 4]), 8)
    with pytest.raises(ValueError, match="perspective_correct"):
        pb.MeshRasterizer(pb.FoVPerspectiveCameras(), pb.RasterizationSettings(perspective_correct=True))(
            pb.TriMeshes(torch.rand(3, 3), torch.tensor([[0, 1, 2]])))
