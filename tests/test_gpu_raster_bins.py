"""The bounded coarse bins (pert_rasterize_bin_bounded + PERT_RAST_BIN_WIDE): fragments bit-identical to the unbinned walk
and to pert_rasterize_bin's bins on every key-kernel case of the path tests, at the benchmark's headline shape, with faces
at +-1e9, +-inf and NaN, and in scenes where every face or no face is wide; the invariants of the lists read back from
the buffers; a large-mesh forward that never synchronises with the host; and a large-mesh render captured in a CUDA
graph, forward and backward, equal to the eager run."""

import math

import pytest
import torch

import test_gpu_raster_paths as P
from conftest import rel_err
from oracle import raster_oracle as RO

pytestmark = pytest.mark.gpu

DEV = "cuda"
EVAL_BLUR = P.EVAL_BLUR


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _bounded(rs, N):
    """pert_rasterize_bin_bounded's two passes around the prefix sum, with nothing read back in between: (count, offset,
    lists), lists sized by pert_rasterize_bin_capacity and prefilled with -1."""
    from pertrenderer_b200 import _cabi
    lib = _cabi.load()
    fill, capacity = _cabi.raster_bin_fns()
    nb = int(lib.pert_rasterize_num_bins(rs)) + N
    count = torch.zeros((nb,), dtype=torch.int32, device=DEV)
    _cabi.check(fill(rs, _cabi.ptr(count), None, None, None, _cabi.stream_ptr(DEV)), "pert_rasterize_bin_bounded")
    offset = (torch.cumsum(count, 0, dtype=torch.int64) - count).contiguous()
    lists = torch.full((max(int(capacity(rs)), 1),), -1, dtype=torch.int64, device=DEV)
    cursor = torch.zeros((nb,), dtype=torch.int32, device=DEV)
    _cabi.check(fill(rs, _cabi.ptr(count), _cabi.ptr(offset), _cabi.ptr(cursor), _cabi.ptr(lists), _cabi.stream_ptr(DEV)),
                "pert_rasterize_bin_bounded")
    torch.cuda.synchronize()
    assert torch.equal(cursor, count)
    return count, offset, lists


def _fwd_bounded(fv, start, H, W, K, blur=0.0, cull=False):
    """pert_rasterize_fwd on the bounded bins; outputs start as garbage (-7 / NaN) as in the path tests."""
    from pertrenderer_b200 import _cabi
    lib = _cabi.load()
    fvd, fs = fv.to(DEV).contiguous(), torch.tensor(start, dtype=torch.int64, device=DEV)
    N = len(start) - 1
    p2f = torch.full((N, H, W, K), -7, dtype=torch.int64, device=DEV)
    zbuf, dists = (torch.full((N, H, W, K), float("nan"), device=DEV) for _ in range(2))
    bary = torch.full((N, H, W, K, 3), float("nan"), device=DEV)
    rs = P._struct(fvd, fs, H, W, K, blur, cull)
    lists = _bounded(rs, N)
    rs.bin_count, rs.bin_offset, rs.bin_faces = (t.data_ptr() for t in lists)
    rs.flags |= _cabi.RAST_BIN_WIDE
    _cabi.check(lib.pert_rasterize_fwd(rs, _cabi.ptr(p2f), _cabi.ptr(zbuf), _cabi.ptr(bary), _cabi.ptr(dists),
                                       _cabi.stream_ptr(DEV)), "pert_rasterize_fwd")
    torch.cuda.synchronize()
    return (p2f, zbuf, bary, dists), lists


def _bin_cap():
    from pertrenderer_b200 import _cabi
    rs = _cabi.PertRaster()
    rs.num_faces = 1
    return int(_cabi.raster_bin_fns()[1](rs))


def _open_box(v, r):
    """The forward's grown box along one axis of corners v (F,3): fminf / fmaxf ignore a NaN corner, and an axis whose
    three corners are NaN is open on both sides (the tile test never culls on a NaN)."""
    nan = v.isnan()
    lo = torch.where(nan, torch.full_like(v, float("inf")), v).amin(1) - r
    hi = torch.where(nan, torch.full_like(v, float("-inf")), v).amax(1) + r
    every = nan.all(1)
    return torch.where(every, torch.full_like(lo, float("-inf")), lo), torch.where(every, torch.full_like(hi, float("inf")), hi)


def _check_lists(lists, fv, start, H, W, blur, cull):
    """The invariants of the bounded layout, read from the buffers; returns the number of wide faces.
      - every slot up to the total was written, the total is at most the capacity, every entry belongs to its image;
      - no tile meets a face twice (own list and wide list together);
      - a wide face has no tile entry, any other face at most C;
      - every tile with a pixel centre inside the grown bounding box of a face that is not culled lists the face in its
        own list or in its image's wide list, and a face with more than C such tiles is wide.  Faces within rounding of
        a culling threshold (area at +-1e-8 or 0) are not required."""
    count, offset, faces = lists
    N = len(start) - 1
    tx, ty = (W + 31) // 32, (H + 3) // 4
    T = tx * ty
    nb = N * T
    C = _bin_cap()
    F = fv.shape[0]
    total = int(count.long().sum())
    assert total <= C * F and faces.numel() == max(C * F, 1)
    faces = faces[:total]
    assert (faces >= 0).all(), "a slot of the lists was never written"
    bin_of = torch.repeat_interleave(torch.arange(count.numel(), device=DEV), count.long(), output_size=total)
    wide = bin_of >= nb
    img = torch.where(wide, bin_of - nb, bin_of // T)
    fs = torch.tensor(start, device=DEV)
    assert ((faces >= fs[img]) & (faces < fs[img + 1])).all()
    tile_entries = torch.bincount(faces[~wide], minlength=F)
    wide_entries = torch.bincount(faces[wide], minlength=F)
    assert (wide_entries <= 1).all(), "a face is twice in a wide list"
    assert (tile_entries[wide_entries > 0] == 0).all(), "a wide face is also in a tile list"
    assert (tile_entries <= C).all(), "a face has more than C tile entries"
    # every (tile, face) pair the lists give, wide lists expanded to every tile of their image
    own_key = bin_of[~wide] * (F + 1) + faces[~wide]
    wf, wn = faces[wide], img[wide]
    tiles = torch.arange(T, device=DEV)
    key = torch.cat((own_key, ((wn[:, None] * T + tiles[None, :]) * (F + 1) + wf[:, None]).flatten()))
    assert torch.unique(key).numel() == key.numel(), "a tile meets a face twice"
    # the forward's tile test on every (face, tile) of the face's image
    v = fv.to(DEV).float()
    r = float(torch.tensor(blur, dtype=torch.float32).sqrt())
    xmin, xmax = _open_box(v[:, :, 0], r)
    ymin, ymax = _open_box(v[:, :, 1], r)
    area = RO.edge_function(v[:, 0, :2].double(), v[:, 1, :2].double(), v[:, 2, :2].double())  # NaN: never culled
    live = ~(v[:, :, 2].amax(1) < 0) & ~(area.abs() <= 1e-6)
    if cull:
        live &= ~(area <= 1e-6)
    c = RO.pixel_centers(H, W, torch.float64).to(DEV)  # (H, W, 2); x falls with the column, y with the row
    ys, xs = torch.arange(ty, device=DEV) * 4, torch.arange(tx, device=DEV) * 32
    y1, x1 = (ys + 3).clamp(max=H - 1), (xs + 31).clamp(max=W - 1)
    T_xhi, T_xlo = c[0, xs, 0][None, :].expand(ty, tx).flatten(), c[0, x1, 0][None, :].expand(ty, tx).flatten()
    T_yhi, T_ylo = c[ys, 0, 1][:, None].expand(ty, tx).flatten(), c[y1, 0, 1][:, None].expand(ty, tx).flatten()
    hit = ~((T_xlo[None] > xmax[:, None].double()) | (T_xhi[None] < xmin[:, None].double()) |
            (T_ylo[None] > ymax[:, None].double()) | (T_yhi[None] < ymin[:, None].double()))
    hit &= live[:, None]
    face_img = torch.bucketize(torch.arange(F, device=DEV), fs[1:], right=True)
    f_idx, t_idx = hit.nonzero(as_tuple=True)
    need = (face_img[f_idx] * T + t_idx) * (F + 1) + f_idx
    assert torch.isin(need, key).all(), "a tile that can see a face lists it in neither list"
    assert (wide_entries[hit.sum(1) > C] == 1).all(), "a face with more than C tiles is not wide"
    return int((wide_entries > 0).sum())


def _three_ways(fv, start, H, W, K, blur, cull):
    """Unbinned, pert_rasterize_bin's bins and the bounded bins: the same fragments, bit for bit."""
    plain, _ = P._fwd(fv, start, H, W, K, blur, cull)
    binned, _ = P._fwd(fv, start, H, W, K, blur, cull, bins=True)
    bounded, lists = _fwd_bounded(fv, start, H, W, K, blur, cull)
    P._same_bits(bounded, plain)
    P._same_bits(bounded, binned)
    return plain, lists


# ---------------------------------------------------------------------------------------------------------------
# bit-identical fragments
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", P.KEY_CASES, ids=[c[0] for c in P.KEY_CASES])
def test_bounded_bins_match_unbinned_and_tile_bins(case):
    """Partial tiles, unequal and empty images, culling on and off, depth ties, faces at z = 0 and behind the camera."""
    _, scene, H, W, K, blur, cull = case
    fv, start = P._scene(scene)
    _, lists = _three_ways(fv, start, H, W, K, blur, cull)
    _check_lists(lists, fv, start, H, W, blur, cull)


def test_bounded_bins_at_the_benchmark_headline_shape(monkeypatch):
    """8 views of the 1280-face icosphere, 256x256, K = 50, eval.py's blur: through the C ABI, and through
    rasterize_meshes with the bins forced on."""
    import pertrenderer_b200 as pb
    from pertrenderer_b200 import rasterizer
    verts, faces = pb.synthetic_mesh(1280, device="cpu")
    R, T = pb.look_at_view_transform(dist=2.7, elev=30.0, azim=torch.linspace(0, 315, 8))
    ndc = pb.FoVPerspectiveCameras(R=R, T=T).transform_points_ndc(verts)
    fv = ndc[:, faces].reshape(-1, 3, 3).contiguous()
    start = [i * faces.shape[0] for i in range(9)]
    plain, lists = _three_ways(fv, start, 256, 256, 50, EVAL_BLUR, False)
    _check_lists(lists, fv, start, 256, 256, EVAL_BLUR, False)
    fs = torch.tensor(start, device=DEV)
    monkeypatch.setattr(rasterizer, "BIN_MIN_FACES", 1)
    forced = pb.rasterize_meshes(fv.to(DEV), fs, 256, EVAL_BLUR, 50)
    P._same_bits(forced, plain)


@pytest.mark.parametrize("big", [1e9, float("inf")], ids=["1e9", "inf"])
def test_bounded_bins_with_vertices_at_huge_and_infinite_ndc(big):
    """Wedges from the image centre to +-big: listed in every tile they can reach, in the wide list where that is more
    than C tiles (the infinite ones: half an axis of a 70-pixel-wide or 36-pixel-high image)."""
    ext = P._extreme_faces(big)
    fv = torch.cat((P._soup(200, 8), ext, P._soup(150, 9), ext.flip(0))).contiguous()
    start = [0, 204, fv.shape[0]]
    for H, W, K in ((36, 70, 8), (29, 29, 50), (80, 160, 16)):
        for cull in (False, True):
            _, lists = _three_ways(fv, start, H, W, K, EVAL_BLUR, cull)
            n_wide = _check_lists(lists, fv, start, H, W, EVAL_BLUR, cull)
            if H == 80:  # a wedge reaches half an axis: 40 pixel rows or 80 columns
                assert n_wide >= 1


def test_bounded_bins_with_nan_coordinates():
    """Faces whose three x (or three y) coordinates are NaN cover the whole NaN axis: listed in every tile along it,
    in the wide list where that is more than C tiles."""
    nan = float("nan")
    odd = torch.tensor([[[nan, -0.3, 1.0], [nan, 0.2, 1.0], [nan, 0.1, 1.5]],
                        [[-0.4, nan, 1.0], [0.3, nan, 1.2], [0.0, nan, 1.0]],
                        [[nan, 0.4, 2.0], [0.2, -0.1, 2.0], [-0.3, 0.0, 2.0]]])
    fv = torch.cat((P._soup(100, 10), odd, P._soup(80, 11))).contiguous()
    start = [0, 103, fv.shape[0]]
    for H, W, K in ((36, 70, 8), (17, 40, 64), (96, 64, 8)):
        for cull in (False, True):
            _, lists = _three_ways(fv, start, H, W, K, EVAL_BLUR, cull)
            n_wide = _check_lists(lists, fv, start, H, W, EVAL_BLUR, cull)
            if H == 96:  # 24 tile rows along the NaN y axis
                assert n_wide >= 1


def _big_triangles(F, seed):
    """Triangles of circumradius 2.5 around points near the centre: each contains a disc of radius 1.25 around its
    centre, so it covers far more than C tiles of a 64x128 image."""
    g = torch.Generator().manual_seed(seed)
    c = torch.rand(F, 1, 2, generator=g) * 0.6 - 0.3
    th = torch.rand(F, 1, generator=g) * 2 * math.pi + torch.tensor([0.0, 2 * math.pi / 3, 4 * math.pi / 3])
    xy = c + 2.5 * torch.stack((th.cos(), th.sin()), -1)
    z = 0.5 + 2.5 * torch.rand(F, 3, 1, generator=g)
    return torch.cat((xy, z), -1)


def test_every_face_wide():
    fv = torch.cat((_big_triangles(120, 1), _big_triangles(90, 2)))
    fv[::2] = fv[::2].flip(1)  # both windings: culling keeps half
    fv = fv.contiguous()
    start = [0, 120, 210]
    for cull in (False, True):
        plain, lists = _three_ways(fv, start, 64, 128, 50, EVAL_BLUR, cull)
        n_wide = _check_lists(lists, fv, start, 64, 128, EVAL_BLUR, cull)
        count = lists[0]
        assert int(count[:-2].sum()) == 0 and n_wide == int(count[-2:].sum()) > 0
        assert n_wide == (210 if not cull else int((RO.edge_function(fv[:, 0, :2], fv[:, 1, :2], fv[:, 2, :2]) > 0).sum()))
        assert (plain[0] >= 0).any(-1).float().mean() > 0.5


def test_no_face_wide():
    """Faces of about a pixel: none spans more than four tiles."""
    fv = torch.cat((P._soup(3000, 12, spread=0.01), P._soup(2000, 13, spread=0.01))).contiguous()
    start = [0, 3000, 5000]
    for cull in (False, True):
        plain, lists = _three_ways(fv, start, 64, 64, 8, 0.0, cull)
        assert _check_lists(lists, fv, start, 64, 64, 0.0, cull) == 0
        count = lists[0]
        assert int(count[-2:].sum()) == 0 and int(count.sum()) > 0
        assert (plain[0] >= 0).any()


# ---------------------------------------------------------------------------------------------------------------
# no host synchronisation, graph capture
# ---------------------------------------------------------------------------------------------------------------
def _big_scene(imsize=128, K=50, n_faces=20480):
    import pertrenderer_b200 as pb
    verts, faces = pb.synthetic_mesh(n_faces, device=DEV)
    R, T = pb.look_at_view_transform(dist=2.7, elev=30.0, azim=40.0, device=DEV)
    cameras = pb.FoVPerspectiveCameras(R=R, T=T, device=DEV)
    settings = pb.RasterizationSettings(image_size=imsize, blur_radius=EVAL_BLUR, faces_per_pixel=K)
    return verts, faces, cameras, settings


def test_large_mesh_forward_does_not_synchronise(monkeypatch):
    """An eager MeshRasterizer forward of a 20480-face mesh (coarse bins) never waits for the device: torch's sync debug
    mode turns any synchronising call into an error.  Its fragments are the unbinned walk's."""
    import pertrenderer_b200 as pb
    from pertrenderer_b200 import rasterizer
    verts, faces, cameras, settings = _big_scene()
    mesh = pb.TriMeshes(verts, faces)
    rast = pb.MeshRasterizer(cameras=cameras, raster_settings=settings)
    assert faces.shape[0] >= rasterizer.BIN_MIN_FACES
    rast(mesh)  # first call: module loading, allocator warm-up
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        fr = rast(mesh)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    monkeypatch.setattr(rasterizer, "BIN_MIN_FACES", 10 ** 9)
    plain = rast(mesh)
    for a, b in zip(P._bits((fr.pix_to_face, fr.zbuf, fr.bary_coords, fr.dists)),
                    P._bits((plain.pix_to_face, plain.zbuf, plain.bary_coords, plain.dists))):
        assert torch.equal(a, b)
    assert (fr.pix_to_face >= 0).any()


def test_large_mesh_render_captured_in_a_cuda_graph():
    """MeshRenderer(MeshRasterizer, RandomPhongShader with the Gaussian pair) on a 20480-face mesh, forward and backward,
    captured in one CUDA graph inside ops.device_seeds: a replay gives the eager run's fragments and image bit for bit
    and its vertex gradient up to the order of the atomic adds (same host seeds, same device seeds)."""
    import pertrenderer_b200 as pb
    from pertrenderer_b200 import ops
    verts, faces, cameras, settings = _big_scene()
    lights = pb.PointLights(location=[[0.0, 2.0, -2.0]], device=DEV)
    sigma, gamma = 1e-3, 1e-2
    settings.blur_radius = math.log(1.0 / 1e-4 - 1.0) * sigma
    renderer = pb.MeshRenderer(
        rasterizer=pb.MeshRasterizer(cameras=cameras, raster_settings=settings),
        shader=pb.RandomPhongShader(device=DEV, cameras=cameras, lights=lights,
                                    blend_params=pb.BlendParams(sigma=sigma, gamma=gamma, background_color=(0.0, 0.0, 0.0)),
                                    smoothrast=pb.GaussianRast(nb_samples=16, sigma=sigma),
                                    smoothagg=pb.GaussianAgg(nb_samples=16, gamma=gamma, alpha=1.0)))
    for t in renderer.shader.get_smoothing():
        t.requires_grad_(False)
    colors = torch.rand((faces.shape[0], 3), device=DEV, generator=torch.Generator(device=DEV).manual_seed(3))
    mesh = pb.TriMeshes(verts, faces, face_colors=colors)
    # the vertex normals are summed by index_add, in no fixed order on CUDA: every run uses the same ones
    normals = mesh.verts_normals_packed().detach()
    stash = []
    renderer.rasterizer.register_forward_hook(lambda mod, inp, out: stash.append(out))
    v = verts.clone().requires_grad_(True)
    G = torch.randn((1, 128, 128, 4), device=DEV, generator=torch.Generator(device=DEV).manual_seed(4))
    seeds = torch.tensor([0x1234567, 0x7654321], dtype=torch.int64, device=DEV)

    def step():
        m = mesh.update_padded(v)
        m.verts_normals_packed = lambda: normals
        stash.clear()
        img = renderer(m)
        fr = stash[0]
        (g,) = torch.autograd.grad(img, v, G)
        return fr.pix_to_face, fr.zbuf, fr.bary_coords, fr.dists, img, g

    with ops.device_seeds(seeds):
        torch.manual_seed(7)
        eager = [t.detach().clone() for t in step()]
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            torch.manual_seed(7)
            step()
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        torch.manual_seed(7)
        with torch.cuda.graph(graph):
            captured = step()
        graph.replay()
    torch.cuda.synchronize()
    assert (eager[0] >= 0).any() and eager[4].abs().sum() > 0
    for a, b in zip(P._bits(captured[:5]), P._bits(eager[:5])):
        assert torch.equal(a, b)
    assert eager[5].abs().sum() > 0 and rel_err(captured[5], eager[5]) <= 1e-5


def test_pose_iteration_on_a_large_mesh_captured_in_one_cuda_graph():
    """examples/pose_optimisation.py --graph (render + loss + backward + Adam as one CUDA graph per iteration) on the
    20480-face mesh with face colours, at eval.py's 128x128: it runs and gives finite poses."""
    import os
    import runpy
    import pertrenderer_b200 as pb
    from conftest import ROOT
    ex = runpy.run_path(os.path.join(ROOT, "examples", "pose_optimisation.py"), run_name="pose_example")
    torch.manual_seed(0)
    verts, faces = pb.synthetic_mesh(20480, device=DEV)
    colors = torch.rand((faces.shape[0], 3), device=DEV, generator=torch.Generator(device=DEV).manual_seed(5))
    mesh = pb.TriMeshes(verts, faces, face_colors=colors)
    R, T = pb.look_at_view_transform(dist=2.7, elev=30.0, azim=120.0, device=DEV)
    cameras = pb.OpenGLPerspectiveCameras(R=R, T=T, fov=60, device=DEV)
    lights = pb.PointLights(location=[[0.0, 2.0, -2.0]], device=DEV)
    hard = ex["make_renderer"]("hard", cameras, lights, 1e-4, 1e-4, 1, 128, DEV)
    w_true = torch.tensor([0.3, -0.5, 0.2], device=DEV)
    R_true = ex["so3_exp"](w_true)
    with torch.no_grad():
        target = hard(mesh.update_padded(verts @ R_true))[..., :3]
    w0 = ex["so3_log"](R_true @ ex["so3_exp"](math.radians(15.0) * torch.tensor([0.6, 0.0, 0.8], device=DEV)))
    renderer = ex["make_renderer"]("gaussian", cameras, lights, 1e-3, 1e-2, 16, 128, DEV)
    w = ex["optimize_pose_graphed"](mesh, verts, renderer, target, w0, 12, 5e-2)
    torch.cuda.synchronize()
    assert torch.isfinite(w).all()
