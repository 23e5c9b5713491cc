"""Every code path of the fragment producer (csrc/raster.cu) against the float64 oracle (oracle/raster_oracle.py):
the shared-key forward (K <= 64) and the rows forward (K > 64) at partial tiles, batches with unequal and empty face
ranges, depth ties, faces at z = 0, faces behind and across the camera plane, back-face culling; the traversal order
(face_order) and the coarse bins (pert_rasterize_bin), including faces reaching +-1e9 and +-inf; and the backward's
shared-table and global-atomics kernels, with each gradient input alone and the others NULL."""

import math

import pytest
import torch

from conftest import rel_err
from oracle import raster_oracle as RO
from raster_util import TAU, abs_edge_terms, check_fragments, pair_stats

pytestmark = pytest.mark.gpu

DEV = "cuda"
EVAL_BLUR = math.log(1.0 / 1e-4 - 1.0) * 1e-3  # eval.py:137 at sigma = 1e-3


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


# ---------------------------------------------------------------------------------------------------------------
# scenes: a list of per-image (F_n,3,3) float32 face tensors in NDC x, y and view depth, on the CPU
# ---------------------------------------------------------------------------------------------------------------
def _sphere(n_faces, azims, dist=2.7, elev=20.0):
    import pertrenderer_b200 as pb
    verts, faces = pb.synthetic_mesh(n_faces, device="cpu")
    R, T = pb.look_at_view_transform(dist=dist, elev=elev, azim=torch.tensor(azims, dtype=torch.float32))
    ndc = pb.FoVPerspectiveCameras(R=R, T=T).transform_points_ndc(verts)
    return [ndc[i][faces].contiguous() for i in range(len(azims))]


def _soup(F, seed, spread=0.9):
    """F random triangles of either winding around the image centre, corners up to ``spread`` from their centre (1.8:
    most faces cover a large part of the image, so the K-lists are deep)."""
    g = torch.Generator().manual_seed(seed)
    c = torch.rand(F, 1, 2, generator=g) * 1.2 - 0.6
    xy = c + (torch.rand(F, 3, 2, generator=g) * 2.0 - 1.0) * spread
    z = 0.5 + 2.5 * torch.rand(F, 3, 1, generator=g)
    return torch.cat((xy, z), -1)


def _ties():
    """Every face three times in a row: exact depth ties, truncated at K inside a run of equal keys."""
    return [_soup(60, 5, 1.8).repeat_interleave(3, 0)]


def _z0():
    """Faces with all corners at z = 0, and faces whose depth crosses 0 inside them (one corner at 0, one behind)."""
    fv = _soup(120, 6)
    fv[:20, :, 2] = 0.0
    fv[20:40, 0, 2] = 0.0
    fv[20:40, 1, 2] = -1.0
    return [fv]


def _inside():
    """The camera inside the sphere: faces behind it, and faces straddling its plane (huge or flipped NDC)."""
    return _sphere(1280, [0.0, 120.0], dist=0.5, elev=10.0)


SCENES = {
    "soup": lambda: [_soup(300, 0)],
    "soup3": lambda: [_soup(300, 1), _soup(0, 0), _soup(120, 2)],  # unequal face counts, empty middle image
    "deep": lambda: [_soup(900, 3, 1.8)],
    "deep3": lambda: [_soup(400, 4, 1.8), _soup(0, 0), _soup(250, 7, 1.8)],
    "sphere3": lambda: (lambda v: [v[0], v[1][:0], v[2][:200]])(_sphere(320, [10.0, 70.0, 140.0])),
    "ties": _ties,
    "z0": _z0,
    "inside": _inside,
}

# (id, scene, H, W, K, blur, cull_backfaces): K <= 64 runs the shared-key kernel, K > 64 the rows kernel
CASES = [
    ("k1-wide", "soup", 21, 45, 1, 0.0, False),
    ("k2-tall-cull", "soup", 45, 37, 2, EVAL_BLUR, True),
    ("k50-batch", "deep3", 36, 36, 50, EVAL_BLUR, False),
    ("k64-cull", "deep", 34, 66, 64, EVAL_BLUR, True),
    ("k64-sphere-cull", "sphere3", 34, 66, 64, EVAL_BLUR, True),
    ("k64-sphere", "sphere3", 34, 66, 64, 0.0, False),
    ("k65-batch", "deep3", 22, 40, 65, 0.0, False),
    ("k100-cull", "deep", 30, 33, 100, EVAL_BLUR, True),
    ("k300", "deep", 13, 35, 300, EVAL_BLUR, False),
    ("ties-k2", "ties", 20, 36, 2, 0.0, False),
    ("ties-k65", "ties", 20, 36, 65, EVAL_BLUR, False),
    ("z0-k8", "z0", 24, 40, 8, EVAL_BLUR, False),
    ("z0-k80", "z0", 24, 40, 80, 0.0, False),
    ("inside-k8", "inside", 32, 48, 8, EVAL_BLUR, False),
    ("inside-k8-cull", "inside", 32, 48, 8, EVAL_BLUR, True),
    ("inside-k70", "inside", 24, 24, 70, EVAL_BLUR, False),
    ("1x1-k2", "soup", 1, 1, 2, EVAL_BLUR, False),
    ("1x1-k65", "deep3", 1, 1, 65, 0.0, True),
]
KEY_CASES = [c for c in CASES if c[4] <= 64]
TRUNCATING = {"k1-wide", "k2-tall-cull", "k50-batch", "k64-cull", "k100-cull", "ties-k2", "z0-k8", "inside-k8", "inside-k8-cull"}


def _scene(name):
    meshes = SCENES[name]()
    start = [0]
    for m in meshes:
        start.append(start[-1] + m.shape[0])
    return torch.cat(meshes).contiguous(), start


# ---------------------------------------------------------------------------------------------------------------
# the C ABI, called directly
# ---------------------------------------------------------------------------------------------------------------
def _struct(fv, fs, H, W, K, blur, cull, face_order=None):
    from pertrenderer_b200.rasterizer import _raster_struct
    return _raster_struct(fv, fs, fs.numel() - 1, H, W, K, blur, cull, face_order)


def _bins(rs):
    """pert_rasterize_bin's two passes around the prefix sum: (count, offset, lists)."""
    from pertrenderer_b200 import _cabi
    lib = _cabi.load()
    nb = int(lib.pert_rasterize_num_bins(rs))
    count = torch.zeros((nb,), dtype=torch.int32, device=DEV)
    _cabi.check(lib.pert_rasterize_bin(rs, _cabi.ptr(count), None, None, None, _cabi.stream_ptr(DEV)), "pert_rasterize_bin")
    ends = torch.cumsum(count, 0, dtype=torch.int64)
    offset = (ends - count).contiguous()
    lists = torch.full((max(int(ends[-1].item()), 1),), -1, dtype=torch.int64, device=DEV)
    cursor = torch.zeros((nb,), dtype=torch.int32, device=DEV)
    _cabi.check(lib.pert_rasterize_bin(rs, _cabi.ptr(count), _cabi.ptr(offset), _cabi.ptr(cursor), _cabi.ptr(lists),
                                       _cabi.stream_ptr(DEV)), "pert_rasterize_bin")
    torch.cuda.synchronize()
    assert torch.equal(cursor, count)
    return count, offset, lists


def _fwd(fv, start, H, W, K, blur=0.0, cull=False, face_order=None, bins=False):
    """pert_rasterize_fwd; the outputs start as garbage (-7 / NaN) so that an entry the kernel skips shows."""
    from pertrenderer_b200 import _cabi
    lib = _cabi.load()
    fvd, fs = fv.to(DEV).contiguous(), torch.tensor(start, dtype=torch.int64, device=DEV)
    N = len(start) - 1
    p2f = torch.full((N, H, W, K), -7, dtype=torch.int64, device=DEV)
    zbuf, dists = (torch.full((N, H, W, K), float("nan"), device=DEV) for _ in range(2))
    bary = torch.full((N, H, W, K, 3), float("nan"), device=DEV)
    rs = _struct(fvd, fs, H, W, K, blur, cull, face_order)
    lists = _bins(rs) if bins else None
    if bins:
        rs.bin_count, rs.bin_offset, rs.bin_faces = (t.data_ptr() for t in lists)
    _cabi.check(lib.pert_rasterize_fwd(rs, _cabi.ptr(p2f), _cabi.ptr(zbuf), _cabi.ptr(bary), _cabi.ptr(dists),
                                       _cabi.stream_ptr(DEV)), "pert_rasterize_fwd")
    torch.cuda.synchronize()
    return (p2f, zbuf, bary, dists), lists


def _bits(out):
    return [t.view(torch.int32) if t.dtype == torch.float32 else t for t in out]


def _same_bits(a, b):
    for x, y in zip(_bits(a), _bits(b)):
        assert torch.equal(x, y)


# ---------------------------------------------------------------------------------------------------------------
# forward
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_forward_matches_float64_oracle(case):
    cid, scene, H, W, K, blur, cull = case
    fv, start = _scene(scene)
    got, _ = _fwd(fv, start, H, W, K, blur, cull)
    ref = check_fragments(got, fv, start, H, W, K, blur, cull)
    assert (ref[0] >= 0).any(-1).float().mean() > 0.1  # the case rasterises something
    if cid in TRUNCATING:
        assert (ref[0] >= 0).all(-1).float().mean() > 0.3  # ... and more than K faces qualify on many pixels
    if len(start) == 4:
        assert (got[0][1] == -1).all()  # the empty middle image


def test_forward_cull_changes_the_selection():
    """The culling cases above do drop faces: back faces are half of the soup."""
    fv, start = _scene("soup")
    plain, _ = _fwd(fv, start, 30, 33, 100, EVAL_BLUR, False)
    cull, _ = _fwd(fv, start, 30, 33, 100, EVAL_BLUR, True)
    area = RO.edge_function(fv[:, 0, :2], fv[:, 1, :2], fv[:, 2, :2])
    back = torch.nonzero(area < 0).flatten().to(DEV)
    assert torch.isin(plain[0], back).any() and not torch.isin(cull[0], back).any()


@pytest.mark.parametrize("case", KEY_CASES, ids=[c[0] for c in KEY_CASES])
def test_face_order_permutation_is_bit_identical(case):
    _, scene, H, W, K, blur, cull = case
    fv, start = _scene(scene)
    base, _ = _fwd(fv, start, H, W, K, blur, cull)
    g = torch.Generator().manual_seed(11)
    perm = torch.cat([s + torch.randperm(e - s, generator=g) for s, e in zip(start[:-1], start[1:])]).to(DEV)
    got, _ = _fwd(fv, start, H, W, K, blur, cull, face_order=perm)
    _same_bits(got, base)


# ---------------------------------------------------------------------------------------------------------------
# coarse bins
# ---------------------------------------------------------------------------------------------------------------
def _check_bin_lists(lists, p2f, start, H, W):
    """Every face of a fragment at (n, y, x) is in the list of tile (n, y/4, x/32); no list repeats a face; the fill
    pass wrote every slot of the lists (they start at -1, and its cursors end at the counts); every listed face belongs
    to the tile's image."""
    count, offset, faces = lists
    tx, ty = (W + 31) // 32, (H + 3) // 4
    total = int(count.long().sum())
    assert total == faces.numel() or (total == 0 and faces.numel() == 1)
    faces = faces[:total]
    assert (faces >= 0).all(), "a slot of the lists was never written"
    bin_of_entry = torch.repeat_interleave(torch.arange(count.numel(), device=DEV), count.long(), output_size=total)
    img = bin_of_entry // (tx * ty)
    fs = torch.tensor(start, device=DEV)
    assert ((faces >= fs[img]) & (faces < fs[img + 1])).all()
    key = bin_of_entry * (int(fs[-1]) + 1) + faces
    assert torch.unique(key).numel() == total, "a tile lists a face twice"
    n, y, x, _ = torch.meshgrid(*(torch.arange(s, device=DEV) for s in p2f.shape), indexing="ij")
    v = p2f >= 0
    need = ((n * ty + y // 4) * tx + x // 32)[v] * (int(fs[-1]) + 1) + p2f[v]
    assert torch.isin(need, key).all(), "a fragment's face is missing from its tile's list"


@pytest.mark.parametrize("case", KEY_CASES, ids=[c[0] for c in KEY_CASES])
def test_bins_match_unbinned_bit_for_bit(case):
    _, scene, H, W, K, blur, cull = case
    fv, start = _scene(scene)
    plain, _ = _fwd(fv, start, H, W, K, blur, cull)
    binned, lists = _fwd(fv, start, H, W, K, blur, cull, bins=True)
    _same_bits(binned, plain)
    _check_bin_lists(lists, plain[0], start, H, W)


def test_bins_at_the_benchmark_headline_shapes():
    """bench.py's rasterised fragment set (8 views of the 1280-face icosphere, 256x256, K = 50, eval.py's blur) comes
    out the same, bit for bit, through the bins."""
    import pertrenderer_b200 as pb
    verts, faces = pb.synthetic_mesh(1280, device="cpu")
    R, T = pb.look_at_view_transform(dist=2.7, elev=30.0, azim=torch.linspace(0, 315, 8))
    ndc = pb.FoVPerspectiveCameras(R=R, T=T).transform_points_ndc(verts)
    fv = ndc[:, faces].reshape(-1, 3, 3).contiguous()
    start = [i * faces.shape[0] for i in range(9)]
    plain, _ = _fwd(fv, start, 256, 256, 50, EVAL_BLUR)
    binned, lists = _fwd(fv, start, 256, 256, 50, EVAL_BLUR, bins=True)
    _same_bits(binned, plain)
    _check_bin_lists(lists, plain[0], start, 256, 256)


def _extreme_faces(big):
    """Thin wedges from the image centre to a corner at +-big on each axis, in front of the rest (z = 0.2)."""
    out = []
    for axis in (0, 1):
        for s in (1.0, -1.0):
            tip = [0.0, 0.0]
            tip[axis] = s * big
            base0, base1 = [0.1, 0.1], [0.1, 0.1]
            base0[1 - axis], base1[1 - axis] = -0.25, 0.25
            base0[axis] = base1[axis] = -s * 0.1
            out.append(torch.tensor([[tip[0], tip[1], 0.2], [base0[0], base0[1], 0.2], [base1[0], base1[1], 0.2]]))
    return torch.stack(out)


def _check_face_in_tiles(lists, fv, f, n, start, H, W):
    """Face f of image n is listed in every tile that has a pixel centre inside its bounding box.  A NaN bound leaves
    its side of the box open: the unbinned tile test never culls on a NaN."""
    count, offset, faces = lists
    tx, ty = (W + 31) // 32, (H + 3) // 4
    v = fv[f].double()
    c = RO.pixel_centers(H, W, torch.float64)
    inside = torch.ones(H, W, dtype=torch.bool)
    for axis in (0, 1):
        lo, hi = v[:, axis].min(), v[:, axis].max()  # NaN if any corner is NaN: then the coordinate decides nothing
        vals = v[:, axis][~v[:, axis].isnan()]
        if vals.numel() == 3:
            inside &= (c[..., axis] >= lo) & (c[..., axis] <= hi)
        elif vals.numel() > 0:  # the kernels' fminf / fmaxf ignore a NaN corner
            inside &= (c[..., axis] >= vals.min()) & (c[..., axis] <= vals.max())
    y, x = inside.nonzero(as_tuple=True)
    assert y.numel() > 0
    bins = torch.unique((n * ty + y // 4) * tx + x // 32).to(DEV)
    for b in bins.tolist():
        lst = faces[int(offset[b]):int(offset[b]) + int(count[b])]
        assert bool((lst == f).any()), f"face {f} is missing from the list of tile {b}"


def _front_facing(fv, f):
    return not bool(RO.edge_function(fv[f, 0, :2], fv[f, 1, :2], fv[f, 2, :2]) < 0)


@pytest.mark.parametrize("big", [1e9, float("inf")], ids=["1e9", "inf"])
def test_bins_with_vertices_at_huge_and_infinite_ndc(big):
    """A face's box reaching |x| or |y| ~ 1e9 or inf (a vertex at view depth ~ 0) is binned into the tiles it covers,
    like every other face: the binned fragments are the unbinned ones, bit for bit."""
    ext = _extreme_faces(big)
    fv = torch.cat((_soup(200, 8), ext, _soup(150, 9), ext.flip(0))).contiguous()
    start = [0, 204, fv.shape[0]]
    ids = [200, 201, 202, 203, 357, 356, 355, 354]  # the wedges of image 0, then of image 1
    for H, W, K in ((36, 70, 8), (29, 29, 50)):
        for cull in (False, True):
            plain, _ = _fwd(fv, start, H, W, K, EVAL_BLUR, cull)
            binned, lists = _fwd(fv, start, H, W, K, EVAL_BLUR, cull, bins=True)
            _same_bits(binned, plain)
            _check_bin_lists(lists, plain[0], start, H, W)
            for i, f in enumerate(ids):
                if cull and not _front_facing(fv, f):
                    continue
                _check_face_in_tiles(lists, fv, f, i // 4, start, H, W)
                if big < float("inf"):
                    # the wedges are the nearest faces: they own the first slot along their axes, up to the border
                    hit = plain[0][i // 4, ..., 0] == f
                    assert hit.any() and (hit[:, 0].any() or hit[:, -1].any() or hit[0].any() or hit[-1].any())


def test_bins_with_nan_coordinates_match_unbinned():
    """Faces whose three x (or three y) coordinates are NaN: binned and unbinned give the same fragments, bit for bit,
    and such a face is listed along the whole NaN axis."""
    nan = float("nan")
    odd = torch.tensor([[[nan, -0.3, 1.0], [nan, 0.2, 1.0], [nan, 0.1, 1.5]],
                        [[-0.4, nan, 1.0], [0.3, nan, 1.2], [0.0, nan, 1.0]],
                        [[nan, 0.4, 2.0], [0.2, -0.1, 2.0], [-0.3, 0.0, 2.0]]])
    fv = torch.cat((_soup(100, 10), odd, _soup(80, 11))).contiguous()
    start = [0, 103, fv.shape[0]]
    for H, W, K in ((36, 70, 8), (17, 40, 64)):
        for cull in (False, True):
            plain, _ = _fwd(fv, start, H, W, K, EVAL_BLUR, cull)
            binned, lists = _fwd(fv, start, H, W, K, EVAL_BLUR, cull, bins=True)
            _same_bits(binned, plain)
            _check_bin_lists(lists, plain[0], start, H, W)
            for f in (100, 101, 102):
                _check_face_in_tiles(lists, fv, f, 0, start, H, W)


# ---------------------------------------------------------------------------------------------------------------
# backward
# ---------------------------------------------------------------------------------------------------------------
def _bwd(fv, start, p2f, grads, H, W, K):
    """pert_rasterize_bwd with (grad_zbuf, grad_bary, grad_dists), any of them None (NULL)."""
    from pertrenderer_b200 import _cabi
    lib = _cabi.load()
    fvd, fs = fv.to(DEV).contiguous(), torch.tensor(start, dtype=torch.int64, device=DEV)
    g_fv = torch.zeros_like(fvd)
    rs = _struct(fvd, fs, H, W, K, 0.0, False)
    gz, gb, gd = (None if g is None else g.to(DEV).contiguous() for g in grads)
    _cabi.check(lib.pert_rasterize_bwd(rs, _cabi.ptr(p2f), _cabi.ptr(gz), _cabi.ptr(gb), _cabi.ptr(gd), _cabi.ptr(g_fv),
                                       _cabi.stream_ptr(DEV)), "pert_rasterize_bwd")
    torch.cuda.synchronize()
    return g_fv.cpu()


def _bwd_oracle(fv, p2f, grads, H, W):
    """float64 autograd over fragments_from_selection of the kernel's selection: the gradient (F,3,3), and per face a
    bound on the float32 error of the kernel's sum (F,1,1)."""
    p2f = p2f.cpu()
    mask = p2f >= 0
    E = p2f.numel()
    face = p2f.clamp(min=0).flatten()
    fv_e = fv.double()[face].requires_grad_(True)  # one copy of its face per entry: per-entry contributions
    outs = RO.fragments_from_selection(fv_e, torch.where(mask, torch.arange(E).reshape(p2f.shape), -1), H, W)
    loss = 0.0
    for o, g in zip(outs, grads):
        if g is not None:
            m = mask if o.dim() == mask.dim() else mask[..., None].expand_as(o)
            loss = loss + (o * g.double())[m].sum()
    loss.backward()
    F = fv.shape[0]
    ref = torch.zeros(fv.shape, dtype=torch.float64).index_add(0, face, fv_e.grad)
    # float32 error of one entry's nine terms: each is a sum of products of the upstream gradients with
    # gw_i / A (p - v), g_area (v - v) and gd (p - proj), g_area = -sum gw_i w_i / A, gw_i = gb_i + gz z_i.  Every
    # product errs by TAU relative, and 1/A by TAU S_A / |A| (the area's conditioning), so an entry errs by at most
    # TAU (1 + S_A/|A|) times the sum of the magnitudes of its products, mag below.
    z, w = fv_e.detach()[:, :, 2], outs[1].detach().reshape(E, 3)
    gz, gb, gd = (torch.zeros(E, *s, dtype=torch.float64) if g is None else g.double().reshape(E, *s)
                  for g, s in zip(grads, ((), (3,), ())))
    v = fv_e.detach()[:, :, :2]
    pxy = RO.pixel_centers(H, W, torch.float64)[None, :, :, None].expand(*p2f.shape, 2).reshape(E, 1, 2)
    A = RO.edge_function(v[:, 2], v[:, 0], v[:, 1]).abs()
    gw = (gb + gz[:, None] * z).abs()
    d_pv = (pxy - v).abs().amax((-1, -2))
    d_vv = (v[:, :, None] - v[:, None, :]).abs().amax((-1, -2, -3))
    dist = outs[2].detach().abs().reshape(E)
    mag = (gw.sum(-1) * d_pv + (gw * w.abs()).sum(-1) * d_vv) / A + gz.abs() * w.abs().sum(-1) + 4.0 * gd.abs() * (dist.sqrt() + d_pv)
    cond = 1.0 + abs_edge_terms(v[:, 2], v[:, 0], v[:, 1]) / A
    valid = mask.flatten()
    per_entry = torch.where(valid, 4.0 * TAU * cond * mag, torch.zeros_like(mag))
    n_terms = torch.bincount(face[valid], minlength=F).double()
    abs_sum = torch.zeros(fv.shape, dtype=torch.float64).index_add(0, face, fv_e.grad.abs())
    # plus the float32 sum of the entries (atomics, and the table's flush): (m + 1) 2^-24 sum |terms|
    bound = torch.zeros(F, dtype=torch.float64).index_add(0, face, per_entry)[:, None, None] + \
        (n_terms + 1.0)[:, None, None] * 2.0 ** -24 * abs_sum
    return ref, bound, n_terms


def _grads(shape, seed):
    gen = torch.Generator().manual_seed(seed)
    gz, gb, gd = torch.randn(shape, generator=gen), torch.randn(shape + (3,), generator=gen), torch.randn(shape, generator=gen)
    gz[torch.rand(shape, generator=gen) < 0.3] = 0.0
    return gz, gb, gd


def _check_grad(got, oracle, fv, what):
    ref, bound, n_terms = oracle
    assert rel_err(got, ref) <= 2e-4, what  # fp32 atomic sums of terms with 1/area^2 factors
    # entry by entry, within the float32 bound of _bwd_oracle, on well-conditioned faces (projected area at least a
    # quarter of the median)
    area = RO.edge_function(fv[:, 0, :2], fv[:, 1, :2], fv[:, 2, :2]).abs()
    touched = n_terms > 0
    wc = touched & (area >= 0.25 * area[touched].median())
    assert wc.sum() > 0.5 * touched.sum(), what
    err = (got.double() - ref).abs()
    bad = wc[:, None, None] & (err > bound)
    assert not bad.any(), (what, int(bad.sum()), (err / bound.clamp_min(1e-300))[wc].max().item())


def _edge_choice_is_a_rounding(fv, p2f, H, W):
    mask = p2f >= 0
    ent = mask.nonzero()
    v = fv.double()[p2f[mask]][:, :, :2]
    p = RO.pixel_centers(H, W, torch.float64)[ent[:, 1], ent[:, 2]]
    st = pair_stats(fv.double(), p2f[mask], p, max(H, W) / min(H, W))
    d, proj = [], []
    for a, b in ((0, 1), (0, 2), (1, 2)):
        ab = v[:, b] - v[:, a]
        t = ((ab * (p - v[:, a])).sum(-1) / (ab * ab).sum(-1)).clamp(0.0, 1.0)
        q = v[:, a] + t[:, None] * ab
        proj.append(q)
        d.append(((p - q) ** 2).sum(-1))
    d, proj = torch.stack(d, -1), torch.stack(proj, 1)
    order = d.argsort(-1)
    i0, i1 = order[:, 0], order[:, 1]
    r = torch.arange(len(d))
    tie = (d[r, i1] - d[r, i0] <= 2.0 * st["dd"]) & ((proj[r, i0] - proj[r, i1]).abs().amax(-1) > 1e-9)
    out = torch.zeros(p2f.shape, dtype=torch.bool)
    out[mask] = tie
    return out


def _run_backward(meshes, H, W, K, blur, seed):
    start = [0]
    for m in meshes:
        start.append(start[-1] + m.shape[0])
    fv = torch.cat(meshes).contiguous()
    (p2f, *_), _ = _fwd(fv, start, H, W, K, blur)
    gz, gb, gd = _grads(tuple(p2f.shape), seed)
    # dists is the distance to the closest edge.  Where two edges are equally close within the float32 error of
    # dists and their closest points differ, the kernel's choice between them is a rounding: the two gradients differ
    # by about sqrt(float32 ulp) relative.  No upstream gradient is put on such entries.
    gd[_edge_choice_is_a_rounding(fv, p2f.cpu(), H, W)] = 0.0
    grads = (gz, gb, gd)
    for which in (None, 0, 1, 2):  # all three, then each alone with the other two NULL
        gsel = grads if which is None else tuple(g if i == which else None for i, g in enumerate(grads))
        got = _bwd(fv, start, p2f, gsel, H, W, K)
        _check_grad(got, _bwd_oracle(fv, p2f, gsel, H, W), fv, which)
    return fv, start, p2f


def test_backward_table_path_with_spill_to_global_atomics():
    """H*W*K > 64512 takes the shared-table kernel; 5120 faces per mesh exceed its 4096-face table, so the faces past
    it take the global atomics in the same launch; image 1's table is flushed at its own face offset."""
    H = W = 64
    K = 16
    assert H * W * K > 64512
    meshes = _sphere(5120, [0.0, 180.0])
    fv, start, p2f = _run_backward(meshes, H, W, K, EVAL_BLUR, 0)
    for n in range(2):  # both sides of the table cap carry gradient in both images
        loc = p2f[n][p2f[n] >= 0] - start[n]
        assert (loc < 4096).any() and (loc >= 4096).any()


def test_backward_table_path_unequal_face_counts():
    """Meshes of 5120 and 1280 faces: the table holds ceil(6400 / 2) = 3200 faces, so image 0 spills and image 1 does
    not; every image's table lands on its own faces."""
    meshes = [_sphere(5120, [30.0])[0], _sphere(1280, [200.0])[0]]
    _run_backward(meshes, 64, 48, 24, EVAL_BLUR, 1)


def test_backward_global_atomics_unequal_and_empty_images():
    meshes = [_soup(300, 3), _soup(0, 0), _sphere(320, [40.0])[0]]
    H, W, K = 22, 37, 6
    assert H * W * K <= 64512
    _run_backward(meshes, H, W, K, EVAL_BLUR, 2)
