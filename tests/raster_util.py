"""Strict comparison of the rasteriser's fragments (pert_rasterize_fwd) with the float64 oracle
(oracle/raster_oracle.py), shared by the -m gpu raster tests.

The kernels evaluate every (pixel, face) pair in float32; the oracle evaluates the same formulas in float64 on the
same float32 inputs, so it is exact to about 1e-16 relative.  Each float32 quantity q of a pair gets a first-order
error bound dq from the operations that produce it:

    edge e = (p.x-a.x)(b.y-a.y) - (p.y-a.y)(b.x-a.x)   de = TAU * (|p.x-a.x||b.y-a.y| + |p.y-a.y||b.x-a.x|
                                                                  + R (|b.x-a.x| + |b.y-a.y|))
        (R = the long-to-short side ratio: the float32 pixel centre is off by a few ulps of R)
    A = edge(v2; v0, v1) + kEps                         dA = TAU * (|terms of A|)
    w_i = e_i / A                                       dw_i = (de_i + |w_i| dA) / |A| + TAU |w_i|
    pz = sum w_i z_i                                    dpz = sum dw_i |z_i| + TAU sum |w_i z_i|
    dist = |p - proj|^2 on the closest edge             dd = 2 sqrt(dist) dr + dr^2 + TAU dist, dr = TAU L
        (L = largest |coordinate| of the pixel and the face: the error of p - proj)

with TAU = 16 float32 ulps (2^-20): the longest chain above has about eight roundings, each at most half an ulp of a
term no larger than the bounded one, and the factor of two covers the second-order terms.  The 1/|A| factor widens
the bound of sliver faces instead of masking them out.

Selections may differ only where a decision is marginal: every face in the symmetric difference of the kernel's and
the oracle's set at a pixel must sit within its error bound of one of the boundaries the kernels test (an edge
function at 0, dist at the blur radius, pz at 0 or at the K-th kept depth, |area| at kEps or at 0 when culling back
faces).  Within a kept list, depths must ascend up to those bounds, so a changed order is only allowed at a depth tie.
Faces with bit-identical corners are an exact tie, which the kernels break by face index: the earlier one comes first,
and the later one is never kept without it.
"""

import numpy as np
import torch

from oracle import raster_oracle as RO

TAU = 2.0 ** -20
K_EPS32 = float(np.float32(1e-8))


def f32(x):
    """The float32 value the C ABI receives for a Python float."""
    return float(np.float32(x))


def abs_edge_terms(p, a, b):
    return (p[..., 0] - a[..., 0]).abs() * (b[..., 1] - a[..., 1]).abs() + (p[..., 1] - a[..., 1]).abs() * (b[..., 0] - a[..., 0]).abs()


def pair_stats(fv64, faces, pxy, R):
    """float64 values and float32 error bounds of the (pixel, face) pairs faces (M,) x pxy (M,2)."""
    v = fv64[faces]
    v0, v1, v2 = v[:, 0, :2], v[:, 1, :2], v[:, 2, :2]
    z = v[:, :, 2]
    e = torch.stack((RO.edge_function(pxy, v1, v2), RO.edge_function(pxy, v2, v0), RO.edge_function(pxy, v0, v1)), -1)
    de = TAU * torch.stack([abs_edge_terms(pxy, a, b) + R * (b - a).abs().sum(-1) for a, b in ((v1, v2), (v2, v0), (v0, v1))], -1)
    area_raw = RO.edge_function(v0, v1, v2)  # the culling tests' area
    A = RO.edge_function(v2, v0, v1) + RO.K_EPS
    dA = TAU * abs_edge_terms(v2, v0, v1) + TAU * abs(RO.K_EPS)
    w = e / A[:, None]
    dw = (de + w.abs() * dA[:, None]) / A.abs()[:, None] + TAU * w.abs()
    pz = (w * z).sum(-1)
    dpz = (dw * z.abs()).sum(-1) + TAU * (w * z).abs().sum(-1)
    dist = RO.point_triangle_distance(pxy, v0, v1, v2)
    L = torch.cat((pxy.abs(), v[:, :, :2].abs().flatten(1)), -1).amax(-1)
    dr = TAU * L
    dd = 2.0 * dist.sqrt() * dr + dr * dr + TAU * dist
    inside = (w > 0).all(-1)
    return dict(w=w, dw=dw, pz=pz, dpz=dpz, dist=dist, dd=dd, sd=torch.where(inside, -dist, dist),
                edge_marginal=(w.abs() <= dw).any(-1), area_raw=area_raw, dA=dA)


def _ratio(err, bound):
    """err / bound, 0 where the error is 0 (a bound of 0 then allows exactly 0); NaN stays NaN and fails."""
    return torch.where(err == 0, torch.zeros_like(err), err / bound)


def _marginal(st, i, blur, cull, zk_bounds):
    """Is pair i of the stats st within its error bound of a boundary of the kernels' tests?"""
    if bool(st["edge_marginal"][i]):
        return "edge"
    if abs(st["dist"][i].item() - blur) <= st["dd"][i].item() + TAU * blur:
        return "blur"
    if abs(st["pz"][i].item()) <= st["dpz"][i].item():
        return "pz0"
    a = st["area_raw"][i].item()
    if abs(abs(a) - K_EPS32) <= st["dA"][i].item() or (cull and abs(a) <= st["dA"][i].item()):
        return "area"
    for zk, dzk in zk_bounds:
        if abs(st["pz"][i].item() - zk) <= st["dpz"][i].item() + dzk:
            return "depth"
    return None


def check_fragments(got, fv, face_start, H, W, K, blur, cull=False, max_diff_frac=0.01, min_valid=1):
    """Assert that the kernel's fragments got = (pix_to_face, zbuf, bary, dists) are the oracle's on the float32
    faces fv (F,3,3) up to the bounds of the module docstring.  Returns the oracle's float64 fragments."""
    p2f_g, z_g, b_g, d_g = (t.cpu() for t in got)
    N = p2f_g.shape[0]
    assert p2f_g.shape == (N, H, W, K) and b_g.shape == (N, H, W, K, 3)
    fv64 = fv.detach().cpu().double()
    blur = f32(blur)
    ref = RO.rasterize(fv64, [int(s) for s in face_start], H, W, K, blur, cull)
    p2f_r = ref[0]
    valid = p2f_g >= 0
    assert int(valid.sum()) >= min_valid, "too few fragments for the case to test anything"

    # padding: exactly -1, after the kept entries
    assert (valid[..., 1:] <= valid[..., :-1]).all()
    pad = ~valid
    assert (p2f_g[pad] == -1).all() and (z_g[pad] == -1).all() and (d_g[pad] == -1).all() and (b_g[pad] == -1).all()
    # kept faces belong to the pixel's image, once each
    fs = torch.as_tensor([int(s) for s in face_start])
    n_of = torch.arange(N).reshape(N, 1, 1, 1).expand_as(p2f_g)
    assert ((p2f_g >= fs[n_of]) & (p2f_g < fs[n_of + 1]))[valid].all()
    srt = p2f_g.sort(-1).values
    assert not ((srt[..., 1:] == srt[..., :-1]) & (srt[..., 1:] >= 0)).any()

    # values of every kept entry against the float64 formulas of that (pixel, face)
    R = max(H, W) / min(H, W)
    pxy64 = RO.pixel_centers(H, W, torch.float64)
    ent = valid.nonzero()
    st = pair_stats(fv64, p2f_g[valid], pxy64[ent[:, 1], ent[:, 2]], R)
    zg, bg, dg = z_g[valid].double(), b_g[valid].double(), d_g[valid].double()
    ez = _ratio((zg - st["pz"]).abs(), st["dpz"])
    eb = _ratio((bg - st["w"]).abs(), st["dw"]).amax(-1)
    sign_sure = ~st["edge_marginal"]
    ed = _ratio(torch.where(sign_sure, (dg - st["sd"]).abs(), (dg.abs() - st["dist"]).abs()), st["dd"])
    for name, r in (("zbuf", ez), ("bary", eb), ("dists", ed)):
        bad = ~(r <= 1.0)
        if bad.any():
            j = int(r.nan_to_num(float("inf")).argmax())
            raise AssertionError(f"{name}: {int(bad.sum())} of {r.numel()} entries outside the float32 bound; worst at "
                                 f"(n,y,x,k)={ent[j].tolist()} face {int(p2f_g[valid][j])}: error/bound {r[j].item():.3g}")
    # ascending depth up to the bounds: a changed order is a depth tie
    pz = torch.full(p2f_g.shape, float("inf"), dtype=torch.float64)
    dz = torch.zeros(p2f_g.shape, dtype=torch.float64)
    pz[valid], dz[valid] = st["pz"], st["dpz"]
    both = valid[..., 1:]
    assert ((pz[..., :-1] - pz[..., 1:]) <= dz[..., :-1] + dz[..., 1:])[both].all(), "kept depths out of order"
    # faces with bit-identical corners are evaluated identically: their tie is exact and goes to the lower index
    bits = fv.detach().cpu().float().contiguous().view(torch.int32).reshape(-1, 9)
    fb = bits[p2f_g.clamp(min=0)]
    twin = both & (fb[..., :-1, :] == fb[..., 1:, :]).all(-1)
    assert (p2f_g[..., :-1] < p2f_g[..., 1:])[twin].all(), "identical faces kept out of face order"

    # selections: every face kept by one side only is marginal at that pixel
    sel_g, sel_r = srt, p2f_r.sort(-1).values
    differ = (sel_g != sel_r).any(-1)
    n_diff = int(differ.sum())
    assert n_diff <= max_diff_frac * N * H * W, f"{n_diff} pixels select other faces than the oracle"
    for n, y, x in differ.nonzero().tolist():
        g = set(p2f_g[n, y, x][p2f_g[n, y, x] >= 0].tolist())
        r = set(p2f_r[n, y, x][p2f_r[n, y, x] >= 0].tolist())
        union = sorted(g | r)
        sst = pair_stats(fv64, torch.tensor(union), pxy64[y, x][None].expand(len(union), 2), R)
        # a face lost to truncation at K was outranked by a face whose float32 depth erred by at most its own bound
        slack = sst["dpz"].max().item()
        zk = [(ref[1][n, y, x, K - 1].item(), slack)] if len(r) == K else []
        if len(g) == K:
            zk.append((sst["pz"][union.index(int(p2f_g[n, y, x, K - 1]))].item(), slack))
        for i, a in enumerate(union):  # of two identical faces, the later one is never kept without the earlier
            for b in union[i + 1:]:
                if b in g and a not in g and torch.equal(bits[a], bits[b]):
                    raise AssertionError(f"pixel (n,y,x)=({n},{y},{x}): face {b} kept without its identical face {a}")
        for i, f in enumerate(union):
            if f in g and f in r:
                continue
            assert _marginal(sst, i, blur, cull, zk) is not None, \
                (f"pixel (n,y,x)=({n},{y},{x}): face {f} {'kept' if f in g else 'dropped'} by the kernel is not marginal: "
                 f"pz={sst['pz'][i].item():.9g} dist={sst['dist'][i].item():.9g} w={sst['w'][i].tolist()}")
    return ref
