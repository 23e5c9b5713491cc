"""Oracle checks of the kernel instantiations bench.py times (VERDICT r1, weak #1a), at the shapes it times them at:
BASELINE configs 2, 3, 4 and 5 with the default flags -- the sparse-first main pass with tile blobs, and the fallback pass
for the tiles forward defers -- the per-sample flag at the same configs, the Philox4x32-7 stream, the SoftRas pair, the
per-face colour gather and the explicit-noise parity mode at config 2, and BASELINE config 1 at full size.

With default flags the coverage stage is drawn in law (compound sampler), so what the oracle can check sample by sample is
everything DOWNSTREAM of the kernel's own hit counts: logits, the S_agg perturbed argmax draws (pert_noise_fill with the
tile's global pixel offset materialises exactly the noise the kernel drew in registers), histogram, image, grad_colors, and
the gradients of every logit that can win (never-winning logits get their in-law draw in this mode; the argmax of zi also
collects them through -sum_j grad_zeta_j, so those entries are excluded).  The per-sample flag is compared end to end,
sampled tiles at every config and the whole image (in chunks of pixels) at configs 2 and 4, where the oracle's d/dsigma,
d/dgamma and d/dalpha are summed over the chunks and compared with the kernel's."""

import math
import os
import sys
import types

import pytest
import torch

from conftest import ROOT, elementwise_close, rel_err
from oracle import pert_oracle as O

pytestmark = pytest.mark.gpu

SIGMA, GAMMA, ALPHA, EPS = 1e-3, 1e-2, 1.0, 1e-10
BG = (1.0, 1.0, 1.0)

# The BASELINE configs bench.py times (its CONFIGS): (N, HW, K, S); the width `tp` in pixels of the sparse-first main
# pass's tiles the shader picks for them on a 148-SM B200 (csrc/cabi.cu sparse_tp; the fallback pass redoes a deferred
# tile as two tp/2-pixel half-tiles); and, per fragment set, the range (low, high) that the share of main-pass tiles
# forward defers to the fallback pass falls in.  (0, 0) says that no tile defers: the work list must be empty.
CONFIGS = {
    2: dict(shape=(8, 256, 50, 64), tp=16, defer=dict(realistic=(0.0, 0.0), dense=(0.9, 1.0), rasterised=(0.35, 0.6))),
    3: dict(shape=(8, 512, 100, 256), tp=8, defer=dict(realistic=(0.0, 0.0), rasterised=(0.35, 0.6))),
    4: dict(shape=(1, 128, 50, 4096), tp=4, defer=dict(rasterised=(0.35, 0.6))),
    5: dict(shape=(16, 1024, 50, 32), tp=16, defer=dict(realistic=(0.0, 0.0))),
}


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")


_LAST_FRAGMENTS = {}


def _fragments(kind, N, HW, K, S):
    """bench.py's fragment sets.  The last one is kept: the config-5 set alone is 23 GB, and tests in a row share it."""
    import pertrenderer_b200 as pb
    key = (kind, N, HW, K)
    if key not in _LAST_FRAGMENTS:
        _LAST_FRAGMENTS.clear()
        torch.cuda.empty_cache()
        if kind == "rasterised":
            if ROOT not in sys.path:
                sys.path.insert(0, ROOT)
            import bench
            fr = bench.rasterised_fragments(types.SimpleNamespace(views=N, image_size=HW, faces_per_pixel=K, nb_samples=S),
                                            torch.device("cuda"))
        else:
            fr = pb.synthetic_fragments(N, HW, HW, K, kind=kind, sigma=SIGMA, seed=0, device="cuda")
        _LAST_FRAGMENTS[key] = fr
    return _LAST_FRAGMENTS[key]


def _problem(fr, col, S, seed_r, seed_a, flags=0, **extra):
    from pertrenderer_b200 import ops
    return ops.ShadeProblem(pix_to_face=fr.pix_to_face, zbuf=fr.zbuf, dists=fr.dists, colors=col, znear=1.0, zfar=100.0,
                            background=BG, sigma=SIGMA, gamma=GAMMA, alpha=ALPHA, eps=EPS, S_rast=S, S_agg=S,
                            seed_rast=seed_r, seed_agg=seed_a, flags=flags, **extra)


def _grad_image(N, HW, seed=1):
    return torch.randn((N, HW, HW, 4), device="cuda", generator=torch.Generator(device="cuda").manual_seed(seed))


def _tile_rows(P, tiles, tp):
    """Gather (1, n_tiles, tp) + tail CPU tensors of the pixels of the given tp-pixel tiles from (P,) + tail tensors."""
    n_tiles = len(tiles)
    pix = (tiles[:, None] * tp + torch.arange(tp)[None, :]).reshape(-1).to("cuda")

    def rows(t, tail):
        return t.reshape((P,) + tail)[pix].reshape((1, n_tiles, tp) + tail).cpu()
    return rows


def _backward_nan_partials(pr, saved, G):
    """ops.shade_backward with its scalar partials buffer filled with NaN first: a row that neither pass writes reaches
    d/d(sigma, gamma, alpha) as NaN."""
    from pertrenderer_b200 import _cabi
    N, H, W, K = pr.shape
    dev = pr.device
    gd = torch.empty((N, H, W, K), dtype=torch.float32, device=dev)
    gz = torch.empty_like(gd)
    gc = torch.empty((N, H, W, K, 3), dtype=torch.float32, device=dev)
    partials = torch.full((3 * pr.num_tiles(), 4), float("nan"), dtype=torch.float32, device=dev)
    scal = torch.empty((3,), dtype=torch.float32, device=dev)
    p = _cabi.ptr
    rc = _cabi.load().pert_shade_bwd(pr.c_struct(), p(G), p(saved.counts), p(saved.rsum), p(saved.winners),
                                     p(saved.pixstate), p(gd), p(gz), p(gc), p(partials), p(scal), None, None, None,
                                     p(saved.worklist), p(saved.blob), _cabi.stream_ptr(dev))
    _cabi.check(rc, "pert_shade_bwd")
    return gd, gz, gc, scal


def _check_scalar_rows(gd, scal, what):
    """The kernel adds d/dsigma = sum gx over the scalar partials rows of both passes and stores grad_dists = -gx
    (shade_bwd.cu, phase 4): a row missing from the sum, or counted twice, breaks the identity."""
    s = gd.double().sum().item()
    scale = gd.double().abs().sum().item()
    assert scale > 0, what
    assert abs(scal[0].item() + s) <= 1e-6 * scale, (what, scal[0].item(), -s, scale)
    assert torch.isfinite(scal).all(), (what, scal.tolist())


def _downstream_oracle(sub, counts, rsum, V, S, G):
    """The oracle from given hit counts on: (a_s, image, grads dict, zeta)."""
    zeta, prob, aux = O.logits_from_counts(sub["pix_to_face"], sub["zbuf"], counts.float(), S, 1.0, 100.0, GAMMA, ALPHA, EPS)
    hist, a_s, a_0 = O.argmax_shard(zeta, V, GAMMA)
    image, weights = O.blend_from_hist(hist, S, prob, sub["colors"], BG)
    grad_w = O._grad_weights(sub["colors"], G, O._as_background(BG))
    packed = O.argmax_score_sums(grad_w, a_s, a_0, V)
    gr = O.shade_backward_from_sums(prob, weights, dict(aux, bg=BG), G, sub["zbuf"], sub["colors"], SIGMA, GAMMA, ALPHA, EPS,
                                    S, S, rsum, packed)
    return a_s, image, gr, zeta


def _check_tiles(config, kind, n_tiles, seed, flags=0):
    """Default flags (or PERT_F_PHILOX7) at a BASELINE config: the work list forward leaves against CONFIGS, the scalar
    partials rows of both passes, and n_tiles main-pass tiles, half of them deferred to the fallback pass, against the
    downstream oracle.  Returns the share of tiles forward deferred."""
    from pertrenderer_b200 import _cabi, ops
    (N, HW, K, S), tp = CONFIGS[config]["shape"], CONFIGS[config]["tp"]
    lo, hi = CONFIGS[config]["defer"][kind]
    fr, col = _fragments(kind, N, HW, K, S)
    dev = fr.pix_to_face.device
    P = N * HW * HW
    G = _grad_image(N, HW)
    seed_r, seed_a = 0x5EED0001 + seed, 0x5EED0002 + seed
    pr = _problem(fr, col, S, seed_r, seed_a, flags)
    image, saved = ops.shade_forward(pr)
    assert saved.blob is not None and saved.worklist is not None  # the production path: sparse-first tiles, tile blobs
    # backward resets the work list: read forward's first
    n_def = int(saved.worklist[0].item())
    ids = saved.worklist[4:4 + n_def].long().cpu()
    n_main = P // tp
    assert n_def == 0 or int(ids.max()) < n_main, f"config {config}: work-list id beyond {n_main} tiles of {tp} pixels"
    assert ids.unique().numel() == n_def
    share = n_def / n_main
    print(f"config {config} {kind} flags={flags:#x}: {n_def} of {n_main} tiles deferred ({share:.4f})")
    if hi == 0:
        assert n_def == 0, f"config {config} {kind}: {n_def} tiles deferred, CONFIGS says none"
    else:
        assert lo <= share <= hi, (config, kind, share)
    gd, gz, gc, scal = _backward_nan_partials(pr, saved, G)
    torch.cuda.synchronize()
    _check_scalar_rows(gd, scal, f"config {config} {kind}")

    gen = torch.Generator().manual_seed(seed)
    deferred = torch.zeros(n_main, dtype=torch.bool)
    deferred[ids] = True
    pick_d = ids[torch.randperm(n_def, generator=gen)[:n_tiles // 2]]
    others = (~deferred).nonzero().squeeze(1)
    pick_m = others[torch.randperm(others.numel(), generator=gen)[:n_tiles - pick_d.numel()]]
    tiles = torch.cat([pick_d, pick_m]).sort().values
    n_tiles = tiles.numel()
    rows = _tile_rows(P, tiles, tp)

    sub = dict(pix_to_face=rows(fr.pix_to_face, (K,)), zbuf=rows(fr.zbuf, (K,)), colors=rows(col, (K, 3)))
    mask = sub["pix_to_face"] >= 0
    counts = rows(saved.counts.to(torch.int32) & 0xFFFF, (K,)) * mask
    rsum = rows(saved.rsum, (K,)) * mask
    stage = 1 | 16 if flags & _cabi.F_PHILOX7 else 1  # pert_noise_fill: bit 4 selects Philox4x32-7
    V = torch.cat([ops.noise_fill(seed_a, stage, (1, 1, tp, K), S, dev, pixel_offset=int(t) * tp) for t in tiles], dim=2).cpu()
    a_s, img_o, gr, zeta = _downstream_oracle(sub, counts, rsum, V, S, rows(G, (4,)))
    # indices bit-exact, image to rounding, colour gradients (weights * G) to rounding
    win = rows(saved.winners_full(), (S,)).long().permute(3, 0, 1, 2)
    assert torch.equal(win, a_s), f"config {config} {kind}: argmax winners differ from the oracle"
    assert (rows(image, (4,)) - img_o).abs().max().item() <= 2e-6
    assert rel_err(rows(gc, (K, 3)), gr["colors"]) <= 1e-6
    # gradients of the logits that can win, away from the argmax of zi
    zmax = zeta.max(-1, keepdim=True).values
    cut = 2.0 * GAMMA * 5.66 * 1.0001 + 4e-7 * zmax.abs().clamp(min=1.0)
    live = (torch.isfinite(zeta) & (zeta >= zmax - cut + 1e-6))[..., :-1]
    zi = torch.where(mask, (100.0 - sub["zbuf"]) / 99.0, torch.zeros_like(sub["zbuf"]))
    sel = mask & live & (zi < zi.max(-1, keepdim=True).values)
    assert sel.sum().item() > n_tiles  # the comparison is not vacuous
    if pick_d.numel():  # ... on the deferred tiles too
        assert sel[0, torch.isin(tiles, pick_d)].any()
    for name, got, ref in (("grad_zbuf", rows(gz, (K,)), gr["zbuf"]), ("grad_dists", rows(gd, (K,)), gr["dists"])):
        scale = ref.abs().max().item()
        err = (got - ref)[sel].abs().max().item()
        assert err <= 1e-5 * scale, (config, kind, name, err, scale)
        assert elementwise_close(got[sel], ref[sel], 1e-5), (config, kind, name)
    assert (rows(gz, (K,))[~mask] == 0).all() and (rows(gd, (K,))[~mask] == 0).all()
    return share


@pytest.mark.parametrize("kind", ["realistic", "dense", "rasterised"])
def test_config2_default_flags_tiles_match_the_oracle(kind):
    """BASELINE config 2 (8 x 256^2, K = 50, S = 64), default flags, 64 random 16-pixel tiles against the oracle."""
    _check_tiles(2, kind, 64, seed=3)


@pytest.mark.parametrize("config, kind", [(3, "rasterised"), (3, "realistic"), (4, "rasterised"), (5, "realistic")])
def test_default_flags_tiles_match_the_oracle(config, kind):
    """BASELINE configs 3 (K = 100, S = 256: two S_agg chunks per backward tile), 4 (S = 4096 on 4-pixel tiles: sixteen
    chunks, 16 lanes per pixel in the fallback pass) and 5 (16.7 M pixels: 64-bit offsets) as config_legs times them."""
    _check_tiles(config, kind, 64, seed=config)


def test_config2_philox7_tiles_match_the_oracle():
    """The philox7 leg: config 2 with PERT_F_PHILOX7, the aggregation noise of the Philox4x32-7 stream."""
    from pertrenderer_b200 import _cabi
    _check_tiles(2, "rasterised", 64, seed=7, flags=_cabi.F_PHILOX7)


def _check_tiles_per_sample(config, kind, n_tiles, seed_r, seed_a, tile_seed):
    """PERT_F_PER_SAMPLE_NOISE at a BASELINE config: coverage counts, winners, image and ALL gradients of n_tiles random
    tiles against the oracle, U and V materialised per tile."""
    from pertrenderer_b200 import _cabi, ops
    (N, HW, K, S), tp = CONFIGS[config]["shape"], CONFIGS[config]["tp"]
    fr, col = _fragments(kind, N, HW, K, S)
    dev = fr.pix_to_face.device
    P = N * HW * HW
    G = _grad_image(N, HW)
    pr = _problem(fr, col, S, seed_r, seed_a, _cabi.F_PER_SAMPLE_NOISE)
    image, saved = ops.shade_forward(pr)
    gd, gz, gc, scal = ops.shade_backward(pr, saved, G)
    tiles = torch.randperm(P // tp, generator=torch.Generator().manual_seed(tile_seed))[:n_tiles].sort().values
    rows = _tile_rows(P, tiles, tp)
    U = torch.cat([ops.noise_fill(seed_r, 0, (1, 1, tp, K), S, dev, pixel_offset=int(t) * tp) for t in tiles], dim=2).cpu()
    V = torch.cat([ops.noise_fill(seed_a, 1, (1, 1, tp, K), S, dev, pixel_offset=int(t) * tp) for t in tiles], dim=2).cpu()
    st, gr = O.shade_fwd_bwd(rows(fr.pix_to_face, (K,)), rows(fr.zbuf, (K,)), rows(fr.dists, (K,)), rows(col, (K, 3)), BG, 1.0,
                             100.0, SIGMA, GAMMA, ALPHA, EPS, U, V, rows(G, (4,)))
    mask = rows(fr.pix_to_face, (K,)) >= 0
    assert mask.any()
    assert torch.equal((rows(saved.counts.to(torch.int32) & 0xFFFF, (K,)))[mask], st.counts[mask])
    assert torch.equal(rows(saved.winners_full(), (S,)).long().permute(3, 0, 1, 2), st.a_s)
    assert (rows(image, (4,)) - st.image).abs().max().item() <= 2e-6
    for name, got, ref in (("colors", rows(gc, (K, 3)), gr["colors"]), ("zbuf", rows(gz, (K,)), gr["zbuf"]),
                           ("dists", rows(gd, (K,)), gr["dists"])):
        assert rel_err(got, ref) <= 1e-5, (config, name)
        assert elementwise_close(got, ref, 1e-5), (config, name)


def test_config2_per_sample_flag_tiles_match_the_oracle_end_to_end():
    """Same job with PERT_F_PER_SAMPLE_NOISE: coverage counts, winners, image and ALL gradients of 48 random tiles."""
    _check_tiles_per_sample(2, "realistic", 48, 77, 78, 9)


@pytest.mark.parametrize("config, kind", [(3, "realistic"), (4, "rasterised"), (5, "realistic")])
def test_per_sample_flag_tiles_match_the_oracle_end_to_end(config, kind):
    """PERT_F_PER_SAMPLE_NOISE at BASELINE configs 3, 4 and 5, 48 random tiles end to end."""
    _check_tiles_per_sample(config, kind, 48, 77 + config, 78 + config, 9 + config)


def chunked_shade_fwd_bwd(p2f, zbuf, dists, colors, G, noise, chunk):
    """O.shade_fwd_bwd over P pixels, `chunk` pixels at a time, so that the noise of a large image never exists whole.
    Inputs are CPU tensors with the pixels flattened: p2f, zbuf, dists (P,K), colors (P,K,3), G (P,4).  noise(start, n)
    returns U (S_rast,1,1,n,K) and V (S_agg,1,1,n,K+1) of pixels start .. start+n-1.  Returns counts (P,K), a_s (S_agg,P),
    image (P,4), gradients dists, zbuf (P,K) and colors (P,K,3), and d/dsigma, d/dgamma, d/dalpha summed over the
    chunks in float64."""
    P, K = p2f.shape
    parts = dict(counts=[], a_s=[], image=[], dists=[], zbuf=[], colors=[])
    scal = dict(sigma=0.0, gamma=0.0, alpha=0.0)
    for c0 in range(0, P, chunk):
        n = min(chunk, P - c0)
        U, V = noise(c0, n)
        st, gr = O.shade_fwd_bwd(p2f[c0:c0 + n].reshape(1, 1, n, K), zbuf[c0:c0 + n].reshape(1, 1, n, K),
                                 dists[c0:c0 + n].reshape(1, 1, n, K), colors[c0:c0 + n].reshape(1, 1, n, K, 3), BG, 1.0,
                                 100.0, SIGMA, GAMMA, ALPHA, EPS, U, V, G[c0:c0 + n].reshape(1, 1, n, 4))
        parts["counts"].append(st.counts.reshape(n, K))
        parts["a_s"].append(st.a_s.reshape(-1, n))
        parts["image"].append(st.image.reshape(n, 4))
        for k in ("dists", "zbuf"):
            parts[k].append(gr[k].reshape(n, K))
        parts["colors"].append(gr["colors"].reshape(n, K, 3))
        for k in scal:
            scal[k] += float(gr[k].double())
    out = {k: torch.cat(v, dim=1 if k == "a_s" else 0) for k, v in parts.items()}
    out.update(scal)
    return out


@pytest.mark.parametrize("config, kind, chunk", [(2, "realistic", 16384), (4, "rasterised", 256)])
def test_per_sample_flag_whole_image_matches_the_oracle(config, kind, chunk):
    """PERT_F_PER_SAMPLE_NOISE on every pixel of BASELINE configs 2 and 4 against the oracle, run in chunks of pixels:
    every entry of counts, winners, image and gradients, and the kernel's d/dsigma, d/dgamma, d/dalpha against the sums
    of the oracle's per-chunk ones -- what no sample of tiles can show about how the partials rows are reduced."""
    from pertrenderer_b200 import _cabi, ops
    N, HW, K, S = CONFIGS[config]["shape"]
    fr, col = _fragments(kind, N, HW, K, S)
    dev = fr.pix_to_face.device
    P = N * HW * HW
    G = _grad_image(N, HW, seed=2)
    seed_r, seed_a = 0x51 + config, 0x52 + config
    pr = _problem(fr, col, S, seed_r, seed_a, _cabi.F_PER_SAMPLE_NOISE)
    image, saved = ops.shade_forward(pr)
    gd, gz, gc, scal = ops.shade_backward(pr, saved, G)

    def noise(c0, n):
        return tuple(ops.noise_fill(seed, stage, (1, 1, n, K), S, dev, pixel_offset=c0).cpu()
                     for seed, stage in ((seed_r, 0), (seed_a, 1)))
    ref = chunked_shade_fwd_bwd(fr.pix_to_face.reshape(P, K).cpu(), fr.zbuf.reshape(P, K).cpu(), fr.dists.reshape(P, K).cpu(),
                                col.reshape(P, K, 3).cpu(), G.reshape(P, 4).cpu(), noise, chunk)
    mask = fr.pix_to_face.reshape(P, K).cpu() >= 0
    assert torch.equal((saved.counts.to(torch.int32) & 0xFFFF).reshape(P, K).cpu()[mask], ref["counts"][mask])
    # Winners bit for bit, but for near-ties: zeta_j = (gamma/alpha) log(c_j/S) + zi_j - zmax takes the log of the same
    # count on both sides, and the device's logf and the CPU's log may round it 1 ulp apart, which can move zeta by one
    # ulp of zi (6e-8 near 1).  A draw whose two best perturbed scores lie closer than that may go either way; it
    # happens about once in 10^8 draws (S = 4096 gives many distinct counts).  Such a pixel is left out of the per-entry
    # comparisons below, whose values depend on its histogram, and its share of the scalars is taken with the kernel's
    # winner of that draw.
    win = saved.winners_full().reshape(P, S).cpu().long().t()
    flips = (win != ref["a_s"]).nonzero().tolist()
    assert len(flips) <= 1e-7 * P * S + 2, len(flips)
    keep = torch.ones(P, dtype=torch.bool)
    for s, p in flips:
        U, V = noise(p, 1)
        st = O.shade_forward(fr.pix_to_face.reshape(P, K)[p].reshape(1, 1, 1, K).cpu(),
                             fr.zbuf.reshape(P, K)[p].reshape(1, 1, 1, K).cpu(), fr.dists.reshape(P, K)[p].reshape(1, 1, 1, K).cpu(),
                             col.reshape(P, K, 3)[p].reshape(1, 1, 1, K, 3).cpu(), BG, 1.0, 100.0, SIGMA, GAMMA, ALPHA, EPS, U, V)
        score = (st.zeta.reshape(-1) + GAMMA * V[s].reshape(-1)).double()
        gap = (score[ref["a_s"][s, p]] - score[win[s, p]]).item()
        assert 0.0 <= gap <= 1.2e-7, (s, p, int(ref["a_s"][s, p]), int(win[s, p]), gap)
        keep[p] = False
        # the pixel's share of d/d(sigma, gamma, alpha) with the kernel's winner of that draw instead of the oracle's
        G1, col1, zb1 = G.reshape(P, 4)[p].reshape(1, 1, 1, 4).cpu(), col.reshape(P, K, 3)[p].reshape(1, 1, 1, K, 3).cpu(), \
            fr.zbuf.reshape(P, K)[p].reshape(1, 1, 1, K).cpu()
        a_s = st.a_s.clone()
        a_s[s] = win[s, p]
        hist = torch.zeros((K + 1,), dtype=torch.int32).scatter_add_(0, a_s.reshape(-1), torch.ones(S, dtype=torch.int32))
        _, weights = O.blend_from_hist(hist.reshape(1, 1, 1, K + 1), S, st.prob, col1, BG)
        packed = O.argmax_score_sums(O._grad_weights(col1, G1, O._as_background(BG)), a_s, st.a_0, V)
        _, rsum = O.rast_shard_sums(fr.dists.reshape(P, K)[p].reshape(1, 1, 1, K).cpu(), U, SIGMA)
        moved = O.shade_backward_from_sums(st.prob, weights, st.aux, G1, zb1, col1, SIGMA, GAMMA, ALPHA, EPS, S, S, rsum, packed)
        orig = O.shade_backward(st, G1, zb1, col1, SIGMA, GAMMA, ALPHA, EPS, U, V)
        for k in ("sigma", "gamma", "alpha"):
            ref[k] += float(moved[k].double()) - float(orig[k].double())
    assert (image.reshape(P, 4).cpu() - ref["image"])[keep].abs().max().item() <= 2e-6
    for name, got in (("colors", gc.reshape(P, K, 3)), ("zbuf", gz.reshape(P, K)), ("dists", gd.reshape(P, K))):
        assert rel_err(got.cpu()[keep], ref[name][keep]) <= 1e-5, (config, name)
        assert elementwise_close(got.cpu()[keep], ref[name][keep], 1e-5), (config, name)
    for i, k in enumerate(("sigma", "gamma", "alpha")):
        assert abs(scal[i].item() - ref[k]) <= 2e-5 * abs(ref[k]) + 1e-7, (config, k, scal[i].item(), ref[k])


def test_config2_softras_pair_whole_image_matches_the_oracle():
    """The softras_pair leg: SoftRast + SoftAgg on every pixel of BASELINE config 2 (realistic) against the oracle, in
    chunks of pixels; the scalars against the float64 sum of the chunks'."""
    from pertrenderer_b200 import ops
    N, HW, K, S = CONFIGS[2]["shape"]
    fr, col = _fragments("realistic", N, HW, K, S)
    P = N * HW * HW
    G = _grad_image(N, HW)
    pr = _problem(fr, col, S, 0, 0)
    image = ops.soft_shade_forward(pr)
    gd, gz, gc, scal = ops.soft_shade_backward(pr, G)
    got = dict(image=image.reshape(P, 4).cpu(), dists=gd.reshape(P, K).cpu(), zbuf=gz.reshape(P, K).cpu(),
               colors=gc.reshape(P, K, 3).cpu())
    cpu = [t.reshape((P,) + t.shape[3:]).cpu() for t in (fr.pix_to_face, fr.zbuf, fr.dists, col, G)]
    ref = dict(image=[], dists=[], zbuf=[], colors=[])
    sums = dict(sigma=0.0, gamma=0.0, alpha=0.0)
    chunk = 65536
    for c0 in range(0, P, chunk):
        p2f, zb, di, co, g = (t[c0:c0 + chunk].reshape((1, 1, -1) + t.shape[1:]) for t in cpu)
        img, _, _, gr = O.soft_shade_fwd_bwd(p2f, zb, di, co, BG, 1.0, 100.0, SIGMA, GAMMA, ALPHA, EPS, g)
        ref["image"].append(img.reshape(-1, 4))
        for k in ("dists", "zbuf", "colors"):
            ref[k].append(gr[k].reshape((-1,) + got[k].shape[1:]))
        for k in sums:
            sums[k] += float(gr[k].double())
    ref = {k: torch.cat(v) for k, v in ref.items()}
    assert (got["image"] - ref["image"]).abs().max().item() <= 2e-6
    for k in ("dists", "zbuf", "colors"):
        assert rel_err(got[k], ref[k]) <= 1e-5, k
    for i, k in enumerate(("sigma", "gamma", "alpha")):
        assert abs(scal[i].item() - sums[k]) <= 1e-4 * abs(sums[k]) + 1e-7, (k, scal[i].item(), sums[k])


def test_config2_face_colour_gather_gradient_matches_a_float64_scatter():
    """The face_colour_gather leg: BASELINE config 2 (realistic), default flags, texel colours gathered through pix_to_face
    from a 1280-face table inside the kernels.  The (F,3) gradient the kernels scatter with atomics against a float64
    index_add of (hist / S_agg) G_rgb over the whole image, hist counted from the kernel's winners (which the sampled-tile
    tests check bit for bit against the oracle)."""
    from pertrenderer_b200 import ops
    N, HW, K, S = CONFIGS[2]["shape"]
    fr, _ = _fragments("realistic", N, HW, K, S)
    dev = fr.pix_to_face.device
    P, F = N * HW * HW, 1280
    table = torch.rand((F, 3), device=dev, generator=torch.Generator(device=dev).manual_seed(7))
    p2f = fr.pix_to_face.clamp(max=F - 1)
    G = _grad_image(N, HW)
    pr = ops.ShadeProblem(pix_to_face=p2f, zbuf=fr.zbuf, dists=fr.dists, colors=None, face_colors=table, znear=1.0,
                          zfar=100.0, background=BG, sigma=SIGMA, gamma=GAMMA, alpha=ALPHA, eps=EPS, S_rast=S, S_agg=S,
                          seed_rast=21, seed_agg=22)
    image, saved = ops.shade_forward(pr)
    gd, gz, gc, scal = ops.shade_backward(pr, saved, G)
    win = saved.winners_full().reshape(P, S).long()
    hist = torch.zeros((P, K + 1), dtype=torch.float64, device=dev).scatter_add_(1, win, torch.ones_like(win, dtype=torch.float64))
    p2f = p2f.reshape(P, K)
    valid = p2f >= 0
    contrib = (hist[:, :K, None] / S) * G.reshape(P, 1, 4)[..., :3].double()
    ref = torch.zeros((F, 3), dtype=torch.float64, device=dev).index_add_(0, p2f[valid], contrib[valid])
    assert ref.abs().max().item() > 0
    assert rel_err(gc, ref) <= 1e-5


def test_config2_explicit_noise_tiles_match_the_oracle():
    """The explicit_noise leg: BASELINE config 2 with both noise tensors (S,N,H,W,K) and (S,N,H,W,K+1) in HBM, the exact-
    noise parity mode: 48 random tiles end to end against the oracle, U and V sliced from the device tensors."""
    from pertrenderer_b200 import ops
    N, HW, K, S = CONFIGS[2]["shape"]
    tp, n_tiles = 16, 48
    fr, col = _fragments("rasterised", N, HW, K, S)
    dev = fr.pix_to_face.device
    P = N * HW * HW
    G = _grad_image(N, HW)
    gen = torch.Generator(device=dev).manual_seed(5)
    U = torch.randn((S, N, HW, HW, K), device=dev, generator=gen)
    V = torch.randn((S, N, HW, HW, K + 1), device=dev, generator=gen)
    pr = _problem(fr, col, S, 0, 0, noise_rast=U, noise_agg=V)
    image, saved = ops.shade_forward(pr)
    gd, gz, gc, scal = ops.shade_backward(pr, saved, G)
    tiles = torch.randperm(P // tp, generator=torch.Generator().manual_seed(11))[:n_tiles].sort().values
    rows = _tile_rows(P, tiles, tp)
    Ut = torch.stack([rows(U[s], (K,)) for s in range(S)])
    Vt = torch.stack([rows(V[s], (K + 1,)) for s in range(S)])
    del U, V
    st, gr = O.shade_fwd_bwd(rows(fr.pix_to_face, (K,)), rows(fr.zbuf, (K,)), rows(fr.dists, (K,)), rows(col, (K, 3)), BG, 1.0,
                             100.0, SIGMA, GAMMA, ALPHA, EPS, Ut, Vt, rows(G, (4,)))
    mask = rows(fr.pix_to_face, (K,)) >= 0
    assert mask.any()
    assert torch.equal((rows(saved.counts.to(torch.int32) & 0xFFFF, (K,)))[mask], st.counts[mask])
    assert torch.equal(rows(saved.winners_full(), (S,)).long().permute(3, 0, 1, 2), st.a_s)
    assert (rows(image, (4,)) - st.image).abs().max().item() <= 2e-6
    for name, got, ref in (("colors", rows(gc, (K, 3)), gr["colors"]), ("zbuf", rows(gz, (K,)), gr["zbuf"]),
                           ("dists", rows(gd, (K,)), gr["dists"])):
        assert rel_err(got, ref) <= 1e-5, name
        assert elementwise_close(got, ref, 1e-5), name


def test_config1_full_size_matches_the_oracle():
    """BASELINE config 1 at full size (1 x 64^2, K = 50, S = 16): per-sample flag end to end against the oracle on the
    whole image; default flags through the downstream oracle on every pixel."""
    from pertrenderer_b200 import _cabi, ops
    import pertrenderer_b200 as pb
    N, HW, K, S = 1, 64, 50, 16
    for kind in ("realistic", "dense"):
        fr, col = pb.synthetic_fragments(N, HW, HW, K, kind=kind, sigma=SIGMA, seed=4, device="cuda")
        dev = fr.pix_to_face.device
        G = torch.randn((N, HW, HW, 4), device=dev, generator=torch.Generator(device=dev).manual_seed(2))
        cpu = dict(pix_to_face=fr.pix_to_face.cpu(), zbuf=fr.zbuf.cpu(), dists=fr.dists.cpu(), colors=col.cpu())
        mask = cpu["pix_to_face"] >= 0

        def problem(flags):
            return ops.ShadeProblem(pix_to_face=fr.pix_to_face, zbuf=fr.zbuf, dists=fr.dists, colors=col, znear=1.0, zfar=100.0,
                                    background=BG, sigma=SIGMA, gamma=GAMMA, alpha=ALPHA, eps=EPS, S_rast=S, S_agg=S,
                                    seed_rast=5, seed_agg=6, flags=flags)
        U = ops.noise_fill(5, 0, (N, HW, HW, K), S, dev).cpu()
        V = ops.noise_fill(6, 1, (N, HW, HW, K), S, dev).cpu()
        # per-sample path, everything
        pr = problem(_cabi.F_PER_SAMPLE_NOISE)
        image, saved = ops.shade_forward(pr)
        gd, gz, gc, scal = ops.shade_backward(pr, saved, G)
        st, gr = O.shade_fwd_bwd(cpu["pix_to_face"], cpu["zbuf"], cpu["dists"], cpu["colors"], BG, 1.0, 100.0, SIGMA, GAMMA,
                                 ALPHA, EPS, U, V, G.cpu())
        assert torch.equal((saved.counts.to(torch.int32) & 0xFFFF).cpu()[mask], st.counts[mask])
        assert torch.equal(saved.winners_full().cpu().long().permute(3, 0, 1, 2), st.a_s)
        assert (image.cpu() - st.image).abs().max().item() <= 2e-6
        for name, got, ref in (("colors", gc, gr["colors"]), ("zbuf", gz, gr["zbuf"]), ("dists", gd, gr["dists"])):
            assert rel_err(got.cpu(), ref) <= 1e-5, (kind, name)
            assert elementwise_close(got.cpu(), ref, 1e-5), (kind, name)
        for i, k in enumerate(("sigma", "gamma", "alpha")):
            assert abs(scal[i].item() - gr[k].item()) <= 2e-5 * abs(gr[k].item()) + 1e-7, (kind, k)
        # default flags: downstream of the kernel's own counts
        pr = problem(0)
        image, saved = ops.shade_forward(pr)
        gd, gz, gc, scal = ops.shade_backward(pr, saved, G)
        counts = (saved.counts.to(torch.int32) & 0xFFFF).cpu() * mask
        a_s, img_o, gr2, zeta = _downstream_oracle(cpu, counts, saved.rsum.cpu() * mask, V, S, G.cpu())
        assert torch.equal(saved.winners_full().cpu().long().permute(3, 0, 1, 2), a_s)
        assert (image.cpu() - img_o).abs().max().item() <= 2e-6
        assert rel_err(gc.cpu(), gr2["colors"]) <= 1e-6
        assert torch.isfinite(gd).all() and torch.isfinite(gz).all() and torch.isfinite(scal).all()


def test_graph_captured_step_matches_eager_and_redraws_noise():
    """Small-problem path: forward + backward captured in ONE CUDA graph with device-side seeds (pert_problem.seed_device,
    pert_seed_advance).  A replay equals the eager run with the effective seeds (seed ^ device value) bit for bit; the next
    replay draws other noise; inputs written into the static buffers between replays are picked up."""
    import pertrenderer_b200 as pb
    from pertrenderer_b200 import ops
    N, HW, K, S = 1, 64, 50, 16
    fr, col = pb.synthetic_fragments(N, HW, HW, K, kind="realistic", sigma=SIGMA, seed=3, device="cuda")
    dev = fr.pix_to_face.device
    G = torch.randn((N, HW, HW, 4), device=dev, generator=torch.Generator(device=dev).manual_seed(2))
    zbuf, dists, colors = fr.zbuf.clone(), fr.dists.clone(), col.clone()
    step = ops.GraphedShadeStep(fr.pix_to_face, zbuf, dists, colors, G, sigma=SIGMA, gamma=GAMMA, alpha=ALPHA, eps=EPS,
                                S_rast=S, S_agg=S, background=BG, seed=1234)
    seeds_before = step.seed_device.clone()
    out1 = [t.clone() for t in step.replay()]
    torch.cuda.synchronize()
    seeds_used = step.seed_device.clone()  # advance runs first inside the graph: these are the seeds replay 1 drew with
    assert not torch.equal(seeds_before, seeds_used)

    def eager(seeds):
        pr = ops.ShadeProblem(pix_to_face=fr.pix_to_face, zbuf=zbuf, dists=dists, colors=colors, znear=1.0, zfar=100.0,
                              background=BG, sigma=SIGMA, gamma=GAMMA, alpha=ALPHA, eps=EPS, S_rast=S, S_agg=S,
                              seed_rast=int(seeds[0].item()), seed_agg=int(seeds[1].item()))
        image, saved = ops.shade_forward(pr)
        return (image,) + ops.shade_backward(pr, saved, G)
    ref1 = eager(seeds_used)
    for a, b in zip(out1, ref1):
        assert torch.equal(a, b)
    out2 = [t.clone() for t in step.replay()]
    assert not torch.equal(out1[0], out2[0])  # fresh noise
    for a, b in zip(out2, eager(step.seed_device)):
        assert torch.equal(a, b)
    dists.mul_(0.5)  # new inputs through the static buffers
    out3 = [t.clone() for t in step.replay()]
    for a, b in zip(out3, eager(step.seed_device)):
        assert torch.equal(a, b)


def test_in_place_edit_of_an_input_before_backward_is_detected():
    """The backward kernels re-read dists / zbuf / colours: the autograd Function registers them, so an in-place edit
    between forward and backward raises instead of changing the gradients silently."""
    import pertrenderer_b200 as pb
    fr, col = pb.synthetic_fragments(1, 8, 8, 6, kind="dense", device="cuda")
    d = fr.dists.clone().requires_grad_(True)
    dd = d * 1.0  # non-leaf, so that an in-place op is legal
    img = pb.smooth_rgb_blend(col, pb.Fragments(fr.pix_to_face, fr.zbuf, None, dd), pb.GaussianRast(nb_samples=8, sigma=1e-3),
                              pb.GaussianAgg(nb_samples=8, gamma=1e-2), pb.BlendParams())
    dd.mul_(2.0)
    with pytest.raises(RuntimeError, match="modified by an inplace operation"):
        img.sum().backward()


def test_atlas_textured_mesh_through_the_fused_shader():
    """TexturesAtlas meshes (eval.py:216-238): TriMeshes(atlas=...) -> sample_textures -> the fused pair; the gradient reaches
    the atlas cells that were hit, and the image equals the one rendered from the materialised texel tensor."""
    import pertrenderer_b200 as pb
    dev = "cuda"
    N, HW, K, F, R = 2, 16, 8, 20, 4
    fr, _ = pb.synthetic_fragments(N, HW, HW, K, kind="realistic", sigma=SIGMA, n_faces=F, seed=2, device=dev)
    p2f = fr.pix_to_face.clamp(max=F - 1)
    bary = pb.synthetic_bary(p2f, seed=1)
    frag = pb.Fragments(p2f, fr.zbuf, bary, fr.dists)
    verts, faces = pb.synthetic_mesh(F, device=dev)
    atlas = torch.rand((F, R, R, 3), device=dev).requires_grad_(True)
    mesh = pb.TriMeshes(verts, faces, atlas=atlas)
    shader = pb.RandomSimpleShader(device=dev, cameras=pb.DepthCameras(n=N, device=dev),
                                   smoothrast=pb.GaussianRast(nb_samples=16, sigma=SIGMA),
                                   smoothagg=pb.GaussianAgg(nb_samples=16, gamma=GAMMA), blend_params=pb.BlendParams())
    torch.manual_seed(5)
    img = shader(frag, mesh)
    img[..., :3].sum().backward()
    assert atlas.grad is not None and torch.isfinite(atlas.grad).all() and atlas.grad.abs().sum() > 0
    tex = pb.AtlasTexels(atlas.detach()).materialize(p2f, bary)
    torch.manual_seed(5)
    img2 = shader(frag, pb.TexelMeshes(tex))
    assert torch.equal(img.detach(), img2.detach())
