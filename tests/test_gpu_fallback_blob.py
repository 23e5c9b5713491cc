"""The fallback records of the tile blob (csrc/common.cuh): on tiles that the sparse-first main pass hands to the fallback
pass, backward takes the valid list and the per-pixel logit summary from the half-tile's record that forward wrote, and
forward's aggregation launch takes the valid list from the record its coverage launch wrote.  Both must compute exactly
what the re-deriving paths compute (tile_blob = NULL) on the tiles both give to the same pass: BASELINE config 2 at full
size on the rasterised, dense and realistic sets, and with the per-face colour gather."""

import dataclasses
import types

import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda"
N, HW, K, S = 8, 256, 50, 64  # BASELINE config 2


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


_FRAGMENTS = {}


def _fragments(kind):
    if kind not in _FRAGMENTS:
        import bench
        import pertrenderer_b200 as pb
        if kind == "rasterised":
            _FRAGMENTS[kind] = bench.rasterised_fragments(
                types.SimpleNamespace(views=N, image_size=HW, faces_per_pixel=K, nb_samples=S), DEV)
        else:
            _FRAGMENTS[kind] = pb.synthetic_fragments(N, HW, HW, K, kind=kind, sigma=1e-3, seed=0, device=DEV)
    return _FRAGMENTS[kind]


def _problem(kind, face):
    from pertrenderer_b200 import ops
    fr, col = _fragments(kind)
    table = None
    if face:  # one colour per face id of the batch
        table = torch.rand((int(fr.pix_to_face.max()) + 1, 3), device=DEV, generator=torch.Generator(device=DEV).manual_seed(7))
        col = None
    return ops.ShadeProblem(pix_to_face=fr.pix_to_face, zbuf=fr.zbuf, dists=fr.dists, colors=col, face_colors=table, znear=1.0,
                            zfar=100.0, background=(0.2, 0.5, 0.8), sigma=1e-3, gamma=1e-2, alpha=1.0, eps=1e-10,
                            S_rast=S, S_agg=S, seed_rast=1234, seed_agg=5678)


def _grad_image():
    return torch.randn((N, HW, HW, 4), device=DEV, generator=torch.Generator(device=DEV).manual_seed(1))


def _forward_without_blob(pr):
    """pert_shade_fwd with tile_blob = NULL: the aggregation launch of the fallback pass re-scans pix_to_face."""
    from pertrenderer_b200 import _cabi, ops
    lib = _cabi.load()
    image, saved = ops.shade_forward(pr)  # buffers of the right shapes, overwritten with junk and recomputed below
    saved = dataclasses.replace(saved, blob=None)
    image.fill_(float("nan"))
    saved.rsum.fill_(float("nan"))
    for t in (saved.counts, saved.winners, saved.pixstate):
        t.fill_(-1)
    rc = lib.pert_shade_fwd(pr.c_struct(), _cabi.ptr(image), _cabi.ptr(saved.counts), _cabi.ptr(saved.rsum),
                            _cabi.ptr(saved.winners), _cabi.ptr(saved.pixstate), None, _cabi.ptr(saved.worklist), None,
                            _cabi.stream_ptr(torch.device(DEV)))
    _cabi.check(rc, "pert_shade_fwd")
    return image, saved


def _tile_passes(pr, saved):
    """Per tile of the sparse-first main pass (16 pixels at config 2): did forward defer it to the fallback pass, and does
    it overflow the main pass's compact arrays (more than 160 valid entries)?  Read before backward resets the work list."""
    tp, cap = 16, 160
    n = int(saved.worklist[0].item())
    deferred = torch.zeros(N * HW * HW // tp, dtype=torch.bool, device=DEV)
    deferred[saved.worklist[4:4 + n].long()] = True
    overflow = (pr.pix_to_face >= 0).reshape(-1, tp * K).sum(1) > cap
    return deferred, overflow


@pytest.mark.parametrize("face", [False, True], ids=["colors", "face_colors"])
@pytest.mark.parametrize("kind", ["rasterised", "dense", "realistic"])
def test_backward_from_fallback_records_matches_rederive(kind, face):
    """Backward with the tile blob (main-pass blobs, fallback records) against backward with tile_blob = NULL, from one
    forward.  Without a blob, backward's main pass hands over only the tiles that overflow its compact arrays; forward also
    defers tiles with many entries for the compound sampler, which the blob's headers send to the fallback pass.  Every tile
    that both runs give to the same pass must come out bit for bit; the others differ in the association order of float
    sums only (compact against dense per-logit arrays)."""
    from pertrenderer_b200 import ops
    pr = _problem(kind, face)
    image, saved = ops.shade_forward(pr)
    assert saved.blob is not None
    deferred, overflow = _tile_passes(pr, saved)
    if kind != "realistic":
        assert (deferred & overflow).any()  # the fallback pass ran from its records on tiles compared bit for bit
    same = ~deferred | overflow
    G = _grad_image()
    with_blob = ops.shade_backward(pr, saved, G)
    rederived = ops.shade_backward(pr, dataclasses.replace(saved, blob=None), G)
    per_entry = [("grad_dists", 0), ("grad_zbuf", 1)] + ([] if face else [("grad_colors", 2)])
    for name, i in per_entry:
        a, b = (t.reshape(same.numel(), -1) for t in (with_blob[i], rederived[i]))
        assert torch.equal(a[same], b[same]), f"{kind}: {name} differs between the blob and the re-derive path"
        scale = b.abs().max().item()
        assert torch.allclose(a[~same], b[~same], rtol=1e-4, atol=1e-5 * scale), (kind, name)
    if face:  # per-face colour gradients are sums of float atomics: their order is not fixed, from one run to the next too
        scale = rederived[2].abs().max().item()
        assert torch.allclose(with_blob[2], rederived[2], rtol=1e-4, atol=1e-4 * scale)
    # d/d(sigma, gamma, alpha): tile partials summed in double, rows in work-list (atomic) order
    assert torch.isfinite(with_blob[3]).all()
    assert torch.allclose(with_blob[3], rederived[3], rtol=1e-5, atol=0.0)


@pytest.mark.parametrize("kind", ["rasterised", "dense"])
def test_forward_from_fallback_records_is_bit_identical(kind):
    from pertrenderer_b200 import ops
    pr = _problem(kind, False)
    image, saved = ops.shade_forward(pr)
    n_fallback = int(saved.worklist[0].item())
    assert n_fallback > 0
    image0, saved0 = _forward_without_blob(pr)
    assert int(saved0.worklist[0].item()) == n_fallback
    valid = pr.pix_to_face >= 0
    assert torch.equal(image, image0)
    assert torch.equal(saved.pixstate, saved0.pixstate)
    assert torch.equal(saved.winners_full(), saved0.winners_full())
    assert torch.equal(saved.counts[valid], saved0.counts[valid])
    assert torch.equal(saved.rsum[valid], saved0.rsum[valid])
