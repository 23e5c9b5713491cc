"""The phase-split forward-only render (ops.shade_render_phase, pert_shade_render_phase) against the phase-split training
forward (ops.shade_forward with phase bits): W ranks simulated in one process, the all-reduces done with torch between
the phases.  Every shard's counts and histogram and the image are the training ones bit for bit; with per-sample noise
the sums over the shards are the single call's.  Then the public API: smooth_rgb_blend_sample_sharded under no_grad on a
one-rank NCCL group (the grad-mode image bit for bit, memory that does not grow with the sample counts) and on two GPUs."""

import dataclasses
import os
import socket
import types

import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda"
CFG2 = (8, 256, 50, 64)  # BASELINE config 2: views, image size, faces per pixel, samples


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _problem(fr, col, flags=0, S_rast=64, S_agg=64, **over):
    from pertrenderer_b200 import ops
    kw = dict(pix_to_face=fr.pix_to_face, zbuf=fr.zbuf, dists=fr.dists, colors=col, znear=1.0, zfar=100.0,
              background=(0.2, 0.5, 0.8), sigma=1e-3, gamma=1e-2, alpha=1.0, eps=1e-10, S_rast=S_rast, S_agg=S_agg,
              seed_rast=1234, seed_agg=5678, flags=flags)
    kw.update(over)
    return ops.ShadeProblem(**kw)


def _shards(pr, W):
    from pertrenderer_b200.dist import check_sample_sharding, sample_range
    check_sample_sharding(pr.S_rast, pr.S_agg, W)
    return [dataclasses.replace(pr, s_rast=sample_range(pr.S_rast, W, r), s_agg=sample_range(pr.S_agg, W, r))
            for r in range(W)]


def _u16(t):
    return t.to(torch.int32) & 0xFFFF


def _render_sharded(pr, W):
    """The forward-only phases on W simulated ranks: per-shard counts and histograms, their sums, the image."""
    from pertrenderer_b200 import _cabi, ops
    N, H, Wd, K = pr.shape
    shards = _shards(pr, W)
    counts = []
    for p in shards:
        c = torch.zeros((N, H, Wd, K), dtype=torch.int16, device=DEV)
        assert ops.shade_render_phase(p, _cabi.PH_RAST, c) is None
        counts.append(_u16(c))
    csum = sum(counts)
    c16 = csum.to(torch.int16)
    hists = []
    for p in shards:
        h = torch.full((N, H, Wd, K + 1), -7, dtype=torch.int32, device=DEV)  # AGG writes every entry
        ops.shade_render_phase(p, _cabi.PH_AGG, c16, h)
        hists.append(h)
    hsum = sum(hists)
    image = ops.shade_render_phase(shards[0], _cabi.PH_BLEND, c16, hsum)
    if W > 1:  # every rank blends the same image
        assert torch.equal(ops.shade_render_phase(shards[-1], _cabi.PH_BLEND, c16, hsum), image)
    return dict(counts=counts, hists=hists, csum=csum, hsum=hsum, image=image)


def _train_sharded(pr, W):
    """The same with the phase-split training forward (pert_shade_fwd with phase bits)."""
    from pertrenderer_b200 import _cabi, ops
    shards = _shards(pr, W)
    saved = [ops.shade_forward(p, want_hist=True, phases=_cabi.PH_RAST)[1] for p in shards]
    counts = [_u16(s.counts) for s in saved]
    csum = sum(counts)
    hists = []
    for p, s in zip(shards, saved):
        s.counts.copy_(csum)
        ops.shade_forward(p, phases=_cabi.PH_AGG, saved=s)
        hists.append(s.hist.clone())
    hsum = sum(hists)
    saved[0].hist.copy_(hsum)
    image, _ = ops.shade_forward(shards[0], phases=_cabi.PH_BLEND, saved=saved[0])
    return dict(counts=counts, hists=hists, csum=csum, hsum=hsum, image=image)


def _check_against_training(pr, W):
    """Shard by shard: counts at the valid entries, every histogram entry, the image: all bit for bit."""
    ren, tr = _render_sharded(pr, W), _train_sharded(pr, W)
    valid = pr.pix_to_face >= 0
    for r in range(W):
        assert torch.equal(ren["counts"][r][valid], tr["counts"][r][valid]), r
        assert (ren["counts"][r][~valid] == 0).all()  # padding untouched (zeroed by the caller)
        assert torch.equal(ren["hists"][r], tr["hists"][r]), r
    assert torch.equal(ren["image"], tr["image"])
    return ren


# ---- small geometry: every flag, shard count and sample count -------------------------------------------------------
_SMALL = {}


def _small():
    """2 x 45 x 37, K = 50, realistic: 40 % empty pixels, and a partial last tile (3330 pixels, 4-pixel tiles)."""
    if not _SMALL:
        import pertrenderer_b200 as pb
        _SMALL["frag"] = pb.synthetic_fragments(2, 45, 37, 50, kind="realistic", sigma=1e-3, seed=7, device=DEV)
    return _SMALL["frag"]


def _explicit(pr, seed=3):
    gen = torch.Generator(device=DEV).manual_seed(seed)
    N, H, W, K = pr.shape
    return dataclasses.replace(pr, noise_rast=torch.randn((pr.S_rast, N, H, W, K), device=DEV, generator=gen),
                               noise_agg=torch.randn((pr.S_agg, N, H, W, K + 1), device=DEV, generator=gen))


FLAGS = ["F_DEFAULT", "F_PER_SAMPLE_NOISE", "F_CAUCHY", "F_NO_VR", "explicit"]


def _flagged(fr, col, flag, S, **over):
    from pertrenderer_b200 import _cabi
    if flag == "explicit":
        return _explicit(_problem(fr, col, S_rast=S, S_agg=S, **over))
    return _problem(fr, col, 0 if flag == "F_DEFAULT" else getattr(_cabi, flag), S_rast=S, S_agg=S, **over)


@pytest.mark.parametrize("S", [64, 61])
@pytest.mark.parametrize("W", [1, 2, 3, 8])
@pytest.mark.parametrize("flag", FLAGS)
def test_render_phases_equal_training_phases(flag, W, S):
    from pertrenderer_b200 import ops
    fr, col = _small()
    pr = _flagged(fr, col, flag, S)
    ren = _check_against_training(pr, W)
    if flag in ("F_PER_SAMPLE_NOISE", "explicit"):
        # per-sample noise: a shard draws exactly its samples of the single call's stream
        image, saved = ops.shade_forward(pr, want_hist=True)
        valid = pr.pix_to_face >= 0
        assert torch.equal(ren["csum"][valid], _u16(saved.counts)[valid])
        assert torch.equal(ren["hsum"], saved.hist)
        # the blend sums the all-shard histogram in another order than the on-chip one of the single call
        assert (ren["image"] - ops.shade_render(pr)).abs().max().item() <= 1e-6
        assert torch.equal(ren["image"][..., 3], image[..., 3])


@pytest.mark.parametrize("flag", ["F_DEFAULT", "F_CAUCHY", "explicit"])
def test_render_phases_face_colors_pixel_offset_device_seeds(flag):
    fr, _ = _small()
    nf = int(fr.pix_to_face.max()) + 1
    fc = torch.rand((nf, 3), device=DEV, generator=torch.Generator(device=DEV).manual_seed(4))
    sd = torch.tensor([0x1234567, 0x7654321], dtype=torch.int64, device=DEV)
    pr = _flagged(fr, None, flag, 64, face_colors=fc, pixel_offset=5 * 45 * 37 + 3, seed_device=sd)
    ren = _check_against_training(pr, 3)
    sd.add_(1)
    if flag != "explicit":  # the device seeds are mixed into the in-kernel streams
        assert not torch.equal(_render_sharded(pr, 3)["hsum"], ren["hsum"])


@pytest.mark.parametrize("flag", ["F_DEFAULT", "F_PER_SAMPLE_NOISE", "F_CAUCHY"])
@pytest.mark.parametrize("H,W,K", [(40, 36, 100), (200, 200, 24)])
def test_render_phases_lanes_per_pixel(H, W, K, flag):
    """Dense fragments (every entry valid).  K = 100: 4-pixel tiles, 8 lanes per pixel; K = 24 on 200^2 pixels: 16-pixel
    tiles, 2 lanes per pixel (the instantiation with runtime lanes)."""
    import pertrenderer_b200 as pb
    fr, col = pb.synthetic_fragments(1, H, W, K, kind="dense", sigma=1e-3, seed=9, device=DEV)
    _check_against_training(_flagged(fr, col, flag, 64), 3)


# ---- config 2, the three fragment sets ----------------------------------------------------------------------------
_FRAGMENTS = {}


def _fragments(kind):
    if kind not in _FRAGMENTS:
        import bench
        import pertrenderer_b200 as pb
        N, HW, K, S = CFG2
        if kind == "rasterised":
            _FRAGMENTS[kind] = bench.rasterised_fragments(
                types.SimpleNamespace(views=N, image_size=HW, faces_per_pixel=K, nb_samples=S), DEV)
        else:
            _FRAGMENTS[kind] = pb.synthetic_fragments(N, HW, HW, K, kind=kind, sigma=1e-3, seed=0, device=DEV)
    return _FRAGMENTS[kind]


@pytest.mark.parametrize("kind", ["realistic", "rasterised", "dense"])
def test_render_phases_config2(kind):
    fr, col = _fragments(kind)
    _check_against_training(_problem(fr, col), 4)


def test_render_phases_million_samples_histogram_rows():
    """2 x 64^2, S_agg = 2^20 over 8 shards: every row of the all-shard histogram counts every sample once."""
    import pertrenderer_b200 as pb
    fr, col = pb.synthetic_fragments(2, 64, 64, 50, kind="realistic", sigma=1e-3, seed=2, device=DEV)
    pr = _problem(fr, col, S_rast=64, S_agg=1 << 20)
    ren = _render_sharded(pr, 8)
    assert (ren["hsum"].sum(-1) == 1 << 20).all()
    assert torch.isfinite(ren["image"]).all()


# ---- public API ----------------------------------------------------------------------------------------------------
def _blend_args(fr, col, S_agg, requires_grad=False):
    import pertrenderer_b200 as pb
    d, z, c = fr.dists, fr.zbuf, col
    if requires_grad:
        d, z, c = d.clone().requires_grad_(True), z.clone().requires_grad_(True), c.clone().requires_grad_(True)
    rast = pb.GaussianRast(nb_samples=64, sigma=1e-3)
    agg = pb.GaussianAgg(nb_samples=S_agg, gamma=1e-2, alpha=1.0)
    return c, pb.Fragments(fr.pix_to_face, z, None, d), rast, agg, pb.BlendParams(background_color=(0.2, 0.5, 0.8))


def _peak_above(fn):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    out = fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base, out


def test_public_api_no_grad_one_rank(tmp_path):
    import torch.distributed as dist
    import pertrenderer_b200 as pb
    from pertrenderer_b200 import _cabi, ops
    from pertrenderer_b200.dist import smooth_rgb_blend_sample_sharded
    dist.init_process_group("nccl", init_method=f"file://{tmp_path / 'pg'}", rank=0, world_size=1,
                            device_id=torch.device(DEV, 0))
    try:
        fr, col = pb.synthetic_fragments(2, 64, 64, 50, kind="realistic", sigma=1e-3, seed=1, device=DEV)
        for flags, sync in ((0, False), (_cabi.F_PER_SAMPLE_NOISE, True), (_cabi.F_CAUCHY, False)):
            with ops.kernel_flags(flags & _cabi.F_PER_SAMPLE_NOISE):
                args = _blend_args(fr, col, 64, requires_grad=True)
                if flags & _cabi.F_CAUCHY:
                    args = args[:2] + (pb.ArctanRast(nb_samples=64, sigma=1e-3), pb.CauchyAgg(nb_samples=64, gamma=1e-2)) + args[4:]
                torch.manual_seed(21)
                img = smooth_rgb_blend_sample_sharded(*args, sync_seeds=sync)
                assert img.grad_fn is not None
                after = torch.randint(0, 2 ** 62, ()).item()
                torch.manual_seed(21)
                with torch.no_grad():
                    out = smooth_rgb_blend_sample_sharded(*args, sync_seeds=sync)
                assert out.grad_fn is None
                assert torch.equal(out, img.detach()), hex(flags)
                assert torch.randint(0, 2 ** 62, ()).item() == after  # the generator moved as in grad mode

        # memory: nothing grows with S_agg; below counts + int32 counts + histogram + image + 1 MiB
        N, HW, K = 2, 256, 50
        fr, col = pb.synthetic_fragments(N, HW, HW, K, kind="realistic", sigma=1e-3, seed=0, device=DEV)
        peaks = {}
        for S in (64, 65536):
            args = _blend_args(fr, col, S)
            with torch.no_grad():
                peaks[S], img = _peak_above(lambda: smooth_rgb_blend_sample_sharded(*args))
            assert torch.isfinite(img).all()
            del img
        P = N * HW * HW
        bound = P * K * 2 + P * K * 4 + P * (K + 1) * 4 + P * 16 + (1 << 20)
        assert abs(peaks[64] - peaks[65536]) <= 1 << 20, peaks
        assert peaks[65536] <= bound, (peaks, bound)
    finally:
        dist.destroy_process_group()


# ---- two GPUs --------------------------------------------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _two_gpu_case(dev):
    import pertrenderer_b200 as pb
    fr, col = pb.synthetic_fragments(2, 48, 48, 50, kind="realistic", sigma=1e-3, seed=3, device="cpu")
    return pb.Fragments(fr.pix_to_face.to(dev), fr.zbuf.to(dev), None, fr.dists.to(dev)), col.to(dev)


def _two_gpu_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    from pertrenderer_b200 import _cabi, ops
    from pertrenderer_b200.dist import smooth_rgb_blend_sample_sharded
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        fr, col = _two_gpu_case(dev)
        out = {}
        with ops.kernel_flags(_cabi.F_PER_SAMPLE_NOISE):
            for S in (64, 4096):
                args = _blend_args(fr, col, S, requires_grad=True)
                torch.manual_seed(77)
                grad_img = smooth_rgb_blend_sample_sharded(*args, sync_seeds=True)
                torch.manual_seed(77)
                with torch.no_grad():
                    img = smooth_rgb_blend_sample_sharded(*args, sync_seeds=True)
                out[S] = dict(grad=grad_img.detach().cpu(), nograd=img.cpu())
        torch.save(out, os.path.join(out_dir, f"rank{rank}.pt"))
    finally:
        dist.destroy_process_group()


def test_nccl_render_world2(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least 2 CUDA devices")
    import torch.multiprocessing as mp
    import pertrenderer_b200 as pb
    from pertrenderer_b200 import _cabi, ops
    world = 2
    mp.spawn(_two_gpu_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    outs = [torch.load(tmp_path / f"rank{r}.pt") for r in range(world)]
    fr, col = _two_gpu_case(DEV)
    for S in (64, 4096):
        assert torch.equal(outs[0][S]["nograd"], outs[1][S]["nograd"])  # ranks agree exactly
        assert torch.equal(outs[0][S]["nograd"], outs[0][S]["grad"])
        c, frag, rast, agg, bp = _blend_args(fr, col, S)
        torch.manual_seed(77)
        with ops.kernel_flags(_cabi.F_PER_SAMPLE_NOISE), torch.no_grad():
            whole = pb.smooth_rgb_blend(c, frag, rast, agg, bp).cpu()
        assert (outs[0][S]["nograd"] - whole).abs().max().item() <= 1e-6
