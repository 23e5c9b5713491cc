"""The shader without control variates (GaussianRast_wovr + GaussianAgg_wovr, PERT_F_NO_VR) in the fused kernels:
explicit noise against the CPU oracle (wovr_oracle.py), empty tiles and images (the gamma term of pixels without any
valid entry), the in-kernel stream against its materialised copy, the fused path against the operator-by-operator
composition it replaces (same seeds, same noise), CUDA-graph capture with device-side seeds, noise-sample shards and the
estimator's statistics.  Tolerances as in test_gpu_parity.py: images 2e-6, gradients 1e-5 (element-wise), scalar
gradients 1e-4 relative; hit counts and winners bit-exact."""

import math

import pytest
import torch

import wovr_oracle as W
from conftest import elementwise_close, rel_err
from oracle import pert_oracle as O

pytestmark = pytest.mark.gpu

RTOL = 1e-5
DEV = "cuda"


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _scalars_close(got, ref, what, rtol=1e-4):
    assert abs(got - ref) <= rtol * max(abs(ref), 1e-12) + 1e-8, (what, got, ref)


def _run_oracle(g):
    zn, zf = g["znear"].reshape(-1, 1, 1, 1), g["zfar"].reshape(-1, 1, 1, 1)
    return W.shade_fwd_bwd(g["pix_to_face"], g["zbuf"], g["dists"], g["colors"], g["background"], zn, zf, g["sigma"],
                           g["gamma"], g["alpha"], g["eps"], g["U"], g["V"], g["grad_image"])


def _check_against_oracle(g):
    from gpu_util import problem_from_case, run_cuda
    from pertrenderer_b200 import _cabi
    st, gr = _run_oracle(g)
    out = run_cuda(problem_from_case(g, flags=_cabi.F_NO_VR), g["grad_image"])
    mask = g["pix_to_face"] >= 0
    assert torch.equal(out["counts"][mask], st.counts[mask])
    assert torch.equal(out["winners"].permute(3, 0, 1, 2).long(), st.a_s)
    assert (out["image"] - st.image).abs().max() <= 2e-6
    for k in ("colors", "dists", "zbuf"):
        assert elementwise_close(out["grad_" + k], gr[k], RTOL), k
    for i, k in enumerate(("sigma", "gamma", "alpha")):
        _scalars_close(out["scalars"][i].item(), gr[k].item(), k)
    return out, gr


def test_explicit_noise_matches_wovr_oracle_on_golden_geometries(shade_case):
    _check_against_oracle(dict(shade_case))


@pytest.mark.parametrize("shape", [(1, 8, 8, 50, 16, 16), (1, 6, 7, 50, 12, 20), (1, 5, 5, 17, 7, 9), (2, 4, 6, 50, 8, 8)])
def test_explicit_noise_matches_wovr_oracle_synthetic(shape):
    """K = 50 with holes in the mask, S_rast != S_agg, S not a multiple of 4, N > 1 with per-view znear / zfar."""
    from test_gpu_parity import _holey_case
    N, H, W_, K, S_r, S_a = shape
    g = _holey_case(N, H, W_, K, S_r, S_a, seed=3000 + K + S_r)
    g["U"], g["V"] = O.draw_noise((N, H, W_, K), S_r, S_a, generator=torch.Generator().manual_seed(K + S_a))
    _check_against_oracle(g)


def _empty_case(all_empty):
    """16 x 16 pixels whose first eight rows (128 pixels: whole tiles at every tile size) have no valid entry, or an
    image without any."""
    from gpu_util import synthetic_case
    N, H, W_, K, S = 1, 16, 16, 8, 12
    g = synthetic_case(N, H, W_, K, S, S, kind="realistic", seed=17, background=(0.3, 0.6, 0.9))
    rows = H if all_empty else 8
    g["pix_to_face"][:, :rows] = -1
    g["U"], g["V"] = O.draw_noise((N, H, W_, K), S, S, generator=torch.Generator().manual_seed(18))
    return g


@pytest.mark.parametrize("all_empty", [False, True])
def test_empty_tiles_contribute_their_gamma_term(all_empty):
    """Pixels without a valid entry: the background wins every sample, c_s = <G, bg>, and their gamma term
    (1/(S gamma)) sum_s c_s (||V_s||^2 - 1) is not zero (the variance-reduced pair gives exactly 0 there)."""
    from gpu_util import problem_from_case, run_cuda
    g = _empty_case(all_empty)
    out, gr = _check_against_oracle(g)
    assert out["scalars"][1].item() != 0.0
    gauss = run_cuda(problem_from_case(g), g["grad_image"])
    if all_empty:
        assert gauss["scalars"][1].item() == 0.0
        assert (out["grad_dists"] == 0).all() and (out["grad_zbuf"] == 0).all()
    else:
        assert gauss["scalars"][1].item() != out["scalars"][1].item()


@pytest.mark.parametrize("kind", ["realistic", "dense"])
def test_in_kernel_stream_equals_its_materialised_copy(kind):
    """In-kernel Philox noise == the explicit-noise kernels fed with pert_noise_fill (stages 0 and 1).  Bit for bit with
    PERT_F_NO_SKIP (the same entries and logits take part); with the exact skips of the default (entries with
    x < -sigma*Umax, logits that cannot win) integer state, image and colour gradients stay bit for bit and the sums
    differ only in the order of their terms."""
    from gpu_util import problem_from_case, run_cuda, synthetic_case
    from pertrenderer_b200 import _cabi, ops
    N, H, W_, K, S_r, S_a = 2, 10, 10, 50, 16, 24
    g = synthetic_case(N, H, W_, K, S_r, S_a, kind=kind, seed=8)
    seed_r, seed_a = 0x1234567890ABCDEF, 0x0FEDCBA987654321
    g["U"] = ops.noise_fill(seed_r, 0, (N, H, W_, K), S_r, DEV).cpu()
    g["V"] = ops.noise_fill(seed_a, 1, (N, H, W_, K), S_a, DEV).cpu()
    F = _cabi.F_NO_VR
    b = run_cuda(problem_from_case(g, explicit=True, flags=F), g["grad_image"])
    a = run_cuda(problem_from_case(g, explicit=False, seed_rast=seed_r, seed_agg=seed_a, flags=F | _cabi.F_NO_SKIP),
                 g["grad_image"])
    mask = g["pix_to_face"] >= 0
    assert torch.equal(a["counts"][mask], b["counts"][mask])
    for k in ("rsum", "winners", "hist", "image", "grad_dists", "grad_zbuf", "grad_colors", "scalars"):
        assert torch.equal(a[k], b[k]), k
    d = run_cuda(problem_from_case(g, explicit=False, seed_rast=seed_r, seed_agg=seed_a, flags=F), g["grad_image"])
    assert torch.equal(d["counts"][mask], b["counts"][mask])
    for k in ("winners", "hist", "grad_colors"):
        assert torch.equal(d[k], b[k]), k
    assert (d["image"] - b["image"]).abs().max() <= 1e-6
    for k in ("rsum", "grad_dists", "grad_zbuf"):
        assert elementwise_close(d[k], b[k], RTOL), k
    assert torch.allclose(d["scalars"], b["scalars"], rtol=1e-4, atol=1e-6)
    st, gr = _run_oracle(g)
    assert elementwise_close(b["grad_dists"], gr["dists"], RTOL) and elementwise_close(b["grad_zbuf"], gr["zbuf"], RTOL)


def _config2_inputs():
    import types
    import bench
    return bench.rasterised_fragments(types.SimpleNamespace(views=8, image_size=256, faces_per_pixel=50, nb_samples=64), DEV)


def _public_run(blend_fn, fr, colors, G, S, fixed_noise, face, seed=123):
    """One forward + backward through a smooth_rgb_blend-like function; returns every output the caller sees."""
    import pertrenderer_b200 as pb
    rast = pb.GaussianRast_wovr(nb_samples=S, sigma=1e-3)
    agg = pb.GaussianAgg_wovr(nb_samples=S, gamma=1e-2, alpha=1.0, fixed_noise=fixed_noise)
    d, z = fr.dists.clone().requires_grad_(True), fr.zbuf.clone().requires_grad_(True)
    c = colors.clone().requires_grad_(True)
    frag = pb.Fragments(fr.pix_to_face, z, None, d)
    torch.manual_seed(seed)
    img = blend_fn(pb.FaceTexels(c) if face else c, frag, rast, agg, pb.BlendParams(background_color=(0.2, 0.5, 0.8)))
    (img * G).sum().backward()
    return dict(image=img.detach(), dists=d.grad, zbuf=z.grad, colors=c.grad,
                scal=[rast.sigma.grad.item(), agg.gamma.grad.item(), agg.alpha.grad.item()])


@pytest.mark.parametrize("face,fixed_noise", [(False, False), (True, False), (False, True)])
def test_fused_equals_composition_config2_rasterised(face, fixed_noise):
    """BASELINE config 2 (8 x 256^2, K = 50, S = 64) on rasterised fragments: the fused path and the composition draw the
    same seeds in the same order.  Counts and winners bit-exact; image and gradients to rounding."""
    import pertrenderer_b200 as pb
    from pertrenderer_b200 import _cabi, ops
    from pertrenderer_b200.random_rasterizer import _composed_rgb_blend
    from gpu_util import counts_u16
    fr, col = _config2_inputs()
    S = 64
    G = torch.randn(fr.zbuf.shape[:3] + (4,), device=DEV, generator=torch.Generator(device=DEV).manual_seed(3))
    if face:
        colors = torch.rand((int(fr.pix_to_face.max()) + 1, 3), device=DEV, generator=torch.Generator(device=DEV).manual_seed(4))
    else:
        colors = col
    fused = _public_run(pb.smooth_rgb_blend, fr, colors, G, S, fixed_noise, face)
    comp = _public_run(_composed_rgb_blend, fr, colors, G, S, fixed_noise, face)
    assert (fused["image"] - comp["image"]).abs().max().item() <= 2e-6
    for k in ("dists", "zbuf", "colors"):
        assert elementwise_close(fused[k], comp[k], RTOL), k
    for i in range(3):
        _scalars_close(fused["scal"][i], comp["scal"][i], i)
    if face or fixed_noise:
        return
    # the integer state behind both: hit counts of the coverage stage, winners of the argmax stage
    torch.manual_seed(123)
    seed_r, seed_a = ops.draw_seed(), ops.draw_seed()
    mask = fr.pix_to_face >= 0
    prob, _ = ops.rast_forward(-fr.dists, S, 1e-3, seed=seed_r, flags=_cabi.F_NO_VR)
    agg = pb.GaussianAgg_wovr(nb_samples=S, gamma=1e-2, alpha=1.0)
    zeta = agg._logits(fr.zbuf, 100.0, 1.0, prob * mask, mask).detach()
    _, winners = ops.argmax_forward(zeta, S, 1e-2, seed=seed_a, flags=_cabi.F_NO_VR)

    def problem(flags):
        return ops.ShadeProblem(pix_to_face=fr.pix_to_face, zbuf=fr.zbuf, dists=fr.dists, colors=col, znear=1.0,
                                zfar=100.0, background=(0.2, 0.5, 0.8), sigma=1e-3, gamma=1e-2, alpha=1.0, eps=1e-10,
                                S_rast=S, S_agg=S, seed_rast=seed_r, seed_agg=seed_a, flags=flags)

    img_w, saved = ops.shade_forward(problem(_cabi.F_NO_VR))
    assert saved.blob is None  # no sparse-first pass, no tile blob
    assert torch.equal(counts_u16(saved)[mask], (prob * S).round().to(torch.int32)[mask])
    assert torch.equal(saved.winners_full(), winners.to(torch.int32))
    # forward is the Gaussian pair's per-sample path: same counts, winners and image; only the saved score sums differ
    img_g, saved_g = ops.shade_forward(problem(_cabi.F_PER_SAMPLE_NOISE))
    assert torch.equal(img_g, img_w)
    assert torch.equal(counts_u16(saved_g)[mask], counts_u16(saved)[mask])
    assert torch.equal(saved_g.winners_full(), saved.winners_full())
    assert not torch.equal(saved_g.rsum[mask], saved.rsum[mask])


def _cube_scene():
    import os
    import runpy
    import pertrenderer_b200 as pb
    from conftest import ROOT
    ex = runpy.run_path(os.path.join(ROOT, "examples", "pose_optimisation.py"), run_name="pose_example")
    verts, faces, colors = ex["cube_mesh"](DEV)
    R, T = pb.look_at_view_transform(dist=6.7, elev=30.0, azim=120.0, device=DEV)
    cameras = pb.OpenGLPerspectiveCameras(R=R, T=T, fov=60, device=DEV)
    lights = pb.PointLights(location=[[0.0, 2.0, -2.0]], device=DEV)
    return ex, verts, faces, colors, cameras, lights


def test_phong_shader_fused_equals_composition(monkeypatch):
    """RandomPhongShader with the wovr pair (sparse Phong: valid entries only) against the same shader forced onto the
    composition (dense Phong), same seeds."""
    import pertrenderer_b200 as pb
    from pertrenderer_b200 import random_rasterizer as rr
    ex, verts, faces, colors, cameras, lights = _cube_scene()

    def run():
        renderer = ex["make_renderer"]("gaussian_wovr", cameras, lights, 1e-3, 1e-2, 16, 64, DEV)
        v = verts.clone().requires_grad_(True)
        torch.manual_seed(9)
        img = renderer(pb.TriMeshes(v, faces, face_colors=colors))
        img[..., :3].sum().backward()
        return img.detach(), v.grad

    img_f, gv_f = run()
    monkeypatch.setattr(rr, "_perturbed_pair_flags", lambda smoothrast, smoothagg: None)
    img_c, gv_c = run()
    assert (img_f - img_c).abs().max().item() <= 2e-6
    assert rel_err(gv_f, gv_c) <= 1e-4  # through the rasteriser's backward: atomic adds in another order


def test_graph_captured_wovr_step_matches_eager_and_redraws_noise():
    import pertrenderer_b200 as pb
    from pertrenderer_b200 import _cabi, ops
    N, HW, K, S = 1, 64, 50, 16
    fr, col = pb.synthetic_fragments(N, HW, HW, K, kind="realistic", sigma=1e-3, seed=3, device=DEV)
    G = torch.randn((N, HW, HW, 4), device=DEV, generator=torch.Generator(device=DEV).manual_seed(2))
    zbuf, dists, colors = fr.zbuf.clone(), fr.dists.clone(), col.clone()
    kw = dict(sigma=1e-3, gamma=1e-2, alpha=1.0, eps=1e-10, S_rast=S, S_agg=S, background=(1.0, 1.0, 1.0))
    step = ops.GraphedShadeStep(fr.pix_to_face, zbuf, dists, colors, G, seed=99, flags=_cabi.F_NO_VR, **kw)

    def eager(seeds):
        pr = ops.ShadeProblem(pix_to_face=fr.pix_to_face, zbuf=zbuf, dists=dists, colors=colors, znear=1.0, zfar=100.0,
                              seed_rast=int(seeds[0].item()), seed_agg=int(seeds[1].item()), flags=_cabi.F_NO_VR, **kw)
        image, saved = ops.shade_forward(pr)
        return (image,) + ops.shade_backward(pr, saved, G)

    out1 = [t.clone() for t in step.replay()]
    torch.cuda.synchronize()
    for a, b in zip(out1, eager(step.seed_device)):
        assert torch.equal(a, b)
    out2 = [t.clone() for t in step.replay()]
    assert not torch.equal(out1[0], out2[0])  # fresh noise
    for a, b in zip(out2, eager(step.seed_device)):
        assert torch.equal(a, b)


def test_wovr_pose_iteration_captured_in_one_cuda_graph():
    """examples/pose_optimisation.py --graph with the wovr pair: the captured loop runs, stays finite, moves the pose and
    draws fresh noise at every replay."""
    import pertrenderer_b200 as pb
    ex, verts, faces, colors, cameras, lights = _cube_scene()
    torch.manual_seed(0)
    mesh = pb.TriMeshes(verts, faces, face_colors=colors)
    hard = ex["make_renderer"]("hard", cameras, lights, 1e-4, 1e-4, 1, 64, DEV)
    w_true = torch.tensor([0.3, -0.5, 0.2], device=DEV)
    R_true = ex["so3_exp"](w_true)
    with torch.no_grad():
        target = hard(mesh.update_padded(verts @ R_true))[..., :3]
    axis = torch.tensor([0.6, 0.0, 0.8], device=DEV)
    w0 = ex["so3_log"](R_true @ ex["so3_exp"](math.radians(15.0) * axis))

    def run():
        renderer = ex["make_renderer"]("gaussian_wovr", cameras, lights, 1e-3, 1e-2, 16, 64, DEV)
        return ex["optimize_pose_graphed"](mesh, verts, renderer, target, w0, 60, 5e-2)

    w1, w2 = run(), run()
    torch.cuda.synchronize()
    assert torch.isfinite(w1).all() and torch.isfinite(w2).all()
    assert (w1 - w0).abs().max().item() > 1e-3 and (w2 - w0).abs().max().item() > 1e-3
    assert not torch.equal(w1, w2)  # fresh seeds per run and per replay


def test_wovr_sample_shards_reproduce_the_whole_job():
    """Phase-split shards run one after another, exchange buffers summed by hand: integer state exactly, gradients to
    rounding.  Half of the image has no valid entry, so the shards carry the gamma term of empty tiles too."""
    from gpu_util import counts_u16, problem_from_case, run_cuda, synthetic_case
    from pertrenderer_b200 import _cabi, ops
    g = synthetic_case(1, 8, 8, 50, 32, 32, kind="dense", seed=41)
    g["pix_to_face"][:, :4] = -1
    F = _cabi.F_NO_VR
    whole = run_cuda(problem_from_case(g, explicit=False, seed_rast=9, seed_agg=10, flags=F), g["grad_image"])
    R = 2
    prs = [problem_from_case(g, explicit=False, seed_rast=9, seed_agg=10, s_rast=(16 * r, 16 * r + 16),
                             s_agg=(16 * r, 16 * r + 16), flags=F) for r in range(R)]
    saved = [ops.shade_forward(pr, want_hist=True, phases=_cabi.PH_RAST)[1] for pr in prs]
    counts = sum(counts_u16(s) for s in saved)
    rsum = sum(s.rsum for s in saved)
    for s in saved:
        s.counts.copy_(counts.to(torch.int16))
        s.rsum.copy_(rsum)
    for pr, s in zip(prs, saved):
        ops.shade_forward(pr, phases=_cabi.PH_AGG, saved=s)
    hist = sum(s.hist for s in saved)
    for s in saved:
        s.hist.copy_(hist)
    images = [ops.shade_forward(pr, phases=_cabi.PH_BLEND, saved=s)[0] for pr, s in zip(prs, saved)]
    mask = g["pix_to_face"] >= 0
    assert torch.equal(counts.cpu()[mask], whole["counts"][mask])
    assert torch.equal(hist.cpu(), whole["hist"])
    assert torch.equal(torch.cat([s.winners_full() for s in saved], -1).cpu(), whole["winners"])
    for im in images:
        assert (im.cpu() - whole["image"]).abs().max() <= 1e-6
    assert torch.allclose(rsum.cpu()[mask], whole["rsum"][mask], rtol=1e-6, atol=1e-5)
    P, K1 = 64, 51
    gi = g["grad_image"].cuda()
    accs = [torch.empty((P, K1), device=DEV) for _ in range(R)]
    stats = [torch.empty((P, 2), device=DEV) for _ in range(R)]
    for pr, s, a, t in zip(prs, saved, accs, stats):
        ops.shade_backward(pr, s, gi, phases=_cabi.PH_BWD_SAMPLE, acc=a, pixstat=t, use_hist=True)
    acc, stat = sum(accs), sum(stats)
    for pr, s in zip(prs, saved):
        gd, gz, gc, scal = ops.shade_backward(pr, s, gi, phases=_cabi.PH_BWD_FINISH, acc=acc, pixstat=stat, use_hist=True)
        assert rel_err(gd.cpu(), whole["grad_dists"]) <= RTOL
        assert rel_err(gz.cpu(), whole["grad_zbuf"]) <= RTOL
        assert torch.equal(gc.cpu(), whole["grad_colors"])
        assert torch.allclose(scal.cpu(), whole["scalars"], rtol=1e-4, atol=1e-6)


def test_graph_captured_sample_sharded_wovr_step_single_rank(tmp_path):
    """GraphedSampleShardedStep with F_NO_VR on a one-rank NCCL group: every replay equals the unsharded eager job with
    the seeds the replay drew."""
    import torch.distributed as dist
    import pertrenderer_b200 as pb
    from pertrenderer_b200 import _cabi, ops
    from pertrenderer_b200.dist import GraphedSampleShardedStep
    dist.init_process_group("nccl", init_method=f"file://{tmp_path / 'pg'}", rank=0, world_size=1,
                            device_id=torch.device(DEV, 0))
    try:
        N, HW, K, S = 1, 32, 50, 64
        fr, col = pb.synthetic_fragments(N, HW, HW, K, kind="realistic", sigma=1e-3, seed=5, device=DEV)
        G = torch.randn((N, HW, HW, 4), device=DEV, generator=torch.Generator(device=DEV).manual_seed(6))
        kw = dict(sigma=1e-3, gamma=1e-2, alpha=1.0, eps=1e-10, S_rast=S, S_agg=S, background=(1.0, 1.0, 1.0))
        step = GraphedSampleShardedStep(fr.pix_to_face, fr.zbuf, fr.dists, col, G, seed=5, flags=_cabi.F_NO_VR, **kw)
        try:
            for _ in range(2):
                out = [t.clone() for t in step.replay()]
                torch.cuda.synchronize()
                sd = step.seed_device
                pr = ops.ShadeProblem(pix_to_face=fr.pix_to_face, zbuf=fr.zbuf, dists=fr.dists, colors=col, znear=1.0,
                                      zfar=100.0, seed_rast=int(sd[0].item()), seed_agg=int(sd[1].item()),
                                      flags=_cabi.F_NO_VR, **kw)
                image, saved = ops.shade_forward(pr)
                gd, gz, gc, scal = ops.shade_backward(pr, saved, G)
                assert (out[0] - image).abs().max().item() <= 1e-6
                assert rel_err(out[1], gd) <= RTOL and rel_err(out[2], gz) <= RTOL and rel_err(out[3], gc) <= RTOL
                assert torch.allclose(out[4], scal, rtol=1e-4, atol=1e-6)
        finally:
            step.close()
    finally:
        dist.destroy_process_group()


def test_fused_wovr_statistics_over_seeds():
    """Same expectation as the variance-reduced pair, larger spread (the point of the ablation): over 48 seeds, the mean
    of sum(grad_dists) agrees within 6 standard errors, and the per-entry variance of grad_dists is larger."""
    import pertrenderer_b200 as pb
    N, HW, K, S = 1, 32, 8, 16
    fr, col = pb.synthetic_fragments(N, HW, HW, K, kind="realistic", sigma=1e-3, seed=11, device=DEV)
    G = torch.randn((N, HW, HW, 4), device=DEV, generator=torch.Generator(device=DEV).manual_seed(12))
    mask = fr.pix_to_face >= 0

    def grads(rast_cls, agg_cls, seed):
        d = fr.dists.clone().requires_grad_(True)
        torch.manual_seed(seed)
        img = pb.smooth_rgb_blend(col, pb.Fragments(fr.pix_to_face, fr.zbuf, None, d), rast_cls(nb_samples=S, sigma=1e-3),
                                  agg_cls(nb_samples=S, gamma=1e-2, alpha=1.0), pb.BlendParams())
        (img * G).sum().backward()
        return d.grad[mask].double()

    R = 48
    gw = torch.stack([grads(pb.GaussianRast_wovr, pb.GaussianAgg_wovr, s) for s in range(R)])
    gg = torch.stack([grads(pb.GaussianRast, pb.GaussianAgg, 1000 + s) for s in range(R)])
    tw, tg = gw.sum(dim=1), gg.sum(dim=1)
    se = (tw.var() / R + tg.var() / R).sqrt()
    assert abs(tw.mean() - tg.mean()) <= 6 * se
    assert gw.var(dim=0).mean() > 2 * gg.var(dim=0).mean()
