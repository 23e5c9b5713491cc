"""The forward-only render (ops.shade_render, pert_shade_render) against the training forward (ops.shade_forward): the same
image bit for bit on every kernel configuration it runs (Gaussian sparse-first main and fallback passes, Philox-7, the
per-sample path, Cauchy, the pair without control variates, explicit noise, per-face colours, pixel offsets, device
seeds), explicit noise against the CPU oracle, the automatic dispatch of the public API under torch.no_grad, memory that
does not depend on the sample counts, and CUDA-graph capture."""

import types

import pytest
import torch

from oracle import pert_oracle as O

pytestmark = pytest.mark.gpu

DEV = "cuda"
CFG2 = (8, 256, 50, 64)  # BASELINE config 2: views, image size, faces per pixel, samples


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


_FRAGMENTS = {}


def _fragments(kind):
    """Config-2 fragments of one set: synthetic realistic / dense, or an actual rasterisation (bench.py)."""
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


def _problem(fr, col, flags=0, S_rast=64, S_agg=64, seed_rast=1234, seed_agg=5678, **over):
    from pertrenderer_b200 import ops
    kw = dict(pix_to_face=fr.pix_to_face, zbuf=fr.zbuf, dists=fr.dists, colors=col, znear=1.0, zfar=100.0,
              background=(0.2, 0.5, 0.8), sigma=1e-3, gamma=1e-2, alpha=1.0, eps=1e-10, S_rast=S_rast, S_agg=S_agg,
              seed_rast=seed_rast, seed_agg=seed_agg, flags=flags)
    kw.update(over)
    return ops.ShadeProblem(**kw)


FLAGS = ["F_DEFAULT", "F_PHILOX7", "F_PER_SAMPLE_NOISE", "F_CAUCHY", "F_NO_VR"]


def _flag(name):
    from pertrenderer_b200 import _cabi
    return 0 if name == "F_DEFAULT" else getattr(_cabi, name)


@pytest.mark.parametrize("kind", ["realistic", "dense", "rasterised"])
@pytest.mark.parametrize("flag", FLAGS)
def test_render_equals_training_forward_config2(kind, flag):
    from pertrenderer_b200 import ops
    fr, col = _fragments(kind)
    pr = _problem(fr, col, _flag(flag))
    image, saved = ops.shade_forward(pr)
    rendered, worklist = ops.shade_render(pr, return_worklist=True)
    assert torch.equal(rendered, image)
    if flag in ("F_DEFAULT", "F_PHILOX7"):
        # sparse-first mode: the render hands the same tiles to its fallback pass as the training forward
        n = int(worklist[0].item())
        assert n == int(saved.worklist[0].item())
        if kind == "dense":  # the dense set overflows the main pass's tiles
            assert n > 0
    else:
        assert worklist is None


@pytest.mark.parametrize("kind", ["realistic", "dense"])
@pytest.mark.parametrize("flag", FLAGS)
def test_render_face_colors_pixel_offset_device_seeds(kind, flag):
    from pertrenderer_b200 import ops
    fr, _ = _fragments(kind)
    nf = int(fr.pix_to_face.max()) + 1
    fc = torch.rand((nf, 3), device=DEV, generator=torch.Generator(device=DEV).manual_seed(4))
    sd = torch.tensor([0x1234567, 0x7654321], dtype=torch.int64, device=DEV)
    pr = _problem(fr, None, _flag(flag), face_colors=fc, pixel_offset=3 * 256 * 256 + 17, seed_device=sd)
    image, _ = ops.shade_forward(pr)
    assert torch.equal(ops.shade_render(pr), image)
    # the device seeds are mixed in: another pair gives another image
    sd.add_(1)
    assert not torch.equal(ops.shade_render(pr), image)


def test_render_explicit_noise_matches_forward_and_oracle(shade_case):
    from gpu_util import problem_from_case, run_oracle
    from pertrenderer_b200 import ops
    g = shade_case
    pr = problem_from_case(g)
    image, _ = ops.shade_forward(pr)
    rendered = ops.shade_render(pr)
    assert torch.equal(rendered, image)
    st, _ = run_oracle(g, g["U"], g["V"])
    assert (rendered.cpu() - st.image).abs().max().item() <= 2e-6
    # explicit noise in one stage, the in-kernel stream in the other
    for over in (dict(noise_rast=None), dict(noise_agg=None)):
        pr = problem_from_case(g, seed_rast=7, seed_agg=8, **over)
        assert torch.equal(ops.shade_render(pr), ops.shade_forward(pr)[0])


def test_render_explicit_noise_cauchy_and_wovr():
    from gpu_util import problem_from_case, synthetic_case
    from pertrenderer_b200 import _cabi, ops
    g = synthetic_case(1, 12, 10, 50, 16, 20, kind="dense", seed=2)
    gen = torch.Generator().manual_seed(3)
    g["U"] = torch.randn((16, 1, 12, 10, 50), generator=gen)
    g["V"] = torch.randn((20, 1, 12, 10, 51), generator=gen)
    for flags in (_cabi.F_CAUCHY, _cabi.F_NO_VR):
        pr = problem_from_case(g, flags=flags)
        assert torch.equal(ops.shade_render(pr), ops.shade_forward(pr)[0])


# ---- public API: torch.no_grad dispatches to the render, same image, same seeds --------------------------------------
PAIRS = {"gaussian": ("GaussianRast", "GaussianAgg"), "cauchy": ("ArctanRast", "CauchyAgg"),
         "wovr": ("GaussianRast_wovr", "GaussianAgg_wovr")}


def _pair(name, S, fixed_noise):
    import pertrenderer_b200 as pb
    r, a = PAIRS[name]
    return getattr(pb, r)(nb_samples=S, sigma=1e-3), getattr(pb, a)(nb_samples=S, gamma=1e-2, alpha=1.0,
                                                                   fixed_noise=fixed_noise)


@pytest.mark.parametrize("pair", list(PAIRS))
@pytest.mark.parametrize("fixed_noise", [False, True])
def test_smooth_rgb_blend_no_grad_equals_grad_mode(pair, fixed_noise, monkeypatch):
    import pertrenderer_b200 as pb
    from pertrenderer_b200 import ops
    fr, col = pb.synthetic_fragments(2, 64, 64, 50, kind="realistic", sigma=1e-3, seed=1, device=DEV)
    rast, agg = _pair(pair, 32, fixed_noise)
    d, z, c = fr.dists.clone().requires_grad_(True), fr.zbuf.clone().requires_grad_(True), col.clone().requires_grad_(True)
    frag = pb.Fragments(fr.pix_to_face, z, None, d)
    bp = pb.BlendParams(background_color=(0.2, 0.5, 0.8))
    torch.manual_seed(11)
    img = pb.smooth_rgb_blend(c, frag, rast, agg, bp)
    assert img.grad_fn is not None
    after_grad = torch.randint(0, 2 ** 62, ()).item()
    calls = []
    real = ops.shade_render
    monkeypatch.setattr(ops, "shade_render", lambda pr: calls.append(pr) or real(pr))
    for ctx in (torch.no_grad, torch.inference_mode):
        torch.manual_seed(11)
        with ctx():
            out = pb.smooth_rgb_blend(c, frag, rast, agg, bp)
        assert out.grad_fn is None
        assert torch.equal(out, img.detach())
        assert torch.randint(0, 2 ** 62, ()).item() == after_grad  # the generator moved as in grad mode
    assert len(calls) == 2


@pytest.mark.parametrize("pair", list(PAIRS))
def test_shaders_no_grad_equal_grad_mode(pair):
    """RandomSimpleShader (per-face colours) and RandomPhongShader (sparse Phong colours) on a rasterised cube."""
    import os
    import runpy
    import pertrenderer_b200 as pb
    from conftest import ROOT
    ex = runpy.run_path(os.path.join(ROOT, "examples", "pose_optimisation.py"), run_name="pose_example")
    verts, faces, colors = ex["cube_mesh"](DEV)
    R, T = pb.look_at_view_transform(dist=6.7, elev=30.0, azim=120.0, device=DEV)
    cameras = pb.OpenGLPerspectiveCameras(R=R, T=T, fov=60, device=DEV)
    lights = pb.PointLights(location=[[0.0, 2.0, -2.0]], device=DEV)
    phong = ex["make_renderer"](pair if pair != "wovr" else "gaussian_wovr", cameras, lights, 1e-3, 1e-2, 16, 64, DEV)
    rast, agg = _pair(pair, 16, False)
    simple = pb.MeshRenderer(rasterizer=phong.rasterizer,
                             shader=pb.RandomSimpleShader(device=DEV, cameras=cameras, smoothrast=rast, smoothagg=agg,
                                                          blend_params=pb.BlendParams(background_color=(0.0, 0.0, 0.0))))
    for renderer in (phong, simple):
        v = verts.clone().requires_grad_(True)
        mesh = pb.TriMeshes(v, faces, face_colors=colors)
        torch.manual_seed(5)
        img = renderer(mesh)
        assert img.grad_fn is not None
        torch.manual_seed(5)
        with torch.no_grad():
            out = renderer(mesh)
        assert out.grad_fn is None
        assert torch.equal(out, img.detach())
        assert out[..., 3].max().item() > 0  # the cube is in view


# ---- memory ------------------------------------------------------------------------------------------------------------
def _peak_above(fn):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    out = fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base, out


def test_render_memory_does_not_depend_on_samples():
    import pertrenderer_b200 as pb
    from pertrenderer_b200 import ops
    N, HW, K = 2, 256, 50
    fr, col = pb.synthetic_fragments(N, HW, HW, K, kind="realistic", sigma=1e-3, seed=0, device=DEV)
    frag = pb.Fragments(fr.pix_to_face, fr.zbuf, None, fr.dists)
    bp = pb.BlendParams()
    peaks = {}
    for S in (64, 65536):
        rast, agg = _pair("gaussian", 64, False)
        agg.update_nb_samples(S)
        with torch.no_grad():
            peaks[S], img = _peak_above(lambda: pb.smooth_rgb_blend(col, frag, rast, agg, bp))
        assert torch.isfinite(img).all()
        del img
    P = N * HW * HW
    pr = _problem(fr, col, S_agg=64)
    bound = P * 4 * 4 + P * K * 2 + 4 * (4 + pr.num_tiles()) + (1 << 20)  # image, counts workspace, work list, slack
    assert abs(peaks[64] - peaks[65536]) <= 1 << 20, peaks
    assert peaks[65536] <= bound, (peaks, bound)  # the training forward's winners alone would take P * 65536 bytes


def test_render_million_samples_and_alpha_of_counts():
    """S_agg = 2^20 at 1 x 128^2: 16 GiB of winners in a training forward.  The alpha channel depends on the coverage
    counts only: it equals the training forward's at the same S_rast and coverage seed."""
    import pertrenderer_b200 as pb
    from pertrenderer_b200 import ops
    fr, col = pb.synthetic_fragments(1, 128, 128, 50, kind="realistic", sigma=1e-3, seed=2, device=DEV)
    big = _problem(fr, col, S_rast=64, S_agg=1 << 20)
    peak, image = _peak_above(lambda: ops.shade_render(big))
    assert torch.isfinite(image).all()
    assert peak < 64 << 20
    rgb_sum = image[..., :3]
    assert (rgb_sum >= 0).all() and (rgb_sum <= 1.0 + 1e-5).all()
    small_image, _ = ops.shade_forward(_problem(fr, col, S_rast=64, S_agg=64))
    assert torch.equal(image[..., 3], small_image[..., 3])
    assert (small_image[..., 3] > 0).any()


# ---- CUDA graph --------------------------------------------------------------------------------------------------------
def test_render_captured_in_a_cuda_graph_with_device_seeds():
    import pertrenderer_b200 as pb
    from pertrenderer_b200 import ops
    fr, col = pb.synthetic_fragments(1, 96, 96, 50, kind="dense", sigma=1e-3, seed=3, device=DEV)
    sd = torch.tensor([99, 12345], dtype=torch.int64, device=DEV)
    pr = _problem(fr, col, S_rast=16, S_agg=16, seed_rast=0, seed_agg=0, seed_device=sd)

    def run():
        ops.seed_advance(sd)
        return ops.shade_render(pr)

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        run()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static = run()

    def eager():
        s = [int(v) for v in sd.tolist()]
        return ops.shade_render(_problem(fr, col, S_rast=16, S_agg=16, seed_rast=s[0], seed_agg=s[1]))

    graph.replay()
    torch.cuda.synchronize()
    first = static.clone()
    assert torch.equal(first, eager())
    graph.replay()
    torch.cuda.synchronize()
    assert not torch.equal(static, first)  # fresh noise at every replay
    assert torch.equal(static, eager())


def test_no_grad_blend_captured_under_device_seeds(monkeypatch):
    """smooth_rgb_blend under torch.no_grad inside ops.device_seeds, captured with a seed_advance node: the render picks up
    the device seeds, a replay equals the eager no-grad call at the same device seeds, and the next replay differs."""
    import pertrenderer_b200 as pb
    from pertrenderer_b200 import ops
    fr, col = pb.synthetic_fragments(1, 96, 96, 50, kind="dense", sigma=1e-3, seed=4, device=DEV)
    frag = pb.Fragments(fr.pix_to_face, fr.zbuf, None, fr.dists)
    rast, agg = _pair("gaussian", 16, False)
    bp = pb.BlendParams()
    sd = torch.tensor([5, 77], dtype=torch.int64, device=DEV)
    calls = []
    real = ops.shade_render

    def blend():
        with torch.no_grad():
            return pb.smooth_rgb_blend(col, frag, rast, agg, bp)

    def run():
        ops.seed_advance(sd)
        return blend()

    def eager():  # the host seeds the capture froze (torch.manual_seed cannot run inside a capture)
        torch.manual_seed(21)
        return blend()

    monkeypatch.setattr(ops, "shade_render", lambda pr, **kw: calls.append(pr.seed_device is sd) or real(pr, **kw))
    with ops.device_seeds(sd):
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            run()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        torch.manual_seed(21)
        with torch.cuda.graph(graph):
            static = run()
        graph.replay()
        torch.cuda.synchronize()
        first = static.clone()
        assert torch.equal(first, eager())
        graph.replay()
        torch.cuda.synchronize()
        assert not torch.equal(static, first)
        assert torch.equal(static, eager())
    assert calls and all(calls)  # every call went to the render with the device seeds
