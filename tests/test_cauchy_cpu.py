"""The Cauchy-perturbed pair (ArctanRast + CauchyAgg) without a GPU: the Cauchy oracle (cauchy_oracle.py) against the unmodified
reference's own draws and gradients (tests/golden/ops_cauchy.npz), the sample-sharded orchestration driven by the
oracle with Cauchy noise over gloo, and the C ABI's handling of PERT_F_CAUCHY on the fused entry points."""

import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import load_golden, rel_err
import cauchy_oracle as C
from oracle import pert_oracle as O
from pertrenderer_b200 import _cabi, ops
from pertrenderer_b200 import dist as pdist
from test_dist_cpu import OracleStages, _free_port


def test_cauchy_oracle_matches_reference_golden():
    g = load_golden("ops_cauchy")
    prob, h, h0 = O.random_heaviside_fwd(g["x"], g["U"], g["sigma"])
    assert torch.equal(prob, g["prob"])
    gx, gs = C.random_heaviside_bwd(g["grad_l"], h, h0, g["U"], g["sigma"])
    assert rel_err(gx, g["grad_x"]) <= 1e-6
    assert abs(gs.item() - g["grad_sigma"]) <= 1e-5 * abs(g["grad_sigma"])
    w, a_s, a_0 = O.random_argmax_fwd(g["z"], g["V"], g["gamma"])
    assert torch.equal(w, g["weights"])
    gz, gg = C.random_argmax_bwd(g["grad_w"], a_s, a_0, g["V"], g["gamma"])
    assert rel_err(gz, g["grad_z"]) <= 1e-6
    assert abs(gg.item() - g["grad_gamma"]) <= 1e-5 * abs(g["grad_gamma"])
    # the golden has a -inf logit: its gradient is the score sum of its own noise, not zero
    assert (gz[..., 0] != 0).any()
    # the Gaussian score gives other gradients on the same draws
    gz_n, _ = O.random_argmax_bwd(g["grad_w"], a_s, a_0, g["V"], g["gamma"])
    assert rel_err(gz_n, g["grad_z"]) > 1e-3
    # the shard helpers carry the same score: one shard = the whole estimator
    _, rsum = C.rast_shard_sums(-g["x"], g["U"], g["sigma"])
    assert rel_err(rsum / (int(g["S"]) * g["sigma"]) * g["grad_l"], g["grad_x"]) <= 1e-6
    packed = C.argmax_score_sums(g["grad_w"], a_s, a_0, g["V"])
    K1 = g["z"].shape[-1]
    assert rel_err(packed[..., :K1] / (int(g["S"]) * g["gamma"]), g["grad_z"]) <= 1e-6
    ggs = ((packed[..., K1] - packed[..., K1 + 1]) / (int(g["S"]) * g["gamma"])).sum()
    assert abs(ggs.item() - g["grad_gamma"]) <= 1e-5 * abs(g["grad_gamma"])


def cauchy_case(name="small", seed=5):
    """A golden shader geometry with clamped standard Cauchy draws in place of the Gaussian ones."""
    g = load_golden("shade_" + name)
    g["znear_t"], g["zfar_t"] = g["znear"].reshape(-1, 1, 1, 1), g["zfar"].reshape(-1, 1, 1, 1)
    gen = torch.Generator().manual_seed(seed)
    for k in ("U", "V"):
        u = torch.rand(g[k].shape, generator=gen, dtype=torch.float64)
        g[k] = torch.tan(torch.pi * (u - 0.5)).clamp(-1e7, 1e7).float()
    return g


class CauchyOracleStages(OracleStages):
    def rast(self):
        counts, self.rsum_local = C.rast_shard_sums(self.g["dists"], self.U, self.g["sigma"])
        return counts

    def bwd_sample(self, grad_image):
        g = self.g
        grad_w = O._grad_weights(g["colors"], grad_image, g["background"])
        self.packed_shape = tuple(grad_w.shape[:-1]) + (grad_w.shape[-1] + 2,)
        packed = C.argmax_score_sums(grad_w, self.a_s, self.a_0, self.V)
        return torch.cat((packed.flatten(), self.rsum_local.flatten()))


def _cauchy_worker(rank, world, port, case, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.set_num_threads(1)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        g = cauchy_case(case)
        stages = CauchyOracleStages(g, pdist.sample_range(int(g["S_r"]), world, rank),
                                    pdist.sample_range(int(g["S_a"]), world, rank))
        image = pdist.sharded_forward(stages)
        gd, gz, gc, scal = pdist.sharded_backward(stages, g["grad_image"])
        torch.save(dict(image=image, gd=gd, gz=gz, gc=gc, scal=scal), os.path.join(out_dir, f"rank{rank}.pt"))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("case", ["small", "uneven"])
def test_cauchy_sample_sharded_orchestration_gloo_world2(case, tmp_path):
    world = 2
    mp.spawn(_cauchy_worker, args=(world, _free_port(), case, str(tmp_path)), nprocs=world, join=True)
    g = cauchy_case(case)
    st, gr = C.shade_fwd_bwd(g["pix_to_face"], g["zbuf"], g["dists"], g["colors"], g["background"], g["znear_t"],
                             g["zfar_t"], g["sigma"], g["gamma"], g["alpha"], g["eps"], g["U"], g["V"], g["grad_image"])
    outs = [torch.load(tmp_path / f"rank{r}.pt") for r in range(world)]
    for o in outs:
        assert (o["image"] - st.image).abs().max() <= 1e-6
        assert rel_err(o["gd"], gr["dists"]) <= 1e-5
        assert rel_err(o["gz"], gr["zbuf"]) <= 1e-5
        assert rel_err(o["gc"], gr["colors"]) <= 1e-6
        for i, k in enumerate(("sigma", "gamma", "alpha")):
            ref = gr[k].item()
            assert abs(o["scal"][i].item() - ref) <= 2e-5 * max(abs(ref), 1e-12) + 1e-8, k
    for k in ("image", "gd", "gz", "gc", "scal"):
        assert torch.equal(outs[0][k], outs[1][k]), k


def _problem(flags):
    p = _cabi.PertProblem()
    p.N, p.H, p.W, p.K = 1, 4, 4, 4
    p.S_rast = p.S_agg = 8
    p.s_rast_begin, p.s_rast_end, p.s_agg_begin, p.s_agg_end = 0, 8, 0, 8
    p.depth_len = 1
    p.sigma, p.gamma, p.alpha, p.eps = 1e-3, 1e-2, 1.0, 1e-10
    fake = 1 << 20  # aligned, never dereferenced: validation rejects the call before any launch
    p.pix_to_face = p.zbuf = p.dists = p.colors = p.znear = p.zfar = fake
    p.flags = flags
    return p, fake


@pytest.mark.parametrize("other", ["F_PHILOX7", "F_NO_VR", "F_SKIP_DEAD_NOISE", "F_UNIFORM", "F_GUMBEL"])
def test_fused_entry_points_reject_unsupported_cauchy_combinations(other):
    lib = _cabi.load()
    assert lib.pert_version() == _cabi.ABI_VERSION == 15
    p, f = _problem(_cabi.F_CAUCHY | getattr(_cabi, other))
    assert lib.pert_shade_fwd(p, f, f, f, f, f, None, None, None, None) == -3
    assert lib.pert_shade_bwd(p, f, f, f, f, f, f, f, f, f, f, None, None, None, None, None, None) == -3


def test_cauchy_pair_is_a_fused_pair():
    from pertrenderer_b200 import random_rasterizer as rr
    import pertrenderer_b200 as pb
    assert rr._perturbed_pair_flags(pb.ArctanRast(), pb.CauchyAgg()) == _cabi.F_CAUCHY
    assert rr._perturbed_pair_flags(pb.GaussianRast(), pb.GaussianAgg()) == 0
    assert rr._perturbed_pair_flags(pb.GaussianRast(), pb.CauchyAgg()) is None
    with ops.device_seeds(torch.zeros(2, dtype=torch.int64)):
        with pytest.raises(RuntimeError, match="ArctanRast \\+ CauchyAgg"):
            ops.refuse_device_seeds("randomArgmax")
    with pytest.raises(ValueError, match="ArctanRast, CauchyAgg"):
        pdist.smooth_rgb_blend_sample_sharded(None, None, pb.GaussianRast(), pb.CauchyAgg(), pb.BlendParams())
