"""The pair without control variates (GaussianRast_wovr + GaussianAgg_wovr) without a GPU: the wovr oracle's shard sums
(wovr_oracle.py) against the unmodified reference's own draws and gradients (tests/golden/ops_wovr.npz), the
sample-sharded orchestration driven by the oracle over gloo, the C ABI's handling of PERT_F_NO_VR on the fused entry
points, the operator-pair dispatch and the check that refuses a library whose fused kernels ignore the flag."""

import os
import types

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import load_golden, rel_err
import wovr_oracle as W
from oracle import pert_oracle as O
from pertrenderer_b200 import _cabi, ops
from pertrenderer_b200 import dist as pdist
from test_cauchy_cpu import _problem
from test_dist_cpu import OracleStages, _free_port


def test_wovr_shard_sums_match_reference_golden():
    g = load_golden("ops_wovr")
    S = int(g["S"])
    counts, rsum = W.rast_shard_sums(-g["x"], g["U"], g["sigma"])
    assert torch.equal(counts / S, g["prob"])
    assert rel_err(rsum / (S * g["sigma"]) * g["grad_l"], g["grad_x"]) <= 1e-6
    gs = (rsum / (S * g["sigma"]) * g["grad_l"]).sum()
    assert abs(gs.item() - g["grad_sigma"]) <= 1e-5 * abs(g["grad_sigma"])
    w, a_s, _ = O.random_argmax_fwd(g["z"], g["V"], g["gamma"])
    assert torch.equal(w, g["weights"])
    packed = W.argmax_score_sums(g["grad_w"], a_s, g["V"])
    K1 = g["z"].shape[-1]
    assert rel_err(packed[..., :K1] / (S * g["gamma"]), g["grad_z"]) <= 1e-6
    gg = ((packed[..., K1] - packed[..., K1 + 1]) / (S * g["gamma"])).sum()
    assert abs(gg.item() - g["grad_gamma"]) <= 1e-5 * abs(g["grad_gamma"])
    # the variance-reduced sums differ on the same draws
    assert rel_err(O.argmax_score_sums(g["grad_w"], a_s, torch.max(g["z"], -1).indices, g["V"])[..., :K1], packed[..., :K1]) > 1e-3


def wovr_case(name="small"):
    g = load_golden("shade_" + name)
    g["znear_t"], g["zfar_t"] = g["znear"].reshape(-1, 1, 1, 1), g["zfar"].reshape(-1, 1, 1, 1)
    return g


class WovrOracleStages(OracleStages):
    def rast(self):
        counts, self.rsum_local = W.rast_shard_sums(self.g["dists"], self.U, self.g["sigma"])
        return counts

    def bwd_sample(self, grad_image):
        g = self.g
        grad_w = O._grad_weights(g["colors"], grad_image, g["background"])
        self.packed_shape = tuple(grad_w.shape[:-1]) + (grad_w.shape[-1] + 2,)
        packed = W.argmax_score_sums(grad_w, self.a_s, self.V)
        return torch.cat((packed.flatten(), self.rsum_local.flatten()))


def _wovr_worker(rank, world, port, case, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.set_num_threads(1)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        g = wovr_case(case)
        stages = WovrOracleStages(g, pdist.sample_range(int(g["S_r"]), world, rank),
                                  pdist.sample_range(int(g["S_a"]), world, rank))
        image = pdist.sharded_forward(stages)
        gd, gz, gc, scal = pdist.sharded_backward(stages, g["grad_image"])
        torch.save(dict(image=image, gd=gd, gz=gz, gc=gc, scal=scal), os.path.join(out_dir, f"rank{rank}.pt"))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("case", ["small", "uneven"])
def test_wovr_sample_sharded_orchestration_gloo_world2(case, tmp_path):
    world = 2
    mp.spawn(_wovr_worker, args=(world, _free_port(), case, str(tmp_path)), nprocs=world, join=True)
    g = wovr_case(case)
    st, gr = W.shade_fwd_bwd(g["pix_to_face"], g["zbuf"], g["dists"], g["colors"], g["background"], g["znear_t"],
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


@pytest.mark.parametrize("other", ["F_PHILOX7", "F_SKIP_DEAD_NOISE", "F_UNIFORM", "F_GUMBEL", "F_CAUCHY"])
def test_fused_entry_points_reject_unsupported_no_vr_combinations(other):
    lib = _cabi.load()
    p, f = _problem(_cabi.F_NO_VR | getattr(_cabi, other))
    assert lib.pert_shade_fwd(p, f, f, f, f, f, None, None, None, None) == -3
    assert lib.pert_shade_bwd(p, f, f, f, f, f, f, f, f, f, f, None, None, None, None, None, None) == -3


def test_library_reports_the_fused_estimator_flags():
    _cabi.load()
    _cabi.require_fused_flags(_cabi.F_NO_VR)  # the library built from this tree implements it
    have = _cabi._fused_flags[1]
    assert have & _cabi.F_NO_VR and have & _cabi.F_CAUCHY
    assert not have & (_cabi.F_UNIFORM | _cabi.F_GUMBEL)  # forward-only noises: stand-alone argmax only


def test_wovr_pair_dispatch():
    from pertrenderer_b200 import random_rasterizer as rr
    import pertrenderer_b200 as pb
    assert rr._perturbed_pair_flags(pb.GaussianRast_wovr(), pb.GaussianAgg_wovr()) == _cabi.F_NO_VR
    # mixed pairs stay on the operator-by-operator composition
    assert rr._perturbed_pair_flags(pb.GaussianRast(), pb.GaussianAgg_wovr()) is None
    assert rr._perturbed_pair_flags(pb.GaussianRast_wovr(), pb.GaussianAgg()) is None
    assert rr._fused_pair(pb.GaussianRast_wovr(), pb.GaussianAgg_wovr())
    assert not rr._fused_pair(pb.GaussianRast(), pb.GaussianAgg_wovr())
    with ops.device_seeds(torch.zeros(2, dtype=torch.int64)):
        with pytest.raises(RuntimeError, match="GaussianRast_wovr \\+ GaussianAgg_wovr"):
            ops.refuse_device_seeds("randomArgmax_wovr")
    with pytest.raises(ValueError, match="GaussianRast_wovr, GaussianAgg_wovr"):
        pdist.smooth_rgb_blend_sample_sharded(None, None, pb.GaussianRast(), pb.GaussianAgg_wovr(), pb.BlendParams())


@pytest.mark.parametrize("fake", [types.SimpleNamespace(),
                                  types.SimpleNamespace(pert_shade_fused_flags=lambda: _cabi.F_CAUCHY)])
def test_library_without_fused_no_vr_is_refused(fake, monkeypatch):
    """A library built before the fused pair (no pert_shade_fused_flags, or without the bit) would silently return the
    variance-reduced gradients: the first fused call asks for a rebuild instead.  Other flags never consult it."""
    monkeypatch.setattr(_cabi, "_lib", fake)
    monkeypatch.setattr(_cabi, "_fused_flags", None)
    _cabi.require_fused_flags(_cabi.F_CAUCHY | _cabi.F_PER_SAMPLE_NOISE)
    with pytest.raises(_cabi.PertLibraryError, match="rebuild"):
        _cabi.require_fused_flags(_cabi.F_NO_VR)
