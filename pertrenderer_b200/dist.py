"""Multi-GPU partitioning of the perturbed shader (SURVEY.md §8e): one process per GPU.

Batch sharding (BASELINE config 3)
    Pixels are independent, so a batch of views is split over ranks with NO collective on the data
    path; ``pixel_offset`` keeps the Philox counters global, so the union of the shards is bit-
    identical to the single-GPU job.  Only d/d(sigma, gamma, alpha) are summed (3 floats).

Noise-sample sharding (BASELINE config 4: few pixels, thousands of samples)
    Inputs are replicated; rank r draws samples [s0_r, s1_r).  Forward is two-stage and the second
    stage consumes log(mean over ALL samples of stage one) (smoothagg.py:200-201), so there are
    three exchanges per forward+backward, each ONE all-reduce:
        AR1  hit counts + score sums      (2,P,K)    float   after the coverage phase
        AR2  winner histogram             (P,K1)     int32   after the argmax phase
        AR3  score sums of the argmax     (P,K1+2)   float   in backward
    after which every rank finishes identically.  The collective plumbing is torch.distributed
    (NCCL over NVLink on the GPU box, gloo in the CPU tests); the phases are the PERT_PH_* phases of
    the fused kernels.  The orchestration is written against a small ``stages`` interface so that
    the CPU tests can drive it with the oracle while production drives it with the CUDA kernels.
    Without gradients (``torch.no_grad``) the same AR1 / AR2 sequence drives the forward-only phases
    (``pert_shade_render_phase``), which store nothing for backward: no buffer grows with the sample counts.
"""

from __future__ import annotations

from typing import Optional, Tuple

import torch
import torch.distributed as dist
from torch.autograd import Function

# ------------------------------------------------------------------------------------------------
# partitioning
# ------------------------------------------------------------------------------------------------


def batch_range(n_items: int, world: int, rank: int) -> Tuple[int, int]:
    """Contiguous, balanced split of ``n_items`` batch elements: the first ``n % world`` ranks get
    one more."""
    if not (0 <= rank < world):
        raise ValueError("rank out of range")
    base, extra = divmod(n_items, world)
    start = rank * base + min(rank, extra)
    return start, start + base + (1 if rank < extra else 0)


def sample_range(n_samples: int, world: int, rank: int) -> Tuple[int, int]:
    """Contiguous split of the noise samples in whole quads (the kernels draw four samples per
    Philox call, so shard boundaries are multiples of 4).  Ranks past the last quad get an empty
    range."""
    if not (0 <= rank < world):
        raise ValueError("rank out of range")
    quads = (n_samples + 3) // 4
    q0, q1 = batch_range(quads, world, rank)
    return min(4 * q0, n_samples), min(4 * q1, n_samples)


def check_sample_sharding(n_rast: int, n_agg: int, world: int) -> None:
    """Every rank needs at least one quad of each stage's samples.  Raises the same ValueError on every rank."""
    for name, n in (("GaussianRast", n_rast), ("GaussianAgg", n_agg)):
        if (n + 3) // 4 < world:
            raise ValueError(f"{name}.nb_samples = {n} is too small to shard over {world} ranks "
                             "(the kernels draw four samples per Philox call: one quad per rank at least)")


def all_reduce_scalar_grads(tensors, group=None, device=None):
    """Batch sharding: sum the gradients of the 0-dim CPU leaves (sigma, gamma, alpha) over ranks
    with one 3-float all-reduce."""
    grads = [t.grad if t.grad is not None else torch.zeros_like(t) for t in tensors]
    buf = torch.stack([g.detach().float().reshape(()) for g in grads])
    if device is not None:
        buf = buf.to(device)
    dist.all_reduce(buf, group=group)
    buf = buf.cpu()
    for t, v in zip(tensors, buf):
        t.grad = v.to(t.dtype).reshape(t.shape)


# ------------------------------------------------------------------------------------------------
# sample-sharded orchestration
# ------------------------------------------------------------------------------------------------
class CudaStages:
    """The phases of the fused kernels (include/pertshade.h PERT_PH_*) on one rank's sample shard.

    Everything that is exchanged lives in persistent buffers laid out for the collectives, so that no phase packs or
    copies: the hit counts are reduced as int32 (AR1; NCCL has no 16-bit integer type), the winner histogram in place
    (AR2), and ONE flat float buffer holds, back to back, the argmax score sums (P,K1), the two per-pixel sums (P,2) and
    the coverage score sums rsum (P,K) -- the kernels write / read its three regions through separate pointers and AR3
    reduces it in one call (rsum is only needed by the last backward phase, SURVEY.md §8e, so it rides along there
    instead of doubling AR1).

    ``render=True``: the forward-only phases (pert_shade_render_phase), for calls that need no gradient.  They keep only
    the uint16 counts, their int32 all-reduce copy and the histogram, none of which depends on the sample counts; there
    is no backward."""

    def __init__(self, pr, render=False):
        from . import _cabi, ops
        self.ops, self.cabi, self.pr, self.render = ops, _cabi, pr, render
        N, H, W, K = pr.shape
        dev = pr.device
        P, K1 = N * H * W, K + 1
        if render:
            self.saved = ops.ShadeSaved(counts=torch.zeros((N, H, W, K), dtype=torch.int16, device=dev), rsum=None,
                                        winners=None, pixstate=None,
                                        hist=torch.empty((N, H, W, K1), dtype=torch.int32, device=dev))
        else:
            self.flat = torch.zeros((P * K1 + 2 * P + P * K,), dtype=torch.float32, device=dev)
            self.acc = self.flat[:P * K1].view(N, H, W, K1)
            self.pixstat = self.flat[P * K1:P * K1 + 2 * P].view(N, H, W, 2)
            rsum = self.flat[P * K1 + 2 * P:].view(N, H, W, K)
            sa_loc = pr.s_agg[1] - pr.s_agg[0]
            self.saved = ops.ShadeSaved(
                counts=torch.zeros((N, H, W, K), dtype=torch.int16, device=dev), rsum=rsum,
                winners=torch.empty((N, H, W, sa_loc), dtype=pr.winner_dtype(), device=dev),
                pixstate=torch.empty((N, H, W), dtype=torch.int16, device=dev),
                hist=torch.empty((N, H, W, K1), dtype=torch.int32, device=dev))
        self.counts32 = torch.empty((N, H, W, K), dtype=torch.int32, device=dev)

    def _phase(self, phase):
        if self.render:
            return self.ops.shade_render_phase(self.pr, phase, self.saved.counts, self.saved.hist)
        return self.ops.shade_forward(self.pr, phases=phase, saved=self.saved)[0]

    def rast(self):
        # entries the kernel does not touch (padding) must be defined: they are summed over ranks
        self.saved.counts.zero_()
        if not self.render:
            self.saved.rsum.zero_()
        self._phase(self.cabi.PH_RAST)
        # widened in place (no (P,K) int32 temporary): int16 -> int32 sign-extends, the mask restores the uint16 value
        self.counts32.copy_(self.saved.counts).bitwise_and_(0xFFFF)
        return self.counts32

    def agg(self, counts32):
        self.saved.counts.copy_(counts32)  # int32 -> the uint16 bit pattern (S_rast <= 65535)
        self._phase(self.cabi.PH_AGG)
        return self.saved.hist

    def blend(self, hist):
        if hist is not self.saved.hist:
            self.saved.hist.copy_(hist)
        return self._phase(self.cabi.PH_BLEND)

    def bwd_sample(self, grad_image):
        self.ops.shade_backward(self.pr, self.saved, grad_image, phases=self.cabi.PH_BWD_SAMPLE, acc=self.acc,
                                pixstat=self.pixstat, use_hist=True)
        return self.flat  # [acc | pixstat | rsum]: reduced in one call

    def bwd_finish(self, grad_image, flat, need_colors=True):
        if flat is not self.flat:
            self.flat.copy_(flat)
        return self.ops.shade_backward(self.pr, self.saved, grad_image, need_colors=need_colors,
                                       phases=self.cabi.PH_BWD_FINISH, acc=self.acc, pixstat=self.pixstat, use_hist=True)


def sharded_forward(stages, group=None):
    """AR1 and AR2 around the three forward phases.  Returns the image (identical on every rank)."""
    counts = stages.rast()
    dist.all_reduce(counts, group=group)  # exact: integers
    hist = stages.agg(counts)
    dist.all_reduce(hist, group=group)
    return stages.blend(hist)


def sharded_backward(stages, grad_image, group=None, need_colors=True):
    """AR3 between the two backward phases.  Every rank returns the full gradients."""
    packed = stages.bwd_sample(grad_image)
    dist.all_reduce(packed, group=group)
    return stages.bwd_finish(grad_image, packed, need_colors=need_colors)


def _sharded_problem(colors, dists, zbuf, sigma, gamma, alpha, pix_to_face, znear, zfar, cfg):
    """This rank's ShadeProblem of a sample-sharded call: its two seeds (broadcast from rank 0 with ``sync_seeds``) and
    its sample shards.  Shared by the training and the forward-only path, so that the same ``torch.manual_seed`` gives
    the same image with and without gradients."""
    from . import ops
    group = cfg.get("group")
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    dev = pix_to_face.device
    if cfg.get("sync_seeds", False):
        # reproduce the single-GPU sample path: rank 0 draws the two seeds, everyone receives them
        # (one broadcast and one host read per forward)
        seeds = torch.zeros(2, dtype=torch.int64)
        if rank == 0:
            seeds[0] = ops.draw_seed()
            if cfg["fixed_noise"]:
                torch.manual_seed(1)
            seeds[1] = ops.draw_seed()
        seeds = seeds.to(dev)
        dist.broadcast(seeds, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
        seed_r, seed_a = (int(v) for v in seeds.cpu())
    else:
        # every rank draws its own seeds from its own torch generator: the shards own disjoint sample
        # indices, so whatever the seeds are the union is S independent samples (no communication)
        seed_r = ops.draw_seed()
        if cfg["fixed_noise"]:
            torch.manual_seed(1)
        seed_a = ops.draw_seed()
    S_r, S_a = int(cfg["S_rast"]), int(cfg["S_agg"])
    # decided on data every rank has, so that either all ranks raise or none does (a rank that raised alone would
    # leave the others blocked in the first all-reduce)
    check_sample_sharding(S_r, S_a, world)
    sr, sa = sample_range(S_r, world, rank), sample_range(S_a, world, rank)
    return ops.ShadeProblem(
        pix_to_face=pix_to_face, zbuf=zbuf, dists=dists, colors=colors, znear=znear, zfar=zfar,
        background=cfg["background"], sigma=float(sigma), gamma=float(gamma), alpha=float(alpha),
        eps=float(cfg["eps"]), S_rast=S_r, S_agg=S_a, seed_rast=seed_r, seed_agg=seed_a,
        flags=ops.current_flags() | int(cfg.get("flags", 0)), s_rast=sr, s_agg=sa)


class _SampleShardedShade(Function):
    """Autograd wrapper of the sample-sharded shader; same differentiable inputs as the fused
    single-GPU Function (random_rasterizer._PerturbedShade)."""

    @staticmethod
    def forward(ctx, colors, dists, zbuf, sigma, gamma, alpha, pix_to_face, znear, zfar, cfg):
        group = cfg.get("group")
        stages = CudaStages(_sharded_problem(colors, dists, zbuf, sigma, gamma, alpha, pix_to_face, znear, zfar, cfg))
        image = sharded_forward(stages, group)
        ctx.stages, ctx.group, ctx.scalars = stages, group, (sigma, gamma, alpha)
        return image

    @staticmethod
    def backward(ctx, grad_image):
        need = ctx.needs_input_grad
        gd, gz, gc, scal = sharded_backward(ctx.stages, grad_image.contiguous(), ctx.group, need_colors=need[0])
        out = [None, None, None]
        if any(need[3:6]):
            host = scal.cpu()
            for i, t in enumerate(ctx.scalars):
                if need[3 + i] and torch.is_tensor(t):
                    out[i] = host[i].to(dtype=t.dtype).reshape(t.shape).to(t.device)
        return (gc if need[0] else None, gd if need[1] else None, gz if need[2] else None,
                out[0], out[1], out[2], None, None, None, None)


def smooth_rgb_blend_sample_sharded(colors, fragments, smoothrast, smoothagg, blend_params, znear=1.0, zfar=100,
                                    group=None, sync_seeds=False) -> torch.Tensor:
    """``smooth_rgb_blend`` with the noise samples split over the ranks of ``group`` (inputs
    replicated on every rank; every rank returns the same image and, after backward, the same
    gradients).  ``sync_seeds=True`` makes rank 0's torch generator drive the noise of every rank, which
    reproduces the single-GPU sample path exactly (one broadcast + host read per call); by default each
    rank seeds its own disjoint sample shard from its own generator."""
    from .random_rasterizer import _background_tuple, _perturbed_pair_flags
    flags = _perturbed_pair_flags(smoothrast, smoothagg)
    if flags is None:
        raise ValueError("sample sharding is implemented for the (GaussianRast, GaussianAgg), (ArctanRast, CauchyAgg) and "
                         "(GaussianRast_wovr, GaussianAgg_wovr) pairs")
    cfg = dict(background=_background_tuple(blend_params), eps=smoothagg.eps, S_rast=smoothrast.nb_samples,
               S_agg=smoothagg.nb_samples, fixed_noise=bool(smoothagg.fixed_noise), group=group, sync_seeds=sync_seeds,
               flags=flags)
    args = (colors, fragments.dists, fragments.zbuf, smoothrast.sigma, smoothagg.gamma, smoothagg.alpha,
            fragments.pix_to_face, znear, zfar, cfg)
    # no gradient wanted: the forward-only phases, whose buffers do not grow with the sample counts.  Decided here:
    # inside Function.forward grad mode is always off
    if not torch.is_grad_enabled():
        return sharded_forward(CudaStages(_sharded_problem(*args), render=True), group)
    return _SampleShardedShade.apply(*args)


class GraphedSampleShardedStep:
    """Noise-sample sharded forward + backward captured in ONE CUDA graph per rank (BASELINE config 4: few pixels,
    thousands of samples): seed advance, the three forward phases, the two backward phases and the three NCCL all-reduces
    between them are graph nodes, so a step costs the kernels and the collectives, not ~1 ms of host orchestration.

    Inputs are replicated: every rank passes the same ``pix_to_face, zbuf, dists, colors, grad_image`` (the graph's static
    buffers; write new values into them between replays).  Rank r draws the samples ``sample_range(S, world, r)``.  The
    noise seeds live on the device, start equal on every rank (broadcast from rank 0 at construction) and are stepped by
    the same ``pert_seed_advance`` node everywhere, so all ranks draw from one stream without exchanging seeds.
    Every rank ends a replay with the same ``image, grad_dists, grad_zbuf, grad_colors, grad_scalars``."""

    def __init__(self, pix_to_face, zbuf, dists, colors, grad_image, *, sigma, gamma, alpha=1.0, eps=1e-10, S_rast, S_agg,
                 background=(1.0, 1.0, 1.0), znear=1.0, zfar=100.0, group=None, seed=None, flags=0, need_colors=True):
        from . import ops
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        dev = pix_to_face.device
        check_sample_sharding(int(S_rast), int(S_agg), world)
        seeds = torch.zeros(2, dtype=torch.int64, device=dev)
        if rank == 0:
            s0 = ops.draw_seed() if seed is None else int(seed)
            seeds.copy_(torch.tensor([s0, (s0 * 0x9E3779B1 + 12345) & (2 ** 62 - 1)], dtype=torch.int64))
        dist.broadcast(seeds, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
        self.seed_device = seeds
        self.group, self.grad_image, self.need_colors = group, grad_image, need_colors
        self.problem = ops.ShadeProblem(
            pix_to_face=pix_to_face, zbuf=zbuf, dists=dists, colors=colors, znear=znear, zfar=zfar, background=tuple(background),
            sigma=float(sigma), gamma=float(gamma), alpha=float(alpha), eps=float(eps), S_rast=int(S_rast), S_agg=int(S_agg),
            seed_rast=0, seed_agg=0, flags=int(flags), s_rast=sample_range(int(S_rast), world, rank),
            s_agg=sample_range(int(S_agg), world, rank), seed_device=self.seed_device)
        self.stages = CudaStages(self.problem)

        def run():
            ops.seed_advance(self.seed_device)
            image = sharded_forward(self.stages, group)
            return (image,) + tuple(sharded_backward(self.stages, self.grad_image, group, need_colors=need_colors))

        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):  # warm-up outside the capture: NCCL communicator, function attributes
            for _ in range(2):
                run()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        dist.barrier(group=group)
        self.graph = torch.cuda.CUDAGraph()
        # thread_local: the NCCL watchdog thread queries events while this thread captures
        with torch.cuda.graph(self.graph, capture_error_mode="thread_local"):
            self.image, self.grad_dists, self.grad_zbuf, self.grad_colors, self.grad_scalars = run()

    def replay(self):
        self.graph.replay()
        return self.image, self.grad_dists, self.grad_zbuf, self.grad_colors, self.grad_scalars

    def close(self):
        """Release the captured graph.  Call before ``destroy_process_group``: tearing the NCCL communicator down while a
        graph that holds its kernels is alive blocks (measured on the GPU box: both ranks stop in
        destroy_process_group)."""
        if getattr(self, "graph", None) is not None:
            torch.cuda.synchronize(self.seed_device.device)
            self.graph.reset()
            self.graph = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
