#!/usr/bin/env python
"""The sample-sharded render without gradients (smooth_rgb_blend_sample_sharded under torch.no_grad: the forward-only
phases of pert_shade_render_phase, AR1 and AR2 between them) on W GPUs, one process per GPU over NCCL on localhost.

    python tools/time_render_sharded.py [--sets realistic rasterised dense] [--s-agg 4096 65536 1048576]
                                        [--worlds 1 2 4 8] [--steps 5] [--warmup 1] [--out FILE]

BASELINE config 2 (8 x 256^2, K = 50), S_rast = 64.  Per case and rank: device time per call (CUDA events around each
call, which includes both all-reduces; every call bracketed by a barrier and a synchronize, after the warm-up calls;
median over the timed calls, max over ranks), peak memory above the inputs of one call (torch.cuda.max_memory_allocated),
and the max image difference against W = 1 with per-sample noise and synchronised seeds (then every W draws the same
samples and only the summation order of the blend differs).  Where its winners fit in memory, the training sharded
forward (_SampleShardedShade) is timed beside the render under torch.no_grad.  Worlds larger than the number of visible
GPUs are skipped and reported."""

import argparse
import json
import os
import socket
import statistics
import subprocess
import sys
import tempfile
import types

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N, HW, K, S_RAST = 8, 256, 50, 64


def _fragments(kind, dev):
    import bench
    import pertrenderer_b200 as pb
    if kind == "rasterised":
        return bench.rasterised_fragments(types.SimpleNamespace(views=N, image_size=HW, faces_per_pixel=K, nb_samples=S_RAST), dev)
    return pb.synthetic_fragments(N, HW, HW, K, kind=kind, sigma=1e-3, seed=0, device=dev)


def _training_bytes(S_agg, world):
    """What the training sharded forward allocates per rank: winners (uint8, K1 <= 256), the flat backward buffer, the
    counts (uint16 + int32), pixstate and the histogram."""
    P = N * HW * HW
    return P * (-(-S_agg // world)) + P * (2 * K + 3) * 4 + P * K * 6 + P * 2 + P * (K + 1) * 4


def _worker(rank, world, port, args, out_dir):
    import torch.distributed as dist
    import pertrenderer_b200 as pb
    from pertrenderer_b200 import _cabi, ops
    from pertrenderer_b200.dist import _SampleShardedShade, smooth_rgb_blend_sample_sharded
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    total_mem = torch.cuda.get_device_properties(dev).total_memory
    rows = []

    def timed(fn, n):
        times = []
        for _ in range(n):
            dist.barrier()
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn()
            e1.record()
            torch.cuda.synchronize(dev)
            times.append(e0.elapsed_time(e1))
            del out
        return statistics.median(times)

    def peak(fn):
        torch.cuda.synchronize(dev)
        torch.cuda.reset_peak_memory_stats(dev)
        base = torch.cuda.memory_allocated(dev)
        out = fn()
        torch.cuda.synchronize(dev)
        return torch.cuda.max_memory_allocated(dev) - base, out

    try:
        for kind in args.sets:
            fr, col = _fragments(kind, dev)
            frag = pb.Fragments(fr.pix_to_face, fr.zbuf, None, fr.dists)
            bp = pb.BlendParams(background_color=(1.0, 1.0, 1.0))
            for S in args.s_agg:
                rast = pb.GaussianRast(nb_samples=S_RAST, sigma=1e-3)
                agg = pb.GaussianAgg(nb_samples=S, gamma=1e-2)
                n = args.steps if S < (1 << 20) else args.big_steps

                def render():
                    with torch.no_grad():
                        return smooth_rgb_blend_sample_sharded(col, frag, rast, agg, bp)

                for _ in range(args.warmup):
                    render()
                ms = timed(render, n)
                mem, _ = peak(render)
                # the image compared across worlds: per-sample noise, seeds from rank 0's generator
                torch.manual_seed(123)
                with ops.kernel_flags(_cabi.F_PER_SAMPLE_NOISE), torch.no_grad():
                    img = smooth_rgb_blend_sample_sharded(col, frag, rast, agg, bp, sync_seeds=True)
                if rank == 0:
                    torch.save(img.cpu(), os.path.join(out_dir, f"img_{kind}_{S}_{world}.pt"))
                del img
                row = dict(kind=kind, S_agg=S, world=world, rank=rank, render_ms=ms, render_peak=mem, steps=n)
                if _training_bytes(S, world) < 0.6 * total_mem:
                    cfg = dict(background=(1.0, 1.0, 1.0), eps=agg.eps, S_rast=S_RAST, S_agg=S, fixed_noise=False,
                               group=None, sync_seeds=False, flags=0)

                    def train():
                        with torch.no_grad():  # the call as it ran before the forward-only phases existed
                            return _SampleShardedShade.apply(col, fr.dists, fr.zbuf, rast.sigma, agg.gamma, agg.alpha,
                                                             fr.pix_to_face, 1.0, 100.0, cfg)

                    for _ in range(args.warmup):
                        train()
                    row["train_ms"] = timed(train, n)
                    row["train_peak"], _ = peak(train)
                    torch.cuda.empty_cache()
                rows.append(row)
            del fr, col, frag
            torch.cuda.empty_cache()
        with open(os.path.join(out_dir, f"rows_{world}_{rank}.json"), "w") as f:
            json.dump(rows, f)
    finally:
        dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60).stdout.strip().splitlines()
        return q[0] if q else "nvidia-smi: no answer"
    except Exception as e:  # the device name below still identifies the card
        return f"nvidia-smi unavailable ({e.__class__.__name__})"


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--sets", nargs="+", default=["realistic", "rasterised", "dense"])
    ap.add_argument("--s-agg", nargs="+", type=int, default=[4096, 65536, 1 << 20])
    ap.add_argument("--worlds", nargs="+", type=int, default=[1, 2, 4, 8])
    ap.add_argument("--steps", type=int, default=5, help="timed calls per case")
    ap.add_argument("--big-steps", type=int, default=2, help="timed calls per case at S_agg >= 2^20")
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None, help="also write the report here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_render_sharded.py measures on CUDA devices: none is visible")
    import torch.multiprocessing as mp
    ngpu = torch.cuda.device_count()
    lines = [f"# tools/time_render_sharded.py {' '.join(sys.argv[1:])}".rstrip(),
             f"# BASELINE config 2 ({N} x {HW}^2, K = {K}, S_rast = {S_RAST}), smooth_rgb_blend_sample_sharded under "
             "torch.no_grad (forward-only phases, two all-reduces); device ms per call = median of the timed calls, max over "
             "ranks; peak = max over ranks of the memory above the inputs of one call; diff = max |image - image(W=1)| with "
             "per-sample noise and synchronised seeds; training = the sharded training forward under no_grad where its "
             "winners fit",
             f"# {torch.cuda.get_device_name(0)} x {ngpu} visible; nvidia-smi name, power limit: {_card()}"]
    rows, images = [], {}
    with tempfile.TemporaryDirectory() as tmp:
        for world in args.worlds:
            if world > ngpu:
                lines.append(f"# W = {world}: skipped, {ngpu} GPU(s) visible")
                continue
            mp.spawn(_worker, args=(world, _free_port(), args, tmp), nprocs=world, join=True)
            for r in range(world):
                with open(os.path.join(tmp, f"rows_{world}_{r}.json")) as f:
                    rows += json.load(f)
        for kind in args.sets:
            for S in args.s_agg:
                ref_path = os.path.join(tmp, f"img_{kind}_{S}_1.pt")
                ref = torch.load(ref_path) if os.path.exists(ref_path) else None
                for world in args.worlds:
                    rr = [r for r in rows if r["kind"] == kind and r["S_agg"] == S and r["world"] == world]
                    if not rr:
                        continue
                    img = torch.load(os.path.join(tmp, f"img_{kind}_{S}_{world}.pt"))
                    diff = f"{(img - ref).abs().max().item():.1e}" if ref is not None else "n/a"
                    line = (f"{kind:10s} S_agg {S:8d} W {world}  render {max(r['render_ms'] for r in rr):10.3f} ms  "
                            f"peak {max(r['render_peak'] for r in rr) / 2**20:9.1f} MiB  diff vs W=1 {diff}")
                    if all("train_ms" in r for r in rr):
                        line += (f"   training {max(r['train_ms'] for r in rr):10.3f} ms  "
                                 f"peak {max(r['train_peak'] for r in rr) / 2**20:9.1f} MiB")
                    else:
                        line += f"   training: not run, would allocate {_training_bytes(S, world) / 2**30:.0f} GiB per rank"
                    lines.append(line)
    report = "\n".join(lines)
    print(report)
    if args.out:
        with open(args.out, "w") as f:
            f.write(report + "\n")


if __name__ == "__main__":
    main()
