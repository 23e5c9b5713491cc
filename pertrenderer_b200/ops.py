"""Host-side launchers: torch tensors in, C-ABI calls out (include/pertshade.h).

These functions allocate outputs with torch, fill a ``pert_problem`` and call libpertshade.so on the
current CUDA stream.  They hold no state and do not synchronise.  The reference-facing classes in
smoothrast.py / smoothagg.py / random_rasterizer.py are thin autograd wrappers over them.
"""

from __future__ import annotations

import contextlib
import threading
from dataclasses import dataclass, field
from typing import Optional, Tuple

import torch

from . import _cabi
from ._cabi import (F_CAUCHY, F_GUMBEL, F_NO_SKIP, F_NO_VR, F_PHILOX7, F_UNIFORM, F_PER_SAMPLE_NOISE, F_SKIP_DEAD_NOISE, PH_AGG, PH_BLEND, PH_BWD_FINISH, PH_BWD_SAMPLE, PH_RAST,
                    TEX_ATLAS, TEX_UV, TEX_VERTEX, PertProblem, PertTexture, check, ptr, require_cuda, stream_ptr)

_tls = threading.local()


def draw_seed() -> int:
    """A fresh 63-bit seed from torch's default CPU generator: ``torch.manual_seed`` controls the
    noise exactly as it controls the reference's ``torch.normal`` draws (smoothrast.py:21,
    smoothagg.py:21), without touching the device."""
    return int(torch.randint(0, 2 ** 63 - 1, (), dtype=torch.int64).item())


@contextlib.contextmanager
def explicit_noise(noise_rast=None, noise_agg=None):
    """Feed explicit noise tensors, ``noise_rast`` (S_rast,N,H,W,K) and ``noise_agg``
    (S_agg,N,H,W,K+1), to every perturbed op executed inside the block instead of the in-kernel
    Philox stream.  This is the exact-noise parity mode: with the reference's own draws the kernels
    reproduce the reference's images, indices and gradients."""
    prev = getattr(_tls, "noise", (None, None))
    _tls.noise = (noise_rast, noise_agg)
    try:
        yield
    finally:
        _tls.noise = prev


def current_explicit_noise():
    return getattr(_tls, "noise", (None, None))


@contextlib.contextmanager
def kernel_flags(flags: int):
    """Extra PERT_F_* flags for every op inside the block (e.g. F_NO_SKIP for brute-force audits)."""
    prev = getattr(_tls, "flags", 0)
    _tls.flags = flags
    try:
        yield
    finally:
        _tls.flags = prev


def current_flags() -> int:
    return getattr(_tls, "flags", 0)


@contextlib.contextmanager
def device_seeds(seed_device: Optional[torch.Tensor]):
    """Within the block every fused perturbed op reads its seeds as ``host seed ^ seed_device[i]`` (``pert_problem.
    seed_device``; int64 (2,) on the device: coverage stage, aggregation stage).  Inside a captured CUDA graph the
    host seeds are frozen, so the loop steps the device pair with :func:`seed_advance` (a graph node) and every
    replay draws fresh noise: this is what lets a whole render + backward + optimiser iteration be captured
    (examples/pose_optimisation.py)."""
    prev = getattr(_tls, "seed_device", None)
    _tls.seed_device = seed_device
    try:
        yield
    finally:
        _tls.seed_device = prev


def current_seed_device() -> Optional[torch.Tensor]:
    return getattr(_tls, "seed_device", None)


def refuse_device_seeds(op: str):
    """The stand-alone operators take host seeds only: inside ``device_seeds`` (i.e. a CUDA-graph capture) they would
    replay the same noise for ever.  Fail loudly instead."""
    if current_seed_device() is not None:
        raise RuntimeError(f"{op}: device-side seeds (ops.device_seeds) are implemented for the fused operator pairs "
                           "(GaussianRast + GaussianAgg, ArctanRast + CauchyAgg, GaussianRast_wovr + GaussianAgg_wovr, "
                           "SoftRast + SoftAgg) only; run this pair outside the block")


def _f32c(t):
    return t if (t.dtype == torch.float32 and t.is_contiguous()) else t.to(torch.float32).contiguous()


def depth_plane(v, N, device):
    """znear / zfar as a float32 device vector of length 1 or N.  Accepts python floats
    (smooth_rgb_blend's defaults, random_rasterizer.py:35) and (N,), (N,1,1,1) or 0-dim tensors
    (random_rasterizer.py:172-173)."""
    if torch.is_tensor(v):
        t = v.detach().reshape(-1).to(device=device, dtype=torch.float32).contiguous()
    else:
        t = torch.full((1,), float(v), dtype=torch.float32, device=device)
    if t.numel() not in (1, N):
        raise ValueError(f"znear/zfar must have 1 or N={N} elements, got {t.numel()}")
    return t


@dataclass
class ShadeTexture:
    """A texture the fused kernels sample themselves (``pert_texture``): the colour of entry (n,h,w,k) is computed from
    ``bary[n,h,w,k]`` and a per-face table where the kernels blend it, and no (N,H,W,K,3) colour tensor exists.
    ``kind``: "vert" (``table`` (F,3,3) corner colours), "uv" (``table`` (M,Hm,Wm,3) maps, M = 1 or N, ``face_uvs``
    (F,3,2)) or "atlas" (``table`` (F,R,R,3)).  ``bary`` (N,H,W,K,3) is ``fragments.bary_coords``."""
    kind: str
    bary: torch.Tensor
    table: torch.Tensor
    face_uvs: Optional[torch.Tensor] = None

    _KINDS = {"vert": TEX_VERTEX, "uv": TEX_UV, "atlas": TEX_ATLAS}

    def __post_init__(self):
        if self.kind not in self._KINDS:
            raise ValueError(f"texture kind must be one of {sorted(self._KINDS)}, got {self.kind!r}")
        require_cuda(self.bary, self.table, self.face_uvs)
        self.bary, self.table = _f32c(self.bary.detach()), _f32c(self.table.detach())
        if self.face_uvs is not None:
            self.face_uvs = _f32c(self.face_uvs.detach())
        t = self.table
        if self.kind == "vert" and (t.dim() != 3 or tuple(t.shape[1:]) != (3, 3)):
            raise ValueError("vertex colours must be (F,3,3)")
        if self.kind == "uv" and (t.dim() != 4 or t.shape[3] != 3 or self.face_uvs is None or self.face_uvs.dim() != 3
                                  or tuple(self.face_uvs.shape[1:]) != (3, 2)):
            raise ValueError("a UV texture needs maps (M,Hm,Wm,3) and face_uvs (F,3,2)")
        if self.kind == "atlas" and (t.dim() != 4 or t.shape[1] != t.shape[2] or t.shape[3] != 3):
            raise ValueError("an atlas must be (F,R,R,3)")

    @property
    def num_faces(self) -> int:
        return self.face_uvs.shape[0] if self.kind == "uv" else self.table.shape[0]

    def c_struct(self) -> PertTexture:
        tx = PertTexture()
        tx.kind = self._KINDS[self.kind]
        tx.bary, tx.table = self.bary.data_ptr(), self.table.data_ptr()
        tx.num_faces = self.num_faces
        if self.kind == "uv":
            tx.face_uvs = self.face_uvs.data_ptr()
            tx.map_count, tx.map_h, tx.map_w = self.table.shape[0], self.table.shape[1], self.table.shape[2]
        if self.kind == "atlas":
            tx.atlas_size = self.table.shape[1]
        return tx


@dataclass
class ShadeProblem:
    """Everything a forward/backward pair shares.  Built once per forward call."""
    pix_to_face: torch.Tensor
    zbuf: torch.Tensor
    dists: torch.Tensor
    colors: torch.Tensor
    znear: torch.Tensor
    zfar: torch.Tensor
    background: Tuple[float, float, float]
    sigma: float
    gamma: float
    alpha: float
    eps: float
    S_rast: int
    S_agg: int
    seed_rast: int = 0
    seed_agg: int = 0
    pixel_offset: int = 0
    flags: int = 0
    s_rast: Optional[Tuple[int, int]] = None
    s_agg: Optional[Tuple[int, int]] = None
    noise_rast: Optional[torch.Tensor] = None
    noise_agg: Optional[torch.Tensor] = None
    face_colors: Optional[torch.Tensor] = None  # (F,3): colours gathered through pix_to_face inside the kernels
    seed_device: Optional[torch.Tensor] = None  # int64 (2,) on the device: effective seeds = seed_* ^ seed_device (graphs)
    texture: Optional[ShadeTexture] = None  # sampled inside the kernels (pert_shade_tex_*); colors / face_colors are then None
    _keep: list = field(default_factory=list)

    def __post_init__(self):
        require_cuda(self.pix_to_face, self.zbuf, self.dists, self.colors, self.noise_rast, self.noise_agg,
                     self.face_colors)
        if self.pix_to_face.dim() != 4:
            raise ValueError("pix_to_face must be (N,H,W,K)")
        if self.pix_to_face.dtype != torch.int64:
            self.pix_to_face = self.pix_to_face.to(torch.int64)
        self.pix_to_face = self.pix_to_face.contiguous()
        self.zbuf, self.dists = _f32c(self.zbuf.detach()), _f32c(self.dists.detach())
        self.colors = _f32c(self.colors.detach()) if self.colors is not None else None
        N, H, W, K = self.pix_to_face.shape
        if tuple(self.zbuf.shape) != (N, H, W, K) or tuple(self.dists.shape) != (N, H, W, K):
            raise ValueError("zbuf and dists must have the shape of pix_to_face")
        if self.colors is not None and tuple(self.colors.shape) != (N, H, W, K, 3):
            raise ValueError("colors must be (N,H,W,K,3)")
        if self.face_colors is not None:
            self.face_colors = _f32c(self.face_colors.detach())
            if self.face_colors.dim() != 2 or self.face_colors.shape[1] != 3:
                raise ValueError("face_colors must be (F,3)")
        elif self.colors is None and self.texture is None:
            raise ValueError("one of colors (N,H,W,K,3), face_colors (F,3) or texture is required")
        if self.texture is not None:
            if self.colors is not None or self.face_colors is not None:
                raise ValueError("a texture is the only colour source of its problem: colors and face_colors must be None")
            if tuple(self.texture.bary.shape) != (N, H, W, K, 3):
                raise ValueError("the texture's bary must be (N,H,W,K,3)")
        dev = self.pix_to_face.device
        self.znear = depth_plane(self.znear, N, dev)
        self.zfar = depth_plane(self.zfar, N, dev)
        if self.znear.numel() != self.zfar.numel():
            n = max(self.znear.numel(), self.zfar.numel())
            self.znear, self.zfar = self.znear.expand(n).contiguous(), self.zfar.expand(n).contiguous()
        if self.noise_rast is not None:
            self.noise_rast = _f32c(self.noise_rast)
            if tuple(self.noise_rast.shape) != (self.S_rast, N, H, W, K):
                raise ValueError("noise_rast must be (S_rast,N,H,W,K)")
        if self.noise_agg is not None:
            self.noise_agg = _f32c(self.noise_agg)
            if tuple(self.noise_agg.shape) != (self.S_agg, N, H, W, K + 1):
                raise ValueError("noise_agg must be (S_agg,N,H,W,K+1)")
        if self.s_rast is None:
            self.s_rast = (0, self.S_rast)
        if self.s_agg is None:
            self.s_agg = (0, self.S_agg)

    @property
    def shape(self):
        return tuple(self.pix_to_face.shape)

    @property
    def device(self):
        return self.pix_to_face.device

    def c_struct(self, flags=None) -> PertProblem:
        N, H, W, K = self.shape
        pb = PertProblem()
        pb.N, pb.H, pb.W, pb.K = N, H, W, K
        pb.sigma, pb.gamma, pb.alpha, pb.eps = self.sigma, self.gamma, self.alpha, self.eps
        pb.background[0], pb.background[1], pb.background[2] = self.background
        pb.S_rast, pb.S_agg = self.S_rast, self.S_agg
        pb.s_rast_begin, pb.s_rast_end = self.s_rast
        pb.s_agg_begin, pb.s_agg_end = self.s_agg
        pb.seed_rast, pb.seed_agg = self.seed_rast, self.seed_agg
        pb.pixel_offset = self.pixel_offset
        pb.flags = self.flags if flags is None else flags
        pb.depth_len = self.znear.numel()
        pb.pix_to_face, pb.zbuf, pb.dists = self.pix_to_face.data_ptr(), self.zbuf.data_ptr(), self.dists.data_ptr()
        pb.colors = self.colors.data_ptr() if self.colors is not None else None
        pb.znear, pb.zfar = self.znear.data_ptr(), self.zfar.data_ptr()
        pb.noise_rast = self.noise_rast.data_ptr() if self.noise_rast is not None else None
        pb.noise_agg = self.noise_agg.data_ptr() if self.noise_agg is not None else None
        if self.face_colors is not None:
            pb.face_colors, pb.num_faces = self.face_colors.data_ptr(), self.face_colors.shape[0]
        if self.seed_device is not None:
            if self.seed_device.dtype != torch.int64 or self.seed_device.numel() != 2 or not self.seed_device.is_cuda:
                raise ValueError("seed_device must be an int64 CUDA tensor with two elements")
            pb.seed_device = self.seed_device.data_ptr()
        return pb

    def winner_dtype(self):
        return torch.uint8 if self.shape[3] + 1 <= 256 else torch.int16  # int16 storage, read as uint16

    def num_tiles(self) -> int:
        return _geometry(self)[0]

    def blob_bytes(self) -> int:
        return _geometry(self)[1]


_GEOMETRY = {}


def _geometry(pr: "ShadeProblem"):
    """(pert_num_tiles, pert_blob_bytes) of a problem: functions of the shape only, cached per shape (the host side of a
    small problem is a few hundred microseconds: every ctypes call counts)."""
    key = pr.shape
    g = _GEOMETRY.get(key)
    if g is None:
        lib = _cabi.load()
        pb = pr.c_struct()
        g = _GEOMETRY[key] = (int(lib.pert_num_tiles(pb)), int(lib.pert_blob_bytes(pb)))
    return g


@dataclass
class ShadeSaved:
    """State forward leaves for backward.  counts / rsum are defined only where pix_to_face >= 0;
    winners rows only for pixels whose pixstate has the ACTIVE bit (0x8000)."""
    counts: torch.Tensor  # int16 storage of uint16 (N,H,W,K)
    rsum: torch.Tensor  # float (N,H,W,K)
    winners: torch.Tensor  # (N,H,W,S_agg_local) uint8 / int16
    pixstate: torch.Tensor  # int16 storage of uint16 (N,H,W): a0 | 0x8000 * active
    worklist: Optional[torch.Tensor] = None  # int32 (4 + tiles): sparse-first mode work list (see pertshade.h)
    blob: Optional[torch.Tensor] = None  # uint8 (pert_blob_bytes): per-tile valid lists and logit summaries
    hist: Optional[torch.Tensor] = None  # int32 (N,H,W,K1), only when requested

    def winners_full(self) -> torch.Tensor:
        """(N,H,W,S_agg_local) int32 winner of every sample: inactive pixels picked a0 every time."""
        w = self.winners.to(torch.int32)
        if self.winners.dtype == torch.int16:
            w = w & 0xFFFF
        st = self.pixstate.to(torch.int32) & 0xFFFF
        active = (st & 0x8000) != 0
        a0 = (st & 0x7FFF)[..., None].expand_as(w)
        return torch.where(active[..., None], w, a0)


def _sparse_first(pr: ShadeProblem) -> bool:
    """The noise and flags of the sparse-first mode of a single forward call (csrc/cabi.cu sparse_first_ok)."""
    return pr.noise_rast is None and pr.noise_agg is None and \
        not (pr.flags & (F_NO_SKIP | F_PER_SAMPLE_NOISE | F_CAUCHY | F_NO_VR))


def shade_forward(pr: ShadeProblem, want_hist: bool = False, phases: int = 0, saved: Optional[ShadeSaved] = None):
    """Launch pert_shade_fwd.  Returns (image (N,H,W,4), ShadeSaved)."""
    lib = _cabi.load()
    _cabi.require_fused_flags(pr.flags)
    N, H, W, K = pr.shape
    dev = pr.device
    with torch.cuda.device(dev):
        sa_loc = pr.s_agg[1] - pr.s_agg[0]
        if saved is None:
            # phase-split (sample-sharded) jobs all-reduce counts / rsum as whole tensors: define every entry
            alloc = torch.zeros if phases else torch.empty
            # the tile blobs are written by the production path only (in-kernel Gaussian noise, all phases in one call, no
            # global histogram, default noise flags and estimator: csrc/cabi.cu sparse_first_ok); the buffer only exists
            # then, so that a backward with other flags can never read what forward did not write
            prod = not phases and not want_hist and _sparse_first(pr)
            saved = ShadeSaved(
                counts=alloc((N, H, W, K), dtype=torch.int16, device=dev),
                rsum=alloc((N, H, W, K), dtype=torch.float32, device=dev),
                winners=torch.empty((N, H, W, sa_loc), dtype=pr.winner_dtype(), device=dev),
                pixstate=torch.empty((N, H, W), dtype=torch.int16, device=dev),
                worklist=None if phases else torch.empty((4 + pr.num_tiles(),), dtype=torch.int32, device=dev),
                blob=torch.empty((pr.blob_bytes(),), dtype=torch.uint8, device=dev) if prod else None,
                hist=torch.empty((N, H, W, K + 1), dtype=torch.int32, device=dev) if want_hist else None)
        do_blend = (phases == 0) or bool(phases & PH_BLEND)
        image = torch.empty((N, H, W, 4), dtype=torch.float32, device=dev) if do_blend else None
        pb = pr.c_struct(flags=pr.flags | phases)
        args = (ptr(image), ptr(saved.counts), ptr(saved.rsum), ptr(saved.winners), ptr(saved.pixstate), ptr(saved.hist),
                ptr(saved.worklist), ptr(saved.blob), stream_ptr(dev))
        if pr.texture is not None:
            rc = _cabi.shade_tex_fns()[0](pb, pr.texture.c_struct(), *args)
        else:
            rc = lib.pert_shade_fwd(pb, *args)
    check(rc, "pert_shade_tex_fwd" if pr.texture is not None else "pert_shade_fwd")
    return image, saved


def shade_render(pr: ShadeProblem, return_worklist: bool = False):
    """Launch pert_shade_render: the image (N,H,W,4) of :func:`shade_forward` for the same problem, bit for bit, without
    the state backward would need.  Nothing it allocates depends on the sample counts: the sparse-first work list and
    the uint16 (N,H,W,K) counts workspace of its fallback pass (only where that mode runs), and the image.
    ``return_worklist``: return ``(image, worklist)``; word 0 of the work list is the number of tiles the fallback pass
    redid (None where the sparse-first mode does not run)."""
    fn = _cabi.shade_render_fn()
    tex_fn = _cabi.shade_tex_fns()[2] if pr.texture is not None else None
    _cabi.require_fused_flags(pr.flags)
    if pr.s_rast != (0, pr.S_rast) or pr.s_agg != (0, pr.S_agg):
        raise ValueError("shade_render renders all samples in one call: the sample-sharded forward needs shade_forward")
    N, H, W, K = pr.shape
    dev = pr.device
    with torch.cuda.device(dev):
        sparse = _sparse_first(pr)
        worklist = torch.empty((4 + pr.num_tiles(),), dtype=torch.int32, device=dev) if sparse else None
        counts_ws = torch.empty((N, H, W, K), dtype=torch.int16, device=dev) if sparse else None
        image = torch.empty((N, H, W, 4), dtype=torch.float32, device=dev)
        args = (ptr(image), ptr(counts_ws), ptr(worklist), stream_ptr(dev))
        rc = tex_fn(pr.c_struct(), pr.texture.c_struct(), *args) if tex_fn else fn(pr.c_struct(), *args)
    check(rc, "pert_shade_tex_render" if tex_fn else "pert_shade_render")
    return (image, worklist) if return_worklist else image


def shade_render_phase(pr: ShadeProblem, phase: int, counts: torch.Tensor, hist: Optional[torch.Tensor] = None):
    """Launch pert_shade_render_phase: one phase (PH_RAST, PH_AGG or PH_BLEND) of the sample-sharded forward on the shards
    ``pr.s_rast`` / ``pr.s_agg``, without the state backward would need.  ``counts`` int16 storage of uint16 (N,H,W,K): the
    shard's hit counts (PH_RAST writes the valid entries only), then the all-shard counts (PH_AGG, PH_BLEND read them).
    ``hist`` int32 (N,H,W,K+1): PH_AGG writes the shard's winner histogram, PH_BLEND reads the all-shard one.  Returns the
    image (N,H,W,4) for PH_BLEND, else None."""
    fn = _cabi.shade_render_phase_fn()
    require_cuda(counts, hist)
    N, H, W, K = pr.shape
    dev = pr.device
    with torch.cuda.device(dev):
        image = torch.empty((N, H, W, 4), dtype=torch.float32, device=dev) if phase & PH_BLEND else None
        rc = fn(pr.c_struct(flags=pr.flags | phase), ptr(image), ptr(counts), ptr(hist), stream_ptr(dev))
    check(rc, "pert_shade_render_phase")
    return image


def shade_backward(pr: ShadeProblem, saved: ShadeSaved, grad_image: torch.Tensor, need_colors: bool = True,
                   phases: int = 0, acc=None, pixstat=None, use_hist: bool = False, need_bary: bool = False):
    """Launch pert_shade_bwd.  Returns (grad_dists, grad_zbuf, grad_colors | None, grad_scalars(3)).  With ``pr.texture``
    (pert_shade_tex_bwd) the third element is the pair (grad_table | None, grad_bary | None): the gradient of the texture's
    table (``need_colors``) and of its ``bary`` (N,H,W,K,3) (``need_bary``; zero at the entries no sample picked)."""
    lib = _cabi.load()
    _cabi.require_fused_flags(pr.flags)
    N, H, W, K = pr.shape
    dev = pr.device
    require_cuda(grad_image)
    grad_image = _f32c(grad_image)
    with torch.cuda.device(dev):
        finish = (phases == 0) or bool(phases & PH_BWD_FINISH)
        gd = torch.empty((N, H, W, K), dtype=torch.float32, device=dev) if finish else None
        gz = torch.empty((N, H, W, K), dtype=torch.float32, device=dev) if finish else None
        gb = None
        if pr.texture is not None:  # scatter targets of the in-kernel sampling: atomics into zeros
            gc = torch.zeros_like(pr.texture.table) if (finish and need_colors) else None
            gb = torch.zeros_like(pr.texture.bary) if (finish and need_bary) else None
        elif pr.face_colors is not None:  # scatter target of the in-kernel gather: atomics into zeros
            gc = torch.zeros_like(pr.face_colors) if (finish and need_colors) else None
        else:
            gc = torch.empty((N, H, W, K, 3), dtype=torch.float32, device=dev) if (finish and need_colors) else None
        partials = torch.empty((3 * pr.num_tiles(), 4), dtype=torch.float32, device=dev) if finish else None
        scal = torch.empty((3,), dtype=torch.float32, device=dev) if finish else None
        pb = pr.c_struct(flags=pr.flags | phases)
        saved_in = (ptr(grad_image), ptr(saved.counts), ptr(saved.rsum), ptr(saved.winners), ptr(saved.pixstate), ptr(gd), ptr(gz))
        rest = (ptr(partials), ptr(scal), ptr(acc), ptr(pixstat), ptr(saved.hist) if use_hist else None,
                None if phases else ptr(saved.worklist), None if phases else ptr(saved.blob), stream_ptr(dev))
        if pr.texture is not None:
            rc = _cabi.shade_tex_fns()[1](pb, pr.texture.c_struct(), *saved_in, ptr(gc), ptr(gb), *rest)
        else:
            rc = lib.pert_shade_bwd(pb, *saved_in, ptr(gc), *rest)
    check(rc, "pert_shade_tex_bwd" if pr.texture is not None else "pert_shade_bwd")
    return gd, gz, (gc, gb) if pr.texture is not None else gc, scal


# ---------------------------------------------------------------------------------------------
# SoftRas pair (SoftRast + SoftAgg): deterministic fused kernels, nothing saved between the passes
# ---------------------------------------------------------------------------------------------
def soft_shade_forward(pr: ShadeProblem):
    """Launch pert_soft_shade_fwd.  Returns the image (N,H,W,4)."""
    lib = _cabi.load()
    N, H, W, K = pr.shape
    dev = pr.device
    with torch.cuda.device(dev):
        image = torch.empty((N, H, W, 4), dtype=torch.float32, device=dev)
        rc = lib.pert_soft_shade_fwd(pr.c_struct(), ptr(image), stream_ptr(dev))
    check(rc, "pert_soft_shade_fwd")
    return image


def soft_shade_backward(pr: ShadeProblem, grad_image: torch.Tensor, need_colors: bool = True):
    """Launch pert_soft_shade_bwd.  Returns (grad_dists, grad_zbuf, grad_colors | None, grad_scalars(3))."""
    lib = _cabi.load()
    N, H, W, K = pr.shape
    dev = pr.device
    require_cuda(grad_image)
    grad_image = _f32c(grad_image)
    with torch.cuda.device(dev):
        gd = torch.empty((N, H, W, K), dtype=torch.float32, device=dev)
        gz = torch.empty((N, H, W, K), dtype=torch.float32, device=dev)
        gc = torch.empty((N, H, W, K, 3), dtype=torch.float32, device=dev) if need_colors else None
        partials = torch.empty((pr.num_tiles(), 4), dtype=torch.float32, device=dev)
        scal = torch.empty((3,), dtype=torch.float32, device=dev)
        rc = lib.pert_soft_shade_bwd(pr.c_struct(), ptr(grad_image), ptr(gd), ptr(gz), ptr(gc), ptr(partials), ptr(scal),
                                     stream_ptr(dev))
    check(rc, "pert_soft_shade_bwd")
    return gd, gz, gc, scal


# ---------------------------------------------------------------------------------------------
# stand-alone operators
# ---------------------------------------------------------------------------------------------
def rast_forward(x, S, sigma, seed=0, noise=None, pixel_offset=0, flags=0, s_range=None):
    """pert_rast_fwd on x (..., K): returns (prob, rsum)."""
    lib = _cabi.load()
    require_cuda(x, noise)
    x = _f32c(x.detach())
    K = x.shape[-1]
    P = x.numel() // K
    s0, s1 = s_range if s_range is not None else (0, S)
    if noise is not None:
        noise = _f32c(noise)
        if noise.numel() != S * x.numel():
            raise ValueError("noise must be (S,) + x.shape")
    dev = x.device
    with torch.cuda.device(dev):
        prob, rsum = torch.empty_like(x), torch.empty_like(x)
        rc = lib.pert_rast_fwd(ptr(x), P, K, S, s0, s1, float(sigma), seed, pixel_offset, ptr(noise), flags,
                               ptr(prob), ptr(rsum), stream_ptr(dev))
    check(rc, "pert_rast_fwd")
    return prob, rsum


def rast_backward(grad_l, rsum, S, sigma):
    lib = _cabi.load()
    require_cuda(grad_l, rsum)
    grad_l = _f32c(grad_l)
    n = rsum.numel()
    dev = rsum.device
    with torch.cuda.device(dev):
        gx = torch.empty_like(rsum)
        partials = torch.empty(((n + 255) // 256,), dtype=torch.float32, device=dev)
        gs = torch.empty((), dtype=torch.float32, device=dev)
        rc = lib.pert_rast_bwd(ptr(grad_l), ptr(rsum), n, S, float(sigma), ptr(gx), ptr(partials), ptr(gs),
                               stream_ptr(dev))
    check(rc, "pert_rast_bwd")
    return gx, gs


def _winner_dtype_k1(K1):
    return torch.uint8 if K1 <= 256 else torch.int16


def argmax_forward(z, S, gamma, seed=0, noise=None, pixel_offset=0, flags=0, s_range=None):
    """pert_argmax_fwd on logits z (..., K1): returns (weights, winners)."""
    lib = _cabi.load()
    require_cuda(z, noise)
    z = _f32c(z.detach())
    K1 = z.shape[-1]
    P = z.numel() // K1
    s0, s1 = s_range if s_range is not None else (0, S)
    if noise is not None:
        noise = _f32c(noise)
        if noise.numel() != S * z.numel():
            raise ValueError("noise must be (S,) + z.shape")
    dev = z.device
    with torch.cuda.device(dev):
        weights = torch.empty_like(z)
        winners = torch.empty(z.shape[:-1] + (s1 - s0,), dtype=_winner_dtype_k1(K1), device=dev)
        rc = lib.pert_argmax_fwd(ptr(z), P, K1, S, s0, s1, float(gamma), seed, pixel_offset, ptr(noise), flags,
                                 ptr(weights), ptr(winners), stream_ptr(dev))
    check(rc, "pert_argmax_fwd")
    return weights, winners


def argmax_backward(grad_l, z, winners, S, gamma, seed=0, noise=None, pixel_offset=0, flags=0, s_range=None):
    lib = _cabi.load()
    require_cuda(grad_l, z, winners, noise)
    grad_l, z = _f32c(grad_l), _f32c(z.detach())
    K1 = z.shape[-1]
    P = z.numel() // K1
    s0, s1 = s_range if s_range is not None else (0, S)
    if noise is not None:
        noise = _f32c(noise)
    dev = z.device
    with torch.cuda.device(dev):
        gz = torch.empty_like(z)
        partials = torch.empty(((P + 3) // 4,), dtype=torch.float32, device=dev)
        gg = torch.empty((), dtype=torch.float32, device=dev)
        rc = lib.pert_argmax_bwd(ptr(grad_l), ptr(z), ptr(winners), P, K1, S, s0, s1, float(gamma), seed,
                                 pixel_offset, ptr(noise), flags, ptr(gz), ptr(partials), ptr(gg), stream_ptr(dev))
    check(rc, "pert_argmax_bwd")
    return gz, gg


def noise_fill(seed, stage, shape4, S, device, pixel_offset=0, s_range=None):
    """Materialise the counter-based noise of one stage: stage 0 -> (S,N,H,W,K), stage 1 ->
    (S,N,H,W,K+1).  Test aid: the fused kernels never store this tensor."""
    lib = _cabi.load()
    N, H, W, K = shape4
    slots = K if (stage & 1) == 0 else K + 1  # bit 0: stage; higher bits: noise variant (pertshade.h pert_noise_fill)
    s0, s1 = s_range if s_range is not None else (0, S)
    dev = torch.device(device)
    with torch.cuda.device(dev):
        out = torch.empty((s1 - s0, N, H, W, slots), dtype=torch.float32, device=dev)
        rc = lib.pert_noise_fill(seed, stage, N * H * W, slots, s0, s1, pixel_offset, ptr(out), stream_ptr(dev))
    check(rc, "pert_noise_fill")
    return out


# ---------------------------------------------------------------------------------------------
# small problems: forward + backward captured in one CUDA graph
# ---------------------------------------------------------------------------------------------
def seed_advance(seed_device: torch.Tensor):
    """pert_seed_advance: one splitmix64 step of the two device-side seeds (capturable)."""
    lib = _cabi.load()
    require_cuda(seed_device)
    with torch.cuda.device(seed_device.device):
        rc = lib.pert_seed_advance(ptr(seed_device), stream_ptr(seed_device.device))
    check(rc, "pert_seed_advance")


class GraphedShadeStep:
    """One fused forward + backward of the perturbed shader captured in a CUDA graph, for loops over a FIXED shape where
    launch overhead dominates (BASELINE config 1; the pose optimisation of experiments/eval.py:341-394 at 64x64..128x128).

    The caller keeps writing its inputs into the tensors it passed (``pix_to_face, zbuf, dists, colors, grad_image``:
    they are the graph's static inputs) and calls :meth:`replay`; the results appear in ``image, grad_dists, grad_zbuf,
    grad_colors, grad_scalars`` (static outputs, overwritten by the next replay).  The noise seeds live on the device
    (``pert_problem.seed_device``) and a ``pert_seed_advance`` node steps them inside the graph, so every replay draws
    fresh noise although all launch parameters are frozen.  sigma / gamma / alpha / the sample counts are frozen too:
    re-capture after ``update_smoothing`` / ``update_nb_samples``."""

    def __init__(self, pix_to_face, zbuf, dists, colors, grad_image, *, sigma, gamma, alpha=1.0, eps=1e-10, S_rast, S_agg,
                 background=(1.0, 1.0, 1.0), znear=1.0, zfar=100.0, seed=None, flags=0, face_colors=None, need_colors=True):
        dev = pix_to_face.device
        require_cuda(pix_to_face, zbuf, dists, colors, grad_image, face_colors)
        s0, s1 = (draw_seed(), draw_seed()) if seed is None else (int(seed), int(seed) ^ 0x9E3779B97F4A7C15 & (2 ** 63 - 1))
        self.seed_device = torch.tensor([s0, s1], dtype=torch.int64, device=dev)
        self.problem = ShadeProblem(pix_to_face=pix_to_face, zbuf=zbuf, dists=dists, colors=colors, face_colors=face_colors,
                                    znear=znear, zfar=zfar, background=tuple(background), sigma=float(sigma), gamma=float(gamma),
                                    alpha=float(alpha), eps=float(eps), S_rast=int(S_rast), S_agg=int(S_agg), seed_rast=0,
                                    seed_agg=0, flags=int(flags), seed_device=self.seed_device)
        if self.problem.zbuf.data_ptr() != zbuf.data_ptr() or self.problem.dists.data_ptr() != dists.data_ptr() or \
                (colors is not None and self.problem.colors.data_ptr() != colors.data_ptr()):
            raise ValueError("GraphedShadeStep needs contiguous float32 inputs (they are the graph's static buffers)")
        self.grad_image = grad_image
        self.need_colors = need_colors

        def run():
            seed_advance(self.seed_device)
            image, saved = shade_forward(self.problem)
            return (image,) + shade_backward(self.problem, saved, self.grad_image, need_colors=self.need_colors)

        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):  # warm-up outside the capture (function attributes, cached device properties)
            for _ in range(2):
                run()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.image, self.grad_dists, self.grad_zbuf, self.grad_colors, self.grad_scalars = run()

    def replay(self):
        self.graph.replay()
        return self.image, self.grad_dists, self.grad_zbuf, self.grad_colors, self.grad_scalars
