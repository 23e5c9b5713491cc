"""Shader layer — the reference-facing mirror of ``randomras/random_rasterizer.py``.

``smooth_rgb_blend`` (random_rasterizer.py:34-56) and ``RandomSimpleShader`` (:132-191) keep the
reference's signatures, so ``MeshRenderer(rasterizer=..., shader=RandomSimpleShader(...))`` works
unchanged.  With the (GaussianRast, GaussianAgg) pair, the Cauchy pair (ArctanRast, CauchyAgg) and the pair
without control variates (GaussianRast_wovr, GaussianAgg_wovr) the whole chain — coverage sampling, mask, alpha, logits, perturbed argmax, blend, and the score-function
backward — is ONE forward and ONE backward sm_100a kernel (``pert_shade_fwd`` / ``pert_shade_bwd``).  A call made
without gradients (``torch.no_grad`` / ``torch.inference_mode``) renders with ``pert_shade_render`` instead: the same
image, nothing saved for backward, no buffer that grows with the sample counts.  A CUDA ``VertexTexels`` / ``UVTexels`` /
``AtlasTexels`` texture is sampled inside those kernels (``pert_shade_tex_*``): no (N,H,W,K,3) colour tensor is built.
Any other operator pair falls through to the operator-by-operator composition of the reference, where
the perturbed operators still run on their own CUDA kernels.
"""

from __future__ import annotations

import torch
import torch.nn as nn
from torch.autograd import Function

from . import ops
from .smoothagg import CauchyAgg, GaussianAgg, GaussianAgg_wovr, SoftAgg  # noqa: F401
from .smoothrast import ArctanRast, GaussianRast, GaussianRast_wovr, SoftRast
from .structures import AtlasTexels, BlendParams, FaceTexels, UVTexels, VertexTexels


def _background_tuple(blend_params):
    bg = blend_params.background_color
    if torch.is_tensor(bg):
        bg = bg.detach().reshape(-1).tolist()
    bg = tuple(float(v) for v in bg)
    if len(bg) != 3:
        raise ValueError("background_color must have 3 components")
    return bg


def _perturbed_problem(colors, dists, zbuf, sigma, gamma, alpha, pix_to_face, znear, zfar, cfg, texture=None) -> ops.ShadeProblem:
    """The fused kernels' problem for one call of a perturbed pair, with its noise seeds drawn from torch's generator in
    the reference's order: coverage draw first (smoothrast.py:21), then the optional global reseed (smoothagg.py:18-19),
    then the aggregation draw (smoothagg.py:21).  The training forward and the forward-only render both build it here,
    so that the same ``torch.manual_seed`` gives both the same noise.  ``texture`` (an ``ops.ShadeTexture``): the colour
    source the kernels sample themselves; ``colors`` is then None."""
    noise_r, noise_a = ops.current_explicit_noise()
    seed_r = 0 if noise_r is not None else ops.draw_seed()
    if cfg["fixed_noise"]:
        torch.manual_seed(1)
    seed_a = 0 if noise_a is not None else ops.draw_seed()
    face = bool(cfg.get("face_colors", False))  # `colors` is then the (F,3) per-face table
    return ops.ShadeProblem(
        pix_to_face=pix_to_face, zbuf=zbuf, dists=dists, colors=None if face else colors,
        face_colors=colors if face else None, znear=znear, zfar=zfar,
        background=cfg["background"], sigma=float(sigma), gamma=float(gamma), alpha=float(alpha),
        eps=float(cfg["eps"]), S_rast=int(cfg["S_rast"]), S_agg=int(cfg["S_agg"]),
        seed_rast=seed_r, seed_agg=seed_a, pixel_offset=int(cfg.get("pixel_offset", 0)),
        flags=ops.current_flags() | int(cfg.get("flags", 0)), noise_rast=noise_r, noise_agg=noise_a,
        seed_device=None if (noise_r is not None or noise_a is not None) else ops.current_seed_device(), texture=texture)


class _PerturbedShade(Function):
    """Fused GaussianRast -> mask/alpha -> GaussianAgg -> blend (``cfg["flags"]`` = F_CAUCHY: ArctanRast / CauchyAgg;
    F_NO_VR: GaussianRast_wovr / GaussianAgg_wovr).

    Differentiable inputs: colors, dists, zbuf and the three 0-dim scalars sigma, gamma, alpha
    (CPU leaves in the reference: smoothrast.py:116, smoothagg.py:153-154).  Saved for backward:
    uint16 hit counts and float score sums per pixel·face, one winner index per pixel·sample —
    nothing of size (S,N,H,W,K)."""

    @staticmethod
    def forward(ctx, colors, dists, zbuf, sigma, gamma, alpha, pix_to_face, znear, zfar, cfg):
        pr = _perturbed_problem(colors, dists, zbuf, sigma, gamma, alpha, pix_to_face, znear, zfar, cfg)
        image, saved = ops.shade_forward(pr)
        ctx.pr, ctx.saved = pr, saved
        ctx.scalars = (sigma, gamma, alpha)
        # the kernels of backward re-read the inputs through the pointers in ctx.pr: registering the tensors with autograd
        # makes an in-place edit between forward and backward raise instead of silently changing the gradients
        ctx.save_for_backward(colors, dists, zbuf, pix_to_face)
        return image

    @staticmethod
    def backward(ctx, grad_image):
        need = ctx.needs_input_grad
        ctx.saved_tensors  # noqa: B018  (version check of the inputs)
        gd, gz, gc, scal = ops.shade_backward(ctx.pr, ctx.saved, grad_image, need_colors=need[0])
        out_scal = [None, None, None]
        if any(need[3:6]):
            host = scal.cpu()  # one 12-byte read; the reference moves each scalar grad to the CPU leaf
            for i, t in enumerate(ctx.scalars):
                if need[3 + i] and torch.is_tensor(t):
                    out_scal[i] = host[i].to(dtype=t.dtype).reshape(t.shape).to(t.device)
        return (gc if need[0] else None, gd if need[1] else None, gz if need[2] else None,
                out_scal[0], out_scal[1], out_scal[2], None, None, None, None)


class _PerturbedTexShade(Function):
    """:class:`_PerturbedShade` with a texture the fused kernels sample themselves (``pert_shade_tex_fwd`` / ``_bwd``): the
    (N,H,W,K,3) colour tensor and its gradient are never materialised.  Differentiable inputs: the texture's table
    ((F,3,3) vertex colours, (M,Hm,Wm,3) maps or (F,R,R,3) atlas), ``bary`` (fragments.bary_coords), dists, zbuf and the
    three scalars; ``face_uvs`` and ``kind`` are constants."""

    @staticmethod
    def forward(ctx, table, bary, dists, zbuf, sigma, gamma, alpha, pix_to_face, znear, zfar, face_uvs, kind, cfg):
        tex = ops.ShadeTexture(kind=kind, bary=bary, table=table, face_uvs=face_uvs)
        pr = _perturbed_problem(None, dists, zbuf, sigma, gamma, alpha, pix_to_face, znear, zfar, cfg, texture=tex)
        image, saved = ops.shade_forward(pr)
        ctx.pr, ctx.saved = pr, saved
        ctx.scalars = (sigma, gamma, alpha)
        ctx.save_for_backward(table, bary, dists, zbuf, pix_to_face)  # in-place edits before backward raise (see _PerturbedShade)
        return image

    @staticmethod
    def backward(ctx, grad_image):
        need = ctx.needs_input_grad
        ctx.saved_tensors  # noqa: B018
        # an atlas texel is piecewise constant in bary: its gradient is None (zero), nothing is allocated for it
        gd, gz, (gt, gb), scal = ops.shade_backward(ctx.pr, ctx.saved, grad_image, need_colors=need[0],
                                                    need_bary=need[1] and ctx.pr.texture.kind != "atlas")
        out_scal = [None, None, None]
        if any(need[4:7]):
            host = scal.cpu()
            for i, t in enumerate(ctx.scalars):
                if need[4 + i] and torch.is_tensor(t):
                    out_scal[i] = host[i].to(dtype=t.dtype).reshape(t.shape).to(t.device)
        return (gt if need[0] else None, gb if need[1] else None, gd if need[2] else None, gz if need[3] else None,
                out_scal[0], out_scal[1], out_scal[2], None, None, None, None, None, None)


def _fused_texture(colors, fragments):
    """(kind, table, face_uvs) of a lazy texture the fused perturbed kernels can sample themselves, or None (today's
    materialising path): a CUDA VertexTexels / UVTexels / AtlasTexels with fragments.bary_coords."""
    bary = fragments.bary_coords
    if bary is None:
        return None
    if isinstance(colors, VertexTexels):
        kind, table, face_uvs = "vert", colors.face_vert_colors(), None
    elif isinstance(colors, UVTexels):
        kind, table, face_uvs = "uv", colors.maps, colors.face_uvs()
    else:
        kind, table, face_uvs = "atlas", colors.atlas, None
    if not all(t is None or t.is_cuda for t in (table, face_uvs, bary, fragments.pix_to_face)):
        return None
    return kind, table, face_uvs


class _SoftShade(Function):
    """Fused SoftRast -> mask/alpha -> SoftAgg -> blend (the shaders' DEFAULT operator pair;
    smoothrast.py:126-134, smoothagg.py:165-182): one deterministic streaming kernel per pass,
    backward recomputes forward instead of saving it."""

    @staticmethod
    def forward(ctx, colors, dists, zbuf, sigma, gamma, alpha, pix_to_face, znear, zfar, cfg):
        pr = ops.ShadeProblem(
            pix_to_face=pix_to_face, zbuf=zbuf, dists=dists, colors=colors, znear=znear, zfar=zfar,
            background=cfg["background"], sigma=float(sigma), gamma=float(gamma), alpha=float(alpha),
            eps=float(cfg["eps"]), S_rast=4, S_agg=4)
        ctx.pr = pr
        ctx.scalars = (sigma, gamma, alpha)
        ctx.save_for_backward(colors, dists, zbuf, pix_to_face)  # in-place edits before backward raise (see _PerturbedShade)
        return ops.soft_shade_forward(pr)

    @staticmethod
    def backward(ctx, grad_image):
        need = ctx.needs_input_grad
        ctx.saved_tensors  # noqa: B018
        gd, gz, gc, scal = ops.soft_shade_backward(ctx.pr, grad_image, need_colors=need[0])
        out_scal = [None, None, None]
        if any(need[3:6]):
            host = scal.cpu()
            for i, t in enumerate(ctx.scalars):
                if need[3 + i] and torch.is_tensor(t):
                    out_scal[i] = host[i].to(dtype=t.dtype).reshape(t.shape).to(t.device)
        return (gc if need[0] else None, gd if need[1] else None, gz if need[2] else None,
                out_scal[0], out_scal[1], out_scal[2], None, None, None, None)


def _perturbed_pair_flags(smoothrast, smoothagg):
    """PERT_F_* noise flags of the fused perturbed kernels for this operator pair: 0 for (GaussianRast, GaussianAgg),
    F_CAUCHY for (ArctanRast, CauchyAgg), F_NO_VR for (GaussianRast_wovr, GaussianAgg_wovr); None for a pair without
    them (mixed pairs such as GaussianRast + GaussianAgg_wovr run op by op)."""
    if isinstance(smoothrast, GaussianRast) and isinstance(smoothagg, GaussianAgg):
        return 0
    if isinstance(smoothrast, ArctanRast) and isinstance(smoothagg, CauchyAgg):
        return ops.F_CAUCHY
    if isinstance(smoothrast, GaussianRast_wovr) and isinstance(smoothagg, GaussianAgg_wovr):
        return ops.F_NO_VR
    return None


def _fused_pair(smoothrast, smoothagg) -> bool:
    """The pair runs on fused kernels, which read the colours of valid entries only."""
    return _perturbed_pair_flags(smoothrast, smoothagg) is not None or \
        (type(smoothrast) is SoftRast and type(smoothagg) is SoftAgg)


def smooth_rgb_blend(colors, fragments, smoothrast, smoothagg, blend_params, znear: float = 1.0,
                     zfar: float = 100) -> torch.Tensor:
    """random_rasterizer.py:34-56.  Returns the (N,H,W,4) RGBA image.

    ``colors`` (N,H,W,K,3); ``fragments`` with ``pix_to_face`` / ``zbuf`` / ``dists`` (N,H,W,K);
    ``znear`` / ``zfar`` python floats or tensors broadcastable to (N,1,1,1)."""
    flags = _perturbed_pair_flags(smoothrast, smoothagg)
    if isinstance(colors, (VertexTexels, UVTexels, AtlasTexels)):
        tex = _fused_texture(colors, fragments) if flags is not None else None
        if tex is not None:
            # TexturesVertex / TexturesUV / TexturesAtlas with a perturbed pair: the fused kernels sample the texels where
            # they blend them, and scatter the gradient into the table and bary_coords
            ops.require_cuda(fragments.zbuf, fragments.dists)
            kind, table, face_uvs = tex
            cfg = dict(background=_background_tuple(blend_params), eps=smoothagg.eps,
                       S_rast=smoothrast.nb_samples, S_agg=smoothagg.nb_samples,
                       fixed_noise=bool(smoothagg.fixed_noise), flags=flags)
            args = (table, fragments.bary_coords, fragments.dists, fragments.zbuf, smoothrast.sigma, smoothagg.gamma,
                    smoothagg.alpha, fragments.pix_to_face, znear, zfar, face_uvs, kind, cfg)
            if not torch.is_grad_enabled():
                return ops.shade_render(_perturbed_problem(None, *args[2:10], cfg, texture=ops.ShadeTexture(
                    kind=kind, bary=fragments.bary_coords, table=table, face_uvs=face_uvs)))
            return _PerturbedTexShade.apply(*args)
        # otherwise sample the texels with the texture-only mode of the Phong kernel; the fused pairs read colours of
        # valid entries only, so the padded ones need not be written
        from .shading import sample_lazy_textures
        colors = sample_lazy_textures(colors, fragments, sparse=_fused_pair(smoothrast, smoothagg))
    face = isinstance(colors, FaceTexels)
    ops.require_cuda(colors.face_colors if face else colors, fragments.pix_to_face, fragments.zbuf, fragments.dists)
    if flags is not None:
        cfg = dict(background=_background_tuple(blend_params), eps=smoothagg.eps,
                   S_rast=smoothrast.nb_samples, S_agg=smoothagg.nb_samples,
                   fixed_noise=bool(smoothagg.fixed_noise), face_colors=face, flags=flags)
        args = (colors.face_colors if face else colors, fragments.dists, fragments.zbuf, smoothrast.sigma, smoothagg.gamma,
                smoothagg.alpha, fragments.pix_to_face, znear, zfar, cfg)
        # no gradient wanted (torch.no_grad / inference_mode): the forward-only kernels, which store nothing for backward.
        # Decided here: inside Function.forward grad mode is always off
        if not torch.is_grad_enabled():
            return ops.shade_render(_perturbed_problem(*args))
        return _PerturbedShade.apply(*args)

    if type(smoothrast) is SoftRast and type(smoothagg) is SoftAgg and not face:
        cfg = dict(background=_background_tuple(blend_params), eps=smoothagg.eps)
        return _SoftShade.apply(colors, fragments.dists, fragments.zbuf, smoothrast.sigma, smoothagg.gamma,
                                smoothagg.alpha, fragments.pix_to_face, znear, zfar, cfg)
    return _composed_rgb_blend(colors, fragments, smoothrast, smoothagg, blend_params, znear, zfar)


def _composed_rgb_blend(colors, fragments, smoothrast, smoothagg, blend_params, znear=1.0, zfar=100) -> torch.Tensor:
    """random_rasterizer.py:44-56 operator by operator: every pair without fused kernels runs here (e.g. GaussianRast +
    SoftAgg), and for a fused pair it draws the same seeds in the same order, hence the same noise, as the fused path.
    ``colors`` is a (N,H,W,K,3) tensor or a ``FaceTexels``."""
    if isinstance(colors, FaceTexels):
        colors = colors.materialize(fragments.pix_to_face)
    device = fragments.pix_to_face.device
    background = blend_params.background_color
    if not torch.is_tensor(background):
        background = torch.tensor(background, dtype=torch.float32, device=device)
    else:
        background = background.to(device)
    mask = fragments.pix_to_face >= 0
    prob_map = smoothrast.rasterize(fragments.dists) * mask
    transmittance = torch.prod(1.0 - prob_map, dim=-1)
    weights = smoothagg.aggregate(fragments.zbuf, zfar, znear, prob_map, mask)
    rgb = (weights[..., :-1, None] * colors).sum(dim=-2) + weights[..., -1:] * background
    return torch.cat((rgb, (1.0 - transmittance)[..., None]), dim=-1).to(colors.dtype)


def _default_lights_materials(device):
    """The reference builds pytorch3d PointLights / Materials defaults (random_rasterizer.py:145-148);
    they are stored but never read on the Simple path.  pytorch3d is optional here."""
    try:
        from pytorch3d.renderer import Materials, PointLights  # type: ignore
        return PointLights(device=device), Materials(device=device)
    except Exception:
        return None, None


class SimpleShader(nn.Module):
    """random_rasterizer.py:194-203: texels of the closest face, background where the pixel is empty
    (pytorch3d's hard_rgb_blend: RGB of face k = 0, alpha = coverage)."""

    def __init__(self, device="cpu", blend_params=None):
        super().__init__()
        self.blend_params = blend_params if blend_params is not None else BlendParams()

    def forward(self, fragments, meshes, **kwargs) -> torch.Tensor:
        blend_params = kwargs.get("blend_params", self.blend_params)
        texels = meshes.sample_textures(fragments)
        if isinstance(texels, (FaceTexels, VertexTexels, UVTexels, AtlasTexels)):
            from .shading import sample_lazy_textures
            texels = sample_lazy_textures(texels, fragments)
        covered = fragments.pix_to_face[..., 0] >= 0
        bg = torch.as_tensor(blend_params.background_color, dtype=texels.dtype, device=texels.device)
        rgb = torch.where(covered[..., None], texels[..., 0, :], bg.expand_as(texels[..., 0, :]))
        return torch.cat((rgb, covered[..., None].to(texels.dtype)), dim=-1)


class SoftSimpleShader(nn.Module):
    """random_rasterizer.py:205-215: texels blended by pytorch3d's ``softmax_rgb_blend`` with ``blend_params.sigma`` /
    ``.gamma`` (znear = 1, zfar = 100).  That blend is the SoftRast + SoftAgg pair at alpha = 1 (same probability
    sigmoid(-dists/sigma), same weights P exp((z_inv - z_max)/gamma) and background term exp((eps - z_max)/gamma), same
    alpha channel), so it runs on the fused soft kernels; pytorch3d additionally clamps the background term to
    >= 1e-10, a relative difference of at most 1e-10 in the image."""

    def __init__(self, device="cpu", blend_params=None):
        super().__init__()
        self.blend_params = blend_params if blend_params is not None else BlendParams()

    def forward(self, fragments, meshes, **kwargs) -> torch.Tensor:
        blend_params = kwargs.get("blend_params", self.blend_params)
        texels = meshes.sample_textures(fragments)
        return smooth_rgb_blend(texels, fragments, SoftRast(sigma=float(blend_params.sigma)),
                                SoftAgg(gamma=float(blend_params.gamma), alpha=1.0), blend_params,
                                znear=kwargs.get("znear", 1.0), zfar=kwargs.get("zfar", 100.0))


class RandomSimpleShader(nn.Module):
    """random_rasterizer.py:132-191: texels -> smooth_rgb_blend.  Same constructor, ``forward``,
    ``to``, ``get_smoothing``, ``get_nb_samples``, ``update_smoothing``, ``update_nb_samples``."""

    def __init__(self, device="cpu", cameras=None, lights=None, materials=None, smoothrast=SoftRast(),
                 smoothagg=SoftAgg(), blend_params=None):
        super().__init__()
        d_lights, d_materials = (None, None) if (lights is not None and materials is not None) \
            else _default_lights_materials(device)
        self.lights = lights if lights is not None else d_lights
        self.materials = materials if materials is not None else d_materials
        if cameras is None:
            try:  # reference default: a camera 2.7 units away (random_rasterizer.py:152-153)
                from pytorch3d.renderer import OpenGLPerspectiveCameras, look_at_view_transform  # type: ignore
                R, T = look_at_view_transform(dist=2.7, elev=torch.zeros((1)), azim=torch.zeros((1)))
                cameras = OpenGLPerspectiveCameras(device=device, R=R, T=T)
            except Exception:
                from .structures import DepthCameras
                cameras = DepthCameras(znear=1.0, zfar=100.0, n=1, device=device)
        self.cameras = cameras
        self.blend_params = blend_params if blend_params is not None else BlendParams()
        self.smoothrast = smoothrast
        self.smoothagg = smoothagg

    def to(self, device):
        # like the reference (random_rasterizer.py:158-162) this moves the non-Module members and
        # returns None
        self.cameras = None if self.cameras is None else self.cameras.to(device)
        self.materials = None if self.materials is None else self.materials.to(device)
        self.lights = None if self.lights is None else self.lights.to(device)

    def forward(self, fragments, meshes, **kwargs) -> torch.Tensor:
        cameras = kwargs.get("cameras", self.cameras)
        if cameras is None:
            raise ValueError("Cameras must be specified either at initialization "
                             "or in the forward pass of RandomSimpleShader")
        texels = meshes.sample_textures(fragments)
        blend_params = kwargs.get("blend_params", self.blend_params)
        znear = kwargs.get("znear", getattr(cameras, "znear", 1.0))
        zfar = kwargs.get("zfar", getattr(cameras, "zfar", 100.0))
        if torch.is_tensor(znear):
            znear = znear[:, None, None, None]
        if torch.is_tensor(zfar):
            zfar = zfar[:, None, None, None]
        return smooth_rgb_blend(texels, fragments, self.smoothrast, self.smoothagg, blend_params,
                                znear=znear, zfar=zfar)

    def get_smoothing(self):
        return self.smoothrast.sigma, self.smoothagg.gamma, self.smoothagg.alpha

    def get_nb_samples(self):
        return self.smoothagg.nb_samples

    def update_smoothing(self, sigma=4e-4, gamma=4e-2, alpha=1.):
        self.smoothrast.update_smoothing(sigma)
        self.smoothagg.update_smoothing(gamma, alpha)

    def update_nb_samples(self, nb_samples=16):
        self.smoothrast.update_nb_samples(nb_samples)
        self.smoothagg.update_nb_samples(nb_samples)


class RandomPhongShader(RandomSimpleShader):
    """random_rasterizer.py:60-130, the shader experiments/eval.py:170-176 uses: per-pixel Phong lighting of
    every fragment entry (``phong_shading``, kernels ``pert_phong_fwd/bwd``), then ``smooth_rgb_blend``.
    Same constructor, ``forward``, ``to`` and smoothing / sample-count accessors as the reference class."""

    def __init__(self, device="cpu", cameras=None, lights=None, materials=None, smoothrast=SoftRast(),
                 smoothagg=SoftAgg(), blend_params=None):
        from .structures import Materials, PointLights
        super().__init__(device=device, cameras=cameras, lights=lights, materials=materials, smoothrast=smoothrast,
                         smoothagg=smoothagg, blend_params=blend_params)
        if cameras is None:  # the reference keeps None here and fails in forward (random_rasterizer.py:83,95-99)
            self.cameras = None
        if self.lights is None:
            self.lights = PointLights(device=device)
        if self.materials is None:
            self.materials = Materials(device=device)

    def forward(self, fragments, meshes, **kwargs) -> torch.Tensor:
        from .shading import phong_shading
        cameras = kwargs.get("cameras", self.cameras)
        if cameras is None:
            raise ValueError("Cameras must be specified either at initialization "
                             "or in the forward pass of SoftPhongShader")
        texels = meshes.sample_textures(fragments)
        lights = kwargs.get("lights", self.lights)
        materials = kwargs.get("materials", self.materials)
        blend_params = kwargs.get("blend_params", self.blend_params)
        # every consumer below reads colours of valid entries only when the blend is one of the fused pairs
        colors = phong_shading(meshes=meshes, fragments=fragments, texels=texels, lights=lights, cameras=cameras,
                               materials=materials, sparse=_fused_pair(self.smoothrast, self.smoothagg))
        znear = kwargs.get("znear", getattr(cameras, "znear", 1.0))
        zfar = kwargs.get("zfar", getattr(cameras, "zfar", 100.0))
        if torch.is_tensor(znear):
            znear = znear[:, None, None, None]
        if torch.is_tensor(zfar):
            zfar = zfar[:, None, None, None]
        return smooth_rgb_blend(colors, fragments, self.smoothrast, self.smoothagg, blend_params, znear=znear, zfar=zfar)
