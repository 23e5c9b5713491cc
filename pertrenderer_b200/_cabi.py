"""ctypes binding of the C ABI declared in include/pertshade.h (libpertshade.so, sm_100a).

PyTorch is plumbing here: it owns device memory and streams; every entry point receives raw device
pointers (``tensor.data_ptr()``), sizes and the current CUDA stream handle.  There is no CPU
fallback: if the library is missing or the tensors are not on a CUDA device, calls raise.
"""

from __future__ import annotations

import ctypes as C
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpertshade.so")
ABI_VERSION = 15

# flags (include/pertshade.h)
F_NO_SKIP = 1
F_SKIP_DEAD_NOISE = 2
F_PER_SAMPLE_NOISE = 4
F_CAUCHY = 8
F_NO_VR = 0x400
F_UNIFORM = 0x800
F_GUMBEL = 0x1000
F_PHILOX7 = 0x2000
PH_RAST, PH_AGG, PH_BLEND = 0x10, 0x20, 0x40
PH_BWD_SAMPLE, PH_BWD_FINISH = 0x100, 0x200

EXPORTS = [
    "pert_version", "pert_shade_fused_flags", "pert_strerror", "pert_last_cuda_error", "pert_num_tiles", "pert_winner_bytes", "pert_blob_bytes",
    "pert_shade_fwd", "pert_shade_render", "pert_shade_render_phase", "pert_shade_bwd", "pert_shade_tex_fwd", "pert_shade_tex_bwd", "pert_shade_tex_render", "pert_soft_shade_fwd", "pert_soft_shade_bwd", "pert_rast_fwd", "pert_rast_bwd", "pert_argmax_fwd",
    "pert_argmax_bwd", "pert_noise_fill", "pert_seed_advance", "pert_phong_fwd", "pert_phong_bwd", "pert_phong_atlas_fwd", "pert_phong_atlas_bwd",
    "pert_rasterize_fwd", "pert_rasterize_bwd", "pert_rasterize_num_bins", "pert_rasterize_bin", "pert_rasterize_bin_bounded",
    "pert_rasterize_bin_capacity",
]

RAST_CULL_BACKFACES = 1  # PERT_RAST_CULL_BACKFACES
RAST_BIN_WIDE = 2  # PERT_RAST_BIN_WIDE

TEX_VERTEX, TEX_UV, TEX_ATLAS = 1, 2, 3  # PERT_TEX_* (pert_texture.kind)

PHONG_STRIDE = 20  # PERT_PHONG_STRIDE
PHONG_SPARSE = 1  # PERT_PHONG_SPARSE
PHONG_UNLIT = 2  # PERT_PHONG_UNLIT


class PertProblem(C.Structure):
    """Mirror of ``struct pert_problem``."""
    _fields_ = [
        ("N", C.c_int64), ("H", C.c_int64), ("W", C.c_int64),
        ("K", C.c_int32),
        ("sigma", C.c_float), ("gamma", C.c_float), ("alpha", C.c_float), ("eps", C.c_float),
        ("background", C.c_float * 3),
        ("S_rast", C.c_int32), ("S_agg", C.c_int32),
        ("s_rast_begin", C.c_int32), ("s_rast_end", C.c_int32),
        ("s_agg_begin", C.c_int32), ("s_agg_end", C.c_int32),
        ("seed_rast", C.c_uint64), ("seed_agg", C.c_uint64),
        ("pixel_offset", C.c_int64),
        ("flags", C.c_uint32),
        ("depth_len", C.c_int32),
        ("pix_to_face", C.c_void_p), ("zbuf", C.c_void_p), ("dists", C.c_void_p), ("colors", C.c_void_p),
        ("znear", C.c_void_p), ("zfar", C.c_void_p),
        ("noise_rast", C.c_void_p), ("noise_agg", C.c_void_p),
        ("face_colors", C.c_void_p), ("num_faces", C.c_int64),
        ("seed_device", C.c_void_p),
    ]


class PertTexture(C.Structure):
    """Mirror of ``struct pert_texture``."""
    _fields_ = [
        ("kind", C.c_int32), ("atlas_size", C.c_int32),
        ("bary", C.c_void_p), ("table", C.c_void_p), ("face_uvs", C.c_void_p),
        ("map_h", C.c_int32), ("map_w", C.c_int32), ("map_count", C.c_int32),
        ("num_faces", C.c_int64),
    ]


class PertPhong(C.Structure):
    """Mirror of ``struct pert_phong``."""
    _fields_ = [
        ("P", C.c_int64), ("HW", C.c_int64),
        ("K", C.c_int32), ("light_rows", C.c_int32),
        ("num_faces", C.c_int64),
        ("flags", C.c_uint32),
        ("pix_to_face", C.c_void_p), ("bary", C.c_void_p), ("face_verts", C.c_void_p), ("face_normals", C.c_void_p),
        ("texels", C.c_void_p), ("face_colors", C.c_void_p), ("lighting", C.c_void_p),
        ("face_vert_colors", C.c_void_p),
        ("face_uvs", C.c_void_p), ("uv_map", C.c_void_p),
        ("map_h", C.c_int32), ("map_w", C.c_int32), ("map_count", C.c_int32),
        ("faces_per_mesh", C.c_int64),
    ]


class PertRaster(C.Structure):
    """Mirror of ``struct pert_raster``."""
    _fields_ = [
        ("N", C.c_int64),
        ("H", C.c_int32), ("W", C.c_int32), ("K", C.c_int32),
        ("flags", C.c_uint32),
        ("blur_radius", C.c_float),
        ("num_faces", C.c_int64),
        ("face_verts", C.c_void_p), ("face_start", C.c_void_p), ("face_order", C.c_void_p),
        ("bin_count", C.c_void_p), ("bin_offset", C.c_void_p), ("bin_faces", C.c_void_p),
    ]


_lock = threading.Lock()
_lib = None


class PertLibraryError(RuntimeError):
    pass


def load():
    """Load libpertshade.so (once).  Raises PertLibraryError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise PertLibraryError(
                f"{LIB_PATH} is missing: build it with `python -m pertrenderer_b200.build` "
                "(there is no CPU or PyTorch fallback for the perturbed shading path)")
        lib = C.CDLL(LIB_PATH)
        vp, i32, i64, u32, u64, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint32, C.c_uint64, C.c_float
        pp = C.POINTER(PertProblem)
        lib.pert_version.restype = C.c_int
        lib.pert_version.argtypes = []
        lib.pert_strerror.restype = C.c_char_p
        lib.pert_strerror.argtypes = [C.c_int]
        lib.pert_last_cuda_error.restype = C.c_char_p
        lib.pert_last_cuda_error.argtypes = []
        lib.pert_num_tiles.restype = i64
        lib.pert_num_tiles.argtypes = [pp]
        lib.pert_blob_bytes.restype = i64
        lib.pert_blob_bytes.argtypes = [pp]
        lib.pert_winner_bytes.restype = C.c_int
        lib.pert_winner_bytes.argtypes = [i32]
        lib.pert_shade_fwd.restype = C.c_int
        lib.pert_shade_fwd.argtypes = [pp] + [vp] * 9
        lib.pert_shade_bwd.restype = C.c_int
        lib.pert_shade_bwd.argtypes = [pp] + [vp] * 16
        lib.pert_soft_shade_fwd.restype = C.c_int
        lib.pert_soft_shade_fwd.argtypes = [pp, vp, vp]
        lib.pert_soft_shade_bwd.restype = C.c_int
        lib.pert_soft_shade_bwd.argtypes = [pp] + [vp] * 7
        lib.pert_rast_fwd.restype = C.c_int
        lib.pert_rast_fwd.argtypes = [vp, i64, i32, i32, i32, i32, f32, u64, i64, vp, u32, vp, vp, vp]
        lib.pert_rast_bwd.restype = C.c_int
        lib.pert_rast_bwd.argtypes = [vp, vp, i64, i32, f32, vp, vp, vp, vp]
        lib.pert_argmax_fwd.restype = C.c_int
        lib.pert_argmax_fwd.argtypes = [vp, i64, i32, i32, i32, i32, f32, u64, i64, vp, u32, vp, vp, vp]
        lib.pert_argmax_bwd.restype = C.c_int
        lib.pert_argmax_bwd.argtypes = [vp, vp, vp, i64, i32, i32, i32, i32, f32, u64, i64, vp, u32, vp, vp, vp, vp]
        lib.pert_seed_advance.restype = C.c_int
        lib.pert_seed_advance.argtypes = [vp, vp]
        lib.pert_noise_fill.restype = C.c_int
        lib.pert_noise_fill.argtypes = [u64, i32, i64, i32, i32, i32, i64, vp, vp]
        lib.pert_phong_fwd.restype = C.c_int
        lib.pert_phong_fwd.argtypes = [C.POINTER(PertPhong), vp, vp]
        lib.pert_phong_bwd.restype = C.c_int
        lib.pert_phong_bwd.argtypes = [C.POINTER(PertPhong)] + [vp] * 7
        lib.pert_rasterize_fwd.restype = C.c_int
        lib.pert_rasterize_fwd.argtypes = [C.POINTER(PertRaster)] + [vp] * 5
        lib.pert_rasterize_num_bins.restype = i64
        lib.pert_rasterize_num_bins.argtypes = [C.POINTER(PertRaster)]
        lib.pert_rasterize_bin.restype = C.c_int
        lib.pert_rasterize_bin.argtypes = [C.POINTER(PertRaster)] + [vp] * 5
        lib.pert_rasterize_bwd.restype = C.c_int
        lib.pert_rasterize_bwd.argtypes = [C.POINTER(PertRaster)] + [vp] * 6
        if lib.pert_version() != ABI_VERSION:
            raise PertLibraryError(f"libpertshade.so ABI {lib.pert_version()} != expected {ABI_VERSION}: rebuild")
        _lib = lib
    return _lib


_fused_flags = None  # (library, pert_shade_fused_flags()) of the library that answered


def require_fused_flags(flags: int):
    """Raise PertLibraryError unless the loaded library's pert_shade_fwd / pert_shade_bwd implement F_NO_VR when
    ``flags`` asks for it.  Libraries built before it ignore the flag there and would return the variance-reduced
    gradients; they also lack ``pert_shade_fused_flags``, which is therefore bound lazily here rather than in
    :func:`load`, so that such a library keeps serving every other call."""
    global _fused_flags
    if not flags & F_NO_VR:
        return
    lib = load()
    if _fused_flags is None or _fused_flags[0] is not lib:
        fn = getattr(lib, "pert_shade_fused_flags", None)
        if fn is not None:
            fn.restype = C.c_uint32
            fn.argtypes = []
        _fused_flags = (lib, int(fn()) if fn is not None else 0)
    if not _fused_flags[1] & F_NO_VR:
        raise PertLibraryError(
            f"{LIB_PATH} predates the fused GaussianRast_wovr + GaussianAgg_wovr pair (PERT_F_NO_VR in pert_shade_fwd / "
            "pert_shade_bwd): rebuild it with `python -m pertrenderer_b200.build --force`")


_render = None  # (library, its bound pert_shade_render)
_render_phase = None  # (library, its bound pert_shade_render_phase)


def _bind_render(name: str, what: str):
    """(library, ``name`` bound) for one of the render entry points, which are bound on first use rather than in
    :func:`load`, so that a library built before them keeps serving every other call; with such a library this raises
    PertLibraryError asking for a rebuild."""
    lib = load()
    fn = getattr(lib, name, None)
    if fn is None:
        raise PertLibraryError(f"{LIB_PATH} predates {what} ({name}): rebuild it with "
                               "`python -m pertrenderer_b200.build --force`")
    fn.restype = C.c_int
    fn.argtypes = [C.POINTER(PertProblem)] + [C.c_void_p] * 4
    return lib, fn


def shade_render_fn():
    """``pert_shade_render`` of the loaded library (see :func:`_bind_render`)."""
    global _render
    if _render is None or _render[0] is not load():
        _render = _bind_render("pert_shade_render", "the forward-only render")
    return _render[1]


def shade_render_phase_fn():
    """``pert_shade_render_phase`` of the loaded library (see :func:`_bind_render`)."""
    global _render_phase
    if _render_phase is None or _render_phase[0] is not load():
        _render_phase = _bind_render("pert_shade_render_phase", "the sample-sharded forward-only render")
    return _render_phase[1]


_phong_atlas = None  # (library, its bound pert_phong_atlas_fwd, pert_phong_atlas_bwd)


def phong_atlas_fns():
    """(``pert_phong_atlas_fwd``, ``pert_phong_atlas_bwd``) of the loaded library, bound on first use rather than in
    :func:`load`, so that a library built before them keeps serving every other call; with such a library this raises
    PertLibraryError asking for a rebuild."""
    global _phong_atlas
    lib = load()
    if _phong_atlas is None or _phong_atlas[0] is not lib:
        fwd, bwd = getattr(lib, "pert_phong_atlas_fwd", None), getattr(lib, "pert_phong_atlas_bwd", None)
        if fwd is None or bwd is None:
            raise PertLibraryError(f"{LIB_PATH} predates the texture-atlas Phong kernels (pert_phong_atlas_fwd / _bwd): "
                                   "rebuild it with `python -m pertrenderer_b200.build --force`")
        fwd.restype = bwd.restype = C.c_int
        fwd.argtypes = [C.POINTER(PertPhong), C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
        bwd.argtypes = [C.POINTER(PertPhong), C.c_void_p, C.c_int32] + [C.c_void_p] * 7
        _phong_atlas = (lib, fwd, bwd)
    return _phong_atlas[1], _phong_atlas[2]


_shade_tex = None  # (library, its bound pert_shade_tex_fwd, pert_shade_tex_bwd, pert_shade_tex_render)


def shade_tex_fns():
    """(``pert_shade_tex_fwd``, ``pert_shade_tex_bwd``, ``pert_shade_tex_render``) of the loaded library, bound on first use
    rather than in :func:`load`, so that a library built before them keeps serving every other call; with such a library
    this raises PertLibraryError asking for a rebuild (the texture is never materialised behind the caller's back)."""
    global _shade_tex
    lib = load()
    if _shade_tex is None or _shade_tex[0] is not lib:
        names = ("pert_shade_tex_fwd", "pert_shade_tex_bwd", "pert_shade_tex_render")
        fns = [getattr(lib, n, None) for n in names]
        if any(f is None for f in fns):
            raise PertLibraryError(f"{LIB_PATH} predates the textures sampled inside the fused shading kernels "
                                   "(pert_shade_tex_fwd / _bwd / _render): rebuild it with "
                                   "`python -m pertrenderer_b200.build --force`")
        fwd, bwd, render = fns
        pp, pt, vp = C.POINTER(PertProblem), C.POINTER(PertTexture), C.c_void_p
        fwd.restype = bwd.restype = render.restype = C.c_int
        fwd.argtypes = [pp, pt] + [vp] * 9
        bwd.argtypes = [pp, pt] + [vp] * 17
        render.argtypes = [pp, pt] + [vp] * 4
        _shade_tex = (lib, fwd, bwd, render)
    return _shade_tex[1], _shade_tex[2], _shade_tex[3]


_raster_bins = None  # (library, its bound pert_rasterize_bin_bounded, pert_rasterize_bin_capacity)


def raster_bin_fns():
    """(``pert_rasterize_bin_bounded``, ``pert_rasterize_bin_capacity``) of the loaded library, bound on first use rather
    than in :func:`load`, so that a library built before them keeps serving every other call.  Such a library would
    ignore RAST_BIN_WIDE and drop the faces of the wide lists, so this raises PertLibraryError asking for a rebuild."""
    global _raster_bins
    lib = load()
    if _raster_bins is None or _raster_bins[0] is not lib:
        fill, cap = getattr(lib, "pert_rasterize_bin_bounded", None), getattr(lib, "pert_rasterize_bin_capacity", None)
        if fill is None or cap is None:
            raise PertLibraryError(f"{LIB_PATH} predates the bounded coarse bins (pert_rasterize_bin_bounded / "
                                   "pert_rasterize_bin_capacity): rebuild it with `python -m pertrenderer_b200.build --force`")
        fill.restype, cap.restype = C.c_int, C.c_int64
        fill.argtypes = [C.POINTER(PertRaster)] + [C.c_void_p] * 5
        cap.argtypes = [C.POINTER(PertRaster)]
        _raster_bins = (lib, fill, cap)
    return _raster_bins[1], _raster_bins[2]


def check(rc: int, what: str):
    """Map a C return code to the Python exception the reference-facing API promises."""
    if rc == 0:
        return
    lib = load()
    msg = lib.pert_strerror(rc).decode()
    if rc == -6:
        raise RuntimeError(f"{what}: {msg} ({lib.pert_last_cuda_error().decode()})")
    if rc in (-2, -3, -5, -7):
        raise ValueError(f"{what}: {msg}")
    raise RuntimeError(f"{what}: {msg}")


def ptr(t):
    """Device pointer of a tensor (or NULL)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError(
                "pertrenderer_b200 runs on CUDA (sm_100a) only: got a tensor on "
                f"{t.device}; there is no CPU fallback for the perturbed shading path")
