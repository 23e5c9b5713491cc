"""Textures sampled inside the fused shading kernels, without a GPU: pert_shade_tex_fwd / _bwd / _render are exported and
bound once, the ctypes mirror of pert_texture matches the header, every refusal of the texture's validation comes before
any device work, and a library built before the entry points is refused with a request to rebuild.  No call here launches
a kernel: the pointers are fake."""

import ctypes
import types

import pytest

from pertrenderer_b200 import _cabi

FAKE = 1 << 20  # aligned, never dereferenced
NAMES = ("pert_shade_tex_fwd", "pert_shade_tex_bwd", "pert_shade_tex_render")


def _problem(N=2, flags=0):
    p = _cabi.PertProblem()
    p.N, p.H, p.W, p.K = N, 4, 4, 8
    p.sigma, p.gamma, p.alpha, p.eps = 1e-3, 1e-2, 1.0, 1e-10
    p.S_rast = p.S_agg = p.s_rast_end = p.s_agg_end = 8
    p.depth_len = 1
    p.flags = flags
    p.pix_to_face = p.zbuf = p.dists = p.znear = p.zfar = FAKE
    return p


def _texture(kind, F=6):
    t = _cabi.PertTexture()
    t.kind, t.bary, t.table, t.num_faces = kind, FAKE, FAKE, F
    if kind == _cabi.TEX_UV:
        t.face_uvs = FAKE
        t.map_h, t.map_w, t.map_count = 8, 8, 1
    if kind == _cabi.TEX_ATLAS:
        t.atlas_size = 4
    return t


def _calls(p, t):
    """Return codes of the three entry points for one problem / texture, every output pointer set."""
    fwd, bwd, render = _cabi.shade_tex_fns()
    f = FAKE
    return (fwd(p, t, f, f, f, f, f, None, f, f, None),
            bwd(p, t, f, f, f, f, f, f, f, f, f, f, f, None, None, None, f, f, None),
            render(p, t, f, f, f, None))


def test_symbols_are_exported_and_bound_once():
    lib = _cabi.load()
    for name in NAMES:
        assert hasattr(lib, name) and name in _cabi.EXPORTS
    fns = _cabi.shade_tex_fns()
    assert len(fns) == 3 and all(a is b for a, b in zip(_cabi.shade_tex_fns(), fns))


def test_texture_layout_matches_header():
    """ctypes mirror of pert_texture: field order / sizes as in the header (LP64)."""
    T = _cabi.PertTexture
    assert ctypes.sizeof(T) == 56
    assert (T.kind.offset, T.atlas_size.offset, T.bary.offset, T.table.offset, T.face_uvs.offset) == (0, 4, 8, 16, 24)
    assert (T.map_h.offset, T.map_w.offset, T.map_count.offset, T.num_faces.offset) == (32, 36, 40, 48)
    assert ctypes.sizeof(_cabi.PertProblem) == 200  # the problem record is unchanged: the texture travels beside it


def test_library_without_texture_kernels_is_refused(monkeypatch):
    """A library built before the entry points keeps serving every other call; the first textured call asks for a rebuild
    instead of falling back to materialised colours."""
    monkeypatch.setattr(_cabi, "_lib", types.SimpleNamespace())
    monkeypatch.setattr(_cabi, "_shade_tex", None)
    with pytest.raises(_cabi.PertLibraryError, match="rebuild"):
        _cabi.shade_tex_fns()


@pytest.mark.parametrize("phase", [_cabi.PH_RAST, _cabi.PH_AGG, _cabi.PH_BLEND, _cabi.PH_BWD_SAMPLE, _cabi.PH_BWD_FINISH,
                                   _cabi.PH_RAST | _cabi.PH_AGG | _cabi.PH_BLEND])
def test_phase_bits_are_refused(phase):
    assert _calls(_problem(flags=phase), _texture(_cabi.TEX_VERTEX)) == (-3, -3, -3)


@pytest.mark.parametrize("kind", [_cabi.TEX_VERTEX, _cabi.TEX_UV, _cabi.TEX_ATLAS])
def test_refusals(kind):
    p, t = _problem(), _texture(kind)
    fwd, bwd, render = _cabi.shade_tex_fns()
    assert _calls(None, t) == (-1, -1, -1)
    assert _calls(p, None) == (-1, -1, -1)
    # a second colour source as well
    p.colors = FAKE
    assert _calls(p, t) == (-3, -3, -3)
    p.colors, p.face_colors, p.num_faces = None, FAKE, 6
    assert _calls(p, t) == (-3, -3, -3)
    p.face_colors = None
    # NULL bary or table (or face_uvs of a UV texture)
    for field in ("bary", "table") + (("face_uvs",) if kind == _cabi.TEX_UV else ()):
        t = _texture(kind)
        setattr(t, field, None)
        assert _calls(p, t) == (-1, -1, -1), field
    # shapes
    t = _texture(kind, F=0)
    assert _calls(p, t) == (-2, -2, -2)
    t = _texture(kind)
    t.kind = 4
    assert _calls(p, t) == (-2, -2, -2)
    if kind == _cabi.TEX_UV:
        for field, value in (("map_h", 0), ("map_w", -1), ("map_count", 0), ("map_count", 3)):
            t = _texture(kind)
            setattr(t, field, value)
            assert _calls(p, t) == (-2, -2, -2), (field, value)
        t = _texture(kind)
        t.map_count = 2  # one map per image (N = 2) passes: the missing image is what is refused
        assert fwd(p, t, None, FAKE, FAKE, FAKE, FAKE, None, FAKE, FAKE, None) == -1
    if kind == _cabi.TEX_ATLAS:
        t = _texture(kind)
        t.atlas_size = 0
        assert _calls(p, t) == (-2, -2, -2)
        t.num_faces, t.atlas_size = 1 << 20, 32  # F R^2 3 > 2^31 - 1: 32-bit atlas offsets
        assert _calls(p, t) == (-3, -3, -3)
        t.num_faces, t.atlas_size = 699050, 32  # F R^2 3 = 2^31 - 2048 passes: the missing image is what is refused
        assert fwd(p, t, None, FAKE, FAKE, FAKE, FAKE, None, FAKE, FAKE, None) == -1
    # alignment
    for field in ("bary", "table") + (("face_uvs",) if kind == _cabi.TEX_UV else ()):
        t = _texture(kind)
        setattr(t, field, FAKE + 2)
        assert _calls(p, t) == (-4, -4, -4), field
    # the counterpart's own rules still hold: a missing output, a misaligned grad_bary
    t = _texture(kind)
    assert fwd(p, t, None, FAKE, FAKE, FAKE, FAKE, None, FAKE, FAKE, None) == -1
    f = FAKE
    assert bwd(p, t, f, f, f, f, f, f, f, f, f + 2, f, f, None, None, None, f, f, None) == -4
    assert render(p, t, None, f, f, None) == -1
