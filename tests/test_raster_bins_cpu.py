"""The bounded coarse bins without a GPU: pert_rasterize_bin_bounded and pert_rasterize_bin_capacity are exported and bound
once, the capacity is C * num_faces, every refusal of the new entry point and of the PERT_RAST_BIN_WIDE flag comes before
any device work, a library built before them is refused with a request to rebuild, and an eager forward picks the bounded
bins exactly where a face's blur margin fits C tiles.  No call here launches a kernel: the pointers are fake."""

import types

import pytest

from pertrenderer_b200 import _cabi

FAKE = 1 << 20  # aligned, never dereferenced
BIN_CAP = 8  # RASTER_BIN_CAP of csrc/kernels.h


def _raster(N=2, H=64, W=96, K=50, F=1000):
    rs = _cabi.PertRaster()
    rs.N, rs.H, rs.W, rs.K, rs.num_faces = N, H, W, K, F
    rs.face_verts = rs.face_start = FAKE
    return rs


def test_bin_symbols_are_exported_and_bound_once():
    lib = _cabi.load()
    for name in ("pert_rasterize_bin_bounded", "pert_rasterize_bin_capacity"):
        assert hasattr(lib, name) and name in _cabi.EXPORTS
    fill, cap = _cabi.raster_bin_fns()
    assert _cabi.raster_bin_fns()[0] is fill and _cabi.raster_bin_fns()[1] is cap
    assert _cabi.RAST_BIN_WIDE == 2 and _cabi.RAST_CULL_BACKFACES == 1
    assert lib.pert_version() == _cabi.ABI_VERSION == 15


def test_raster_struct_keeps_its_layout():
    import ctypes
    assert ctypes.sizeof(_cabi.PertRaster) == 88
    assert _cabi.PertRaster.bin_faces.offset == 80


@pytest.mark.parametrize("N,H,W,F", [(1, 128, 128, 20480), (8, 256, 256, 8 * 20480), (16, 1024, 1024, 16 * 100000),
                                     (3, 1, 1, 1), (1, 7, 33, 0x7fffffff // 9)])
def test_capacity_is_c_faces(N, H, W, F):
    _, cap = _cabi.raster_bin_fns()
    assert cap(_raster(N, H, W, 50, F)) == BIN_CAP * F


def test_capacity_of_no_problem_is_zero():
    _, cap = _cabi.raster_bin_fns()
    assert cap(None) == 0
    assert cap(_raster(F=0)) == 0
    assert cap(_raster(F=-5)) == 0


def test_bounded_bin_refusals():
    fill, _ = _cabi.raster_bin_fns()
    lib = _cabi.load()
    f = FAKE
    rs = _raster()
    assert fill(None, f, None, None, None, None) == -1
    assert fill(rs, None, None, None, None, None) == -1  # count pass without counts
    assert fill(rs, f, None, f, f, None) == -1  # fill pass without offsets
    assert fill(rs, f, f, None, f, None) == -1  # ... or without cursors
    assert fill(rs, f + 2, None, None, None, None) == -4  # int32 counts
    assert fill(rs, f, f + 4, f, f, None) == -4  # int64 offsets
    assert fill(rs, f, f, f + 2, f, None) == -4  # int32 cursors
    assert fill(rs, f, f, f, f + 4, None) == -4  # int64 faces
    # the shared problem rules of pert_rasterize_bin
    for field, value, rc in (("N", 0, -2), ("K", 0, -2), ("num_faces", 0, -2), ("N", 70000, -3), ("K", 2000, -3),
                             ("blur_radius", -1.0, -7), ("blur_radius", float("inf"), -7), ("blur_radius", float("nan"), -7),
                             ("face_verts", None, -1), ("face_start", None, -1), ("face_verts", FAKE + 2, -4),
                             ("face_start", FAKE + 4, -4)):
        bad = _raster()
        setattr(bad, field, value)
        assert fill(bad, f, None, None, None, None) == rc, field
        assert fill(bad, f, f, f, f, None) == rc, field
        assert lib.pert_rasterize_bin(bad, f, None, None, None, None) == rc, field


def test_wide_flag_refusals():
    lib = _cabi.load()
    f = FAKE
    rs = _raster()
    rs.flags = _cabi.RAST_BIN_WIDE
    assert lib.pert_rasterize_fwd(rs, f, f, f, f, None) == -1  # the flag without bin_faces
    rs.flags |= _cabi.RAST_CULL_BACKFACES
    assert lib.pert_rasterize_fwd(rs, f, f, f, f, None) == -1
    rs.bin_faces = f
    assert lib.pert_rasterize_fwd(rs, f, f, f, f, None) == -1  # bin_faces without counts / offsets
    rs.bin_count = rs.bin_offset = f
    rs.bin_faces = f + 4
    assert lib.pert_rasterize_fwd(rs, f, f, f, f, None) == -4
    rs.bin_faces, rs.bin_count = f, f + 2
    assert lib.pert_rasterize_fwd(rs, f, f, f, f, None) == -4
    rs.bin_count = f
    assert lib.pert_rasterize_fwd(rs, f + 4, f, f, f, None) == -4  # the outputs' rules still apply
    assert lib.pert_rasterize_fwd(rs, None, f, f, f, None) == -1


def test_library_without_bounded_bins_is_refused(monkeypatch):
    """A library built before the bounded bins would ignore PERT_RAST_BIN_WIDE and lose the wide faces: it keeps serving
    every other call, and the first bounded-bin call asks for a rebuild."""
    monkeypatch.setattr(_cabi, "_lib", types.SimpleNamespace(pert_rasterize_bin_capacity=lambda rs: 0))
    monkeypatch.setattr(_cabi, "_raster_bins", None)
    with pytest.raises(_cabi.PertLibraryError, match="rebuild"):
        _cabi.raster_bin_fns()


def test_large_mesh_forward_refuses_an_old_library(monkeypatch):
    """The rasteriser's large-mesh path asks for the bounded bins before it launches anything."""
    import torch
    from pertrenderer_b200 import rasterizer
    old = types.SimpleNamespace(pert_version=lambda: _cabi.ABI_VERSION,
                                pert_rasterize_num_bins=lambda rs: 1)
    monkeypatch.setattr(_cabi, "_lib", old)
    monkeypatch.setattr(_cabi, "_raster_bins", None)
    monkeypatch.setattr(rasterizer, "require_cuda", lambda *t: None)
    monkeypatch.setattr(torch.cuda, "device", lambda d: __import__("contextlib").nullcontext())
    fv = torch.zeros((rasterizer.BIN_MIN_FACES, 3, 3))
    fs = torch.tensor([0, fv.shape[0]])
    with pytest.raises(_cabi.PertLibraryError, match="rebuild"):
        rasterizer._Rasterize.apply(fv, fs, 8, 8, 4, 0.0, False)


def test_bins_are_bounded_where_the_blur_margin_fits_c_tiles():
    """Outside a CUDA-graph capture the rasteriser takes the bounded bins where a face's blur margin alone spans at most C
    tiles (there they are the faster ones), and the synchronising bins where every face would be wide."""
    import math
    from pertrenderer_b200 import rasterizer
    _, cap = _cabi.raster_bin_fns()
    blur = math.log(1.0 / 1e-4 - 1.0) * 1e-3  # eval.py at sigma = 1e-3
    for N, HW, F, bounded in ((1, 128, 20480, True), (8, 256, 8 * 20480, False), (16, 1024, 16 * 100000, False),
                              (8, 256, 8 * 20480, True), (1, 64, 20480, True)):
        rs = _raster(N, HW, HW, 50, F)
        b = blur if (N, HW, bounded) != (8, 256, True) else 0.0
        assert rasterizer._bounded_bins_pay(rs, cap, HW, HW, b) is bounded, (N, HW, b)
