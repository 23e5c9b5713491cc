"""The phase-split forward-only render (pert_shade_render_phase) without a GPU: the library exports it, every refusal of
its argument validation comes before any device work, and a library built before it is refused with a request to
rebuild.  No call here passes validation: the pointers are fake."""

import types

import pytest

from pertrenderer_b200 import _cabi, ops
from test_cauchy_cpu import _problem

PHASES = ["PH_RAST", "PH_AGG", "PH_BLEND"]


def test_render_phase_symbol_is_exported():
    lib = _cabi.load()
    assert hasattr(lib, "pert_shade_render_phase")
    assert "pert_shade_render_phase" in _cabi.EXPORTS
    assert _cabi.shade_render_phase_fn() is _cabi.shade_render_phase_fn()  # bound once per library
    assert lib.pert_version() == _cabi.ABI_VERSION == 15


def test_render_phase_null_arguments():
    fn = _cabi.shade_render_phase_fn()
    assert fn(None, None, None, None, None) == -1
    for ph in PHASES:
        p, f = _problem(getattr(_cabi, ph))
        assert fn(p, f, None, f, None) == -1, ph  # every phase reads or writes the counts
    p, f = _problem(_cabi.PH_AGG)
    assert fn(p, f, f, None, None) == -1  # AGG writes the histogram
    p, f = _problem(_cabi.PH_BLEND)
    assert fn(p, f, f, None, None) == -1  # BLEND reads the all-shard histogram
    assert fn(p, None, f, f, None) == -1  # ... and writes the image
    p.colors = None
    assert fn(p, f, f, f, None) == -1  # ... from colors or face_colors
    p, f = _problem(_cabi.PH_RAST)
    p.dists = None
    assert fn(p, None, f, None, None) == -1


@pytest.mark.parametrize("flags", [0, _cabi.PH_RAST | _cabi.PH_AGG, _cabi.PH_AGG | _cabi.PH_BLEND,
                                   _cabi.PH_RAST | _cabi.PH_AGG | _cabi.PH_BLEND, _cabi.PH_RAST | _cabi.PH_BWD_SAMPLE,
                                   _cabi.PH_BLEND | _cabi.PH_BWD_FINISH, _cabi.PH_BWD_SAMPLE])
def test_render_phase_needs_exactly_one_forward_phase(flags):
    fn = _cabi.shade_render_phase_fn()
    p, f = _problem(flags)
    assert fn(p, f, None, None, None) == -3, hex(flags)


@pytest.mark.parametrize("phase", PHASES)
def test_render_phase_rejects_bad_flag_combinations(phase):
    fn = _cabi.shade_render_phase_fn()
    ph = getattr(_cabi, phase)
    # Philox-7 is refused by every phase-split call; the Cauchy / no-control-variate rules are those of pert_shade_fwd
    for flags in (_cabi.F_PHILOX7, _cabi.F_CAUCHY | _cabi.F_PHILOX7, _cabi.F_CAUCHY | _cabi.F_NO_VR,
                  _cabi.F_NO_VR | _cabi.F_PHILOX7, _cabi.F_NO_VR | _cabi.F_SKIP_DEAD_NOISE, _cabi.F_CAUCHY | _cabi.F_GUMBEL,
                  _cabi.F_CAUCHY | _cabi.F_SKIP_DEAD_NOISE, _cabi.F_NO_VR | _cabi.F_UNIFORM):
        p, f = _problem(ph | flags)
        assert fn(p, f, f, f, None) == -3, hex(flags)


@pytest.mark.parametrize("phase", PHASES)
def test_render_phase_rejects_misaligned_buffers(phase):
    fn = _cabi.shade_render_phase_fn()
    p, f = _problem(getattr(_cabi, phase))
    assert fn(p, f + 4, f, f, None) == -4  # image rows are float4
    assert fn(p, f, f + 1, f, None) == -4  # uint16 counts
    assert fn(p, f, f, f + 2, None) == -4  # int32 histogram
    p.colors = f + 2
    assert fn(p, f, f, f, None) == -4
    p, f = _problem(getattr(_cabi, phase))
    p.pix_to_face = f + 4
    assert fn(p, f, f, f, None) == -4
    p, f = _problem(getattr(_cabi, phase))
    p.face_colors, p.num_faces = f + 2, 4
    assert fn(p, f, f, f, None) == -4


@pytest.mark.parametrize("phase", PHASES)
def test_render_phase_checks_sample_shards(phase):
    fn = _cabi.shade_render_phase_fn()
    for field, value in (("s_rast_begin", 2), ("s_agg_begin", 6), ("s_agg_end", 9), ("s_rast_end", 0),
                         ("s_agg_begin", 8)):
        p, f = _problem(getattr(_cabi, phase))
        setattr(p, field, value)
        assert fn(p, f, f, f, None) == -5, (field, value)


def test_library_without_render_phase_is_refused(monkeypatch):
    """A library built before pert_shade_render_phase keeps serving every other call; the first phase-split render asks
    for a rebuild."""
    monkeypatch.setattr(_cabi, "_lib", types.SimpleNamespace())
    monkeypatch.setattr(_cabi, "_render_phase", None)
    with pytest.raises(_cabi.PertLibraryError, match="rebuild"):
        ops.shade_render_phase(types.SimpleNamespace(), _cabi.PH_RAST, None)
