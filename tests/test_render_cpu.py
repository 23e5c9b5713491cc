"""The forward-only render (pert_shade_render) without a GPU: the library exports it, its argument validation runs before
any device work, and a library built before it is refused with a request to rebuild."""

import types

import pytest

from pertrenderer_b200 import _cabi, ops
from test_cauchy_cpu import _problem


def test_render_symbol_is_exported():
    lib = _cabi.load()
    assert hasattr(lib, "pert_shade_render")
    assert "pert_shade_render" in _cabi.EXPORTS
    assert _cabi.shade_render_fn() is _cabi.shade_render_fn()  # bound once per library


def test_render_null_arguments():
    fn = _cabi.shade_render_fn()
    p, f = _problem(0)
    assert fn(None, f, None, None, None) == -1
    assert fn(p, None, None, None, None) == -1
    # the sparse-first work list needs the counts workspace of its fallback pass
    assert fn(p, f, None, f, None) == -1
    p.colors = None
    assert fn(p, f, f, f, None) == -1


@pytest.mark.parametrize("bit", ["PH_RAST", "PH_AGG", "PH_BLEND", "PH_BWD_SAMPLE", "PH_BWD_FINISH"])
def test_render_rejects_phase_bits(bit):
    fn = _cabi.shade_render_fn()
    p, f = _problem(getattr(_cabi, bit))
    assert fn(p, f, f, f, None) == -3


def test_render_rejects_sample_shards_and_bad_flag_combinations():
    fn = _cabi.shade_render_fn()
    p, f = _problem(0)
    p.s_agg_end = 4  # a shard of the aggregation samples: a render covers them all
    assert fn(p, f, f, f, None) == -3
    for flags in (_cabi.F_CAUCHY | _cabi.F_PHILOX7, _cabi.F_CAUCHY | _cabi.F_NO_VR, _cabi.F_NO_VR | _cabi.F_PHILOX7,
                  _cabi.F_NO_VR | _cabi.F_SKIP_DEAD_NOISE, _cabi.F_CAUCHY | _cabi.F_GUMBEL):
        p, f = _problem(flags)
        assert fn(p, f, f, f, None) == -3, hex(flags)
    p, f = _problem(_cabi.F_PHILOX7)
    p.noise_agg = f  # Philox-7 is an in-kernel stream: explicit noise excludes it
    assert fn(p, f, f, f, None) == -3
    p, f = _problem(0)
    assert fn(p, f + 4, f, f, None) == -4  # image rows are float4
    assert fn(p, f, f + 1, f, None) == -4
    assert fn(p, f, f, f + 4, None) == -4


def test_library_without_render_is_refused(monkeypatch):
    """A library built before pert_shade_render keeps serving every other call; the first render asks for a rebuild."""
    monkeypatch.setattr(_cabi, "_lib", types.SimpleNamespace())
    monkeypatch.setattr(_cabi, "_render", None)
    with pytest.raises(_cabi.PertLibraryError, match="rebuild"):
        ops.shade_render(types.SimpleNamespace())
