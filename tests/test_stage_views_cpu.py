"""CPU-only checks of region views of staged sessions (bsg_stage_view, Stage.view): the entry point is exported, the
handle arguments are checked before anything else, the Python wrapper validates its input as Stage() does, and without
a device no session (so no view) can be opened."""
import ctypes as C

import numpy as np
import pytest

import bamsignals_b200 as B
from bamsignals_b200 import api

BSG_EARG, BSG_ECUDA = -8, -6


def _region_args(gr):
    m = api.marshal_regions(gr)
    return m, (m.R, m.levels, m.n_levels, api._p(m.seq_idx, C.c_int32), api._p(m.loc, C.c_int32),
               api._p(m.width, C.c_int32), api._p(m.strand, C.c_int8))


def test_stage_view_exported():
    assert hasattr(B.lib(), "bsg_stage_view")


def test_null_view_or_session_is_earg():
    L = B.lib()
    _m, args = _region_args(B.GRanges(["chr1", "chr2"], [1, 100], [10, 0], ["+", "-"]))
    assert L.bsg_stage_view(None, None, *args) == BSG_EARG
    h = C.c_void_p(12345)
    assert L.bsg_stage_view(C.byref(h), None, *args) == BSG_EARG
    assert not h, "*view must be cleared on failure"
    assert L.bsg_last_error()


def _closed_stage():
    st = B.Stage.__new__(B.Stage)
    st._m, st._h = api.marshal_regions(B.GRanges(["chr1"], [1], [10])), C.c_void_p()
    return st


@pytest.mark.parametrize("bad", ["chr1:1-10", None, [("chr1", 1, 10)], np.zeros(3)])
def test_view_rejects_non_granges(bad):
    with pytest.raises(TypeError, match="must provide a GRanges object"):
        _closed_stage().view(bad)


def test_view_of_closed_stage_is_earg():
    with pytest.raises(B.BamsignalsError) as e:
        _closed_stage().view(B.GRanges(["chr1"], [1], [10]))
    assert e.value.code == BSG_EARG


def test_no_session_without_a_device(fixture_bam):
    if B.lib().bsg_device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(B.BamsignalsError, match="no CUDA device") as e:
        B.Stage(fixture_bam, B.GRanges(["chr1"], [1], [10]))
    assert e.value.code == BSG_ECUDA
