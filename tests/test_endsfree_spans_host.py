"""Per-pair ends-free spans, host side (no GPU): the C entry points and their ctypes signatures, and the checks that
reject a malformed span list before anything is aligned."""
import ctypes as C

import numpy as np
import pytest


def _aligner(n=3):
    import wfagpu
    a = wfagpu.Aligner()
    for i in range(n):
        assert a.add_sequences("ACGT" * (i + 2), "ACGTT" * (i + 2))
    assert a.initialize_parameters(2, 3, 1)
    return a


def test_entry_points_and_signatures(lib):
    import wfagpu
    for name in ("wfagpu_align_spans", "wfagpu_launch_alignments_spans", "wfagpu_device_align_spans",
                 "wfagpu_device_rescore_spans"):
        assert name in wfagpu.EXPORTS
        assert getattr(lib, name) is not None
    P = C.POINTER
    assert lib.wfagpu_align_spans.argtypes == [P(wfagpu.AlignerStruct), P(wfagpu.Span), P(wfagpu.Coords)]
    assert lib.wfagpu_align_spans.restype is C.c_bool
    assert lib.wfagpu_launch_alignments_spans.argtypes[-2:] == [P(wfagpu.Span), P(wfagpu.Coords)]
    assert lib.wfagpu_device_align_spans.argtypes[-1] == P(wfagpu.Span)
    assert lib.wfagpu_device_rescore_spans.argtypes[-2:] == [P(wfagpu.Span), P(C.c_int32)]


def test_spans_of_accepts_tuples_and_arrays():
    import wfagpu
    rows = [(0, 0, 0, 0), (1, 2, 3, 4), (10 ** 6,) * 4]
    for given in (rows, [list(r) for r in rows], np.array(rows), np.array(rows, np.int64)):
        sp = wfagpu.spans_of(given, 3)
        assert [(s.pattern_begin_free, s.pattern_end_free, s.text_begin_free, s.text_end_free) for s in sp] == rows
    assert wfagpu._per_pair(rows) and wfagpu._per_pair(np.array(rows))
    assert not wfagpu._per_pair((1, 2, 3, 4)) and not wfagpu._per_pair(np.array([1, 2, 3, 4]))
    assert not wfagpu._per_pair(None)


@pytest.mark.parametrize("bad", [
    [(0, 0, 0, 0)] * 2,                      # one span short
    [(0, 0, 0, 0)] * 4,                      # one too many
    [(0, 0, 0)] * 3,                         # three values a pair
    [(0, 0, 0, 0, 0)] * 3,
    np.zeros((3, 3), np.int64),
    np.zeros((2, 4), np.int64),
    np.zeros((3, 4, 1), np.int64),
    [],
])
def test_a_wrong_count_or_shape_raises_before_aligning(bad):
    a = _aligner()
    with pytest.raises(ValueError):
        a.align(ends_free=bad)
    with pytest.raises(ValueError):
        a.align(ends_free=bad, coords=True)


def test_per_pair_spans_do_not_combine_with_affine2p():
    a = _aligner()
    with pytest.raises(ValueError):
        a.align(ends_free=[(1, 1, 1, 1)] * 3, affine2p=(2, 3, 1, 10, 1))


def test_negative_or_banded_spans_are_rejected_by_the_library(lib):
    # checked in the driver before any device is touched
    import wfagpu
    a = _aligner()
    sp = (wfagpu.Span * 3)(wfagpu.Span(0, 0, 0, 0), wfagpu.Span(1, 0, -1, 0), wfagpu.Span(0, 0, 0, 0))
    assert not lib.wfagpu_align_spans(C.byref(a.s), sp, None)
    a.options.band = 10
    sp = (wfagpu.Span * 3)(wfagpu.Span(0, 0, 0, 0), wfagpu.Span(0, 0, 2, 2), wfagpu.Span(0, 0, 0, 0))
    assert not lib.wfagpu_align_spans(C.byref(a.s), sp, None)
