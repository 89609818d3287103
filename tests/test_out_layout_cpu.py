"""The layout of SeekerEngine's output block (seeker.OutLayout): every region the kernels write has room of its own,
aligned for its dtype, and the block is no larger than its regions packed back to back."""
import itertools

import numpy as np
import pytest

from findnpropagate_b200 import quality, synth
from findnpropagate_b200.seeker import OutLayout, SeekerEngine

N_QUALITY = quality.QualitySpec(synth.CLASS_NAMES).n_counters


def _packed_total(F, T, S, n_quality):
    """The block's size written out by hand: per slot boxes(7) score best count, per candidate npts nvalid, status
    (8 int32), the recall counters, the keep flags padded to 8 bytes, then per setting boxes(7) score best count per
    candidate, the recall, precision and quality counters."""
    FT, NC, NP = F * T, SeekerEngine.N_COUNTERS, SeekerEngine.N_PRECISION
    return 4 * (10 * FT + 2 * F + 8) + 8 * NC + (FT + 7) // 8 * 8 + 40 * S * F + 8 * S * (NC + NP + n_quality)


@pytest.mark.parametrize("F,T,S,n_quality", list(itertools.product((0, 1, 7, 300), (1, 3), (0, 1, 257), (0, N_QUALITY))))
def test_regions_are_disjoint_aligned_and_inside_the_block(F, T, S, n_quality):
    lay = OutLayout(F, T, S, n_quality)
    assert lay.regions["status"][1:] == (np.dtype(np.int32), (8,))        # include/fnp.h: the C side uses 8
    spans = sorted(((lay.span(k), k) for k in lay.regions), key=lambda sk: sk[0].start)
    assert [k for _, k in spans] == list(lay.regions)                      # in the order of the table
    assert spans[0][0].start == 0 and spans[-1][0].stop <= lay.nbytes
    for (a, ka), (b, kb) in zip(spans, spans[1:]):
        assert a.stop <= b.start, (ka, kb)
    raw = np.zeros(lay.nbytes, np.uint8)
    for k, (off, dt, shape) in lay.regions.items():
        assert off % dt.itemsize == 0, k
        assert lay.span(k).stop - off == dt.itemsize * int(np.prod(shape)), k
        v = lay.view(raw, k)
        assert v.dtype == dt and v.shape == shape, k
        if shape[0] > 1 and v.size:            # a row's address, host view and device pointer alike
            assert lay.ptr(raw.ctypes.data, k, 1) == v[1:].ctypes.data, k
    assert lay.span("sel_recall", "sel_precision") == slice(lay.span("sel_recall").start, lay.span("sel_precision").stop)
    assert abs(lay.nbytes - _packed_total(F, T, S, n_quality)) < 8
