"""The staging rule of the host-buffer pipelines (libflacarray._group_bytes): which host bytes stage one group of
streams, and where each stream starts in them.  The covering range [min start, max end) is copied as it is while it is
at most twice the streams' own bytes; beyond that only the streams' bytes are gathered."""
import numpy as np
import pytest

CASES = {
    # name: (starts, nbytes, buffer size, covering range expected)
    "back_to_back_in_order": ([0, 100, 250, 260], [100, 150, 10, 40], 300, True),
    "back_to_back_out_of_order": ([250, 0, 260, 100], [10, 100, 40, 150], 300, True),
    "gaps_below_the_streams_bytes": ([5, 130, 300, 420], [100, 150, 90, 70], 600, True),
    "ends_of_a_large_buffer": ([0, (1 << 20) - 77], [64, 77], 1 << 20, False),
}


@pytest.mark.parametrize("name", list(CASES))
def test_group_bytes_rebased_starts(name):
    from flacarray_b200 import libflacarray as lf

    starts, nbytes, size, covering = CASES[name]
    comp = np.random.default_rng(5).integers(0, 256, size, dtype=np.uint8)
    st, nb = np.array(starts, np.int64), np.array(nbytes, np.int64)
    part, rel = lf._group_bytes(comp, st, nb)
    lo, hi = int(st.min()), int((st + nb).max())
    if covering:
        assert hi - lo <= 2 * nb.sum()
        assert np.array_equal(part, comp[lo:hi])
    else:
        assert hi - lo > 2 * nb.sum()
        assert part.size == nb.sum()
    assert rel.dtype == np.int64 and rel.shape == st.shape
    assert 0 <= rel.min() and (rel + nb).max() <= part.size
    want = np.concatenate([comp[s:s + n] for s, n in zip(st, nb)])
    got = np.concatenate([part[r:r + n] for r, n in zip(rel, nb)])
    assert np.array_equal(got, want)
