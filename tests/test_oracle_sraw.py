"""Pins the oracle's Cr2sRawInterpolator restatement against the compiled
reference (oracle/_ref): 4:2:2 versions 0-2, 4:2:0 versions 1-2, edge MCUs
(last column / last row), clamping at both ends.  CPU only."""
import numpy as np
import pytest

import oracle
from oracle import port

ref = oracle.ref
pytestmark = pytest.mark.skipif(not oracle.ref.available(), reason="no reference answers (oracle/_ref or tests/golden/ref_calls)")


def sraw_input(num_mcus, rows, per, seed, extreme=False):
    """Subsampled image as Cr2Decompressor leaves it: `per` uint16 per MCU."""
    rng = np.random.default_rng(seed)
    w = num_mcus * per
    pitch = (w * 2 + 15) // 16 * 16
    a = np.zeros((rows, pitch // 2), dtype=np.uint16)
    hi = 65535 if extreme else 16383
    a[:, :w] = rng.integers(0, hi + 1, (rows, w), dtype=np.uint16)
    if not extreme:  # chroma around the 16384 bias like real files
        for c in range(per - 2, per):
            a[:, c:w:per] = rng.integers(16384 - 3000, 16384 + 3000, (rows, num_mcus), dtype=np.uint16)
    return a, w


CASES = [((2, 1), v, n, r) for v in (0, 1, 2) for (n, r) in ((2, 1), (5, 3), (64, 8))] + \
        [((2, 2), v, n, r) for v in (1, 2) for (n, r) in ((2, 1), (2, 2), (5, 3), (64, 8))]


@pytest.mark.parametrize("sub,version,num_mcus,rows", CASES)
@pytest.mark.parametrize("extreme", [False, True])
def test_sraw_interpolate(sub, version, num_mcus, rows, extreme):
    per = 4 if sub == (2, 1) else 6
    inp, in_w = sraw_input(num_mcus, rows, per, seed=version * 100 + num_mcus, extreme=extreme)
    out_w, out_h = 2 * num_mcus, rows * sub[1]
    coeffs, hue = (2100, 1024, 1700), 12 if not extreme else -400
    a = port.new_image(out_w, out_h, 3)
    b = a.copy()
    port.sraw_interpolate(inp, in_w, a, out_w, sub, coeffs, hue, version)
    ref.sraw_interpolate(inp, in_w, b, out_w, sub, coeffs, hue, version)
    assert np.array_equal(a, b)
    assert not np.any(a[:, :out_w * 3] == 0xA5A5) or extreme  # every pixel written
