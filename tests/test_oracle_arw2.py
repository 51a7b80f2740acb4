"""Pins the SonyArw2Decompressor restatement (oracle/rs_oracle.c: rso_sony_arw2) against the
compiled reference (oracle/_ref): plain, curve and dithered-curve tables, the error class of
the one invalid block pattern, truncated input."""
import numpy as np
import pytest

import oracle
from oracle import port, synth

pytestmark = pytest.mark.skipif(not oracle.ref.available(), reason="no reference answers (oracle/_ref or tests/golden/ref_calls)")


@pytest.mark.parametrize("w,h", [(32, 1), (64, 5), (320, 33), (9600, 2)])
@pytest.mark.parametrize("table", ["none", "plain", "dither"])
def test_arw2_matches_reference(w, h, table):
    data = synth.arw2_frame(w, h, seed=w + h)
    a = port.new_image(w, h)
    b = a.copy()
    curve = synth.sony_curve()
    t = None if table == "none" else port.build_table(curve, table == "dither")
    port.sony_arw2(a, w, data, t, table == "dither")
    oracle.ref.sony_arw2(b, w, data, None if table == "none" else curve, table == "dither")
    assert np.array_equal(a, b)
    if table == "none":
        assert int(a[:, :w].max()) <= 0xFFE and not (a[:, :w] & 1).any()


def test_arw2_multithreaded_reference_is_the_same():
    w, h = 640, 48
    data = synth.arw2_frame(w, h, seed=9)
    a = port.new_image(w, h)
    b = a.copy()
    curve = synth.sony_curve()
    port.sony_arw2(a, w, data, port.build_table(curve, True), True)
    oracle.ref.sony_arw2(b, w, data, curve, True, nthreads=4)
    assert np.array_equal(a, b)


def test_arw2_error_classes():
    w, h = 64, 4
    data = synth.arw2_frame(w, h, seed=3).copy()
    # imax == imin in the second block of row 2
    blk = data[2 * w + 16:2 * w + 32]
    v = int(blk[2]) | (int(blk[3]) << 8)
    imax = (v >> 6) & 15
    v = (v & ~(15 << 10)) | (imax << 10)
    blk[2], blk[3] = v & 255, v >> 8
    for f in (lambda: port.sony_arw2(port.new_image(w, h), w, data),
              lambda: oracle.ref.sony_arw2(port.new_image(w, h), w, data)):
        with pytest.raises(port.RawDecoderException):
            f()
    # truncated: fewer than w*h bytes
    good = synth.arw2_frame(w, h, seed=3)
    for f in (lambda: port.sony_arw2(port.new_image(w, h), w, good[:-1]),
              lambda: oracle.ref.sony_arw2(port.new_image(w, h), w, good[:-1])):
        with pytest.raises(port.IOException):
            f()
    # width not a multiple of 32
    for f in (lambda: port.sony_arw2(port.new_image(48, 2), 48, good),
              lambda: oracle.ref.sony_arw2(port.new_image(48, 2), 48, good)):
        with pytest.raises(port.RawDecoderException):
            f()
