"""Pins the PhaseOneDecompressor restatement (oracle/rs_oracle.c: rso_phaseone) against the
compiled reference: encoder round trips (all code lengths, the raw last width % 8 pixels,
shuffled strips at odd offsets), random payloads, error classes."""
import numpy as np
import pytest

import oracle
from oracle import port, synth

pytestmark = pytest.mark.skipif(not oracle.ref.available(), reason="no reference answers (oracle/_ref or tests/golden/ref_calls)")


@pytest.mark.parametrize("w,h,wild", [(8, 1, False), (70, 9, False), (258, 33, True), (1000, 12, False)])
def test_phaseone_round_trip_and_reference(w, h, wild):
    img = synth.image_model(w, h, seed=w, wild=wild, bits=16 if wild else 14)
    blob, strips = synth.make_phaseone(img, shuffle_seed=h, gap=3)
    a = port.new_image(w, h)
    b = a.copy()
    port.phaseone(a, w, blob, strips)
    oracle.ref.phaseone(b, w, blob, strips, nthreads=3)
    assert np.array_equal(a, b)
    assert np.array_equal(a[:, :w], img)


def test_phaseone_random_payloads():
    """Random bits: rows whose first length bit is 1 are errors, the others decode."""
    w, h = 64, 40
    rng = np.random.default_rng(4)
    blob = rng.integers(0, 256, h * 200 + 16, dtype=np.uint8)
    # make every row start with two decodable length codes: first bits 0 (MSB of byte 3)
    strips = [(r * 200, 200, r) for r in range(h)]
    for off, _, _ in strips:
        blob[off + 3] = 0           # at column 0 both length prefixes must be 5 zeros (+ 1 bit):
        blob[off + 2] &= 0x0F       # bits 31..20 of the first chunk = 0
    a = port.new_image(w, h)
    b = a.copy()
    port.phaseone(a, w, blob, strips)
    oracle.ref.phaseone(b, w, blob, strips)
    assert np.array_equal(a, b)


def test_phaseone_error_classes():
    w, h = 16, 4
    img = synth.image_model(w, h, seed=2)
    blob, strips = synth.make_phaseone(img)
    bad = blob.copy()
    bad[strips[2][0] + 3] |= 0x80   # first bit of row 2 is 1: lengths cannot be initialised
    for f in (port.phaseone, oracle.ref.phaseone):
        with pytest.raises(port.RawDecoderException):
            f(port.new_image(w, h), w, bad, strips)
        with pytest.raises(port.RawDecoderException):     # strip count
            f(port.new_image(w, h), w, blob, strips[:-1])
        with pytest.raises(port.RawDecoderException):     # a row twice
            f(port.new_image(w, h), w, blob, strips[:-1] + [strips[0]])
        with pytest.raises(port.RawDecoderException):     # odd width
            f(port.new_image(15, h), 15, blob, strips)
        short = [(o, 4, r) if r == 1 else (o, n, r) for o, n, r in strips]
        with pytest.raises(port.RawDecoderException):     # a strip far too short
            f(port.new_image(w, h), w, blob, short)
