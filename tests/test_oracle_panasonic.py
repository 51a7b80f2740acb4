"""Pins the PanasonicV5/V6/V7 restatements (oracle/rs_oracle.c: rso_panasonic) against the
compiled reference on random payloads (every bit pattern is a valid stream for these
codecs), including partial last blocks (V5), both bit depths and the error classes."""
import numpy as np
import pytest

import oracle
from oracle import port, synth

pytestmark = pytest.mark.skipif(not oracle.ref.available(), reason="no reference answers (oracle/_ref or tests/golden/ref_calls)")


def payload(version, w, h, bps, seed):
    if version == 5:
        ppp = 128 // bps
        nblocks = (w * h // ppp + 1023) // 1024
        return synth.lcg_bytes(nblocks * 0x4000, seed)
    ppb = 9 if version == 7 else (11 if bps == 14 else 14)
    return synth.lcg_bytes(w * h // ppb * 16, seed)


CASES = [(5, 12, 40, 3), (5, 12, 4000, 9), (5, 14, 36, 5), (5, 14, 4005, 7),
         (6, 12, 28, 3), (6, 12, 1400, 11), (6, 14, 22, 4), (6, 14, 1100, 13),
         (7, 14, 18, 2), (7, 14, 1809, 10)]


@pytest.mark.parametrize("version,bps,w,h", CASES)
def test_panasonic_matches_reference(version, bps, w, h):
    data = payload(version, w, h, bps, seed=version * 100 + w)
    a = port.new_image(w, h)
    b = a.copy()
    port.panasonic(version, a, w, data, bps)
    oracle.ref.panasonic(version, b, w, data, bps, nthreads=3)
    assert np.array_equal(a, b)


def test_panasonic_v6_special_values():
    """Blocks of all zeros / all ones exercise the zero-reference and the clamp branches."""
    for bps, ppb in ((12, 14), (14, 11)):
        w, h = ppb * 4, 2
        for fill in (0x00, 0xFF, 0x0F, 0xF0):
            data = np.full(w * h // ppb * 16, fill, dtype=np.uint8)
            a = port.new_image(w, h)
            b = a.copy()
            port.panasonic(6, a, w, data, bps)
            oracle.ref.panasonic(6, b, w, data, bps)
            assert np.array_equal(a, b)


@pytest.mark.parametrize("version,bps,w", [(5, 12, 41), (5, 13, 40), (6, 12, 27), (6, 16, 28), (7, 14, 20)])
def test_panasonic_error_classes(version, bps, w):
    data = synth.lcg_bytes(0x8000, 1)
    for f in (lambda: port.panasonic(version, port.new_image(w, 2), w, data, bps),
              lambda: oracle.ref.panasonic(version, port.new_image(w, 2), w, data, bps)):
        with pytest.raises(port.RawDecoderException):
            f()


@pytest.mark.parametrize("version,bps,w,h", [(5, 12, 40, 3), (6, 14, 22, 4), (7, 14, 18, 2)])
def test_panasonic_truncated_input(version, bps, w, h):
    data = payload(version, w, h, bps, 5)[:-1]
    for f in (lambda: port.panasonic(version, port.new_image(w, h), w, data, bps),
              lambda: oracle.ref.panasonic(version, port.new_image(w, h), w, data, bps)):
        with pytest.raises(port.RawDecoderException):
            f()


@pytest.mark.parametrize("w,h,split,zero_ok", [(14, 1, 0, True), (28, 3, 0, False), (1400, 25, 0x1FF8, True),
                                               (2800, 13, 0x1FF8, False), (1414, 9, 0, False),
                                               (4200, 6, 0x2008, True)])
def test_panasonic_v4_matches_reference(w, h, split, zero_ok):
    """V4 (groundwork, no device kernel yet): random payloads are valid streams; with a
    section split the input is whole 0x4000-byte blocks, without one the last block is short."""
    nbytes = w * h // 14 * 16
    if split:
        nbytes = (nbytes + 0x3FFF) // 0x4000 * 0x4000
    data = synth.lcg_bytes(nbytes, seed=w + h)
    data[::7] = 0     # plenty of zero steps: the zero-reference and bad-pixel branches
    a = port.new_image(w, h)
    b = a.copy()
    za = port.panasonic_v4(a, w, data, zero_ok, split)
    zb = oracle.ref.panasonic_v4(b, w, data, zero_ok, split, nthreads=3)
    assert np.array_equal(a, b)
    assert za == zb and (zero_ok is False or za == [])


def test_panasonic_v4_error_classes():
    data = synth.lcg_bytes(0x8000, 2)
    for f in (port.panasonic_v4, oracle.ref.panasonic_v4):
        with pytest.raises(port.RawDecoderException):       # width not a multiple of 14
            f(port.new_image(15, 2), 15, data)
        with pytest.raises(port.RawDecoderException):       # split beyond the block
            f(port.new_image(14, 2), 14, data, True, 0x4001)
        with pytest.raises(port.IOException):               # not enough data
            f(port.new_image(1400, 40), 1400, data)
