"""Pins the HasselbladDecompressor restatement (oracle/rs_oracle.c: rso_hasselblad_decompress)
against the compiled reference -- groundwork: the codec has no device kernel yet.  Encoder
round trips (all difference lengths incl. 0 and the 65535 -> -32768 case), stream position,
random payloads, error classes."""
import numpy as np
import pytest

import oracle
from oracle import port, synth

pytestmark = pytest.mark.skipif(not oracle.ref.available(), reason="no reference answers (oracle/_ref or tests/golden/ref_calls)")

NCPL, VALS = synth.DEFAULT_NCPL, synth.DEFAULT_VALUES


@pytest.mark.parametrize("w,h,wild", [(2, 1, False), (66, 9, False), (130, 21, True)])
def test_hasselblad_round_trip_and_reference(w, h, wild):
    img = synth.image_model(w, h, seed=w, wild=wild, bits=16 if wild else 14)
    if wild:
        img[0, 0:4] = [0x8000, 0x8000, 0, 0xFFFF]    # differences of -32768 and wrap-around
    ht = port.Huff(NCPL, VALS, full=False)
    data = synth.make_hasselblad(img, ht, 0x8000)
    a = port.new_image(w, h)
    b = a.copy()
    ca = port.hasselblad_decompress(a, w, ht, 0x8000, data)
    cb = oracle.ref.hasselblad_decompress(b, w, NCPL, VALS, False, 0x8000, data)
    assert np.array_equal(a, b) and ca == cb
    assert np.array_equal(a[:, :w], img)


def test_hasselblad_random_payload():
    w, h = 64, 12
    data = synth.lcg_bytes(4096, 9)
    ht = port.Huff(NCPL, VALS, full=False)
    a = port.new_image(w, h)
    b = a.copy()
    ra = rb = None
    try:
        ra = port.hasselblad_decompress(a, w, ht, 0x2000, data)
    except port.OracleError as e:
        ra = type(e)
    try:
        rb = oracle.ref.hasselblad_decompress(b, w, NCPL, VALS, False, 0x2000, data)
    except port.OracleError as e:
        rb = type(e)
    assert ra == rb
    if not isinstance(ra, type):
        assert np.array_equal(a, b)


def test_hasselblad_error_classes():
    ht_full = port.Huff(NCPL, VALS, full=True)
    ht = port.Huff(NCPL, VALS, full=False)
    data = synth.lcg_bytes(256, 1)
    with pytest.raises(port.RawDecoderException):      # full-decode table
        port.hasselblad_decompress(port.new_image(8, 2), 8, ht_full, 0, data)
    with pytest.raises(port.RawDecoderException):
        oracle.ref.hasselblad_decompress(port.new_image(8, 2), 8, NCPL, VALS, True, 0, data)
    with pytest.raises(port.RawDecoderException):      # odd width
        port.hasselblad_decompress(port.new_image(7, 2), 7, ht, 0, data)
    with pytest.raises(port.RawDecoderException):
        oracle.ref.hasselblad_decompress(port.new_image(7, 2), 7, NCPL, VALS, False, 0, data)
    for f in (lambda: port.hasselblad_decompress(port.new_image(64, 64), 64, ht, 0, data[:40]),
              lambda: oracle.ref.hasselblad_decompress(port.new_image(64, 64), 64, NCPL, VALS, False, 0,
                                                       data[:40])):
        with pytest.raises(port.IOException):          # stream ends early
            f()


def test_hasselblad_ljpeg_container_through_the_reference():
    """The container tests/test_gpu_hasselblad.py feeds the host mirror is what the reference's own
    HasselbladLJpegDecoder accepts, and its error classes for the two checks of decodeScan()."""
    w, h = 130, 21
    img = synth.image_model(w, h, seed=3)
    ht = port.Huff(NCPL, VALS, full=False)
    data = synth.make_hasselblad(img, ht, 0x8000)
    o = port.new_image(w, h)
    oracle.ref.hasselblad_ljpeg_decode(synth.hasselblad_ljpeg_container(w, h, data, NCPL, VALS), o, w)
    assert np.array_equal(o[:, :w], img)
    with pytest.raises(port.RawDecoderException):      # frame does not match the image
        oracle.ref.hasselblad_ljpeg_decode(
            synth.hasselblad_ljpeg_container(w, h, data, NCPL, VALS, frame_w=w + 2), port.new_image(w, h), w)
    with pytest.raises(port.RawDecoderException):      # restart interval
        oracle.ref.hasselblad_ljpeg_decode(
            synth.hasselblad_ljpeg_container(w, h, data, NCPL, VALS, dri=4), port.new_image(w, h), w)
