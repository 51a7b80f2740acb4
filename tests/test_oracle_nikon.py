"""Pins the NikonDecompressor restatement (oracle/rs_oracle.c: rso_nikon_*) against the
compiled reference: every maker-note variant of the constructor / createCurve, 12 and 14
bit, both byte orders, dithered curve and uncorrected output, error classes."""
import numpy as np
import pytest

import oracle
from oracle import port, synth

pytestmark = pytest.mark.skipif(not oracle.ref.available(), reason="no reference answers (oracle/_ref or tests/golden/ref_calls)")


def _case(kind, bits, w, h, be=True, seed=1):
    pup = [1 << (bits - 1), (1 << (bits - 1)) + 2, (1 << (bits - 1)) - 8, (1 << (bits - 1)) - 2]
    meta = synth.nikon_meta(kind, bits, (pup[0], pup[2], pup[1], pup[3]), be)
    su = port.nikon_setup(meta, be, bits, w, h)
    assert su["pup"] == pup and su["split"] == 0
    img = (synth.image_model(w, h, seed=seed, bits=bits) & ((1 << bits) - 1)).astype(np.uint16)
    data = synth.make_nikon(img, su["huff_select"], pup)
    return meta, su, img, data


@pytest.mark.parametrize("kind", ["lossless", "table", "segments", "z7", "skip"])
@pytest.mark.parametrize("bits", [12, 14])
@pytest.mark.parametrize("uncorrected", [False, True])
def test_nikon_matches_reference(kind, bits, uncorrected):
    w, h = 130, 37
    meta, su, img, data = _case(kind, bits, w, h, be=(bits == 12), seed=bits)
    a = port.new_image(w, h)
    b = a.copy()
    port.nikon_decompress(a, w, meta, bits == 12, bits, data, uncorrected)
    oracle.ref.nikon_decompress(b, w, meta, bits == 12, bits, data, uncorrected)
    assert np.array_equal(a, b)
    if uncorrected:
        assert np.array_equal(a[:, :w], img)   # round trip of the encoder


def test_nikon_larger_image_dither_sequence():
    w, h = 1024, 300   # 307 200 dither steps in raster order
    meta, su, img, data = _case("table", 14, w, h, seed=5)
    a = port.new_image(w, h)
    b = a.copy()
    port.nikon_decompress(a, w, meta, True, 14, data)
    oracle.ref.nikon_decompress(b, w, meta, True, 14, data)
    assert np.array_equal(a, b)


def test_nikon_error_classes():
    w, h = 64, 8
    meta, su, img, data = _case("table", 12, w, h)
    for f in (port.nikon_decompress, oracle.ref.nikon_decompress):
        with pytest.raises(port.RawDecoderException):   # odd width
            f(port.new_image(63, h), 63, meta, True, 12, data)
        with pytest.raises(port.RawDecoderException):   # bits
            f(port.new_image(w, h), w, meta, True, 13, data)
        with pytest.raises(port.IOException):           # truncated maker note
            f(port.new_image(w, h), w, meta[:9], True, 12, data)
        with pytest.raises(port.IOException):           # stream ends early
            f(port.new_image(w, h), w, meta, True, 12, data[:40])
    bad = bytearray(synth.nikon_meta("segments", 12))
    bad[10:12] = bytes([0, 30])      # csize that does not divide the curve
    for f in (port.nikon_decompress, oracle.ref.nikon_decompress):
        with pytest.raises(port.RawDecoderException):
            f(port.new_image(w, h), w, bytes(bad), True, 12, data)


@pytest.mark.parametrize("bits", [12, 14])
@pytest.mark.parametrize("uncorrected", [False, True])
def test_nikon_split_streams_match_reference(bits, uncorrected):
    """Streams with a split: the rows from `split` on go through the restated
    NikonLASDecompressor ("lossy after split" tree, (len | shl << 4) differences)."""
    w, h, split = 66, 24, 10
    half = 1 << (bits - 1)
    pup = [half, half + 2, half - 8, half - 2]
    meta = synth.nikon_meta("segments", bits, (pup[0], pup[2], pup[1], pup[3]), True, split=split)
    su = port.nikon_setup(meta, True, bits, w, h)
    assert su["split"] == split and su["huff_select"] in (0, 3)
    top = (synth.image_model(w, split, seed=bits, bits=bits) & ((1 << bits) - 1)).astype(np.uint16)
    data = synth.make_nikon_split(top, su["huff_select"], pup, h - split, seed=bits)
    a = port.new_image(w, h)
    b = a.copy()
    port.nikon_decompress(a, w, meta, True, bits, data, uncorrected)
    oracle.ref.nikon_decompress(b, w, meta, True, bits, data, uncorrected)
    assert np.array_equal(a, b)
    if uncorrected:
        assert np.array_equal(a[:split, :w], top)


def test_nikon_split_outside_the_image_is_ignored():
    w, h = 34, 6
    meta = synth.nikon_meta("segments", 12, split=h)     # split >= height: no split
    assert port.nikon_setup(meta, True, 12, w, h)["split"] == 0
