"""Pins the oracle's PentaxDecompressor restatement against the compiled reference:
legacy and "modern" tables (both byte orders), round trip of synthetic images,
out-of-bounds values, corrupt table descriptions, truncated streams.  CPU only."""
import numpy as np
import pytest

import oracle
from oracle import port, synth

ref = oracle.ref
pytestmark = pytest.mark.skipif(not oracle.ref.available(), reason="no reference answers (oracle/_ref or tests/golden/ref_calls)")


def both(img_shape, w, data, meta=None, meta_be=True):
    a = port.new_image(w, img_shape[0])
    b = a.copy()
    ea = eb = None
    try:
        port.pentax_decompress(a, w, data, meta, meta_be)
    except port.OracleError as e:
        ea = e
    try:
        ref.pentax_decompress(b, w, data, meta, meta_be)
    except port.OracleError as e:
        eb = e
    assert type(ea) is type(eb), (ea, eb)
    if ea is not None:
        # (the wording of ByteStream over-reads differs: get<T>() reports through
        #  Buffer::getSubView; the class is what callers see)
        assert isinstance(ea, port.IOException) or ea.msg[:28] in eb.msg, (ea.msg, eb.msg)
    else:  # (after a throw the image content is unspecified: the driver does not copy it out)
        assert np.array_equal(a, b)
    return a, ea


@pytest.mark.parametrize("meta_kind", ["legacy", "modern_be", "modern_le"])
@pytest.mark.parametrize("w,h", [(2, 1), (6, 2), (64, 9), (500, 40)])
def test_pentax_round_trip(meta_kind, w, h):
    meta = None if meta_kind == "legacy" else synth.pentax_modern_meta(meta_kind == "modern_be")
    be = meta_kind != "modern_le"
    table = port.pentax_table(meta, be)
    img = (synth.image_model(w, h, seed=w + h, bits=12) & 0x0FFF).astype(np.uint16)
    data = synth.make_pentax(img, table)
    out, err = both((h, w), w, data, meta, be)
    assert err is None
    assert np.array_equal(out[:, :w], img)


def test_pentax_table_matches_reference_behaviour():
    assert port.pentax_table(None) == ([0, 2, 3, 1, 1, 1, 1, 1, 1, 2, 0, 0, 0, 0, 0, 0],
                                       [3, 4, 2, 5, 1, 6, 0, 7, 8, 9, 10, 11, 12])
    ncpl, vals = port.pentax_table(synth.pentax_modern_meta(True), True)
    assert sum(ncpl) == 15 and sorted(vals) == list(range(15))


def test_pentax_out_of_bounds_value_throws():
    """isIntN(value, 16) (adt/Bit.h:83-90) accepts 0..65535: above or below throws."""
    w, h = 16, 4
    meta = synth.pentax_modern_meta(True)           # differences up to 14 bits
    table = port.pentax_table(meta, True)
    d = np.zeros((h, w), dtype=np.int32)
    d[0, 0:10:2] = 16383                            # 16383 * 4 = 65532 at (0, 6) is fine,
    data = port.encode_diffs_plain(d.reshape(-1), port.Huff(*table))
    _, err = both((h, w), w, data, meta, True)      # 16383 * 5 = 81915 at col 8, row 0 is not
    assert isinstance(err, port.RawDecoderException) and "8:0" in err.msg
    d[0, 8] = 3                                     # 65535 exactly: still fine
    data = port.encode_diffs_plain(d.reshape(-1), port.Huff(*table))
    out, err = both((h, w), w, data, meta, True)
    assert err is None and out[0, 8] == 65535 and out[2, 0] == 16383


def test_pentax_negative_value_throws():
    w, h = 8, 4
    table = port.pentax_table(None)
    d = np.zeros((h, w), dtype=np.int32)
    d[1, 3] = -5
    data = port.encode_diffs_plain(d.reshape(-1), port.Huff(*table))
    _, err = both((h, w), w, data)
    assert isinstance(err, port.RawDecoderException) and "3:1" in err.msg


def test_pentax_bad_dimensions_and_corrupt_meta():
    table = port.pentax_table(None)
    data = port.encode_diffs_plain(np.zeros(64, dtype=np.int32), port.Huff(*table))
    _, err = both((2, 7), 7, data)                     # odd width
    assert isinstance(err, port.RawDecoderException)
    meta = bytearray(synth.pentax_modern_meta(True))
    meta[1] = 9                                        # depth 21 > 15
    _, err = both((2, 8), 8, data, bytes(meta))
    assert isinstance(err, port.RawDecoderException)
    meta = bytearray(synth.pentax_modern_meta(True))
    meta[14 + 30] = 13                                 # a code length of 13
    _, err = both((2, 8), 8, data, bytes(meta))
    assert isinstance(err, port.RawDecoderException)
    _, err = both((2, 8), 8, data, synth.pentax_modern_meta(True)[:20])   # truncated meta
    assert isinstance(err, port.IOException)


def test_pentax_truncated_stream_is_ioe():
    w, h = 64, 16
    table = port.pentax_table(None)
    img = (synth.image_model(w, h, seed=3, bits=12) & 0x0FFF).astype(np.uint16)
    data = synth.make_pentax(img, table)
    _, err = both((h, w), w, data[:len(data) // 3])
    assert isinstance(err, port.IOException)
