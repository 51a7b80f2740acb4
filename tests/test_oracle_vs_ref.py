"""Pins oracle/rs_oracle.c (our restatement) against the UNMODIFIED reference
compiled into oracle/_ref/libref.so -- differential, same seeded inputs,
byte-for-byte over the uncropped buffer.  CPU only."""
import numpy as np
import pytest

import oracle
from oracle import port, synth

ref = oracle.ref
pytestmark = pytest.mark.skipif(not oracle.ref.available(), reason="no reference answers (oracle/_ref or tests/golden/ref_calls)")


@pytest.mark.parametrize("order", [port.LSB, port.MSB, port.MSB16, port.MSB32])
def test_pump_random_access_patterns(order):
    rng = np.random.default_rng(order)
    data = rng.integers(0, 256, 64, dtype=np.uint8)
    for _ in range(20):
        lens = [int(x) for x in rng.integers(1, 33, 12)]
        assert port.pump_getbits(order, data, lens, True) == ref.pump_getbits(order, data, lens, True)


def test_pump_jpeg_stuffing_and_markers():
    rng = np.random.default_rng(7)
    for trial in range(200):
        n = int(rng.integers(8, 40))
        data = rng.integers(0, 256, n, dtype=np.uint8)
        data[rng.integers(0, n, 4)] = 0xFF          # lots of FF
        data[rng.integers(0, n, 3)] = 0x00
        lens = [int(x) for x in rng.integers(1, 33, 10)]
        try:
            a = port.pump_getbits(port.JPEG, data, lens, True)
        except port.OracleError as e:
            with pytest.raises(port.OracleError) as ei:
                ref.pump_getbits(port.JPEG, data, lens, True)
            assert type(ei.value) is type(e)
            continue
        assert a == ref.pump_getbits(port.JPEG, data, lens, True), trial


def test_pump_overread_raises_ioe():
    data = bytes(range(8))
    for order in range(5):
        lens = [32] * 8
        with pytest.raises(port.IOException):
            port.pump_getbits(order, data, lens)
        with pytest.raises(port.IOException):
            ref.pump_getbits(order, data, lens)
        with pytest.raises(port.IOException):   # smaller than MaxProcessBytes
            port.pump_getbits(order, data[:3], [1])
        with pytest.raises(port.IOException):
            ref.pump_getbits(order, data[:3], [1])


@pytest.mark.parametrize("order", [port.LSB, port.MSB, port.MSB16, port.MSB32])
@pytest.mark.parametrize("bps", [1, 7, 8, 10, 12, 13, 14, 16])
def test_unpack(order, bps):
    w, h = 264, 6
    for skip in (0, 3):
        data, pitch = synth.packed_frame(w, h, bps, seed=bps, pitch=w * bps // 8 + skip)
        a = port.new_image(w, h + 2)
        b = a.copy()
        port.unpack(data, a, w, 1, (0, 1, w, h), pitch, bps, order)
        ref.unpack(data, b, w, 1, (0, 1, w, h), pitch, bps, order)
        assert np.array_equal(a, b)


def test_unpack_errors_same_class():
    w, h, bps = 16, 4, 12
    data = synth.lcg_bytes(24 * 4, 1)
    cases = [
        dict(crop=(0, 0, w, h), pitch=23),      # pitch too small
        dict(crop=(0, 0, w, 5), pitch=24),      # truncated
        dict(crop=(1, 0, w, h), pitch=24),      # x offset out of image
        dict(crop=(0, 9, w, h), pitch=24),      # y offset
        dict(crop=(0, 0, 15, h), pitch=24, bps=12 + 1),  # pitch bits not multiple of 8
    ]
    for c in cases:
        b = c.get("bps", bps)
        for fn in (port.unpack, ref.unpack):
            with pytest.raises(port.OracleError):
                fn(data, port.new_image(w, h), w, 1, c["crop"], c["pitch"], b, port.MSB)
    for c in cases:
        b = c.get("bps", bps)
        try:
            port.unpack(data, port.new_image(w, h), w, 1, c["crop"], c["pitch"], b, port.MSB)
        except port.OracleError as e1:
            try:
                ref.unpack(data, port.new_image(w, h), w, 1, c["crop"], c["pitch"], b, port.MSB)
            except port.OracleError as e2:
                assert type(e1) is type(e2), c


def _dng(img, tw, th, cpp=1, **kw):
    h, wc = img.shape
    w = wc // cpp
    fix = kw.get("fix16", False)
    t = synth.make_dng_ljpeg(img, tw, th, cpp=cpp, **kw)
    a = port.new_image(w, h, cpp)
    b = a.copy()
    port.dng_decompress(t.blob, t.offsets, t.lengths, a, w, cpp, tw, th, 7, fix_ljpeg=fix, nthreads=2)
    ref.dng_decompress(t.blob, t.offsets, t.lengths, b, w, cpp, tw, th, 7, fix_ljpeg=fix, nthreads=2)
    assert np.array_equal(a, b)
    assert np.array_equal(a[:, :wc], img)
    return t


def test_dng_ljpeg_variants():
    img = synth.image_model(300, 200, 7)
    _dng(img, 128, 64)
    _dng(synth.image_model(256, 96, 9, wild=True), 128, 32)
    img16 = synth.image_model(128, 64, 11, wild=True, bits=16)
    img16[0, 0:8] = [0, 0x8000, 0, 0x8000, 0xFFFF, 0x7FFF, 0, 0x8000]
    _dng(img16, 64, 64, prec=16)
    _dng(img16, 64, 64, prec=16, fix16=True)
    img = synth.image_model(96, 48, 13)
    _dng(img, 48, 24, ncomp=1)
    _dng(img, 96, 48, ncomp=4)
    _dng(img, 48, 48, ncomp=3)
    _dng(img, 48, 24, ncomp=4, mcu=(2, 2))
    _dng(synth.image_model(96 * 3, 40, 14), 32, 20, ncomp=3, cpp=3)
    tabs = synth.default_tables(2)
    _dng(synth.image_model(200, 100, 15), 100, 50, tabs=tabs, tab_of_comp=[0, 1])
    _dng(synth.image_model(160, 96, 17), 80, 48, restart_rows=1)
    _dng(synth.image_model(160, 96, 17), 80, 48, restart_rows=5)
    _dng(synth.image_model(101, 33, 19), 64, 16)


def test_dng_uncompressed_tiles():
    W, H, tw, th = 100, 60, 32, 16
    for bps, be in [(12, False), (14, False), (16, False), (16, True), (8, True)]:
        pitch = tw * bps // 8
        ntiles = 4 * 4
        blob = synth.lcg_bytes(pitch * th * ntiles + 64, bps)
        offs = [7 + n * pitch * th for n in range(ntiles)]
        a = port.new_image(W, H)
        b = a.copy()
        port.dng_decompress(blob, offs, [pitch * th] * ntiles, a, W, 1, tw, th, 1, bps=bps, big_endian=be)
        ref.dng_decompress(blob, offs, [pitch * th] * ntiles, b, W, 1, tw, th, 1, bps=bps, big_endian=be)
        assert np.array_equal(a, b), (bps, be)


def test_ljpeg_decompressor_consumed_and_restart():
    img = synth.image_model(64, 40, 3)
    hts = synth.default_tables(1)
    for rr in (0, 1, 7):
        blob = port.ljpeg_encode(img, 32, 40, (2, 1), 14, hts, [0, 0], rr)
        from helpers import parse_ljpeg  # noqa
        info = parse_ljpeg(blob)
        data = blob[info["data_off"]:]
        a = port.new_image(64, 40)
        b = a.copy()
        rpr = rr if rr else 40
        ca = port.ljpeg_decompress(a, 64, 1, (0, 0, 64, 40), (2, 1), (32, 40), [hts[0]] * 2,
                                   [1 << 13] * 2, rpr, data)
        cb = ref.ljpeg_decompress(b, 64, 1, (0, 0, 64, 40), (2, 1), (32, 40), [hts[0]],
                                  [0, 0], [1 << 13] * 2, rpr, data)
        assert ca == cb == len(data) - 2
        assert np.array_equal(a, b)
        # garbage between the scan and EOI: position comes from the refill cadence
        data2 = np.concatenate([data[:-2], np.zeros(11, np.uint8), data[-2:]])
        if rr == 0:
            ca = port.ljpeg_decompress(a, 64, 1, (0, 0, 64, 40), (2, 1), (32, 40), [hts[0]] * 2,
                                       [1 << 13] * 2, rpr, data2)
            cb = ref.ljpeg_decompress(b, 64, 1, (0, 0, 64, 40), (2, 1), (32, 40), [hts[0]],
                                      [0, 0], [1 << 13] * 2, rpr, data2)
            assert ca == cb


CR2_CASES = [
    # (w, h, fmt, frame(SOF3 w,h), slicing(numSlices, sliceW, lastSliceW))
    (64, 40, (2, 1, 1), (32, 40), (2, 32, 32)),
    (64, 40, (4, 1, 1), (16, 40), (2, 32, 32)),
    (72, 40, (2, 1, 1), (36, 40), (1, 0, 72)),        # single slice
    (96, 40, (2, 1, 1), (96, 20), (3, 32, 32)),       # Canon double-width/half-height frame
    (80, 48, (2, 1, 1), (40, 48), (3, 24, 32)),       # last slice wider
    (64, 40, (2, 1, 1), (32, 40), (2, 24, 40)),       # frame row not a multiple of slice width
    (64, 40, (2, 1, 1), (40, 40), (2, 32, 32)),       # frame larger than the image
    (96, 40, (2, 1, 1), (48, 40), (2, 32, 32)),       # quirk: slices wrap into two columns
]


@pytest.mark.parametrize("case", CR2_CASES)
def test_cr2(case):
    w, h, fmt, frame, slicing = case
    img = port.new_image(w, h)
    img[:, :w] = synth.image_model(w, h, 31)
    hts = synth.default_tables(2)
    toc = [0, 1, 0, 1][:fmt[0]]
    blob = port.cr2_encode(img, w, fmt, frame, slicing, 14, hts, toc)
    a = port.new_image(w, h)
    b = a.copy()
    port.cr2_ljpeg_decode(blob, a, w, slicing)
    ref.cr2_ljpeg_decode(blob, b, w, slicing)
    assert np.array_equal(a, b)
    assert np.array_equal(a[:, :w], img[:, :w])


def test_cr2_sraw_formats():
    hts = synth.default_tables(2)
    for fmt, w, h, frame, slicing in [((3, 2, 1), 96, 20, (48, 20), (2, 48, 48)),
                                      ((3, 2, 2), 96, 20, (32, 40), (2, 48, 48))]:
        img = port.new_image(w, h)
        img[:, :w] = synth.image_model(w, h, 33)
        blob = port.cr2_encode(img, w, fmt, frame, slicing, 14, hts, [0, 1, 1], is_cfa=False)
        a = port.new_image(w, h)
        b = a.copy()
        sub = (fmt[1], fmt[2])
        port.cr2_ljpeg_decode(blob, a, w, slicing, is_cfa=False, sub=sub)
        ref.cr2_ljpeg_decode(blob, b, w, slicing, is_cfa=False, sub=sub)
        assert np.array_equal(a, b)
        assert np.array_equal(a[:, :w], img[:, :w])


def test_huffman_validation_same_outcome():
    rng = np.random.default_rng(5)
    for trial in range(300):
        ncpl = [0] * 16
        for _ in range(int(rng.integers(1, 6))):
            ncpl[int(rng.integers(0, 16))] += int(rng.integers(1, 4))
        n = sum(ncpl)
        values = [int(v) for v in rng.integers(0, 18, n)]
        ok_a = ok_b = True
        try:
            port.Huff(ncpl, values)
        except port.OracleError:
            ok_a = False
        try:
            ref.huff_check(ncpl, values)
        except port.OracleError:
            ok_b = False
        assert ok_a == ok_b, (ncpl, values)


def test_huffman_decode_random_streams():
    rng = np.random.default_rng(9)
    hts = synth.default_tables(2)
    for ht in hts:
        for fix16 in (False, True):
            h = port.Huff(ht.ncpl, ht.values, True, fix16)
            diffs = rng.integers(-32768, 32768, 400)
            diffs[::7] = rng.integers(-3, 4, len(diffs[::7]))
            enc_a = port.encode_diffs(diffs, [h], [0])
            enc_b = ref.encode_diffs(diffs, ht.ncpl, ht.values, fix16)
            # the reference's vacuumer pads its last 32-bit chunk with zero bits,
            # ours pads the last byte with one bits (T.81): compare the payload
            assert enc_b.startswith(enc_a[:-2]) and len(enc_b) >= len(enc_a) - 1
            buf = enc_a + b"\xff\xd9" + bytes(8)
            assert port.Huff.decode(h, buf, 400) == [int(d) for d in diffs]
            assert ref.huff_decode(ht.ncpl, ht.values, buf, 400, True, fix16) == [int(d) for d in diffs]
