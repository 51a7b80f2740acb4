"""Pins the oracle's restatement of the remaining UncompressedDecompressor members
(decode8BitRaw, decode12BitRawWithControl, decode12BitRawUnpackedLeftAligned, the
F32-image branches of readUncompressedRaw) against the UNMODIFIED reference in
oracle/_ref/libref.so: same seeded inputs, whole uncropped buffers compared
bit-for-bit (float results as uint32 patterns).  CPU only."""
import numpy as np
import pytest

import oracle
from oracle import port, synth

ref = oracle.ref
pytestmark = pytest.mark.skipif(not oracle.ref.available(), reason="no reference answers (oracle/_ref or tests/golden/ref_calls)")


def both(data, mk_img, w, cpp, crop, pitch, bps, order, form, curve=None, dither=False):
    a, b = mk_img(), mk_img()
    table = port.build_table(curve, dither) if curve is not None else None
    ea = eb = None
    try:
        port.unpack_form(data, a, w, cpp, crop, pitch, bps, order, form, table, dither)
    except port.OracleError as e:
        ea = e
    try:
        ref.unpack_form(data, b, w, cpp, crop, pitch, bps, order, form, curve, dither)
    except port.OracleError as e:
        eb = e
    assert type(ea) is type(eb), (ea, eb)
    if ea is not None:
        assert ea.msg[:30] in eb.msg, (ea.msg, eb.msg)  # the reference prepends "func, line N: "
    assert np.array_equal(a, b)
    return a, ea


@pytest.mark.parametrize("form", [port.FORM_8BIT, port.FORM_8BIT_UNCORRECTED])
@pytest.mark.parametrize("curve_kind", ["none", "plain", "dither", "short"])
def test_decode8bit(form, curve_kind):
    w, h = 70, 9
    data = synth.lcg_bytes(w * h + 5, seed=3)
    curve, dither = None, False
    if curve_kind != "none":
        n = 256 if curve_kind != "short" else 100
        curve = (np.arange(n, dtype=np.uint32) ** 2 // 2 % 65536).astype(np.uint16)
        curve[n // 2] = 3  # non-monotonic spot
        dither = curve_kind == "dither"
    img, err = both(data, lambda: port.new_image(w, h), w, 1, (0, 0, w, h), w, 8, port.LSB,
                    form, curve, dither)
    assert err is None
    if form == port.FORM_8BIT_UNCORRECTED or curve is None:
        assert np.array_equal(img[:, :w], data[:w * h].reshape(h, w))


@pytest.mark.parametrize("form", [port.FORM_12BIT_CONTROL_BE, port.FORM_12BIT_CONTROL_LE])
@pytest.mark.parametrize("w", [10, 20, 38, 46, 64, 100])
def test_decode12_with_control(form, w):
    h = 7
    perline = 12 * w // 8 + (w + 2) // 10
    data = synth.lcg_bytes(perline * h, seed=w)
    img, err = both(data, lambda: port.new_image(w, h), w, 1, (0, 0, w, h), perline, 12,
                    port.MSB, form)
    assert err is None
    assert int(img[:, :w].max()) < 4096


@pytest.mark.parametrize("form", [port.FORM_12BIT_LEFT_BE, port.FORM_12BIT_LEFT_LE])
def test_decode12_left_aligned(form):
    w, h = 37, 5
    data = synth.lcg_bytes(2 * w * h, seed=9)
    img, err = both(data, lambda: port.new_image(w, h), w, 1, (0, 0, w, h), 2 * w, 16,
                    port.LSB, form)
    assert err is None


@pytest.mark.parametrize("order", [port.LSB, port.MSB])
@pytest.mark.parametrize("bps", [16, 24, 32])
@pytest.mark.parametrize("cpp", [1, 3])
def test_float_forms(order, bps, cpp):
    w, h, ox, oy = 24, 6, 4, 1
    W, H = w + 8, h + 2
    pitch = w * cpp * bps // 8 + 4
    data = synth.lcg_bytes(pitch * h, seed=bps + cpp).copy()
    # every class of narrow float: zero, subnormal, normal, inf, NaN (both signs)
    specials16 = [0x0000, 0x8000, 0x0001, 0x83FF, 0x0400, 0x7BFF, 0x7C00, 0xFC00, 0x7C01, 0xFE00]
    specials24 = [0x000000, 0x800000, 0x000001, 0x80FFFF, 0x010000, 0x7EFFFF, 0x7F0000,
                  0xFF0000, 0x7F0001, 0xFF8000]
    for i, v in enumerate(specials16 if bps == 16 else specials24 if bps == 24 else []):
        nb = bps // 8
        b = [(v >> (8 * k)) & 255 for k in range(nb)]
        if order == port.MSB:
            b = b[::-1]
        data[i * nb:(i + 1) * nb] = b
    img, err = both(data, lambda: port.new_image_f32(W, H, cpp), W, cpp, (ox, oy, w, h), pitch,
                    bps, order, port.FORM_READ)
    assert err is None
    if bps == 16:  # cross-check against numpy's own half -> float conversion (finite values)
        raw = np.frombuffer(data.tobytes(), dtype=np.uint8).reshape(h, pitch)[:, :w * cpp * 2]
        halfs = raw.reshape(h, -1, 2)
        v16 = (halfs[..., 0].astype(np.uint16) << 8 | halfs[..., 1]) if order == port.MSB else \
              (halfs[..., 1].astype(np.uint16) << 8 | halfs[..., 0])
        want = v16.view(np.float16).astype(np.float32).view(np.uint32)
        col0 = ox  # decodePackedFP writes out(row, offset.x + col): NOT offset.x * cpp
        got = img[oy:oy + h, col0:col0 + w * cpp]
        fin = np.isfinite(v16.view(np.float16)) 
        assert np.array_equal(got[fin], want[fin])


def test_float_unsupported_combination_throws():
    w, h = 8, 2
    data = synth.lcg_bytes(64, seed=1)
    for bps, order in [(16, port.MSB16), (24, port.MSB32), (12, port.MSB)]:
        _, err = both(data, lambda: port.new_image_f32(w, h), w, 1, (0, 0, w, h),
                      w * bps // 8, bps, order, port.FORM_READ)
        assert isinstance(err, port.RawDecoderException)


@pytest.mark.parametrize("form,bpl", [(port.FORM_8BIT, 1.0), (port.FORM_12BIT_CONTROL_BE, 1.6),
                                      (port.FORM_12BIT_LEFT_LE, 2.0)])
def test_truncated_input_is_ioe(form, bpl):
    w, h = 20, 6
    perline = {1.0: w, 1.6: 12 * w // 8 + (w + 2) // 10, 2.0: 2 * w}[bpl]
    ctor_pitch = w  # the constructor is given an 8-bit geometry by these callers
    for have_rows in (0, 3):
        data = synth.lcg_bytes(max(perline * have_rows + 2, ctor_pitch * h), seed=5)
        # ctor wants h*ctor_pitch bytes; the member then needs h*perline
        _, err = both(data, lambda: port.new_image(w, h), w, 1, (0, 0, w, h), ctor_pitch, 8,
                      port.LSB, form)
        if perline * h > data.size:
            assert isinstance(err, port.IOException)
        else:
            assert err is None


def test_odd_width_with_control_is_ioe():
    w, h = 7, 2   # 12*7 % 8 != 0
    data = synth.lcg_bytes(64, seed=2)
    _, err = both(data, lambda: port.new_image(w, h), w, 1, (0, 0, w, h), w, 8, port.LSB,
                  port.FORM_12BIT_CONTROL_LE)
    assert isinstance(err, port.IOException)


@pytest.mark.parametrize("bps", [16, 24, 32])
@pytest.mark.parametrize("big_endian", [False, True])
def test_float_dng_tiles(bps, big_endian):
    """Floating-point DNG, compression 1: AbstractDngDecompressor over an F32 image
    (bps 16/24 are always read MSB; 32 follows the tile byte order... as raw copy)."""
    W, H, tw, th = 100, 60, 32, 16
    pitch = tw * bps // 8
    ntiles = 4 * 4
    blob = synth.lcg_bytes(pitch * th * ntiles + 64, bps)
    offs = [7 + n * pitch * th for n in range(ntiles)]
    lens = [pitch * th] * ntiles
    a, b = port.new_image_f32(W, H), port.new_image_f32(W, H)
    port.dng_decompress(blob, offs, lens, a, W, 1, tw, th, 1, bps=bps, big_endian=big_endian)
    ref.dng_decompress(blob, offs, lens, b, W, 1, tw, th, 1, bps=bps, big_endian=big_endian)
    assert np.array_equal(a, b)
