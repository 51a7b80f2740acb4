"""ctypes binding of oracle/_ref/libref.so -- the UNMODIFIED reference compiled
from /root/reference (see oracle/Makefile, oracle/ref_driver.cpp).
TEST INFRASTRUCTURE ONLY."""
import ctypes as C
import os
import subprocess

import numpy as np

from .port import (Err, raise_for, _u8, Huff, JPEG)  # noqa: F401

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "_ref", "libref.so")
REF_SRC = "/root/reference/src/librawspeed"


class HuffDesc(C.Structure):
    _fields_ = [("ncpl", C.c_uint8 * 16), ("values", C.c_uint8 * 162),
                ("nvalues", C.c_int)]


def build():
    """Build _ref/libref.so when the reference sources are present; elsewhere a
    prebuilt file is used as-is."""
    if os.path.isdir(REF_SRC):
        subprocess.check_call(["make", "-s", "-C", _HERE, "-j8", "ref"])
    return os.path.exists(_LIB)


def live():
    """The compiled reference itself can be called (timings need it)."""
    return os.path.exists(_LIB) and os.environ.get("RSB200_REF") != "replay"


def available():
    """The reference's answers are at hand: live, or replayed from the recorded calls."""
    if live():
        return True
    _watch_port()
    return os.path.isdir(GOLDEN)


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB):
            build()
        _lib = C.CDLL(_LIB)
        _lib.ref_encode_diffs.restype = C.c_int64
    return _lib


def image_pitch(w, h, cpp=1):
    return lib().ref_image_pitch(w, h, cpp)


def pump_getbits(order, data, lens, want_pos=False):
    p, n = _u8(data)
    lens_a = (C.c_int * len(lens))(*lens)
    out = (C.c_uint32 * len(lens))()
    pos = C.c_int(0)
    e = Err()
    rc = lib().ref_pump_getbits(order, p, n, lens_a, len(lens), out, C.byref(pos),
                                C.byref(e))
    e.check(rc)
    return (list(out), pos.value) if want_pos else list(out)


def huff_check(ncpl, values, full=True, fix16=False):
    e = Err()
    rc = lib().ref_huff_check(bytes(ncpl), bytes(values), len(values), int(full),
                              int(fix16), C.byref(e))
    e.check(rc)


def huff_decode(ncpl, values, data, n, full=True, fix16=False, order=JPEG):
    p, sz = _u8(data)
    out = (C.c_int32 * n)()
    e = Err()
    rc = lib().ref_huff_decode(bytes(ncpl), bytes(values), len(values), int(full),
                               int(fix16), order, p, sz, n, out, C.byref(e))
    e.check(rc)
    return list(out)


def encode_diffs(diffs, ncpl, values, fix16=False):
    d = np.ascontiguousarray(diffs, dtype=np.int32)
    cap = d.size * 5 + 64
    out = np.empty(cap, dtype=np.uint8)
    n = lib().ref_encode_diffs(d.ctypes.data_as(C.c_void_p), C.c_uint64(d.size),
                               bytes(ncpl), bytes(values), len(values), int(fix16),
                               out.ctypes.data_as(C.c_void_p), C.c_uint64(cap))
    if n < 0:
        raise ValueError("ref_encode_diffs failed")
    return out[:n].tobytes()


def _descs(tabs):
    arr = (HuffDesc * len(tabs))()
    for i, t in enumerate(tabs):
        for k in range(16):
            arr[i].ncpl[k] = t.ncpl[k]
        for k, v in enumerate(t.values):
            arr[i].values[k] = v
        arr[i].nvalues = len(t.values)
    return arr


def unpack(data, img, w, cpp, crop, in_pitch, bps, order, reps=1):
    p, n = _u8(data)
    ms = C.c_double(0)
    e = Err()
    rc = lib().ref_unpack(p, C.c_uint32(n), C.c_void_p(img.ctypes.data), w,
                          img.shape[0], cpp, img.shape[1] * 2, crop[0], crop[1],
                          crop[2], crop[3], in_pitch, bps, order, reps, C.byref(ms),
                          C.byref(e))
    e.check(rc)
    return ms.value


def unpack_form(data, img, w, cpp, crop, in_pitch, bps, order, form, curve=None,
                dither=False, reps=1):
    """Reference UncompressedDecompressor members other than the packed-int read
    (ref_unpack_form): img uint16, or uint32 (= F32 image bit patterns)."""
    p, n = _u8(data)
    ms = C.c_double(0)
    e = Err()
    cp, nc = None, 0
    if curve is not None:
        curve = np.ascontiguousarray(curve, dtype=np.uint16)
        cp, nc = curve.ctypes.data_as(C.POINTER(C.c_uint16)), curve.size
    L = lib()
    L.ref_unpack_form.argtypes = [C.c_char_p, C.c_uint32, C.c_void_p] + [C.c_int] * 13 + \
        [C.POINTER(C.c_uint16), C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double),
         C.POINTER(Err)]
    rc = L.ref_unpack_form(p, C.c_uint32(n), C.c_void_p(img.ctypes.data),
                           int(img.dtype == np.uint32), w, img.shape[0], cpp,
                           img.shape[1] * img.itemsize, crop[0], crop[1], crop[2], crop[3],
                           in_pitch, bps, order, form, cp, nc, int(dither), reps,
                           C.byref(ms), C.byref(e))
    e.check(rc)
    return ms.value


def ljpeg_decompress(img, w, cpp, img_frame, mcu, frame_dim, tabs, tab_of_comp,
                     init_pred, rows_per_restart, data, fix16=False):
    p, n = _u8(data)
    toc = (C.c_int * len(tab_of_comp))(*tab_of_comp)
    ip = (C.c_uint16 * len(init_pred))(*init_pred)
    consumed = C.c_uint32(0)
    e = Err()
    rc = lib().ref_ljpeg_decompress(
        C.c_void_p(img.ctypes.data), w, img.shape[0], cpp, img.shape[1] * 2,
        img_frame[0], img_frame[1], img_frame[2], img_frame[3], mcu[0], mcu[1],
        frame_dim[0], frame_dim[1], _descs(tabs), toc, ip, len(tab_of_comp),
        int(fix16), rows_per_restart, p, C.c_uint32(n), C.byref(consumed),
        C.byref(e))
    e.check(rc)
    return consumed.value


def ljpeg_decode(blob, img, w, cpp, off, size, max_dim, fix16=False):
    p, n = _u8(blob)
    e = Err()
    rc = lib().ref_ljpeg_decode(p, C.c_uint32(n), C.c_void_p(img.ctypes.data), w,
                                img.shape[0], cpp, img.shape[1] * 2, off[0], off[1],
                                size[0], size[1], max_dim[0], max_dim[1], int(fix16),
                                C.byref(e))
    e.check(rc)
    return img


def dng_decompress(file_bytes, tile_off, tile_len, img, w, cpp, tile_w, tile_h,
                   compression, fix_ljpeg=False, bps=14, big_endian=False,
                   nthreads=1, reps=1):
    """Returns best-of-`reps` wall time (ms) of AbstractDngDecompressor::decompress()."""
    p, n = _u8(file_bytes)
    offs = (C.c_uint64 * len(tile_off))(*tile_off)
    lens = (C.c_uint32 * len(tile_len))(*tile_len)
    ms = C.c_double(0)
    e = Err()
    rc = lib().ref_dng_decompress(p, C.c_uint64(n), offs, lens, len(tile_off),
                                  C.c_void_p(img.ctypes.data), int(img.dtype == np.uint32),
                                  w, img.shape[0], cpp, img.shape[1] * img.itemsize, tile_w,
                                  tile_h, compression, int(fix_ljpeg), bps, int(big_endian),
                                  nthreads, reps, C.byref(ms), C.byref(e))
    e.check(rc)
    return ms.value


def pentax_decompress(img, w, data, meta=None, meta_be=True, reps=1):
    p, n = _u8(data)
    mp, mn = (None, 0) if meta is None else _u8(meta)
    ms = C.c_double(0)
    e = Err()
    L = lib()
    L.ref_pentax_decompress.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_char_p,
                                        C.c_int, C.c_int, C.c_char_p, C.c_uint32, C.c_int,
                                        C.POINTER(C.c_double), C.POINTER(Err)]
    rc = L.ref_pentax_decompress(C.c_void_p(img.ctypes.data), w, img.shape[0],
                                 img.shape[1] * 2, mp, mn, int(meta_be), p, C.c_uint32(n),
                                 reps, C.byref(ms), C.byref(e))
    e.check(rc)
    return ms.value


def nikon_decompress(img, w, meta, meta_be, bits, data, uncorrected=False, reps=1):
    """Reference NikonDecompressor (ref_nikon_decompress)."""
    mp, mn = _u8(meta)
    p, n = _u8(data)
    ms = C.c_double(0)
    e = Err()
    L = lib()
    L.ref_nikon_decompress.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_char_p,
                                       C.c_uint32, C.c_int, C.c_int, C.c_char_p, C.c_uint32,
                                       C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(Err)]
    rc = L.ref_nikon_decompress(C.c_void_p(img.ctypes.data), w, img.shape[0], img.shape[1] * 2,
                                mp, C.c_uint32(mn), int(meta_be), bits, p, C.c_uint32(n),
                                int(uncorrected), reps, C.byref(ms), C.byref(e))
    e.check(rc)
    return ms.value


def hasselblad_ljpeg_decode(blob, img, w):
    """Reference HasselbladLJpegDecoder(blob, img).decode() (ref_hasselblad_ljpeg_decode)."""
    p, n = _u8(blob)
    e = Err()
    L = lib()
    L.ref_hasselblad_ljpeg_decode.argtypes = [C.c_char_p, C.c_uint32, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                              C.c_void_p]
    rc = L.ref_hasselblad_ljpeg_decode(p, C.c_uint32(n), C.c_void_p(img.ctypes.data), w, img.shape[0],
                                       img.shape[1] * 2, C.byref(e))
    e.check(rc)
    return img


def hasselblad_decompress(img, w, ncpl, values, full, init_pred, data):
    """Reference HasselbladDecompressor (ref_hasselblad_decompress); returns the stream position."""
    p, n = _u8(data)
    consumed = C.c_uint32(0)
    ms = C.c_double(0)
    e = Err()
    L = lib()
    L.ref_hasselblad_decompress.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_char_p,
                                            C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_char_p,
                                            C.c_uint32, C.POINTER(C.c_uint32), C.c_int,
                                            C.POINTER(C.c_double), C.POINTER(Err)]
    rc = L.ref_hasselblad_decompress(C.c_void_p(img.ctypes.data), w, img.shape[0],
                                     img.shape[1] * 2, bytes(ncpl), bytes(values), len(values),
                                     int(full), init_pred, p, C.c_uint32(n), C.byref(consumed), 1,
                                     C.byref(ms), C.byref(e))
    e.check(rc)
    return consumed.value


def phaseone(img, w, file, strips, nthreads=1, reps=1):
    """Reference PhaseOneDecompressor (ref_phaseone); strips: [(offset, size, row)]."""
    from .port import _strips
    p, n = _u8(file)
    off, ln, rown, ns = _strips(strips)
    ms = C.c_double(0)
    e = Err()
    L = lib()
    L.ref_phaseone.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_char_p, C.c_uint64,
                               C.POINTER(C.c_uint64), C.POINTER(C.c_uint32), C.POINTER(C.c_int32),
                               C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(Err)]
    rc = L.ref_phaseone(C.c_void_p(img.ctypes.data), w, img.shape[0], img.shape[1] * 2, p,
                        C.c_uint64(n), off, ln, rown, ns, nthreads, reps, C.byref(ms), C.byref(e))
    e.check(rc)
    return ms.value


def panasonic_v4(img, w, data, zero_is_not_bad=True, split=0, cap=1 << 16, nthreads=1):
    """Reference PanasonicV4Decompressor (ref_panasonic_v4); returns the sorted bad-pixel list."""
    p, n = _u8(data)
    z = (C.c_uint32 * cap)()
    nz = C.c_uint32(0)
    e = Err()
    L = lib()
    L.ref_panasonic_v4.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_char_p, C.c_uint32,
                                   C.c_int, C.c_uint32, C.POINTER(C.c_uint32), C.c_uint32,
                                   C.POINTER(C.c_uint32), C.c_int, C.POINTER(Err)]
    rc = L.ref_panasonic_v4(C.c_void_p(img.ctypes.data), w, img.shape[0], img.shape[1] * 2, p,
                            C.c_uint32(n), int(zero_is_not_bad), split, z, cap, C.byref(nz),
                            nthreads, C.byref(e))
    e.check(rc)
    return list(z[:min(nz.value, cap)])


def panasonic(version, img, w, data, bps=14, nthreads=1, reps=1):
    """Reference PanasonicV{5,6,7}Decompressor (ref_panasonic)."""
    p, n = _u8(data)
    ms = C.c_double(0)
    e = Err()
    L = lib()
    L.ref_panasonic.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_char_p,
                                C.c_uint32, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double),
                                C.POINTER(Err)]
    rc = L.ref_panasonic(version, C.c_void_p(img.ctypes.data), w, img.shape[0], img.shape[1] * 2,
                         p, C.c_uint32(n), bps, nthreads, reps, C.byref(ms), C.byref(e))
    e.check(rc)
    return ms.value


def last_ms():
    """Wall ms of the reference call inside the last post-decode driver (scale_values,
    scale_black_white, sixteen_bit_lookup, fix_bad_pixels, dng_opcodes); driver copies excluded."""
    L = lib()
    L.ref_last_ms.restype = C.c_double
    return float(L.ref_last_ms())


def dng_opcodes(img, w, cpp, crop, data, cap=1 << 20):
    """Reference DngOpcodes(ri, data) + applyOpCodes(ri) (ref_dng_opcodes); img: uint16 image or
    uint32 array holding an F32 image.  Returns (crop, mBadPixelPositions); `dng_opcodes.stage`
    = which half threw (1 constructor, 2 apply, 0 none)."""
    p, n = _u8(data)
    cr = (C.c_int * 4)(*[int(v) for v in crop])
    bad = (C.c_uint32 * cap)()
    nbad = C.c_uint32(0)
    stage = C.c_int(0)
    e = Err()
    L = lib()
    is_f32 = img.dtype == np.uint32
    L.ref_dng_opcodes.argtypes = [C.c_void_p] + [C.c_int] * 5 + [C.POINTER(C.c_int), C.c_char_p,
                                  C.c_uint32, C.POINTER(C.c_uint32), C.c_uint32,
                                  C.POINTER(C.c_uint32), C.POINTER(C.c_int), C.POINTER(Err)]
    rc = L.ref_dng_opcodes(C.c_void_p(img.ctypes.data), int(is_f32), w, img.shape[0], cpp,
                           img.shape[1] * (4 if is_f32 else 2), cr, p, C.c_uint32(n), bad, cap,
                           C.byref(nbad), C.byref(stage), C.byref(e))
    dng_opcodes.stage = stage.value
    dng_opcodes.partial = (list(cr), list(bad[:min(nbad.value, cap)]))
    e.check(rc)
    return list(cr), list(bad[:min(nbad.value, cap)])


def sixteen_bit_lookup(img, w, cpp, crop, curve, dither, nthreads=1):
    """Reference setTable(curve, dither) + sixteenBitLookup() (ref_sixteen_bit_lookup)."""
    cr = (C.c_int * 4)(*[int(v) for v in crop])
    cp, nc = None, 0
    if curve is not None:
        curve = np.ascontiguousarray(curve, dtype=np.uint16)
        cp, nc = curve.ctypes.data_as(C.POINTER(C.c_uint16)), curve.size
    e = Err()
    L = lib()
    L.ref_sixteen_bit_lookup.argtypes = [C.c_void_p] + [C.c_int] * 4 + [C.POINTER(C.c_int),
                                         C.POINTER(C.c_uint16), C.c_int, C.c_int, C.c_int, C.POINTER(Err)]
    e.check(L.ref_sixteen_bit_lookup(C.c_void_p(img.ctypes.data), w, img.shape[0], cpp, img.shape[1] * 2,
                                     cr, cp, nc, int(dither), nthreads, C.byref(e)))
    return img


def fix_bad_pixels(img, w, cpp, positions, is_cfa=True, nthreads=1):
    """Reference RawImageData::fixBadPixels() (ref_fix_bad_pixels)."""
    pos = np.ascontiguousarray(positions, dtype=np.uint32)
    e = Err()
    L = lib()
    L.ref_fix_bad_pixels.argtypes = [C.c_void_p] + [C.c_int] * 5 + [C.c_void_p, C.c_uint32, C.c_int,
                                                                    C.POINTER(Err)]
    e.check(L.ref_fix_bad_pixels(C.c_void_p(img.ctypes.data), w, img.shape[0], cpp, img.shape[1] * 2,
                                 int(is_cfa), pos.ctypes.data, pos.size, nthreads, C.byref(e)))
    return img


def scale_values(img, w, crop, black_sep, white, dither=True, nthreads=1):
    """Reference RawImageData::scaleBlackWhite() with blackLevelSeparate / whitePoint given
    (ref_scale_values); crop = (off_x, off_y, crop_w, crop_h)."""
    b = (C.c_int * 4)(*[int(v) for v in black_sep])
    e = Err()
    L = lib()
    L.ref_scale_values.argtypes = [C.c_void_p] + [C.c_int] * 7 + [C.POINTER(C.c_int)] + \
        [C.c_int] * 3 + [C.POINTER(Err)]
    rc = L.ref_scale_values(C.c_void_p(img.ctypes.data), w, img.shape[0], img.shape[1] * 2,
                            crop[0], crop[1], crop[2], crop[3], b, int(white), int(dither),
                            nthreads, C.byref(e))
    e.check(rc)
    return img


def scale_black_white(img, w, crop, black_level=-1, black_sep=None, white=None, areas=(),
                      dither=True, is_cfa=True, nthreads=1, cpp=1):
    """Reference RawImageData::scaleBlackWhite() (ref_scale_black_white); areas:
    [(is_vertical, offset, size)].  Returns (blackLevelSeparate or None, whitePoint)."""
    b = (C.c_int * 4)(*([int(v) for v in black_sep] if black_sep is not None else [-7] * 4))
    wh = C.c_int(int(white) if white is not None else 0)
    flat = [int(x) for a in areas for x in a] or [0]
    ar = (C.c_int * len(flat))(*flat)
    sep_set = C.c_int(0)
    e = Err()
    L = lib()
    L.ref_scale_black_white.argtypes = [C.c_void_p] + [C.c_int] * 10 + [C.POINTER(C.c_int), C.c_int,
                                        C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_int)] + \
        [C.c_int] * 3 + [C.POINTER(C.c_int), C.POINTER(Err)]
    rc = L.ref_scale_black_white(C.c_void_p(img.ctypes.data), w, img.shape[0], cpp, img.shape[1] * 2,
                                 int(is_cfa), crop[0], crop[1], crop[2], crop[3], int(black_level),
                                 b, int(black_sep is not None), C.byref(wh), int(white is not None),
                                 ar, len(areas), int(dither), nthreads, C.byref(sep_set),
                                 C.byref(e))
    e.check(rc)
    return (list(b) if sep_set.value else None), wh.value


def sony_arw2(img, w, data, curve=None, dither=False, nthreads=1, reps=1):
    """Reference SonyArw2Decompressor (ref_sony_arw2); curve: mRaw->setTable(curve, dither)."""
    p, n = _u8(data)
    ms = C.c_double(0)
    e = Err()
    cp, nc = None, 0
    if curve is not None:
        curve = np.ascontiguousarray(curve, dtype=np.uint16)
        cp, nc = curve.ctypes.data_as(C.POINTER(C.c_uint16)), curve.size
    L = lib()
    L.ref_sony_arw2.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_char_p, C.c_uint32,
                                C.POINTER(C.c_uint16), C.c_int, C.c_int, C.c_int, C.c_int,
                                C.POINTER(C.c_double), C.POINTER(Err)]
    rc = L.ref_sony_arw2(C.c_void_p(img.ctypes.data), w, img.shape[0], img.shape[1] * 2, p,
                         C.c_uint32(n), cp, nc, int(dither), nthreads, reps, C.byref(ms),
                         C.byref(e))
    e.check(rc)
    return ms.value


def sraw_interpolate(inp, in_w, out, out_w, sub, coeffs, hue, version, nthreads=1, reps=1):
    """Reference Cr2sRawInterpolator; returns best wall ms."""
    k = (C.c_int * 3)(*coeffs)
    ms = C.c_double(0)
    e = Err()
    L = lib()
    L.ref_sraw_interpolate.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p] + \
        [C.c_int] * 5 + [C.POINTER(C.c_int)] + [C.c_int] * 4 + [C.POINTER(C.c_double),
                                                               C.POINTER(Err)]
    rc = L.ref_sraw_interpolate(inp.ctypes.data, in_w, inp.shape[0], inp.shape[1] * 2,
                                out.ctypes.data, out_w, out.shape[0], out.shape[1] * 2,
                                sub[0], sub[1], k, hue, version, nthreads, reps, C.byref(ms),
                                C.byref(e))
    e.check(rc)
    return ms.value


def cr2_decompress(img, w, fmt, frame, slicing, tabs, tab_of_comp, init_pred, data,
                   is_cfa=True, reps=1, want_ms=False):
    p, n = _u8(data)
    toc = (C.c_int * len(tab_of_comp))(*tab_of_comp)
    ip = (C.c_uint16 * len(init_pred))(*init_pred)
    consumed = C.c_uint32(0)
    ms = C.c_double(0)
    e = Err()
    rc = lib().ref_cr2_decompress(C.c_void_p(img.ctypes.data), w, img.shape[0],
                                  img.shape[1] * 2, int(is_cfa), fmt[0], fmt[1],
                                  fmt[2], frame[0], frame[1], slicing[0], slicing[1],
                                  slicing[2], _descs(tabs), toc, ip,
                                  len(tab_of_comp), p, C.c_uint32(n),
                                  C.byref(consumed), reps, C.byref(ms), C.byref(e))
    e.check(rc)
    return (consumed.value, ms.value) if want_ms else consumed.value


def cr2_ljpeg_decode(blob, img, w, slicing, is_cfa=True, sub=(1, 1), reps=1):
    p, n = _u8(blob)
    ms = C.c_double(0)
    e = Err()
    rc = lib().ref_cr2_ljpeg_decode(p, C.c_uint32(n), C.c_void_p(img.ctypes.data), w,
                                    img.shape[0], img.shape[1] * 2, int(is_cfa),
                                    sub[0], sub[1], slicing[0], slicing[1],
                                    slicing[2], reps, C.byref(ms), C.byref(e))
    e.check(rc)
    return ms.value


# ---- recorded calls -----------------------------------------------------------------------------
# The reference sources are not part of this repository, so libref.so exists only where they were
# at hand.  Elsewhere the tests that pin the oracle against the reference replay what the reference
# answered for the very same inputs.  Each call is keyed by a digest of its arguments; its answer is
# stored under tests/golden/ref_calls/<function>.txt.gz: the return value, the error it raised, the
# attributes it set, and a digest of every array it wrote.  The content of a written array comes
# from the restatement (oracle.port), run on the same inputs in the same test: a port call whose
# array has exactly the digest the reference recorded supplies it, before or after the replayed
# call, and `unmatched()` (checked after every test) lists answers the restatement never produced.
# So the tests still compare oracle and reference bit for bit, through the digest.
#
# RSB200_REF_RECORD=1 (with libref.so built) records every call the suite makes, merged into the
# files when the process exits (so record in one process, not under pytest -n); RSB200_REF=replay
# ignores libref.so.  A call that was never recorded is an error: its inputs changed, so the
# answers must be recorded again.

import ast  # noqa: E402
import atexit  # noqa: E402
import collections  # noqa: E402
import functools  # noqa: E402
import gzip  # noqa: E402
import hashlib  # noqa: E402
import zlib  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(_HERE), "tests", "golden", "ref_calls")
_ATTRS = ("stage", "partial")   # what dng_opcodes leaves on the function object
_WHOLE = ("hasselblad_ljpeg_decode",)   # no restatement to supply the arrays: stored whole
_recorded = {}                  # function name -> {key: answer}, being recorded
_answers = {}                   # function name -> {key: answer}, being replayed
_seen = collections.OrderedDict()   # digest -> bytes of arrays the restatement read or wrote lately
_pending = []                   # (array, digest, function) the reference wrote, content not yet seen


def _feed(h, v):
    if isinstance(v, np.ndarray):
        h.update(b"A%s%s:" % (v.dtype.str.encode(), repr(v.shape).encode()))
        h.update(np.ascontiguousarray(v).tobytes())
    elif isinstance(v, (bytes, bytearray, memoryview)):
        b = bytes(v)
        h.update(b"B%d:" % len(b) + b)
    elif isinstance(v, (list, tuple)):
        h.update(b"L%d[" % len(v))
        for x in v:
            _feed(h, x)
        h.update(b"]")
    elif hasattr(v, "ncpl") and hasattr(v, "values"):   # a Huffman table: all _descs reads
        _feed(h, (v.ncpl, v.values))
    elif isinstance(v, (bool, np.bool_)):
        h.update(b"Z%d" % bool(v))
    elif isinstance(v, (int, np.integer)):
        h.update(b"I%d" % int(v))
    elif isinstance(v, (float, np.floating)):
        h.update(b"F" + float(v).hex().encode())
    elif v is None or isinstance(v, str):
        h.update(b"S" + repr(v).encode())
    else:
        raise TypeError("cannot key a reference call on %r" % type(v))


def _digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:32]


def _arrays(args, kwargs):
    return [("a%d" % i, a) for i, a in enumerate(args) if isinstance(a, np.ndarray)] + \
           [("k_" + k, a) for k, a in sorted(kwargs.items()) if isinstance(a, np.ndarray)]


def _record(name, fn, key, args, kwargs):
    before = {lab: a.tobytes() for lab, a in _arrays(args, kwargs)}
    exc = ret = None
    try:
        ret = fn(*args, **kwargs)
    except (RawDecoderException, IOException) as ex:
        exc = ex
    wrapper = globals()[name]
    argref = [lab for lab, a in _arrays(args, kwargs) if ret is a]
    ans = {"ret": None if argref else ret, "argref": argref[0] if argref else None,
           "exc": None if exc is None else (exc.code, exc.msg),
           "attrs": {k: getattr(wrapper, k) for k in _ATTRS if hasattr(wrapper, k)},
           "out": {lab: _digest(a) for lab, a in _arrays(args, kwargs) if a.tobytes() != before[lab]}}
    if name in _WHOLE:
        ans["whole"] = {lab: zlib.compress(a.tobytes(), 9) for lab, a in _arrays(args, kwargs) if lab in ans["out"]}
    assert ast.literal_eval(repr(ans)) == ans, "reference answer is not a plain literal: %r" % ans
    _recorded.setdefault(name, {})[key] = ans
    if exc is not None:
        raise exc
    return ret


def _fill(a, content):
    a.reshape(-1).view(np.uint8)[:] = np.frombuffer(content, dtype=np.uint8)


def _note(a):
    """The restatement read or wrote `a`: its content may be an answer the reference recorded."""
    if not isinstance(a, np.ndarray) or a.nbytes > (64 << 20):
        return
    d = _digest(a)
    for p in [p for p in _pending if p[1] == d]:
        _fill(p[0], a.tobytes())
        _pending.remove(p)
    _seen[d] = a.tobytes()
    _seen.move_to_end(d)
    while len(_seen) > 256:
        _seen.popitem(last=False)


def _watched(fn):
    @functools.wraps(fn)
    def call(*args, **kwargs):
        arrs = [a for a in list(args) + list(kwargs.values()) if isinstance(a, np.ndarray)]
        for a in arrs:
            _note(a)
        try:
            ret = fn(*args, **kwargs)
        finally:
            for a in arrs:
                _note(a)
        _note(ret)
        return ret
    return call


def _watch_port():
    from . import port
    if getattr(port, "_watched", False):
        return
    import inspect
    for n, f in list(vars(port).items()):
        if inspect.isfunction(f) and f.__module__ == port.__name__ and not n.startswith("_"):
            setattr(port, n, _watched(f))
    port._watched = True


def _play(name, key, args, kwargs):
    _watch_port()
    if name not in _answers:
        path = os.path.join(GOLDEN, name + ".txt.gz")
        _answers[name] = {}
        if os.path.exists(path):
            with gzip.open(path, "rt") as f:
                for ln in f:
                    k, text = ln.split(" ", 1)
                    _answers[name][k] = text
    if key not in _answers[name]:
        raise LookupError("%s: no recorded reference answer for these inputs (key %s); record "
                          "them again with RSB200_REF_RECORD=1 where oracle/_ref is built" % (name, key))
    ans = ast.literal_eval(_answers[name][key])
    arrays = dict(_arrays(args, kwargs))
    for lab, a in arrays.items():
        _note(a)
    for lab, content in ans.get("whole", {}).items():
        _fill(arrays[lab], zlib.decompress(content))
    for lab, d in ans["out"].items():
        if lab in ans.get("whole", {}):
            continue
        if d in _seen:
            _fill(arrays[lab], _seen[d])
        else:
            _pending.append((arrays[lab], d, name))
    for k, v in ans["attrs"].items():
        setattr(globals()[name], k, v)
    if ans["exc"] is not None:
        raise_for(*ans["exc"])
    return arrays[ans["argref"]] if ans["argref"] else ans["ret"]


def unmatched():
    """Replayed reference answers (function names) whose arrays the restatement never produced
    since the last call; clears the list."""
    names = [p[2] for p in _pending]
    del _pending[:]
    return names


def _save():
    os.makedirs(GOLDEN, exist_ok=True)
    for name, calls in _recorded.items():
        path = os.path.join(GOLDEN, name + ".txt.gz")
        lines = {}
        if os.path.exists(path):
            with gzip.open(path, "rt") as f:
                lines = dict(ln.rstrip("\n").split(" ", 1) for ln in f)
        lines.update((k, repr(v)) for k, v in calls.items())
        with gzip.GzipFile(path, "wb", mtime=0) as f:
            f.write("".join("%s %s\n" % kv for kv in sorted(lines.items())).encode())


def _keyed(name, fn):
    @functools.wraps(fn)
    def call(*args, **kwargs):
        h = hashlib.sha256(name.encode())
        _feed(h, list(args))
        _feed(h, sorted(kwargs.items()))
        key = h.hexdigest()[:32]
        if not live():
            return _play(name, key, args, kwargs)
        if os.environ.get("RSB200_REF_RECORD") == "1":
            return _record(name, fn, key, args, kwargs)
        return fn(*args, **kwargs)
    return call


from .port import RawDecoderException, IOException  # noqa: E402

for _name in ("pump_getbits", "huff_check", "huff_decode", "encode_diffs", "unpack", "unpack_form",
              "ljpeg_decompress", "ljpeg_decode", "dng_decompress", "pentax_decompress",
              "nikon_decompress", "hasselblad_ljpeg_decode", "hasselblad_decompress", "phaseone",
              "panasonic_v4", "panasonic", "dng_opcodes", "sixteen_bit_lookup", "fix_bad_pixels",
              "scale_values", "scale_black_white", "sony_arw2", "sraw_interpolate", "cr2_decompress",
              "cr2_ljpeg_decode"):
    globals()[_name] = _keyed(_name, globals()[_name])
if os.environ.get("RSB200_REF_RECORD") == "1":
    atexit.register(_save)
