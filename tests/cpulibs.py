"""ctypes loaders for the two CPU checkers (test infrastructure only):
   - oracle/liboracle.so      : our plain-C restatement (travels, always built by __graft_entry__.build())
   - oracle/_ref/libffref.so  : the unmodified reference compiled by oracle/ref/Makefile (present when built here)
"""
import ctypes as C
import os
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_SO = os.path.join(ROOT, "oracle", "liboracle.so")
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libffref.so")

SWS_FAST_BILINEAR, SWS_BILINEAR, SWS_BICUBIC, SWS_POINT, SWS_AREA, SWS_BICUBLIN = 1, 2, 4, 0x10, 0x20, 0x40
SWS_FULL_CHR_H_INT, SWS_ACCURATE_RND, SWS_BITEXACT = 0x2000, 0x40000, 0x80000

u8p = C.POINTER(C.c_uint8)
i16p = C.POINTER(C.c_int16)
i32p = C.POINTER(C.c_int32)
i64p = C.POINTER(C.c_int64)
u64p = C.POINTER(C.c_uint64)


def ptr(a, t=u8p):
    return a.ctypes.data_as(t)


_oracle = None
_ref = None


def oracle():
    global _oracle
    if _oracle is None:
        L = C.CDLL(ORACLE_SO)
        L.orc_sws_open.restype = C.c_void_p
        L.orc_sws_open.argtypes = [C.c_int] * 5
        L.orc_sws_open_fmt.restype = C.c_void_p
        L.orc_sws_open_fmt.argtypes = [C.c_int] * 6
        L.orc_sws_open_io.restype = C.c_void_p
        L.orc_sws_open_io.argtypes = [C.c_int] * 7
        L.orc_sws_open_range.restype = C.c_void_p
        L.orc_sws_open_range.argtypes = [C.c_int] * 9
        L.orc_sws_set_colorspace_details.argtypes = [C.c_void_p, i32p, C.c_int, i32p, C.c_int, C.c_int, C.c_int, C.c_int]
        L.orc_sws_close.argtypes = [C.c_void_p]
        L.orc_sws_set_colorspace.argtypes = [C.c_void_p, i32p, C.c_int, C.c_int, C.c_int, C.c_int]
        L.orc_sws_scale.argtypes = [C.c_void_p, u8p, C.c_int, u8p, C.c_int, u8p, C.c_int, u8p, C.c_int]
        L.orc_sws_scale_planar.argtypes = [C.c_void_p, u8p, C.c_int, u8p, C.c_int, u8p, C.c_int, u8p, C.c_int, u8p, C.c_int, u8p, C.c_int]
        L.orc_sws_info.argtypes = [C.c_void_p, i32p]
        L.orc_sws_get_filter.argtypes = [C.c_void_p, C.c_int, i16p, i32p, C.c_int]
        L.orc_hscale8to15.argtypes = [i16p, C.c_int, u8p, i16p, i32p, C.c_int]
        if hasattr(L, "orc_idct_batch"):
            L.orc_idct_batch.argtypes = [C.c_int, i16p, C.c_int, u8p, C.c_ssize_t, i64p]
            L.orc_pixels_clamped.argtypes = [C.c_int, i16p, u8p, C.c_ssize_t]
        if hasattr(L, "orc_h264_idct"):
            L.orc_h264_idct.argtypes = [C.c_int, u8p, i16p, C.c_ssize_t]
        if hasattr(L, "orc_me_cmp"):
            L.orc_me_cmp.argtypes = [C.c_int, C.c_int, u8p, u8p, C.c_ssize_t, C.c_int]
            L.orc_esa_frame.argtypes = [u8p, u8p] + [C.c_int] * 7 + [i32p, u64p]
        if hasattr(L, "orc_h264qpel"):
            L.orc_h264qpel.argtypes = [C.c_int, C.c_int, C.c_int, u8p, u8p, C.c_ssize_t]
            L.orc_hpel.argtypes = [C.c_int, C.c_int, C.c_int, u8p, u8p, C.c_ssize_t, C.c_int]
        if hasattr(L, "orc_h264qpel_batch"):
            L.orc_h264qpel_batch.argtypes = [C.c_int, u8p, u8p, i64p, u8p, i64p, C.c_ssize_t]
        if hasattr(L, "orc_emulated_edge_mc"):
            L.orc_emulated_edge_mc.argtypes = [u8p, C.c_void_p, C.c_ssize_t, C.c_ssize_t] + [C.c_int] * 6
            L.orc_emulated_edge_mc.restype = None
        if hasattr(L, "orc_h264_weight"):
            L.orc_h264_weight.argtypes = [C.c_int, u8p, C.c_ssize_t] + [C.c_int] * 4
            L.orc_h264_weight.restype = None
            L.orc_h264_biweight.argtypes = [C.c_int, u8p, u8p, C.c_ssize_t] + [C.c_int] * 5
            L.orc_h264_biweight.restype = None
        if hasattr(L, "orc_h264chroma"):
            L.orc_h264chroma.argtypes = [C.c_int, C.c_int, u8p, u8p, C.c_ssize_t, C.c_int, C.c_int, C.c_int]
        if hasattr(L, "orc_h264chroma_batch"):
            L.orc_h264chroma_batch.argtypes = [C.c_int64, u8p, u8p, u8p, u8p, i64p, u8p, i64p, C.c_ssize_t]
        if hasattr(L, "orc_tx_open"):
            L.orc_tx_open.restype = C.c_void_p
            L.orc_tx_open.argtypes = [C.c_int, C.c_int, C.c_int, C.c_float, C.c_uint]
            L.orc_tx_close.argtypes = [C.c_void_p]
            L.orc_tx_run.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_ssize_t, C.c_int, C.c_ssize_t, C.c_ssize_t]
        _oracle = L
    return _oracle


def have_ref():
    return os.path.exists(REF_SO)


REF_RECORD_DIR = os.path.join(ROOT, "tests", "golden", "ref")


def _digest(a):
    """dtype, shape and contents of an array in 8 hex digits: enough to tell a changed output from the recorded one"""
    import hashlib
    a = np.ascontiguousarray(np.asarray(a))
    return hashlib.sha256(f"{a.dtype.str} {a.shape}".encode() + a.tobytes()).hexdigest()[:8]


class RefRecord:
    """What the compiled reference produced at each comparison point of one test, in the order the test compares, stored as
    digests in tests/golden/ref/<test>.txt.  With oracle/_ref built, same(got, fn) calls fn and compares live, and the reference's
    value must also match the stored digest (FFREF_RECORD=1 rewrites the file instead).  Without it, got is compared with the
    stored digest, so a checkout without the reference keeps every comparison (got must then have the reference value's dtype)."""

    def __init__(self, name):
        self.path = os.path.join(REF_RECORD_DIR, name + ".txt")
        self.live = have_ref()
        self.recording = self.live and os.environ.get("FFREF_RECORD") == "1"
        self.stored = None if self.recording or not os.path.exists(self.path) else open(self.path).read().split("\n")[:-1]
        self.seen = []

    def usable(self):
        return self.live or self.stored is not None

    def same(self, got, fn):
        """True when `got` equals what fn() (a call of the reference) returns; fn is called only when the reference is built"""
        i = len(self.seen)
        if self.live:
            r = np.asarray(fn())
            self.seen.append(_digest(r))
            assert self.stored is None or (i < len(self.stored) and self.stored[i] == self.seen[i]), \
                ("the reference no longer matches " + self.path, i)
            if not np.array_equal(np.asarray(got), r):
                return False
            assert _digest(got) == self.seen[i], ("equal values of another dtype or shape: stored digests could not be checked", i)
            return True
        assert i < len(self.stored), ("more comparisons than " + self.path + " holds", i)
        self.seen.append(self.stored[i])
        return _digest(got) == self.stored[i]

    def close(self):
        if self.recording:
            os.makedirs(REF_RECORD_DIR, exist_ok=True)
            with open(self.path, "w") as f:
                f.write("".join(s + "\n" for s in self.seen))
        elif self.stored is not None:
            assert len(self.seen) == len(self.stored), ("fewer comparisons than " + self.path + " holds", len(self.seen), len(self.stored))


def ref():
    global _ref
    if _ref is None:
        L = C.CDLL(REF_SO)
        L.ffref_set_quiet()
        L.ffref_sws_open.restype = C.c_void_p
        L.ffref_sws_open.argtypes = [C.c_int] * 6
        L.ffref_sws_open_fmt.restype = C.c_void_p
        L.ffref_sws_open_fmt.argtypes = [C.c_int] * 7
        L.ffref_sws_open_io.restype = C.c_void_p
        L.ffref_sws_open_io.argtypes = [C.c_int] * 8
        L.ffref_sws_open_range.restype = C.c_void_p
        L.ffref_sws_open_range.argtypes = [C.c_int] * 10
        L.ffref_sws_close.argtypes = [C.c_void_p]
        L.ffref_sws_set_colorspace.argtypes = [C.c_void_p] + [C.c_int] * 7
        L.ffref_sws_scale.argtypes = [C.c_void_p, u8p, C.c_int, u8p, C.c_int, u8p, C.c_int, C.c_int, C.c_int, u8p, C.c_int]
        L.ffref_sws_scale_planar.argtypes = [C.c_void_p, u8p, C.c_int, u8p, C.c_int, u8p, C.c_int, C.c_int, C.c_int,
                                             u8p, C.c_int, u8p, C.c_int, u8p, C.c_int]
        L.ffref_sws_info.argtypes = [C.c_void_p, i32p]
        L.ffref_sws_get_filter.argtypes = [C.c_void_p, C.c_int, i16p, i32p, C.c_int]
        L.ffref_sws_hscale.argtypes = [C.c_void_p, C.c_int, i16p, C.c_int, u8p, i16p, i32p, C.c_int]
        L.ffref_idct_perm_type.argtypes = [u8p]
        L.ffref_idct_batch.argtypes = [C.c_int, i16p, C.c_int, u8p, C.c_ssize_t, i64p]
        L.ffref_pixels_clamped.argtypes = [C.c_int, i16p, u8p, C.c_ssize_t]
        if hasattr(L, "ffref_h264_idct"):
            L.ffref_h264_idct.argtypes = [C.c_int, u8p, i16p, C.c_ssize_t]
        L.ffref_me_cmp.argtypes = [C.c_int, C.c_int, u8p, u8p, C.c_ssize_t, C.c_int]
        L.ffref_me_cmp_batch.argtypes = [C.c_int, C.c_int, u8p, u8p, C.c_ssize_t, C.c_int, i64p, i64p, C.c_int, i32p]
        L.ffref_esa_frame.argtypes = [u8p, u8p] + [C.c_int] * 7 + [i32p, u64p]
        L.ffref_h264qpel.argtypes = [C.c_int, C.c_int, C.c_int, u8p, u8p, C.c_ssize_t]
        L.ffref_h264qpel_batch.argtypes = [C.c_int, u8p, u8p, i64p, u8p, i64p, C.c_ssize_t]
        L.ffref_hpel.argtypes = [C.c_int, C.c_int, C.c_int, u8p, u8p, C.c_ssize_t, C.c_int]
        if hasattr(L, "ffref_emulated_edge_mc"):
            L.ffref_emulated_edge_mc.argtypes = [u8p, C.c_void_p, C.c_ssize_t, C.c_ssize_t] + [C.c_int] * 6
            L.ffref_emulated_edge_mc.restype = None
        if hasattr(L, "ffref_h264_weight"):
            L.ffref_h264_weight.argtypes = [C.c_int, u8p, C.c_ssize_t] + [C.c_int] * 4
            L.ffref_h264_weight.restype = None
            L.ffref_h264_biweight.argtypes = [C.c_int, u8p, u8p, C.c_ssize_t] + [C.c_int] * 5
            L.ffref_h264_biweight.restype = None
        if hasattr(L, "ffref_h264chroma"):
            L.ffref_h264chroma.argtypes = [C.c_int, C.c_int, u8p, u8p, C.c_ssize_t, C.c_int, C.c_int, C.c_int]
        L.ffref_tx_open.restype = C.c_void_p
        L.ffref_tx_open.argtypes = [C.c_int, C.c_int, C.c_int, C.c_float, C.c_uint]
        L.ffref_tx_close.argtypes = [C.c_void_p]
        L.ffref_tx_run.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_ssize_t, C.c_int, C.c_ssize_t, C.c_ssize_t]
        _ref = L
    return _ref


# ---------------------------------------------------------------- swscale helpers
def yuv_frame(w, h, seed, kind="random", pad=0):
    """Synthetic yuv420p frame; returns (y,u,v) 2-D uint8 arrays (rows padded by `pad` bytes)."""
    rng = np.random.default_rng(seed)
    cw, ch = (w + 1) // 2, (h + 1) // 2
    if kind == "random":
        y = rng.integers(0, 256, (h, w + pad), dtype=np.uint8)
        u = rng.integers(0, 256, (ch, cw + pad), dtype=np.uint8)
        v = rng.integers(0, 256, (ch, cw + pad), dtype=np.uint8)
    elif kind == "limited":
        y = rng.integers(16, 236, (h, w + pad), dtype=np.uint8)
        u = rng.integers(16, 241, (ch, cw + pad), dtype=np.uint8)
        v = rng.integers(16, 241, (ch, cw + pad), dtype=np.uint8)
    else:  # smooth
        yy, xx = np.mgrid[0:h, 0:w + pad]
        y = ((np.sin(xx / 17.0) + np.cos(yy / 11.0)) * 60 + 128).astype(np.uint8)
        yy, xx = np.mgrid[0:ch, 0:cw + pad]
        u = ((np.sin(xx / 9.0 + 1) * np.cos(yy / 13.0)) * 100 + 128).astype(np.uint8)
        v = ((np.cos(xx / 7.0) * np.sin(yy / 5.0 + 2)) * 100 + 128).astype(np.uint8)
    return np.ascontiguousarray(y), np.ascontiguousarray(u), np.ascontiguousarray(v)


PIX_FMT_RGB24, PIX_FMT_BGR24, PIX_FMT_ARGB, PIX_FMT_RGBA, PIX_FMT_ABGR, PIX_FMT_BGRA = 2, 3, 25, 26, 27, 28   # libavutil/pixfmt.h
PACKED_RGB_FORMATS = {"rgb24": PIX_FMT_RGB24, "bgr24": PIX_FMT_BGR24, "argb": PIX_FMT_ARGB, "rgba": PIX_FMT_RGBA,
                      "abgr": PIX_FMT_ABGR, "bgra": PIX_FMT_BGRA}


def fmt_bpp(fmt):
    return 3 if fmt in (PIX_FMT_RGB24, PIX_FMT_BGR24) else 4


PIX_FMT_NV12, PIX_FMT_NV21 = 23, 24


def nv_interleave(u, v, src_fmt, pad=0):
    """U and V planes -> the interleaved plane 1 of an nv12 / nv21 picture (row stride 2*cw + pad)."""
    ch, cw = u.shape[0], u.shape[1]
    uv = np.full((ch, 2 * cw + pad), 0x5C, np.uint8)
    a, b = (u, v) if src_fmt == PIX_FMT_NV12 else (v, u)
    uv[:, 0:2 * cw:2] = a
    uv[:, 1:2 * cw:2] = b
    return uv


def rgb_frame(w, h, seed, bpp, kind="random", pad=0):
    """packed RGB source picture: (h, w*bpp + pad) uint8"""
    rng = np.random.default_rng(seed)
    if kind == "random":
        return rng.integers(0, 256, (h, w * bpp + pad), dtype=np.uint8)
    yy, xx = np.mgrid[0:h, 0:w]
    a = np.full((h, w * bpp + pad), 0x3C, np.uint8)
    for k in range(bpp):
        a[:, k:w * bpp:bpp] = ((xx * 3 + yy * 2 + k * 40) % 256).astype(np.uint8)
    return a


def _open_filters(lib, pre, src_fmt, w, h, sr, fmt, dw, dh, dr, flags, threads, filters, param):
    """filters = (src, dst): src = 4 sequences of doubles (lumH, lumV, chrH, chrV; None = no vector), dst = 4 lengths"""
    src, dst = filters
    arrs = [np.array(v, np.float64) if v is not None and len(v) else None for v in (src or [None] * 4)]
    coef = (C.c_void_p * 4)(*[a.ctypes.data if a is not None else None for a in arrs])
    slen = (C.c_int * 4)(*[len(a) if a is not None else 0 for a in arrs])
    dlen = (C.c_int * 4)(*(dst or [0] * 4))
    pa = (C.c_double * 2)(*param) if param is not None else None
    if pre == "ffref":
        lib.ffref_sws_open_filters.restype, lib.ffref_sws_open_filters.argtypes = C.c_void_p, [C.c_int] * 10 + [C.c_void_p] * 4
        return lib.ffref_sws_open_filters(src_fmt, w, h, sr, fmt, dw, dh, dr, flags, threads, coef, slen, dlen, pa)
    lib.orc_sws_open_filters.restype, lib.orc_sws_open_filters.argtypes = C.c_void_p, [C.c_int] * 9 + [C.c_void_p] * 4
    return lib.orc_sws_open_filters(src_fmt, w, h, sr, fmt, dw, dh, dr, flags, coef, slen, dlen, pa)


def _sws_run(lib, pre, w, h, dw, dh, flags, y, u, v, dst_pad=0, threads=1, colorspace=None, fmt=PIX_FMT_RGB24, src_fmt=0, param=None, filters=None):
    """src_fmt nv12 / nv21: `u` is the interleaved chroma plane, `v` is ignored; param: sws_getContext's two scaler parameters"""
    if filters is not None:
        ctx = _open_filters(lib, pre, src_fmt, w, h, 0, fmt, dw, dh, 0, flags, threads, filters, param)
    elif param is not None:
        pa = (C.c_double * 2)(*param)
        if pre == "ffref":
            lib.ffref_sws_open_params.restype, lib.ffref_sws_open_params.argtypes = C.c_void_p, [C.c_int] * 10 + [C.c_void_p]
            ctx = lib.ffref_sws_open_params(src_fmt, w, h, 0, fmt, dw, dh, 0, flags, threads, pa)
        else:
            lib.orc_sws_open_params.restype, lib.orc_sws_open_params.argtypes = C.c_void_p, [C.c_int] * 9 + [C.c_void_p]
            ctx = lib.orc_sws_open_params(src_fmt, w, h, 0, fmt, dw, dh, 0, flags, pa)
    elif pre == "ffref":
        ctx = lib.ffref_sws_open_io(src_fmt, w, h, fmt, dw, dh, flags, threads)
    else:
        ctx = lib.orc_sws_open_io(src_fmt, w, h, fmt, dw, dh, flags)
    if not ctx:
        return None
    try:
        if colorspace is not None:
            if pre == "ffref":
                lib.ffref_sws_set_colorspace(ctx, *colorspace)
            else:
                tab, tab2 = np.array(COEFFS[colorspace[0]], dtype=np.int32), np.array(COEFFS[colorspace[2]], dtype=np.int32)
                lib.orc_sws_set_colorspace_details.argtypes = [C.c_void_p, i32p, C.c_int, i32p, C.c_int, C.c_int, C.c_int, C.c_int]
                lib.orc_sws_set_colorspace_details(ctx, ptr(tab, i32p), colorspace[1], ptr(tab2, i32p), colorspace[3], colorspace[4], colorspace[5],
                                                   colorspace[6])
        ds = dw * fmt_bpp(fmt) + dst_pad
        # one spare line: rgbToRgbWrapper into argb / abgr from a 24-bit source writes one byte past the last pixel (the alpha of a "next"
        # pixel, swscale_unscaled.c:2030-2042), which real AVFrame buffers absorb in their padding
        dst = np.full((dh + 1, ds), 0xA5, dtype=np.uint8)[:dh]
        if pre == "ffref":
            n = lib.ffref_sws_scale(ctx, ptr(y), y.strides[0], ptr(u), u.strides[0], ptr(v), v.strides[0], 0, h, ptr(dst), ds)
        else:
            n = lib.orc_sws_scale(ctx, ptr(y), y.strides[0], ptr(u), u.strides[0], ptr(v), v.strides[0], ptr(dst), ds)
        assert n == dh, n
        return dst
    finally:
        (lib.ffref_sws_close if pre == "ffref" else lib.orc_sws_close)(ctx)


PIX_FMT_YUV420P = 0


def _sws_run_planar(lib, pre, w, h, dw, dh, flags, y, u, v, dst_pad=0, threads=1, src_fmt=0, ranges=(0, 0), details=None,
                    dst_fmt=PIX_FMT_YUV420P, filters=None):
    """yuv420p / nv12 / nv21 -> yuv420p; returns (Y, U, V) destination planes (pad bytes stay 0xA5).
    ranges = (src_range, dst_range) given before initialisation; details = (src_cs, src_range, dst_cs, dst_range,
    brightness, contrast, saturation) for a sws_setColorspaceDetails() call after it.
    dst_fmt nv12 / nv21: returns (Y, UV) with UV the interleaved plane."""
    if filters is not None:
        ctx = _open_filters(lib, pre, src_fmt, w, h, ranges[0], dst_fmt, dw, dh, ranges[1], flags, threads, filters, None)
    elif pre == "ffref":
        ctx = lib.ffref_sws_open_range(src_fmt, w, h, ranges[0], dst_fmt, dw, dh, ranges[1], flags, threads)
    else:
        ctx = lib.orc_sws_open_range(src_fmt, w, h, ranges[0], dst_fmt, dw, dh, ranges[1], flags)
    if not ctx:
        return None
    try:
        if details is not None:
            if pre == "ffref":
                r = lib.ffref_sws_set_colorspace(ctx, *details)
            else:
                ta, tb = (np.array(COEFFS[k], dtype=np.int32) for k in (details[0], details[2]))
                r = lib.orc_sws_set_colorspace_details(ctx, ptr(ta, i32p), details[1], ptr(tb, i32p), details[3], *details[4:])
            assert r == 0, r
        cw, ch = (dw + 1) // 2, (dh + 1) // 2
        dy = np.full((dh, dw + dst_pad), 0xA5, np.uint8)
        nvd = dst_fmt in (PIX_FMT_NV12, PIX_FMT_NV21)
        du = np.full((ch, (2 * cw if nvd else cw) + dst_pad), 0xA5, np.uint8)
        dv = np.full((ch, cw + dst_pad), 0xA5, np.uint8)
        if pre == "ffref":
            n = lib.ffref_sws_scale_planar(ctx, ptr(y), y.strides[0], ptr(u), u.strides[0], ptr(v), v.strides[0], 0, h,
                                           ptr(dy), dy.strides[0], ptr(du), du.strides[0], ptr(dv), dv.strides[0])
        else:
            n = lib.orc_sws_scale_planar(ctx, ptr(y), y.strides[0], ptr(u), u.strides[0], ptr(v), v.strides[0],
                                         ptr(dy), dy.strides[0], ptr(du), du.strides[0], ptr(dv), dv.strides[0])
        assert n == dh, n
        return (dy, du) if nvd else (dy, du, dv)
    finally:
        (lib.ffref_sws_close if pre == "ffref" else lib.orc_sws_close)(ctx)


def ref_sws_planar(w, h, dw, dh, flags, y, u, v, **kw):
    return _sws_run_planar(ref(), "ffref", w, h, dw, dh, flags, y, u, v, **kw)


def orc_sws_planar(w, h, dw, dh, flags, y, u, v, **kw):
    kw.pop("threads", None)
    return _sws_run_planar(oracle(), "orc", w, h, dw, dh, flags, y, u, v, **kw)


# ---------------------------------------------------------------- mpegvideo inverse quantisers (mpegvideo_unquantize.c)
UNQUANT_VARIANTS = ["mpeg1_intra", "mpeg1_inter", "mpeg2_intra", "mpeg2_intra_bitexact", "mpeg2_inter", "h263_intra", "h263_inter"]
ZIGZAG = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21,
                   28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61,
                   54, 47, 55, 62, 63], np.uint8)                                        # ISO zig-zag scan
ALTERNATE_VERTICAL = np.array([0, 8, 16, 24, 1, 9, 2, 10, 17, 25, 32, 40, 48, 56, 57, 49, 41, 33, 26, 18, 3, 11, 4, 12, 19, 27, 34,
                               42, 50, 58, 35, 43, 51, 59, 20, 28, 5, 13, 6, 14, 21, 29, 36, 44, 52, 60, 37, 45, 53, 61, 22, 30, 7,
                               15, 23, 31, 38, 46, 54, 62, 39, 47, 55, 63], np.uint8)    # ISO 13818-2 figure 7-3


class OrcMpvUnquant(C.Structure):
    _fields_ = [("intra_matrix", C.c_uint16 * 64), ("inter_matrix", C.c_uint16 * 64), ("permutated", C.c_uint8 * 64),
                ("raster_end", C.c_uint8 * 64), ("y_dc_scale", C.c_int32), ("c_dc_scale", C.c_int32), ("q_scale_type", C.c_int32),
                ("h263_aic", C.c_int32), ("ac_pred", C.c_int32)]


def unquant_params(intra_matrix, inter_matrix, alternate_scan, y_dc_scale, c_dc_scale, q_scale_type, h263_aic, ac_pred, struct=OrcMpvUnquant):
    """the oracle's (or, with struct=..., the product's) parameter block; scan tables as ff_init_scantable builds them"""
    p = struct()
    scan = ALTERNATE_VERTICAL if alternate_scan else ZIGZAG
    end = -1
    for i in range(64):
        p.intra_matrix[i], p.inter_matrix[i] = int(intra_matrix[i]), int(inter_matrix[i])
        p.permutated[i] = int(scan[i])
        end = max(end, int(scan[i]))
        p.raster_end[i] = end
    p.y_dc_scale, p.c_dc_scale, p.q_scale_type, p.h263_aic, p.ac_pred = y_dc_scale, c_dc_scale, q_scale_type, h263_aic, ac_pred
    return p


def unquant_case(seed, variant, nblocks=96):
    """seeded quantised blocks the way a decoder leaves them: non-zero only up to last_index in scan order"""
    rng = np.random.default_rng(seed)
    alt = int(rng.integers(0, 2))
    scan = ALTERNATE_VERTICAL if alt else ZIGZAG
    cfg = dict(intra_matrix=rng.integers(8, 84, 64).astype(np.uint16), inter_matrix=rng.integers(8, 60, 64).astype(np.uint16),
               alternate_scan=alt, y_dc_scale=int(rng.integers(1, 9)), c_dc_scale=int(rng.integers(1, 9)),
               q_scale_type=int(rng.integers(0, 2)), h263_aic=int(rng.integers(0, 2)) if variant == 5 else 0,
               ac_pred=int(rng.integers(0, 2)) if variant == 5 else 0)
    cfg["intra_matrix"][0] = 8
    blocks = np.zeros((nblocks, 64), np.int16)
    last = rng.integers(-1 if variant not in (5, 6) else 0, 64, nblocks).astype(np.int8)
    last[:4] = [63, 0, 62, 1]
    for b in range(nblocks):
        k = int(last[b]) + 1
        amp = [3, 40, 300, 2047][b & 3]
        v = rng.integers(-amp, amp + 1, k).astype(np.int16)
        v[rng.random(k) < 0.45] = 0
        blocks[b, scan[:k]] = v
        if b % 7 == 3:
            blocks[b, 63] = int(rng.integers(-5, 6))                  # a coefficient beyond last_index: left alone (unless reached)
    qscale = rng.integers(1, 32, nblocks).astype(np.uint8)
    blk_n = (np.arange(nblocks) % 6).astype(np.uint8) if seed & 1 else rng.integers(0, 6, nblocks).astype(np.uint8)
    return cfg, blocks, blk_n, qscale, last


def orc_unquant(variant, cfg, blocks, blk_n, qscale, last):
    L = oracle()
    L.orc_mpv_unquantize_batch.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
    L.orc_mpv_unquantize_batch.restype = None
    p = unquant_params(**cfg)
    out = np.ascontiguousarray(blocks).copy()
    L.orc_mpv_unquantize_batch(variant, C.byref(p), out.ctypes.data, out.shape[0], blk_n.ctypes.data if blk_n is not None else None,
                               qscale.ctypes.data, last.ctypes.data)
    return out


def ref_unquant(variant, cfg, blocks, blk_n, qscale, last):
    L = ref()
    L.ffref_mpv_unquantize_batch.argtypes = [C.c_int, C.c_void_p, C.c_void_p] + [C.c_int] * 6 + [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
    out = np.ascontiguousarray(blocks).copy()
    im, nm = np.ascontiguousarray(cfg["intra_matrix"], np.uint16), np.ascontiguousarray(cfg["inter_matrix"], np.uint16)
    r = L.ffref_mpv_unquantize_batch(variant, im.ctypes.data, nm.ctypes.data, cfg["alternate_scan"], cfg["y_dc_scale"], cfg["c_dc_scale"],
                                     cfg["q_scale_type"], cfg["h263_aic"], cfg["ac_pred"], out.ctypes.data, out.shape[0],
                                     blk_n.ctypes.data if blk_n is not None else None, qscale.ctypes.data, last.ctypes.data)
    assert r == 0
    return out


# ---------------------------------------------------------------- simple IDCT, 10 / 12 bit
def hbd_picture(depth, kind):
    """(48 x 64 uint16 reference picture, destination picture) for the high-bit-depth h264qpel cases: kind 0 random samples, kind 1 only
    0 and the maximum (the extremes of every intermediate)"""
    rng = np.random.default_rng(1000 * depth + kind)
    mx = (1 << depth) - 1
    img = rng.integers(0, mx + 1, (48, 64)).astype(np.uint16) if kind == 0 else (rng.integers(0, 2, (48, 64)) * mx).astype(np.uint16)
    return img, rng.integers(0, mx + 1, (48, 64)).astype(np.uint16)


def hbd_weight_cases(depth, n=60):
    """(bi, idx, height, log2_denom, wd, ws, offset) for the 16-bit weighted-prediction fixture / tests"""
    rng = np.random.default_rng(4000 + depth)
    return [(int(rng.integers(0, 2)), int(rng.integers(0, 4)), int(rng.choice([2, 4, 8, 16])), int(rng.integers(0, 8)),
             int(rng.integers(-128, 128)), int(rng.integers(-128, 128)), int(rng.integers(-128, 128))) for _ in range(n)]


def h264_idct_hbd_cases(depth, kind, n=24):
    """[(int32 coefficient block, uint16 12 x 16 destination picture)] for the 16-bit H.264 residual-add fixture / tests"""
    rng = np.random.default_rng(6000 + 10 * depth + kind)
    out = []
    for it in range(n):
        N = 64 if kind & 1 else 16
        amp = [300, 4000, 1 << (depth + 6), 1 << 30][it % 4]
        blk = rng.integers(-amp, amp, N).astype(np.int32)
        if it % 7 == 0:
            blk[1:] = 0
        out.append((blk, rng.integers(0, 1 << depth, (12, 16)).astype(np.uint16)))
    return out


def txd_cases():
    """(type, len, inv, scale) of the double-precision tx fixture: AV_TX_DOUBLE_FFT = 2, AV_TX_DOUBLE_MDCT = 3"""
    out = []
    for n in (2, 4, 8, 16, 32, 64, 256, 1024, 4096):
        for inv in (0, 1):
            out.append((2, n, inv, 1.0))
            if n >= 4:
                out += [(3, n, inv, 1.0 / n), (3, n, inv, -1.0)]
    return out


def txd_input(typ, n, inv):
    rng = np.random.default_rng(8000 + 10 * n + 2 * typ + inv)
    return rng.random((3, 2 * n if typ == 2 else (n if inv else 2 * n))) * 2 - 1


def idct_hbd_blocks(seed, depth, n):
    """n coefficient blocks: dense small, full int16 range, sparse, DC only, DC-only rows, decoder-like range"""
    rng = np.random.default_rng(seed)
    out = np.zeros((n, 64), np.int16)
    for i in range(n):
        mode = i % 6
        if mode == 0:
            b = rng.integers(-512, 513, 64)
        elif mode == 1:
            b = rng.integers(-32768, 32768, 64)
        elif mode == 2:
            b = np.zeros(64, np.int64)
            b[rng.integers(0, 64, int(rng.integers(1, 6)))] = rng.integers(-4000, 4000)
        elif mode == 3:
            b = np.zeros(64, np.int64)
            b[0] = rng.integers(-32768, 32768)
        elif mode == 4:
            b = np.zeros(64, np.int64)
            b[::8] = rng.integers(-3000, 3000, 8)
        else:
            b = rng.integers(-(1 << (depth + 3)), 1 << (depth + 3), 64)
        out[i] = b
    return out


def _idct_hbd_run(L, name, depth, kind, blocks, dest, line_size):
    """blocks [n, 64] int16, dest uint16 [8, n*8 (+pad)]: block i at column 8*i.  Returns (blocks after, dest after)."""
    f = getattr(L, name)
    f.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_ssize_t, C.c_void_p]
    b, d = blocks.copy(), dest.copy()
    for i in range(b.shape[0]):
        assert f(depth, kind, d.ctypes.data + 16 * i, line_size, b[i].ctypes.data) == 0
    return b, d


def orc_idct_hbd(depth, kind, blocks, dest, line_size):
    return _idct_hbd_run(oracle(), "orc_idct_hbd", depth, kind, blocks, dest, line_size)


def ref_idct_hbd(depth, kind, blocks, dest, line_size):
    return _idct_hbd_run(ref(), "ffref_idct_hbd", depth, kind, blocks, dest, line_size)


def prores_case(seed, bits, n):
    """(blocks [n, 64] int16, qmat [64] int16): quantised ProRes-like coefficients, several magnitudes, sparse and DC-only blocks"""
    rng = np.random.default_rng(seed)
    blocks = np.zeros((n, 64), np.int16)
    for i in range(n):
        mode = i % 5
        if mode == 0:
            b = rng.integers(-64, 65, 64)
        elif mode == 1:
            b = rng.integers(-2048, 2048, 64)
        elif mode == 2:
            b = np.zeros(64, np.int64)
            b[rng.integers(0, 64, int(rng.integers(1, 6)))] = rng.integers(-500, 500)
        elif mode == 3:
            b = np.zeros(64, np.int64)
            b[0] = rng.integers(-4096, 4096)
        else:
            b = np.zeros(64, np.int64)
            b[::8] = rng.integers(-300, 300, 8)
        blocks[i] = b
    return blocks, rng.integers(1, [64, 5, 255][seed % 3] + 1, 64).astype(np.int16)


def _prores_run(L, name, bits, blocks, qmat, dest, line_size):
    f = getattr(L, name)
    f.argtypes = [C.c_int, C.c_void_p, C.c_ssize_t, C.c_void_p, C.c_void_p]
    b, d = blocks.copy(), dest.copy()
    for i in range(b.shape[0]):
        assert f(bits, d.ctypes.data + 16 * i, line_size, b[i].ctypes.data, qmat.ctypes.data) == 0
    return b, d


def orc_prores(bits, blocks, qmat, dest, line_size):
    return _prores_run(oracle(), "orc_prores_idct_put", bits, blocks, qmat, dest, line_size)


def ref_prores(bits, blocks, qmat, dest, line_size):
    return _prores_run(ref(), "ffref_prores_idct_put", bits, blocks, qmat, dest, line_size)


# ---------------------------------------------------------------- av_pixelutils_get_sad_fn (libavutil/pixelutils.c:43-111)
def pixelutils_case(seed, bits, n):
    """(frame1 [h, s1], frame2 [h, s2], off1, off2): n block pairs of (1 << bits)^2 pixels at random positions, different strides;
    every fourth pair compares a block with a slightly noisy copy of itself"""
    rng = np.random.default_rng(seed)
    size = 1 << bits
    f1 = rng.integers(0, 256, (96, 160)).astype(np.uint8)
    f2 = rng.integers(0, 256, (96, 203)).astype(np.uint8)
    y1, x1 = rng.integers(0, 96 - size + 1, n), rng.integers(0, 160 - size + 1, n)
    y2, x2 = rng.integers(0, 96 - size + 1, n), rng.integers(0, 203 - size + 1, n)
    for i in range(0, min(n, 40), 4):
        blk = f1[y1[i]:y1[i] + size, x1[i]:x1[i] + size].astype(np.int64) + rng.integers(-2, 3, (size, size))
        f2[y2[i]:y2[i] + size, x2[i]:x2[i] + size] = np.clip(blk, 0, 255)
    return f1, f2, (y1 * 160 + x1).astype(np.int64), (y2 * 203 + x2).astype(np.int64)


def _pixelutils_run(L, name, bits, f1, f2, off1, off2):
    f = getattr(L, name)
    f.argtypes = [C.c_int, C.c_void_p, C.c_ssize_t, C.c_void_p, C.c_ssize_t]
    return np.array([f(bits, f1.ctypes.data + int(a), f1.strides[0], f2.ctypes.data + int(b), f2.strides[0]) for a, b in zip(off1, off2)], np.int32)


def orc_pixelutils(bits, f1, f2, off1, off2):
    return _pixelutils_run(oracle(), "orc_pixelutils_sad", bits, f1, f2, off1, off2)


def ref_pixelutils(bits, f1, f2, off1, off2):
    return _pixelutils_run(ref(), "ffref_pixelutils_sad", bits, f1, f2, off1, off2)


# ---------------------------------------------------------------- H.264 deblocking (libavcodec/h264dsp_template.c:103-340)
LF_CELL = 32          # one edge per 32 x 32 cell, q0 of its first line at (8, 8): p3..q3 across and 16 lines along stay inside the cell


def h264lf_case(seed, n, cols=16):
    """(pic uint8 [rows*32, cols*32], kinds uint8 [n], off int64 [n], alpha uint8 [n], beta uint8 [n], tc0 int8 [n, 4]): n independent
    edges of all 16 kinds over noisy, gently and very gently varying content (so that every branch of the filters is taken)"""
    rng = np.random.default_rng(seed)
    rows = (n + cols - 1) // cols
    pic = np.zeros((rows * LF_CELL, cols * LF_CELL), np.uint8)
    for i in range(rows * cols):
        y, x = (i // cols) * LF_CELL, (i % cols) * LF_CELL
        m = (i // 16) % 4
        if m == 0:
            c = rng.integers(0, 256, (LF_CELL, LF_CELL))
        else:
            c = int(rng.integers(0, 256)) + rng.integers(-3 * m, 3 * m + 1, (LF_CELL, LF_CELL))
            if m == 3:
                c[:, 8:] += int(rng.integers(-12, 13))
                c[8:, :] += int(rng.integers(-12, 13))
        pic[y:y + LF_CELL, x:x + LF_CELL] = np.clip(c, 0, 255)
    i = np.arange(n)
    kinds = (i % 16).astype(np.uint8)
    off = ((i // cols) * LF_CELL + 8) * pic.strides[0] + (i % cols) * LF_CELL + 8
    alpha = rng.integers(0, 256, n).astype(np.uint8)
    alpha[rng.random(n) < 0.3] = 255
    beta = rng.integers(0, 19, n).astype(np.uint8)
    tc0 = rng.integers(-1, 14, (n, 4)).astype(np.int8)
    return pic, kinds, off.astype(np.int64), alpha, beta, tc0


def h264lf_hbd_case(seed, n, depth, cols=16):
    """the same layout for 9 / 10 / 12 / 14 bit samples: pic uint16, off in BYTES; the content of the 8-bit case scaled to the depth with
    fresh low bits, so the scaled thresholds see the same mix of branches"""
    pic8, kinds, off8, alpha, beta, tc0 = h264lf_case(seed, n, cols)
    rng = np.random.default_rng(seed + 7777)
    sh = depth - 8
    pic = ((pic8.astype(np.int32) << sh) + rng.integers(0, 1 << sh, pic8.shape)).clip(0, (1 << depth) - 1).astype(np.uint16)
    i = np.arange(n)
    off = (((i // cols) * LF_CELL + 8) * pic.strides[0] + ((i % cols) * LF_CELL + 8) * 2).astype(np.int64)
    return pic, kinds, off, alpha, beta, tc0


def _h264lf_hbd_run(L, name, depth, pic, kinds, off, alpha, beta, tc0):
    f = getattr(L, name)
    f.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_ssize_t, C.c_int, C.c_int, C.c_void_p]
    out = pic.copy()
    for e in range(len(kinds)):
        t = tc0[e].copy()
        assert f(depth, int(kinds[e]), out.ctypes.data + int(off[e]), out.strides[0], int(alpha[e]), int(beta[e]), t.ctypes.data) == 0
    return out


def orc_h264lf_hbd(depth, pic, kinds, off, alpha, beta, tc0):
    return _h264lf_hbd_run(oracle(), "orc_h264_loop_filter_hbd", depth, pic, kinds, off, alpha, beta, tc0)


def ref_h264lf_hbd(depth, pic, kinds, off, alpha, beta, tc0):
    return _h264lf_hbd_run(ref(), "ffref_h264_loop_filter_hbd", depth, pic, kinds, off, alpha, beta, tc0)


def _h264lf_run(L, name, pic, kinds, off, alpha, beta, tc0):
    f = getattr(L, name)
    f.argtypes = [C.c_int, C.c_void_p, C.c_ssize_t, C.c_int, C.c_int, C.c_void_p]
    out = pic.copy()
    for e in range(len(kinds)):
        t = tc0[e].copy()
        assert f(int(kinds[e]), out.ctypes.data + int(off[e]), out.strides[0], int(alpha[e]), int(beta[e]), t.ctypes.data) == 0
    return out


def orc_h264lf(pic, kinds, off, alpha, beta, tc0):
    return _h264lf_run(oracle(), "orc_h264_loop_filter", pic, kinds, off, alpha, beta, tc0)


def ref_h264lf(pic, kinds, off, alpha, beta, tc0):
    return _h264lf_run(ref(), "ffref_h264_loop_filter", pic, kinds, off, alpha, beta, tc0)


# ---------------------------------------------------------------- AVFloatDSPContext (libavutil/float_dsp.c)
FDSP_OPS = ["vector_fmul", "vector_fmac_scalar", "vector_dmac_scalar", "vector_fmul_scalar", "vector_dmul_scalar", "vector_fmul_window",
            "vector_fmul_add", "vector_fmul_reverse", "butterflies_float", "scalarproduct_float", "vector_dmul", "scalarproduct_double"]
FDSP_DOUBLE = (2, 4, 10, 11)


def fdsp_case(seed, op, length):
    """(dst, src0, src1, src2, mul): dst/src2 have 2*length elements for vector_fmul_window; mixed magnitudes, a few
    denormals and signed zeros"""
    rng = np.random.default_rng(seed)
    dt = np.float64 if op in FDSP_DOUBLE else np.float32
    n2 = 2 * length if op == 5 else length

    def mk(n):
        a = (rng.standard_normal(n) * rng.choice([1e-3, 1.0, 1e3], n)).astype(dt)
        if n > 8:
            a[rng.integers(0, n, 3)] = [0.0, -0.0, np.finfo(dt).tiny / 4]
        return a
    return mk(n2), mk(length), mk(length), mk(n2), float(np.float32(rng.standard_normal()))


def _fdsp_run(L, name, op, dst, src0, src1, src2, mul, length):
    f = getattr(L, name)
    f.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_int]
    d, a = dst.copy(), src0.copy()
    assert f(op, d.ctypes.data, a.ctypes.data, src1.ctypes.data, src2.ctypes.data, mul, length) == 0
    return (d[:1] if op in (9, 11) else d), a


def orc_fdsp(op, dst, src0, src1, src2, mul, length):
    """returns (dst after, src0 after) — src0 changes only for butterflies_float; the scalar products return dst[:1]"""
    return _fdsp_run(oracle(), "orc_float_dsp", op, dst, src0, src1, src2, mul, length)


def ref_fdsp(op, dst, src0, src1, src2, mul, length):
    return _fdsp_run(ref(), "ffref_float_dsp", op, dst, src0, src1, src2, mul, length)


NUT_PATH = os.path.join(ROOT, "oracle", "_ref", "libffnut.so")
_nut = None


def have_nut():
    return os.path.exists(NUT_PATH)


def nut_md5(frames, w, h, pix_fmt):
    """md5 of the NUT stream FATE's `-vcodec rawvideo -f nut md5:` writes (oracle/ref/ref_nut.c drives the reference's own
    NUT muxer); frames = one rawvideo packet (planes back to back, no padding) or a list of them."""
    global _nut
    if _nut is None:
        _nut = C.CDLL(NUT_PATH)
        _nut.ffref_nut_md5_frames.argtypes = [C.c_void_p] + [C.c_int] * 5 + [C.c_void_p]
    if not isinstance(frames, (list, tuple)):
        frames = [frames]
    buf = np.concatenate([np.ascontiguousarray(f).ravel() for f in frames])
    m = (C.c_uint8 * 16)()
    n = _nut.ffref_nut_md5_frames(buf.ctypes.data, buf.size // len(frames), len(frames), w, h, pix_fmt, m)
    assert n > buf.size, n
    return bytes(m).hex()


def fate_pixfmts_goldens():
    rows = []
    for line in open(os.path.join(ROOT, "tests", "golden", "fate_pixfmts.txt")):
        if line.startswith("#") or not line.strip():
            continue
        where, test, fmt, size, nframes, md5 = line.split()
        w, h = (int(v) for v in size.split("x"))
        rows.append((where, test, fmt, w, h, int(nframes), md5))
    return rows


VIDEOGEN = os.path.join(ROOT, "oracle", "_ref", "videogen")


def vsynth1_frames(n):
    """frames 0..n-1 of FATE's vsynth1 as (y, u, v): runs the reference's generator (tests/videogen.c, compiled by
    oracle/ref/Makefile) and unpacks its pgmyuv files (Y plane, then rows of U|V)"""
    import subprocess, tempfile
    out = []
    with tempfile.TemporaryDirectory() as td:
        subprocess.run([VIDEOGEN, td + "/"], check=True, stdout=subprocess.DEVNULL)
        for i in range(n):
            raw = open(os.path.join(td, f"{i:02d}.pgm"), "rb").read()
            hdr, rest = raw.split(b"\n255\n", 1)
            assert hdr.split() == [b"P5", b"352", b"432"], hdr
            a = np.frombuffer(rest, np.uint8).reshape(432, 352)
            out.append(tuple(np.ascontiguousarray(p) for p in (a[:288], a[288:, :176], a[288:, 176:])))
    return out


COEFFS = {  # libswscale/yuv2rgb.c:47-59, indexed by SWS_CS_*
    0: (104597, 132201, 25675, 53279), 1: (117489, 138438, 13975, 34925), 2: (104597, 132201, 25675, 53279),
    3: (104597, 132201, 25675, 53279), 4: (104448, 132798, 24759, 53109), 5: (104597, 132201, 25675, 53279),
    6: (104597, 132201, 25675, 53279), 7: (117579, 136230, 16907, 35559), 9: (110013, 140363, 12277, 42626),
    10: (110013, 140363, 12277, 42626),
}


def ref_sws(w, h, dw, dh, flags, y, u, v, **kw):
    return _sws_run(ref(), "ffref", w, h, dw, dh, flags, y, u, v, **kw)


def orc_sws(w, h, dw, dh, flags, y, u, v, **kw):
    kw.pop("threads", None)
    return _sws_run(oracle(), "orc", w, h, dw, dh, flags, y, u, v, **kw)
