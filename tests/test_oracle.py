"""CPU tier: pin the oracle (oracle/liboracle.so) against
   (a) the committed golden fixtures produced by the unmodified reference (scripts/gen_golden.py), always;
   (b) the reference itself (oracle/_ref/libffref.so) on fresh random inputs, wherever that library exists."""
import hashlib
import os

import ctypes as C
import numpy as np
import pytest

import cpulibs as cl
from cases import SWS_SMALL_CASES, SWS_HASH_CASES, FATE, idct_blocks

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def flat(planes):
    return np.concatenate([np.ascontiguousarray(p).ravel() for p in planes])


def test_sws_oracle_vs_golden_small():
    g = np.load(os.path.join(G, "sws_small.npz"))
    for i, (w, h, dw, dh, fl, kind) in enumerate(SWS_SMALL_CASES):
        out = cl.orc_sws(w, h, dw, dh, fl, g[f"c{i}_y"], g[f"c{i}_u"], g[f"c{i}_v"])
        assert out is not None
        assert np.array_equal(out, g[f"c{i}_rgb"]), (i, w, h, dw, dh, hex(fl))


def test_sws_oracle_vs_golden_hashes():
    for line in open(os.path.join(G, "sws_hashes.txt")):
        i, w, h, dw, dh, fl, kind, hin, hout = line.split()
        i, w, h, dw, dh, fl = map(int, (i, w, h, dw, dh, fl))
        y, u, v = cl.yuv_frame(w, h, 200 + i, kind)
        assert sha(np.concatenate([y.ravel(), u.ravel(), v.ravel()])) == hin, "input generator drifted"
        out = cl.orc_sws(w, h, dw, dh, fl, y, u, v)
        assert sha(out) == hout, (i, w, h, dw, dh, hex(fl))


def test_sws_oracle_other_formats_golden_hashes():
    """bgr24 / rgba / bgra / argb / abgr writers against the reference's outputs (sws_format_hashes.txt)."""
    n = 0
    for line in open(os.path.join(G, "sws_format_hashes.txt")):
        name, i, w, h, dw, dh, fl, kind, hout = line.split()
        i, w, h, dw, dh, fl = map(int, (i, w, h, dw, dh, fl))
        y, u, v = cl.yuv_frame(w, h, 500 + i, kind)
        out = cl.orc_sws(w, h, dw, dh, fl, y, u, v, fmt=cl.PACKED_RGB_FORMATS[name])
        assert sha(out) == hout, (name, i, w, h, dw, dh, hex(fl))
        n += 1
    assert n == 50


def test_sws_oracle_formats_are_byte_permutations_of_rgb24():
    """Size-independent property: every format carries the rgb24 values, reordered, plus alpha 255."""
    y, u, v = cl.yuv_frame(96, 64, 9, "random")
    for (dw, dh, fl) in ((96, 64, FATE), (96, 64, cl.SWS_BICUBIC), (50, 40, FATE), (97, 64, FATE)):
        base = cl.orc_sws(96, 64, dw, dh, fl, y, u, v).reshape(dh, dw, 3)
        for name, order in (("bgr24", "bgr"), ("rgba", "rgba"), ("bgra", "bgra"), ("argb", "argb"), ("abgr", "abgr")):
            out = cl.orc_sws(96, 64, dw, dh, fl, y, u, v, fmt=cl.PACKED_RGB_FORMATS[name]).reshape(dh, dw, len(order))
            for k, ch in enumerate(order):
                exp = 255 if ch == "a" else base[:, :, "rgb".index(ch)]
                assert np.array_equal(out[:, :, k], np.broadcast_to(exp, (dh, dw))), (name, ch, dw, dh, hex(fl))


def test_sws_oracle_planar_golden_hashes():
    """yuv420p -> yuv420p scaling (yuv2planeX / yuv2plane1 / plane copy) against the reference's outputs."""
    n = 0
    for line in open(os.path.join(G, "sws_planar_hashes.txt")):
        i, w, h, dw, dh, fl, kind, hout = line.split()
        i, w, h, dw, dh, fl = map(int, (i, w, h, dw, dh, fl))
        y, u, v = cl.yuv_frame(w, h, 600 + i, kind)
        out = cl.orc_sws_planar(w, h, dw, dh, fl, y, u, v)
        assert sha(np.concatenate([p.ravel() for p in out])) == hout, (i, w, h, dw, dh, hex(fl))
        n += 1
    assert n == 14


def test_sws_oracle_planar_vs_ref(refrec):
    rng = np.random.default_rng(8)
    for it in range(25):
        w, h = int(rng.integers(8, 120)), int(rng.integers(8, 90))
        dw, dh = int(rng.integers(8, 160)), int(rng.integers(8, 120))
        fl = int(rng.choice([FATE, cl.SWS_BICUBIC, cl.SWS_BILINEAR, cl.SWS_POINT, cl.SWS_AREA, cl.SWS_BICUBLIN]))
        y, u, v = cl.yuv_frame(w, h, 700 + it, "random", pad=int(rng.integers(0, 9)))
        b = cl.orc_sws_planar(w, h, dw, dh, fl, y, u, v, dst_pad=3)
        assert refrec.same(flat(b), lambda: flat(cl.ref_sws_planar(w, h, dw, dh, fl, y, u, v, dst_pad=3))), (w, h, dw, dh, hex(fl))


def test_sws_oracle_fast_bilinear_golden_hashes():
    """SWS_FAST_BILINEAR (hyscale_fast / hcscale_fast) against the reference's outputs, rgb24 and yuv420p destinations."""
    n = 0
    for line in open(os.path.join(G, "sws_fastbil_hashes.txt")):
        i, w, h, dw, dh, fl, kind, hrgb, hyuv = line.split()
        i, w, h, dw, dh, fl = map(int, (i, w, h, dw, dh, fl))
        y, u, v = cl.yuv_frame(w, h, 800 + i, kind)
        assert sha(cl.orc_sws(w, h, dw, dh, fl, y, u, v)) == hrgb, (i, w, h, dw, dh, hex(fl))
        assert sha(np.concatenate([p.ravel() for p in cl.orc_sws_planar(w, h, dw, dh, fl, y, u, v)])) == hyuv, (i, w, h, dw, dh, hex(fl))
        n += 1
    assert n == 11


def test_sws_oracle_nv12_nv21_golden_hashes():
    """nv12 / nv21 sources to rgb24, bgra and yuv420p against the reference's outputs."""
    n = 0
    for line in open(os.path.join(G, "sws_nv_hashes.txt")):
        name, i, w, h, dw, dh, fl, kind, hrgb, hbgra, hyuv = line.split()
        i, w, h, dw, dh, fl = map(int, (i, w, h, dw, dh, fl))
        sf = cl.PIX_FMT_NV12 if name == "nv12" else cl.PIX_FMT_NV21
        y, u, v = cl.yuv_frame(w, h, 1000 + i, kind)
        uv = cl.nv_interleave(u, v, sf)
        assert sha(cl.orc_sws(w, h, dw, dh, fl, y, uv, uv, src_fmt=sf)) == hrgb, (name, i)
        assert sha(cl.orc_sws(w, h, dw, dh, fl, y, uv, uv, src_fmt=sf, fmt=cl.PIX_FMT_BGRA)) == hbgra, (name, i)
        assert sha(np.concatenate([p.ravel() for p in cl.orc_sws_planar(w, h, dw, dh, fl, y, uv, uv, src_fmt=sf)])) == hyuv, (name, i)
        n += 1
    assert n == 18


def test_sws_oracle_colorspace_golden():
    g = np.load(os.path.join(G, "sws_colorspace.npz"))
    y, u, v = g["y"], g["u"], g["v"]
    css = [(1, 0, 1, 0, 0, 1 << 16, 1 << 16), (5, 1, 5, 1, 0, 1 << 16, 1 << 16),
           (9, 0, 9, 0, 3000, 70000, 80000), (7, 1, 7, 0, -2000, 60000, 50000)]
    for j, cs in enumerate(css):
        for k, fl in enumerate([FATE, cl.SWS_BICUBIC]):
            assert np.array_equal(cl.orc_sws(64, 48, 64, 48, fl, y, u, v, colorspace=cs), g[f"cs{j}_{k}"]), (j, k)
            assert np.array_equal(cl.orc_sws(64, 48, 96, 80, fl, y, u, v, colorspace=cs), g[f"cs{j}_{k}_s"]), (j, k, "s")


def test_idct_oracle_vs_golden():
    g = np.load(os.path.join(G, "idct.npz"))
    O = cl.oracle()
    off = (np.arange(256) * 8).astype(np.int64)
    for kind in ("dense", "wide", "extreme", "sparse", "dc63", "dconly"):
        for op in (0, 1, 2):
            b, de = g[f"{kind}_in"].copy(), g[f"{kind}_dest"].copy()
            O.orc_idct_batch(op, cl.ptr(b, cl.i16p), 256, cl.ptr(de), 256 * 8, cl.ptr(off, cl.i64p))
            assert np.array_equal(b if op == 0 else de, g[f"{kind}_op{op}"]), (kind, op)


@pytest.mark.parametrize("case", [(352, 288, 352, 288, FATE), (352, 288, 352, 288, cl.SWS_BICUBIC),
                                  (352, 288, 200, 100, FATE), (100, 50, 37, 21, FATE), (352, 288, 640, 360, cl.SWS_BILINEAR),
                                  (350, 288, 350, 288, cl.SWS_BICUBIC), (352, 288, 300, 200, cl.SWS_BICUBLIN)])
def test_sws_oracle_vs_reference_live(case, refrec):
    w, h, dw, dh, fl = case
    for seed, kind in ((1, "random"), (2, "smooth"), (3, "limited")):
        y, u, v = cl.yuv_frame(w, h, seed, kind, pad=7)
        b = cl.orc_sws(w, h, dw, dh, fl, y, u, v, dst_pad=5)
        assert refrec.same(b, lambda: cl.ref_sws(w, h, dw, dh, fl, y, u, v, dst_pad=5))


def test_idct_oracle_vs_reference_live(refrec):
    R, O = cl.ref() if cl.have_ref() else None, cl.oracle()
    n = 4096
    off = (np.arange(n) * 8).astype(np.int64)
    for kind in ("dense", "wide", "extreme", "sparse", "dc63", "dconly"):
        for op in (0, 1, 2):
            blk = idct_blocks(kind, n, seed=op + 31)
            d0 = np.random.default_rng(5).integers(0, 256, (8, n * 8), dtype=np.uint8)
            b1, b2, d1, d2 = blk.copy(), blk.copy(), d0.copy(), d0.copy()
            O.orc_idct_batch(op, cl.ptr(b2, cl.i16p), n, cl.ptr(d2), n * 8, cl.ptr(off, cl.i64p))
            out = lambda b, d: np.concatenate([d.ravel(), b.view(np.uint8).ravel() if op == 0 else []]).astype(np.uint8)

            def ref_out():
                R.ffref_idct_batch(op, cl.ptr(b1, cl.i16p), n, cl.ptr(d1), n * 8, cl.ptr(off, cl.i64p))
                return out(b1, d1)
            assert refrec.same(out(b2, d2), ref_out), (kind, op)


def test_host_filter_tables_match_oracle():
    """The product's host-side filter generation (sws_plan.cpp) against the oracle's, no GPU involved."""
    import ffmpeg_b200 as fb
    L, O = fb.lib(), cl.oracle()
    for (w, h, dw, dh, fl, _k) in SWS_SMALL_CASES + SWS_HASH_CASES + [(3840, 2160, 3840, 2160, FATE, ""), (3840, 2160, 1920, 1080, FATE, "")]:
        ctx = O.orc_sws_open(w, h, dw, dh, fl)
        assert ctx
        oi = np.zeros(16, np.int32)
        O.orc_sws_info(ctx, cl.ptr(oi, cl.i32p))
        for which in range(4):
            pi = np.zeros(16, np.int32)
            assert L.b200_sws_plan_probe(w, h, dw, dh, fl, which, None, None, 0, cl.ptr(pi, cl.i32p)) >= 0
            assert list(pi) == list(oi)
            size, cnt = int(pi[which]), [dw, int(pi[6]), dh, int(pi[7])][which]
            if size == 0:
                continue
            f1, p1 = np.zeros(cnt * size, np.int16), np.zeros(cnt, np.int32)
            f2, p2 = f1.copy(), p1.copy()
            L.b200_sws_plan_probe(w, h, dw, dh, fl, which, cl.ptr(f1, cl.i16p), cl.ptr(p1, cl.i32p), cnt, None)
            O.orc_sws_get_filter(ctx, which, cl.ptr(f2, cl.i16p), cl.ptr(p2, cl.i32p), cnt)
            assert np.array_equal(f1, f2) and np.array_equal(p1, p2), (w, h, dw, dh, hex(fl), which)
        O.orc_sws_close(ctx)


def test_sws_oracle_vsynth1_frame0():
    """The FATE picture itself (vsynth1 frame 0, tests/videogen.c) converted by the reference with FATE's sws flags."""
    g = np.load(os.path.join(G, "vsynth1_f0.npz"))
    y, u, v = g["y"], g["u"], g["v"]
    assert np.array_equal(cl.orc_sws(352, 288, 352, 288, FATE, y, u, v), g["rgb_same"])
    assert np.array_equal(cl.orc_sws(352, 288, 200, 100, FATE, y, u, v), g["rgb_200x100"])
    assert np.array_equal(cl.orc_sws(352, 288, 352, 288, cl.SWS_BICUBIC, y, u, v), g["rgb_lut"])


def test_sws_oracle_range_golden_hashes():
    """yuv -> yuv range conversion (lum/chrRangeToJpeg_c, FromJpeg_c) against the reference's outputs, ranges given at
    initialisation or through sws_setColorspaceDetails() afterwards (incl. the context that stays a plain copy)."""
    from cases import SWS_RANGE_CASES
    lines = open(os.path.join(G, "sws_range_hashes.txt")).read().split("\n")[:-1]
    assert len(lines) == len(SWS_RANGE_CASES) == 14
    for line, (w, h, dw, dh, fl, kind, ranges, details) in zip(lines, SWS_RANGE_CASES):
        i, hout = int(line.split()[0]), line.split()[-1]
        y, u, v = cl.yuv_frame(w, h, 1200 + i, kind)
        out = cl.orc_sws_planar(w, h, dw, dh, fl, y, u, v, ranges=ranges, details=details)
        assert sha(np.concatenate([p.ravel() for p in out])) == hout, (i, w, h, dw, dh, hex(fl), ranges, details)


def test_sws_oracle_range_vs_ref(refrec):
    rng = np.random.default_rng(81)
    for it in range(24):
        w, h = int(rng.integers(8, 120)), int(rng.integers(8, 90))
        dw, dh = (w, h) if it % 4 == 0 else (int(rng.integers(8, 160)), int(rng.integers(8, 120)))
        fl = int(rng.choice([FATE, cl.SWS_BICUBIC, cl.SWS_BILINEAR, cl.SWS_POINT, 1]))
        ranges = [(0, 1), (1, 0), (0, 0), (1, 1)][int(rng.integers(0, 4))]
        details = None if it % 3 else (5, int(rng.integers(0, 2)), 5, int(rng.integers(0, 2)), 0, 1 << 16, 1 << 16)
        y, u, v = cl.yuv_frame(w, h, 1300 + it, ["random", "limited"][it & 1], pad=int(rng.integers(0, 9)))
        b = cl.orc_sws_planar(w, h, dw, dh, fl, y, u, v, dst_pad=3, ranges=ranges, details=details)
        assert refrec.same(flat(b), lambda: flat(cl.ref_sws_planar(w, h, dw, dh, fl, y, u, v, dst_pad=3, ranges=ranges, details=details))), \
            (w, h, dw, dh, hex(fl), ranges, details)


FATE_SWS_YUV_RANGE = 0xbc7a0fa2     # tests/ref/fate/sws-yuv-range:6 (framecrc: av_adler32_update(0, ...) over the 152064-byte frame)


def fate_sws_yuv_range_crc(run_planar):
    """tests/fate/libswscale.mak:28-32: vsynth1 frame 0, scale=in_range=limited:out_range=full:flags=+accurate_rnd+bitexact"""
    import zlib
    g = np.load(os.path.join(G, "vsynth1_f0.npz"))
    out = run_planar(352, 288, 352, 288, cl.SWS_BICUBIC | cl.SWS_ACCURATE_RND | cl.SWS_BITEXACT, g["y"], g["u"], g["v"], ranges=(0, 1))
    return zlib.adler32(np.concatenate([p.ravel() for p in out]).tobytes(), 0)


def test_sws_oracle_fate_sws_yuv_range():
    assert fate_sws_yuv_range_crc(cl.orc_sws_planar) == FATE_SWS_YUV_RANGE
    if cl.have_ref():
        assert fate_sws_yuv_range_crc(cl.ref_sws_planar) == FATE_SWS_YUV_RANGE


def test_sws_oracle_yuv_matrix_change_cascades_once():
    """different matrices for yuv -> yuv: the first call builds the bgr24 cascade (utils.c:914-989); later calls go to its first context"""
    L = cl.oracle()
    ctx = L.orc_sws_open_range(0, 64, 48, 0, 0, 100, 70, 0, FATE)
    ta, tb = (np.array(cl.COEFFS[k], dtype=np.int32) for k in (1, 5))
    assert L.orc_sws_set_colorspace_details(ctx, cl.ptr(ta, cl.i32p), 0, cl.ptr(tb, cl.i32p), 1, 0, 1 << 16, 1 << 16) == 0
    assert L.orc_sws_set_colorspace_details(ctx, cl.ptr(ta, cl.i32p), 0, cl.ptr(tb, cl.i32p), 1, 0, 1 << 16, 1 << 16) == 0
    L.orc_sws_close(ctx)


def _all_sws_configs():
    """(src_fmt, w, h, src_range, dst_fmt, dw, dh, dst_range, flags, details) over every case list of tests/cases.py"""
    from cases import SWS_FORMAT_CASES, SWS_PLANAR_CASES, SWS_FASTBIL_CASES, SWS_NV_CASES, SWS_RANGE_CASES
    out = []
    for (w, h, dw, dh, fl, _k) in SWS_FORMAT_CASES:
        for f in cl.PACKED_RGB_FORMATS.values():
            out.append((0, w, h, 0, f, dw, dh, 0, fl, None))
    for (w, h, dw, dh, fl, _k) in SWS_PLANAR_CASES:
        out.append((0, w, h, 0, 0, dw, dh, 0, fl, None))
    for (w, h, dw, dh, fl, _k) in SWS_FASTBIL_CASES:
        out += [(0, w, h, 0, cl.PIX_FMT_RGB24, dw, dh, 0, fl, None), (0, w, h, 0, 0, dw, dh, 0, fl, None)]
    for (w, h, dw, dh, fl, _k) in SWS_NV_CASES:
        for sf in (cl.PIX_FMT_NV12, cl.PIX_FMT_NV21):
            out += [(sf, w, h, 0, cl.PIX_FMT_RGB24, dw, dh, 0, fl, None), (sf, w, h, 0, 0, dw, dh, 0, fl, None)]
    for (w, h, dw, dh, fl, _k, ranges, details) in SWS_RANGE_CASES:
        out.append((0, w, h, ranges[0], 0, dw, dh, ranges[1], fl, details))
        out.append((cl.PIX_FMT_NV12, w, h, ranges[0], 0, dw, dh, ranges[1], fl, details))
        out.append((0, w, h, ranges[0], cl.PIX_FMT_RGB24, dw, dh, ranges[1], fl, None))      # RGB destination: dst_range is ignored
    out += [(0, 3840, 2160, 0, 0, 1920, 1080, 1, FATE, None), (0, 3840, 2160, 1, 0, 3840, 2160, 0, FATE, None)]
    from cases import SWS_RGBSRC_CASES
    for (w, h, dw, dh, fl, _k) in SWS_RGBSRC_CASES:
        for sf in cl.PACKED_RGB_FORMATS.values():
            out += [(sf, w, h, 0, 0, dw, dh, 0, fl, None), (sf, w, h, 0, 0, dw, dh, 1, fl, None)]
            if (w, h) != (dw, dh) and cl.fmt_bpp(sf) == 3:
                out.append((sf, w, h, 0, cl.PIX_FMT_BGRA, dw, dh, 0, fl, None))
        out.append((cl.PIX_FMT_BGR24, w, h, 0, 0, dw, dh, 0, fl, (1, 0, 1, 1, 0, 1 << 16, 1 << 16)))     # bt709 table, full range out
    out += [(cl.PIX_FMT_RGB24, 3840, 2160, 0, 0, 3840, 2160, 0, FATE, None), (cl.PIX_FMT_BGRA, 3840, 2160, 0, 0, 1920, 1080, 0, cl.SWS_BICUBIC, None)]
    for df in (cl.PIX_FMT_NV12, cl.PIX_FMT_NV21):                  # semi-planar destinations from planar and packed sources
        for (w, h, dw, dh, fl, _k) in SWS_PLANAR_CASES:
            out += [(0, w, h, 0, df, dw, dh, 0, fl, None), (0, w, h, 0, df, dw, dh, 1, fl, None)]
        for (w, h, dw, dh, fl, _k) in SWS_RGBSRC_CASES:
            out += [(cl.PIX_FMT_BGR24, w, h, 0, df, dw, dh, 0, fl, None), (cl.PIX_FMT_RGBA, w, h, 0, df, dw, dh, 0, fl, None)]
    from cases import SWS_FLOAT_KERNEL_CASES
    for (w, h, dw, dh, fl, _k) in SWS_FLOAT_KERNEL_CASES:           # gauss / sinc / lanczos / spline / experimental scalers
        out += [(0, w, h, 0, cl.PIX_FMT_RGB24, dw, dh, 0, fl, None), (0, w, h, 0, 0, dw, dh, 0, fl, None), (cl.PIX_FMT_NV12, w, h, 0, cl.PIX_FMT_BGRA, dw, dh, 0, fl, None)]
    return out


def test_host_plan_matches_oracle_and_reference_all_formats():
    """The product's host-side set-up (sws_plan.cpp: converter gates, filter banks, range-conversion constants) for every
    source / destination format, range and flag combination of the case lists, against the oracle and, where built, the
    reference's initialised context.  No GPU involved."""
    import ffmpeg_b200 as fb
    L, O = fb.lib(), cl.oracle()
    R = cl.ref() if cl.have_ref() else None
    O.orc_sws_range_info.argtypes = [C.c_void_p, cl.i32p]
    O.orc_sws_rgb_info.argtypes = [C.c_void_p, cl.i32p]
    if R is not None:
        R.ffref_sws_range_info.argtypes = [C.c_void_p, cl.i32p]
        R.ffref_sws_rgb_info.argtypes = [C.c_void_p, cl.i32p]
    cfgs = _all_sws_configs()
    assert len(cfgs) > 150
    for (sf, w, h, sr, df, dw, dh, dr, fl, details) in cfgs:
        key = (sf, w, h, sr, df, dw, dh, dr, hex(fl), details)
        cfg = np.array([w, h, sf, sr, dw, dh, df, dr, fl], np.int32)
        det = None
        if details is not None:
            det = np.array(list(cl.COEFFS[details[0]]) + [details[1]] + list(cl.COEFFS[details[2]]) + list(details[3:]), np.int32)
        octx = O.orc_sws_open_range(sf, w, h, sr, df, dw, dh, dr, fl)
        assert octx, key
        rctx = R.ffref_sws_open_range(sf, w, h, sr, df, dw, dh, dr, fl, 1) if R is not None else None
        if details is not None:
            ta, tb = (np.array(cl.COEFFS[k], dtype=np.int32) for k in (details[0], details[2]))
            assert O.orc_sws_set_colorspace_details(octx, cl.ptr(ta, cl.i32p), details[1], cl.ptr(tb, cl.i32p), details[3], *details[4:]) == 0
            if rctx:
                assert R.ffref_sws_set_colorspace(rctx, *details) == 0
        oi, ori = np.zeros(16, np.int32), np.zeros(6, np.int32)
        O.orc_sws_info(octx, cl.ptr(oi, cl.i32p))
        O.orc_sws_range_info(octx, cl.ptr(ori, cl.i32p))
        ogi = np.zeros(13, np.int32)
        O.orc_sws_rgb_info(octx, cl.ptr(ogi, cl.i32p))
        if rctx:
            rri, rgi = np.zeros(6, np.int32), np.zeros(13, np.int32)
            R.ffref_sws_range_info(rctx, cl.ptr(rri, cl.i32p))
            R.ffref_sws_rgb_info(rctx, cl.ptr(rgi, cl.i32p))
            assert list(rri) == list(ori), (key, list(rri), list(ori))
            assert list(rgi[:3]) == list(ogi[:3]), (key, list(rgi), list(ogi))
            if ogi[0]:                      # (for yuv -> yuv the reference returns before it fills the table, utils.c:910-989)
                assert list(rgi[4:]) == list(ogi[4:]), (key, list(rgi), list(ogi))
                assert bool(rgi[3]) == bool(ogi[3]), (key, "bgr24 -> yv12 gate")
        for which in range(4):
            pi = np.zeros(48, np.int32)
            n = L.b200_sws_plan_probe2(cl.ptr(cfg, cl.i32p), cl.ptr(det, cl.i32p) if det is not None else None, which, None, None, 0,
                                       cl.ptr(pi, cl.i32p))
            assert n >= 0 and pi[24] == 0, key
            assert list(pi[:8]) == list(oi[:8]) and pi[11] == oi[11], (key, list(pi[:16]), list(oi))
            assert bool(pi[8] or pi[16] or pi[30]) == bool(ori[5]), (key, "unscaled converter gate")
            assert [int(pi[27]), int(pi[28]), int(pi[29]), int(pi[30])] + [int(x) for x in pi[32:41]] == [int(x) for x in ogi], (key, list(pi[27:41]), list(ogi))
            assert [int(pi[17]), int(pi[18]) if pi[17] else 0, int(pi[19]) if pi[17] else 0, int(pi[20]) if pi[17] else 0,
                    int(pi[21]) if pi[17] else 0] == list(ori[:5]), (key, list(pi[16:27]), list(ori))
            size, cnt = int(pi[which]), [dw, int(pi[6]), dh, int(pi[7])][which]
            if size == 0:
                continue
            f1, p1 = np.zeros(cnt * size, np.int16), np.zeros(cnt, np.int32)
            f2, p2 = f1.copy(), p1.copy()
            L.b200_sws_plan_probe2(cl.ptr(cfg, cl.i32p), cl.ptr(det, cl.i32p) if det is not None else None, which,
                                   cl.ptr(f1, cl.i16p), cl.ptr(p1, cl.i32p), cnt, None)
            O.orc_sws_get_filter(octx, which, cl.ptr(f2, cl.i16p), cl.ptr(p2, cl.i32p), cnt)
            assert np.array_equal(f1, f2) and np.array_equal(p1, p2), (key, which)
        O.orc_sws_close(octx)
        if rctx:
            R.ffref_sws_close(rctx)


def test_host_plan_refuses_yuv_matrix_change():
    import ffmpeg_b200 as fb
    L = fb.lib()
    cfg = np.array([64, 48, 0, 0, 100, 70, 0, 0, FATE], np.int32)
    det = np.array(list(cl.COEFFS[1]) + [0] + list(cl.COEFFS[5]) + [1, 0, 1 << 16, 1 << 16], np.int32)
    pi = np.zeros(48, np.int32)
    assert L.b200_sws_plan_probe2(cl.ptr(cfg, cl.i32p), cl.ptr(det, cl.i32p), 0, None, None, 0, cl.ptr(pi, cl.i32p)) >= 0
    assert pi[24] == -38                                            # B200_ENOSYS: the reference would cascade through bgr24
    cfg[6] = cl.PIX_FMT_RGB24                                       # RGB destination: `table` is ignored, like the reference
    assert L.b200_sws_plan_probe2(cl.ptr(cfg, cl.i32p), cl.ptr(det, cl.i32p), 0, None, None, 0, cl.ptr(pi, cl.i32p)) >= 0
    assert pi[24] == 0


def rgbsrc_rows():
    """(case index, case, source name, source format, destination 'yuv420p' / 'rgb24', dst_range, sha256) of sws_rgbsrc_hashes.txt"""
    from cases import SWS_RGBSRC_CASES
    rows = []
    for line in open(os.path.join(G, "sws_rgbsrc_hashes.txt")):
        i, name, dst, dr, h = line.split()
        rows.append((int(i), SWS_RGBSRC_CASES[int(i)], name, cl.PACKED_RGB_FORMATS[name], dst, int(dr), h))
    return rows


def run_rgbsrc_row(run_rgb, run_planar, row):
    i, (w, h, dw, dh, fl, kind), name, sf, dst, dr, _ = row
    src = cl.rgb_frame(w, h, 2000 + i, cl.fmt_bpp(sf), kind)
    if dst == "yuv420p":
        return np.concatenate([p.ravel() for p in run_planar(w, h, dw, dh, fl, src, src, src, src_fmt=sf, ranges=(0, dr))])
    return run_rgb(w, h, dw, dh, fl, src, src, src, fmt=cl.PIX_FMT_RGB24, src_fmt=sf)


def test_sws_oracle_rgb_sources_golden_hashes():
    """packed RGB sources (input readers, 16-bit horizontal pass, bgr24 -> yv12 special converter) against the reference"""
    rows = rgbsrc_rows()
    assert len(rows) == 15 * 6 * 2 + 11 * 2
    for row in rows:
        assert sha(run_rgbsrc_row(cl.orc_sws, cl.orc_sws_planar, row)) == row[-1], row[:6]


def test_sws_oracle_rgb_sources_vs_ref(refrec):
    rng = np.random.default_rng(91)
    names = list(cl.PACKED_RGB_FORMATS)
    for it in range(40):
        w, h = int(rng.integers(8, 120)), int(rng.integers(8, 90))
        dw, dh = (w, h) if it % 5 == 0 else (int(rng.integers(8, 160)), int(rng.integers(8, 120)))
        fl = int(rng.choice([FATE, cl.SWS_BICUBIC, cl.SWS_BILINEAR, cl.SWS_POINT, 1, cl.SWS_BICUBIC | 0x4000]))
        sf = cl.PACKED_RGB_FORMATS[names[it % 6]]
        src = cl.rgb_frame(w, h, 2100 + it, cl.fmt_bpp(sf), "random", pad=int(rng.integers(0, 7)))
        ranges = (0, int(rng.integers(0, 2)))
        b = cl.orc_sws_planar(w, h, dw, dh, fl, src, src, src, dst_pad=3, src_fmt=sf, ranges=ranges)
        assert refrec.same(flat(b), lambda: flat(cl.ref_sws_planar(w, h, dw, dh, fl, src, src, src, dst_pad=3, src_fmt=sf, ranges=ranges))), \
            (w, h, dw, dh, hex(fl), names[it % 6], ranges)
        if (w, h) != (dw, dh):
            df = cl.PIX_FMT_BGR24 if it & 1 else (cl.PIX_FMT_RGBA if cl.fmt_bpp(sf) == 3 else cl.PIX_FMT_RGB24)
            b = cl.orc_sws(w, h, dw, dh, fl, src, src, src, fmt=df, src_fmt=sf, dst_pad=2)
            assert refrec.same(b, lambda: cl.ref_sws(w, h, dw, dh, fl, src, src, src, fmt=df, src_fmt=sf, dst_pad=2)), (w, h, dw, dh, hex(fl), names[it % 6], df)


def test_sws_oracle_alpha_through_the_scaler_vs_ref(refrec):
    """32-bit source and 32-bit destination: c->needAlpha, the alpha plane is read (rgbaToA_c / abgrToA_c), scaled with the luma filters
    and written by the A variants of all six packed writers"""
    rng = np.random.default_rng(4)
    names = ["rgba", "bgra", "argb", "abgr"]
    AO = {"rgba": 3, "bgra": 3, "argb": 0, "abgr": 0}
    for it in range(60):
        w, h = int(rng.integers(8, 90)), int(rng.integers(8, 60))
        dw, dh = int(rng.integers(8, 120)), int(rng.integers(8, 80))
        if it % 7 == 0:
            dh = h
        if it % 11 == 0:
            dw = w
        if (dw, dh) == (w, h):
            dw += 1
        fl = int(rng.choice([4, FATE, 2, 1, 0x10, 0x20, 0x200, 4 | 0x2000, 1 | 0x80000]))
        sn, dn = names[int(rng.integers(0, 4))], names[int(rng.integers(0, 4))]
        src = cl.rgb_frame(w, h, 3000 + it, 4, "random", pad=int(rng.integers(0, 5)))
        if it % 4 == 0:
            src[:, AO[sn]:w * 4:4] = rng.integers(0, 2, (h, w)) * 255
        b = cl.orc_sws(w, h, dw, dh, fl, src, src, src, fmt=cl.PACKED_RGB_FORMATS[dn], src_fmt=cl.PACKED_RGB_FORMATS[sn], dst_pad=1)
        assert refrec.same(b, lambda: cl.ref_sws(w, h, dw, dh, fl, src, src, src, fmt=cl.PACKED_RGB_FORMATS[dn], src_fmt=cl.PACKED_RGB_FORMATS[sn], dst_pad=1)), \
            (w, h, dw, dh, hex(fl), sn, dn)


def rgb2rgb_rows():
    rows = []
    for line in open(os.path.join(G, "sws_rgb2rgb_hashes.txt")):
        w, h, sn, dn, fl, hsh = line.split()
        rows.append((int(w), int(h), sn, dn, int(fl), hsh))
    return rows


def run_rgb2rgb_row(run, row):
    w, h, sn, dn, fl, _ = row
    sf, df = cl.PACKED_RGB_FORMATS[sn], cl.PACKED_RGB_FORMATS[dn]
    src = cl.rgb_frame(w, h, 2600 + w, cl.fmt_bpp(sf), "random", pad=3)
    return run(w, h, w, h, fl, src, src, src, fmt=df, src_fmt=sf)


def test_sws_oracle_same_size_rgb_to_rgb():
    """rgbToRgbWrapper / packedCopyWrapper (and the scaler where SWS_BITEXACT removes the 24 -> 32 bit shuffle): the restatement and the
    product's plan against the reference's outputs for every ordered pair of the six packed formats"""
    import ffmpeg_b200 as fb
    L = fb.lib()
    rows = rgb2rgb_rows()
    assert len(rows) == 2 * 36 * 4
    nshuf = 0
    for row in rows:
        w, h, sn, dn, fl, hsh = row
        assert sha(run_rgb2rgb_row(cl.orc_sws, row)) == hsh, row[:5]
        cfg = np.array([w, h, cl.PACKED_RGB_FORMATS[sn], 0, w, h, cl.PACKED_RGB_FORMATS[dn], 0, fl], np.int32)
        pi = np.zeros(48, np.int32)
        assert L.b200_sws_plan_probe2(cl.ptr(cfg, cl.i32p), None, 0, None, None, 0, cl.ptr(pi, cl.i32p)) >= 0
        through_scaler = (fl & 0x80000) and sn in ("rgb24", "bgr24") and dn in ("rgba", "bgra")
        assert bool(pi[41]) == (not through_scaler), row[:5]
        nshuf += int(pi[41])
    assert nshuf == 2 * (36 * 4 - 4 * 2)
    if cl.have_ref():                                               # other sizes / paddings live
        rng = np.random.default_rng(5)
        names = list(cl.PACKED_RGB_FORMATS)
        for it in range(60):
            w, h = int(rng.integers(1, 70)), int(rng.integers(1, 20))
            sn, dn = names[int(rng.integers(0, 6))], names[int(rng.integers(0, 6))]
            sf, df = cl.PACKED_RGB_FORMATS[sn], cl.PACKED_RGB_FORMATS[dn]
            fl = int(rng.choice([4, 4 | 0x80000, 2, 0x10]))
            if w < 8 and (fl & 0x80000) and sn in ("rgb24", "bgr24") and dn in ("rgba", "bgra"):
                continue                                            # tiny pictures through the scaler: not the point here
            src = cl.rgb_frame(w, h, 2700 + it, cl.fmt_bpp(sf), "random", pad=int(rng.integers(0, 5)))
            a = cl.ref_sws(w, h, w, h, fl, src, src, src, fmt=df, src_fmt=sf, dst_pad=2)
            b = cl.orc_sws(w, h, w, h, fl, src, src, src, fmt=df, src_fmt=sf, dst_pad=2)
            wb = w * cl.fmt_bpp(df)                                 # the reference may write one byte past a line (alpha of the "next" pixel)
            assert np.array_equal(a[:, :wb], b[:, :wb]), (w, h, sn, dn, hex(fl))


def test_sws_oracle_nv_destinations_vs_ref(refrec):
    """nv12 / nv21 as the destination (planarToNv12Wrapper when unscaled, yuv2nv12cX_c through the scaler) from every source kind"""
    from cases import SWS_PLANAR_CASES, SWS_RANGE_CASES, SWS_NV_CASES, SWS_RGBSRC_CASES
    n = 0

    def two(planes):
        assert planes is not None and len(planes) == 2
        return flat(planes)

    def same(*a, **k):
        o = two(cl.orc_sws_planar(*a, **k))
        assert refrec.same(o, lambda: two(cl.ref_sws_planar(*a, **k))), (a[:5], {x: k[x] for x in k if x != "details"})
    for df in (cl.PIX_FMT_NV12, cl.PIX_FMT_NV21):
        for i, (w, h, dw, dh, fl, kind) in enumerate(SWS_PLANAR_CASES):
            same(w, h, dw, dh, fl, *cl.yuv_frame(w, h, 2500 + i, kind), dst_fmt=df, dst_pad=i % 3)
        for i, (w, h, dw, dh, fl, kind, ranges, det) in enumerate(SWS_RANGE_CASES):
            same(w, h, dw, dh, fl, *cl.yuv_frame(w, h, 2600 + i, kind), dst_fmt=df, ranges=ranges, details=det)
        for i, (w, h, dw, dh, fl, kind) in enumerate(SWS_NV_CASES[:6]):
            y, u, v = cl.yuv_frame(w, h, 2700 + i, kind)
            for sf in (cl.PIX_FMT_NV12, cl.PIX_FMT_NV21):
                uv = cl.nv_interleave(u, v, sf)
                same(w, h, dw, dh, fl, y, uv, uv, src_fmt=sf, dst_fmt=df)
        for i, (w, h, dw, dh, fl, kind) in enumerate(SWS_RGBSRC_CASES):
            name = list(cl.PACKED_RGB_FORMATS)[(i + n) % 6]
            sf = cl.PACKED_RGB_FORMATS[name]
            src = cl.rgb_frame(w, h, 2800 + i, cl.fmt_bpp(sf), kind)
            same(w, h, dw, dh, fl, src, src, src, src_fmt=sf, dst_fmt=df)
        n += 1


def test_float_kernel_scalers_oracle_golden_and_ref():
    """SWS_X / GAUSS / SINC / LANCZOS / SPLINE (filter taps from double-precision kernels, utils.c:325-368) against the reference's
    outputs: fixture hashes for both destinations, then the compiled reference on more sizes"""
    from cases import SWS_FLOAT_KERNEL_CASES
    lines = open(os.path.join(G, "sws_float_kernel_hashes.txt")).read().split("\n")[:-1]
    assert len(lines) == len(SWS_FLOAT_KERNEL_CASES)
    for line, (w, h, dw, dh, fl, kind) in zip(lines, SWS_FLOAT_KERNEL_CASES):
        i, hrgb, hyuv = line.split()
        y, u, v = cl.yuv_frame(w, h, 4100 + int(i), kind)
        assert sha(cl.orc_sws(w, h, dw, dh, fl, y, u, v)) == hrgb, (i, hex(fl))
        assert sha(np.concatenate([p.ravel() for p in cl.orc_sws_planar(w, h, dw, dh, fl, y, u, v)])) == hyuv, (i, hex(fl))
    if cl.have_ref():
        for fl in (0x8, 0x80, 0x100, 0x200, 0x400):
            for (w, h, dw, dh) in ((64, 48, 64, 30), (20, 10, 300, 7), (351, 287, 97, 301)):
                y, u, v = cl.yuv_frame(w, h, 4200 + w, "limited")
                assert np.array_equal(cl.orc_sws(w, h, dw, dh, fl | FATE, y, u, v), cl.ref_sws(w, h, dw, dh, fl | FATE, y, u, v)), (hex(fl), w, h, dw, dh)
                src = cl.rgb_frame(w, h, 4300 + w, 4)
                a, b = (f(w, h, dw, dh, fl, src, src, src, src_fmt=cl.PIX_FMT_BGRA, dst_fmt=cl.PIX_FMT_NV12) for f in (cl.orc_sws_planar, cl.ref_sws_planar))
                assert all(np.array_equal(p, q) for p, q in zip(a, b)), (hex(fl), "bgra -> nv12")


def test_sws_oracle_yuv_matrix_cascade_vs_ref(refrec):
    """yuv -> yuv with different source and destination matrices: the reference cascades two contexts through bgr24 (utils.c:914-989)"""
    from cases import SWS_CASCADE_CASES
    for i, (w, h, dw, dh, fl, sf, df, ranges, det) in enumerate(SWS_CASCADE_CASES):
        y, u, v = cl.yuv_frame(w, h, 5200 + i, "random" if i % 2 else "smooth")
        if sf:
            u = v = cl.nv_interleave(u, v, sf)
        b = cl.orc_sws_planar(w, h, dw, dh, fl, y, u, v, src_fmt=sf, dst_fmt=df, ranges=ranges, details=det, dst_pad=i % 3)
        assert refrec.same(flat(b), lambda: flat(cl.ref_sws_planar(w, h, dw, dh, fl, y, u, v, src_fmt=sf, dst_fmt=df, ranges=ranges, details=det, dst_pad=i % 3))), \
            (i, w, h, dw, dh, hex(fl))
        same = cl.orc_sws_planar(w, h, dw, dh, fl, y, u, v, src_fmt=sf, dst_fmt=df, ranges=ranges, details=(det[0], det[1], det[0], det[3]) + det[4:], dst_pad=i % 3)
        assert not all(np.array_equal(p, q) for p, q in zip(b, same)), i        # the second matrix matters


def run_filter_case(run_rgb, run_planar, i, case):
    from cases import SWS_FILTER_CASES  # noqa: F401
    w, h, dw, dh, fl, dst, src, dlen = case
    y, u, v = cl.yuv_frame(w, h, 7100 + i, "random" if i % 2 else "smooth")
    if dst == "yuv420p":
        return run_planar(w, h, dw, dh, fl, y, u, v, filters=(src, dlen))
    return (run_rgb(w, h, dw, dh, fl, y, u, v, filters=(src, dlen), fmt=cl.PACKED_RGB_FORMATS[dst]),)


def test_sws_oracle_src_dst_filters_vs_ref(refrec):
    """sws_getContext's srcFilter / dstFilter (initFilter's filter2 stage, utils.c:384-413, and the unscaled-converter gate :1256-1263)"""
    from cases import SWS_FILTER_CASES
    for i, case in enumerate(SWS_FILTER_CASES):
        b = run_filter_case(cl.orc_sws, cl.orc_sws_planar, i, case)
        assert refrec.same(flat(b), lambda: flat(run_filter_case(cl.ref_sws, cl.ref_sws_planar, i, case))), (i, case[:6])
    plain = run_filter_case(lambda *a, filters=None, **k: cl.orc_sws(*a, **k), lambda *a, filters=None, **k: cl.orc_sws_planar(*a, **k), 0, SWS_FILTER_CASES[0])
    assert not np.array_equal(plain[0], run_filter_case(cl.orc_sws, cl.orc_sws_planar, 0, SWS_FILTER_CASES[0])[0])     # the vectors matter
    one = run_filter_case(cl.orc_sws, cl.orc_sws_planar, 7, SWS_FILTER_CASES[7])
    none = run_filter_case(lambda *a, filters=None, **k: cl.orc_sws(*a, **k), lambda *a, filters=None, **k: cl.orc_sws_planar(*a, **k), 7, SWS_FILTER_CASES[7])
    assert all(np.array_equal(p, q) for p, q in zip(one, none))                                                    # one-tap vectors are the identity
