"""GPU tier, second file: kernels of SURVEY.md 8f rows 2-4 (range conversion, packed-RGB sources, nv12/nv21 destinations, planar
slices, scaler parameters, float_dsp, 10/12-bit IDCT, ProRes, inverse quantisers, DCT / int32 / compound MDCT / full iMDCT, the
H.264 loop filter, pixelutils).  All of them passed on a B200 at the end of round 1 (GPUTEST_r01.json) and are ordinary tests of the
gpu tier: a mismatch fails the tier.  Each compares the CUDA path with the oracle and the reference-generated fixtures.
B200_ISOLATE=1 runs every test body in a child process (useful when bisecting a faulting kernel: the function tables abort()
on a CUDA error like the void C functions they replace)."""
import functools
import os
import subprocess
import sys

import numpy as np
import pytest

import cpulibs as cl
from ctypes import c_int as C_int, c_void_p as C_vp, c_ssize_t as C_ss

pytestmark = [pytest.mark.gpu]
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def isolated(fn):
    """With B200_ISOLATE=1: run the test body in a child pytest process (a faulting kernel poisons its CUDA context and the function
    tables abort() on a CUDA error).  By default the body runs in-process like every other test of the tier."""
    @functools.wraps(fn)
    def wrapper(device):
        if os.environ.get("B200_ISOLATE") != "1" or os.environ.get("B200_ISOLATED_CHILD") == "1":
            return fn(device)
        env = dict(os.environ, B200_ISOLATED_CHILD="1")
        r = subprocess.run([sys.executable, "-m", "pytest", f"{os.path.abspath(__file__)}::{fn.__name__}", "-m", "gpu", "-q", "-x",
                            "-p", "no:cacheprovider"], env=env, capture_output=True, text=True, timeout=600,
                           cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
        assert r.returncode == 0, "child run failed:\n" + r.stdout[-4000:] + r.stderr[-2000:]
    return wrapper


def on_stream(device):
    import torch
    return torch.cuda.stream(torch.cuda.ExternalStream(device.stream))


# ---------------------------------------------------------------------------------------------- swscale yuv -> yuv range conversion
# (the one hardware call these were scheduled on was cut short by its time limit before reaching them)
@isolated
def test_range_conversion_golden_hashes_and_oracle(device):
    """yuv -> yuv range conversion (SWS_RANGE_CASES) against the reference's outputs and the oracle; ranges at initialisation
    or changed through sws_setColorspaceDetails(), incl. the same-size context that stays a plain copy."""
    from cases import SWS_RANGE_CASES
    from test_sws_gpu import gpu_sws_planar, sha
    lines = open(os.path.join(G, "sws_range_hashes.txt")).read().split("\n")[:-1]
    assert len(lines) == len(SWS_RANGE_CASES)
    for line, (w, h, dw, dh, fl, kind, ranges, details) in zip(lines, SWS_RANGE_CASES):
        i, hout = int(line.split()[0]), line.split()[-1]
        y, u, v = cl.yuv_frame(w, h, 1200 + i, kind)
        out = gpu_sws_planar(device, w, h, dw, dh, fl, y, u, v, ranges=ranges, details=details)
        exp = cl.orc_sws_planar(w, h, dw, dh, fl, y, u, v, ranges=ranges, details=details)
        assert all(np.array_equal(p, q) for p, q in zip(out, exp)), (i, [int((p != q).sum()) for p, q in zip(out, exp)])
        assert sha(np.concatenate([p.ravel() for p in out])) == hout, (i, w, h, dw, dh, hex(fl), ranges, details)


@isolated
def test_range_conversion_fate_crc_padded_nv12(device):
    """FATE's sws-yuv-range checksum on the CUDA path; padded strides and an nv12 source."""
    from test_oracle import fate_sws_yuv_range_crc, FATE_SWS_YUV_RANGE
    from test_sws_gpu import gpu_sws_planar, FATE
    assert fate_sws_yuv_range_crc(functools.partial(gpu_sws_planar, device)) == FATE_SWS_YUV_RANGE
    for (w, h, dw, dh, fl, ranges) in [(640, 360, 1280, 720, FATE, (0, 1)), (351, 287, 351, 287, cl.SWS_BICUBIC, (1, 0)),
                                       (1920, 1080, 1280, 720, cl.SWS_BILINEAR, (1, 0))]:
        y, u, v = cl.yuv_frame(w, h, 1400 + w, "random", pad=5)
        out = gpu_sws_planar(device, w, h, dw, dh, fl, y, u, v, dst_pad=7, ranges=ranges)
        exp = cl.orc_sws_planar(w, h, dw, dh, fl, y, u, v, dst_pad=7, ranges=ranges)
        assert all(np.array_equal(p, q) for p, q in zip(out, exp)), (w, h, dw, dh, hex(fl), ranges)
    # nv12 source, limited -> full
    w, h, dw, dh = 640, 360, 800, 450
    y, u, v = cl.yuv_frame(w, h, 1500, "limited")
    uv = cl.nv_interleave(u, v, cl.PIX_FMT_NV12)
    out = gpu_sws_planar(device, w, h, dw, dh, FATE, y, uv, uv, src_fmt=cl.PIX_FMT_NV12, ranges=(0, 1))
    exp = cl.orc_sws_planar(w, h, dw, dh, FATE, y, uv, uv, src_fmt=cl.PIX_FMT_NV12, ranges=(0, 1))
    assert all(np.array_equal(p, q) for p, q in zip(out, exp))


@isolated
def test_range_conversion_batch_device(device):
    """batched device entry point with range conversion (3 frames, full -> limited); a matrix change is accepted"""
    import torch
    import ffmpeg_b200 as fb
    from ffmpeg_b200 import swscale as sw
    from cases import FATE
    w, h, dw, dh, n = 320, 180, 480, 270, 3
    frames = [cl.yuv_frame(w, h, 1600 + k, "random") for k in range(n)]
    cw, ch, dcw, dch = w // 2, h // 2, dw // 2, dh // 2
    ctx = sw.sws_getContext(device, w, h, 0, dw, dh, sw.AV_PIX_FMT_YUV420P, FATE, src_range=1, dst_range=0)
    with torch.cuda.stream(torch.cuda.ExternalStream(device.stream)):
        Y, U, V = (torch.from_numpy(np.stack([f[k] for f in frames])).cuda() for k in range(3))
        DY = torch.zeros((n, dh, dw), dtype=torch.uint8, device="cuda")
        DU = torch.zeros((n, dch, dcw), dtype=torch.uint8, device="cuda")
        DV = torch.zeros((n, dch, dcw), dtype=torch.uint8, device="cuda")
        ctx.scale_batch_device_planar([Y, U, V], [w, cw, cw], [w * h, cw * ch, cw * ch], [DY, DU, DV], [dw, dcw, dcw],
                                      [dw * dh, dcw * dch, dcw * dch], n)
        device.sync()
        got = [t.cpu().numpy() for t in (DY, DU, DV)]
    for i in range(n):
        exp = cl.orc_sws_planar(w, h, dw, dh, FATE, *frames[i], ranges=(1, 0))
        for k in range(3):
            assert np.array_equal(got[k][i], exp[k]), (i, k)
    # different matrices for yuv -> yuv: the reference cascades through bgr24 and so does this path (test_sws_yuv_matrix_cascade)
    assert ctx.setColorspaceDetails(cl.COEFFS[1], 0, cl.COEFFS[5], 1, 0, 1 << 16, 1 << 16) == 0
    ctx.free()


@isolated
def test_sws_float_kernel_scalers(device):
    """SWS_X / GAUSS / SINC / LANCZOS / SPLINE: only the host-side filter banks are new (up to 59 taps vertically here); same kernels"""
    from cases import SWS_FLOAT_KERNEL_CASES
    from test_sws_gpu import gpu_sws, gpu_sws_planar, sha
    lines = open(os.path.join(G, "sws_float_kernel_hashes.txt")).read().split("\n")[:-1]
    for line, (w, h, dw, dh, fl, kind) in zip(lines, SWS_FLOAT_KERNEL_CASES):
        i, hrgb, hyuv = line.split()
        y, u, v = cl.yuv_frame(w, h, 4100 + int(i), kind)
        assert sha(gpu_sws(device, w, h, dw, dh, fl, y, u, v)) == hrgb, (i, hex(fl))
        assert sha(np.concatenate([p.ravel() for p in gpu_sws_planar(device, w, h, dw, dh, fl, y, u, v)])) == hyuv, (i, hex(fl))
    y, u, v = cl.yuv_frame(1920, 1080, 4400, "random")                  # lanczos 1080p -> 720p, the common quality downscale
    fl = 0x200 | 0xc0000
    assert np.array_equal(gpu_sws(device, 1920, 1080, 1280, 720, fl, y, u, v), cl.orc_sws(1920, 1080, 1280, 720, fl, y, u, v))


@isolated
def test_sws_slice_calls_planar_destination(device):
    """sws_scale() band by band into yuv420p / nv12: the lines add up, the planes equal the whole-frame result (the checker's), and
    the per-call counts equal the reference's for the committed slice fixture geometry (64 x 48 source, tests/cases.py)"""
    from ffmpeg_b200 import swscale as sw
    from cases import FATE
    for (w, h, dw, dh, fl, df, bands) in ((64, 48, 100, 70, FATE, 0, [(0, 16), (16, 8), (24, 24)]), (320, 180, 480, 270, cl.SWS_BICUBIC, cl.PIX_FMT_NV12, [(0, 64), (64, 116)]),
                                          (64, 48, 64, 48, cl.SWS_BILINEAR, 0, [(0, 2), (2, 46)])):
        y, u, v = cl.yuv_frame(w, h, 7800 + w, "random")
        exp = cl.orc_sws_planar(w, h, dw, dh, fl, y, u, v, dst_fmt=df)
        cw, ch = (dw + 1) // 2, (dh + 1) // 2
        planes = [np.full((dh, dw), 0xA5, np.uint8), np.full((ch, 2 * cw if df else cw), 0xA5, np.uint8), np.full((ch, cw), 0xA5, np.uint8)]
        ctx = sw.sws_getContext(device, w, h, 0, dw, dh, df, fl)
        for rep in range(2):
            rets = [ctx.scale([y[sy:], u[sy // 2:], v[sy // 2:]], [y.strides[0], u.strides[0], v.strides[0]], sy, sh, planes, [p.strides[0] for p in planes])
                    for (sy, sh) in bands]
            assert sum(rets) == dh and all(r >= 0 for r in rets), rets
        ctx.free()
        assert all(np.array_equal(a, b) for a, b in zip(planes, exp)), (w, h, dw, dh, hex(fl), df)


@isolated
def test_sws_scaler_params(device):
    """sws_getContext's `param`: only the host-side filter banks depend on it"""
    from cases import SWS_PARAM_CASES
    from ffmpeg_b200 import swscale as sw
    for i, (fl, prm) in enumerate(SWS_PARAM_CASES):
        w, h, dw, dh = 352, 288, 200, 100
        y, u, v = cl.yuv_frame(w, h, 4500 + i, "random")
        ctx = sw.sws_getContext(device, w, h, 0, dw, dh, cl.PIX_FMT_RGB24, fl | 0xc0000, param=prm)
        got = ctx.convert(y, u, v)
        ctx.free()
        assert np.array_equal(got, cl.orc_sws(w, h, dw, dh, fl | 0xc0000, y, u, v, param=prm)), (hex(fl), prm)


@isolated
def test_sws_odd_width_unscaled_leaves_last_column(device):
    """same-size yuv420p -> rgb without accurate_rnd at an odd width: the reference's pair-wise LUT converter never writes the last
    column (yuv2rgb.c:137-236); found by differential fuzzing on the emulated device, the host entry points used to copy it back"""
    from test_sws_gpu import gpu_sws
    for (w, h) in ((7, 6), (17, 10), (351, 288)):
        y, u, v = cl.yuv_frame(w, h, 3700 + w, "random")
        for name in ("rgb24", "bgra"):
            f = cl.PACKED_RGB_FORMATS[name]
            got, exp = gpu_sws(device, w, h, w, h, cl.SWS_BICUBIC, y, u, v, fmt=f, dst_pad=2), cl.orc_sws(w, h, w, h, cl.SWS_BICUBIC, y, u, v, fmt=f, dst_pad=2)
            assert np.array_equal(got, exp), (w, h, name)


# ---------------------------------------------------------------------------------------------- mpegvideo inverse quantisers
def gpu_unquant(device, variant, cfg, blocks, blk_n, q, last):
    import torch
    from ffmpeg_b200 import mpegvideo as mv
    from ffmpeg_b200._lib import MpvUnquant
    p = cl.unquant_params(struct=MpvUnquant, **cfg)
    with on_stream(device):
        db = torch.from_numpy(np.ascontiguousarray(blocks)).cuda()
        dn = torch.from_numpy(blk_n).cuda() if blk_n is not None else None
        dq, dl = torch.from_numpy(q).cuda(), torch.from_numpy(last).cuda()
        mv.unquantize_batch_device(device, variant, p, db, blocks.shape[0], dn, dq, dl)
        device.sync()
        return db.cpu().numpy()


@isolated
def test_unquant_golden_and_oracle(device):
    g = np.load(os.path.join(G, "unquant.npz"))
    for variant in range(7):
        for seed in (11, 12):
            cfg, blocks, blk_n, q, last = cl.unquant_case(seed * 7 + variant, variant, nblocks=48)
            out = gpu_unquant(device, variant, cfg, blocks, blk_n, q, last)
            assert np.array_equal(out, g[f"v{variant}_s{seed}"]), (cl.UNQUANT_VARIANTS[variant], seed)
        for seed in range(6):
            cfg, blocks, blk_n, q, last = cl.unquant_case(300 + seed * 7 + variant, variant, nblocks=5000 + seed)
            use_n = blk_n if seed & 1 else None
            out = gpu_unquant(device, variant, cfg, blocks, use_n, q, last)
            assert np.array_equal(out, cl.orc_unquant(variant, cfg, blocks, use_n, q, last)), (cl.UNQUANT_VARIANTS[variant], seed)


@isolated
def test_unquant_errors(device):
    import torch
    import ffmpeg_b200 as fb
    from ffmpeg_b200 import mpegvideo as mv
    from ffmpeg_b200._lib import MpvUnquant
    cfg, blocks, blk_n, q, last = cl.unquant_case(1, 0, nblocks=8)
    p = cl.unquant_params(struct=MpvUnquant, **cfg)
    p.permutated[5] = p.permutated[6]                                  # not a permutation
    with on_stream(device):
        db, dq, dl = torch.from_numpy(blocks).cuda(), torch.from_numpy(q).cuda(), torch.from_numpy(last).cuda()
        with pytest.raises(fb.B200Error):
            mv.unquantize_batch_device(device, 0, p, db, 8, None, dq, dl)
        p = cl.unquant_params(struct=MpvUnquant, **cfg)
        with pytest.raises(fb.B200Error):
            mv.unquantize_batch_device(device, 7, p, db, 8, None, dq, dl)
        assert mv.unquantize_batch_device(device, 0, p, db, 0, None, dq, dl) == 0


# ---------------------------------------------------------------------------------------------- AVFloatDSPContext
@isolated
def test_fdsp_pointer_table_golden(device):
    """AVFloatDSPContext entries called with host pointers, against the reference's outputs (fdsp.npz), bit for bit"""
    import ctypes as C
    from ffmpeg_b200 import float_dsp as fd
    g = np.load(os.path.join(G, "fdsp.npz"))
    c = fd.avpriv_float_dsp_alloc(0)
    F, D = C.POINTER(C.c_float), C.POINTER(C.c_double)
    for op in range(12):
        P = D if op in cl.FDSP_DOUBLE else F
        for length in (16, 100, 1024):
            dst, s0, s1, s2, mul = cl.fdsp_case(40 + op, op, length)
            p = lambda a: a.ctypes.data_as(P)
            name = cl.FDSP_OPS[op]
            fn = getattr(c, name)
            if op in (0, 7, 10):
                fn(p(dst), p(s0), p(s1), length)
            elif op in (1, 2, 3, 4):
                fn(p(dst), p(s0), mul, length)
            elif op in (5, 6):
                fn(p(dst), p(s0), p(s1), p(s2), length)
            elif op == 8:
                fn(p(dst), p(s0), length)
                assert s0.tobytes() == g[f"op{op}_n{length}_v2"].tobytes()
            else:
                dst = np.array([fn(p(s0), p(s1), length)], dst.dtype)
            got = dst[:1] if op in (9, 11) else dst
            assert got.tobytes() == g[f"op{op}_n{length}"].tobytes(), (name, length)


@isolated
def test_fdsp_batch_vs_oracle(device):
    """batched device entry point: many vectors, shared window / operand (stride 0), odd lengths, more than 65535 vectors"""
    import torch
    from ffmpeg_b200 import float_dsp as fd
    for op in range(12):
        for length, nvec in ((1024, 40), (77, 9), (8, 70000 if op in (0, 9) else 300)):
            dt = np.float64 if op in cl.FDSP_DOUBLE else np.float32
            n2 = 2 * length if op == 5 else length
            cases = [cl.fdsp_case(700 + op * 31 + v % 50, op, length) for v in range(min(nvec, 50))]
            idx = np.arange(nvec) % len(cases)
            dst = np.stack([cases[i][0] for i in idx]); s0 = np.stack([cases[i][1] for i in idx]); s1 = np.stack([cases[i][2] for i in idx])
            s2 = cases[0][3]                                            # one window / addend for all vectors (stride 0)
            mul = cases[0][4]
            exp = [cl.orc_fdsp(op, cases[i][0], cases[i][1], cases[i][2], s2, mul, length) for i in range(len(cases))]
            dot = op in (9, 11)
            with on_stream(device):
                dd = torch.from_numpy(np.zeros(nvec, dt) if dot else dst).cuda()
                d0, d1, d2 = torch.from_numpy(s0).cuda(), torch.from_numpy(s1).cuda(), torch.from_numpy(s2).cuda()
                fd.float_dsp_batch_device(device, op, nvec, length, dd, 1 if dot else n2, d0, length, d1, length, d2, 0, mul)
                device.sync()
                got, got0 = dd.cpu().numpy(), d0.cpu().numpy()
            for v in range(nvec):
                e, e0 = exp[idx[v]]
                assert (got[v:v + 1] if dot else got[v]).tobytes() == e.tobytes(), (cl.FDSP_OPS[op], length, v)
                assert got0[v].tobytes() == e0.tobytes(), (cl.FDSP_OPS[op], length, v, "src0")


# ---------------------------------------------------------------------------------------------- simple IDCT, 10 / 12 bit
def gpu_idct_hbd(device, depth, kind, blocks, dest):
    """blocks [n, 64], dest uint16 [8, >= n*8]: block i at column 8*i -> (blocks after, dest after)"""
    import torch
    from ffmpeg_b200 import idctdsp
    n = blocks.shape[0]
    off = (np.arange(n, dtype=np.int64) * 16)
    with on_stream(device):
        db, dd, do = torch.from_numpy(blocks.copy()).cuda(), torch.from_numpy(dest.view(np.int16).copy()).cuda(), torch.from_numpy(off).cuda()
        idctdsp.idct_hbd_batch_device(device, depth, kind, db, n, dd, do, None, dest.strides[0])
        device.sync()
        return db.cpu().numpy(), dd.cpu().numpy().view(np.uint16)


@isolated
def test_idct_hbd_golden_and_oracle(device):
    g = np.load(os.path.join(G, "idct_hbd.npz"))
    for depth in (10, 12):
        blocks = cl.idct_hbd_blocks(70 + depth, depth, 60)
        dest = np.random.default_rng(depth).integers(0, 1 << depth, (8, 60 * 8), dtype=np.uint16)
        for kind in (0, 1, 2):
            b, o = gpu_idct_hbd(device, depth, kind, blocks, dest)
            assert np.array_equal(b if kind == 0 else o, g[f"d{depth}_k{kind}"]), (depth, kind)
            if kind:
                assert np.array_equal(b, blocks)                            # put / add leave the coefficients alone
        for kind in (0, 1, 2):
            blocks = cl.idct_hbd_blocks(400 + depth + kind, depth, 5000)
            dest = np.random.default_rng(kind).integers(0, 1 << depth, (8, 5000 * 8 + 4), dtype=np.uint16)
            b, o = gpu_idct_hbd(device, depth, kind, blocks, dest)
            eb, eo = cl.orc_idct_hbd(depth, kind, blocks, dest, dest.strides[0])
            assert np.array_equal(o, eo) and (kind != 0 or np.array_equal(b, eb)), (depth, kind)


@isolated
def test_idct_hbd_pointer_table(device):
    """IDCTDSPContext for bits_per_raw_sample 9 / 10 / 12 called with host pointers"""
    import ctypes as C
    import ffmpeg_b200 as fb
    from ffmpeg_b200 import idctdsp
    from ffmpeg_b200._lib import u8p, i16p
    for bits, depth in ((9, 10), (10, 10), (12, 12)):
        c = idctdsp.ff_idctdsp_init_hbd(idctdsp.FF_IDCT_SIMPLE, bits, 0)
        blocks = cl.idct_hbd_blocks(bits, depth, 12)
        dest = np.random.default_rng(bits).integers(0, 1 << depth, (8, 12 * 8 + 3), dtype=np.uint16)
        for kind in (0, 1, 2):
            b, d = blocks.copy(), dest.copy()
            for i in range(12):
                blk = b[i].ctypes.data_as(i16p)
                if kind == 0:
                    c.idct(blk)
                else:
                    (c.idct_put if kind == 1 else c.idct_add)(C.cast(d.ctypes.data + 16 * i, u8p), d.strides[0], blk)
            eb, ed = cl.orc_idct_hbd(depth, kind, blocks, dest, dest.strides[0])
            assert np.array_equal(d, ed) and (kind != 0 or np.array_equal(b, eb)), (bits, kind)
    with pytest.raises(fb.B200Error):
        idctdsp.ff_idctdsp_init_hbd(idctdsp.FF_IDCT_SIMPLE, 8, 0)


# ---------------------------------------------------------------------------------------------- swscale: packed RGB sources
@isolated
def test_sws_rgb_sources_golden_and_oracle(device):
    """rgb24 / bgr24 / rgba / bgra / argb / abgr -> yuv420p (input readers fused into the horizontal pass, the bgr24 -> yv12
    converter, range conversion behind them) against the reference's outputs and the oracle"""
    import functools
    from test_oracle import rgbsrc_rows, run_rgbsrc_row, sha
    from test_sws_gpu import gpu_sws_planar, gpu_sws
    rows = rgbsrc_rows()
    assert len(rows) == 15 * 6 * 2 + 11 * 2
    gp, gr = functools.partial(gpu_sws_planar, device), functools.partial(gpu_sws, device)
    for row in rows:                                                    # -> yuv420p, and -> rgb24 through the scaler for rgb24 / bgr24
        got = run_rgbsrc_row(gr, gp, row)
        assert np.array_equal(got, run_rgbsrc_row(cl.orc_sws, cl.orc_sws_planar, row)), row[:6]
        assert sha(got) == row[-1], row[:6]


@isolated
def test_sws_rgb_sources_large_padded_batch(device):
    import torch
    import ffmpeg_b200 as fb
    from ffmpeg_b200 import swscale as sw
    from test_sws_gpu import gpu_sws_planar
    from cases import FATE
    for (w, h, dw, dh, fl, name) in [(1920, 1080, 1920, 1080, FATE, "bgra"), (1920, 1080, 1280, 720, cl.SWS_BICUBIC, "rgb24"),
                                     (1280, 720, 1280, 720, cl.SWS_BICUBIC, "bgr24"), (641, 361, 1280, 720, cl.SWS_BILINEAR, "argb"),
                                     (1281, 721, 1281, 721, cl.SWS_BICUBIC, "bgr24")]:
        sf = cl.PACKED_RGB_FORMATS[name]
        src = cl.rgb_frame(w, h, 2300 + w, cl.fmt_bpp(sf), "random", pad=5)
        out = gpu_sws_planar(device, w, h, dw, dh, fl, src, src, src, dst_pad=3, src_fmt=sf)
        exp = cl.orc_sws_planar(w, h, dw, dh, fl, src, src, src, dst_pad=3, src_fmt=sf)
        assert all(np.array_equal(p, q) for p, q in zip(out, exp)), (w, h, dw, dh, hex(fl), name)
    # batched device entry point, 3 frames of rgba -> yuv420p (scaled) and of bgr24 through the special converter
    for (name, dw, dh, fl) in (("rgba", 480, 270, FATE), ("bgr24", 320, 180, cl.SWS_BICUBIC)):
        sf, w, h, n = cl.PACKED_RGB_FORMATS[name], 320, 180, 3
        bpp = cl.fmt_bpp(sf)
        frames = [cl.rgb_frame(w, h, 2400 + k, bpp) for k in range(n)]
        ctx = sw.sws_getContext(device, w, h, sf, dw, dh, sw.AV_PIX_FMT_YUV420P, fl)
        with torch.cuda.stream(torch.cuda.ExternalStream(device.stream)):
            S = torch.from_numpy(np.stack(frames)).cuda()
            DY = torch.zeros((n, dh, dw), dtype=torch.uint8, device="cuda")
            DU = torch.zeros((n, dh // 2, dw // 2), dtype=torch.uint8, device="cuda")
            DV = torch.zeros((n, dh // 2, dw // 2), dtype=torch.uint8, device="cuda")
            ctx.scale_batch_device_planar([S], [w * bpp], [w * bpp * h], [DY, DU, DV], [dw, dw // 2, dw // 2],
                                          [dw * dh, dw * dh // 4, dw * dh // 4], n)
            device.sync()
            got = [t.cpu().numpy() for t in (DY, DU, DV)]
        for i in range(n):
            exp = cl.orc_sws_planar(w, h, dw, dh, fl, frames[i], frames[i], frames[i], src_fmt=sf)
            for k in range(3):
                assert np.array_equal(got[k][i], exp[k]), (name, i, k)
        ctx.free()
    # packed RGB -> packed RGB through the scaler: batched device entry point, other destination orders
    w, h, dw, dh, n = 320, 180, 200, 100, 3
    frames = [cl.rgb_frame(w, h, 2450 + k, 3) for k in range(n)]
    for dname in ("bgr24", "rgba", "argb"):
        df = cl.PACKED_RGB_FORMATS[dname]
        bpp = cl.fmt_bpp(df)
        ctx = sw.sws_getContext(device, w, h, sw.AV_PIX_FMT_RGB24, dw, dh, df, FATE)
        with torch.cuda.stream(torch.cuda.ExternalStream(device.stream)):
            S = torch.from_numpy(np.stack(frames)).cuda()
            D = torch.zeros((n, dh, dw * bpp), dtype=torch.uint8, device="cuda")
            ctx.scale_batch_device([S], [w * 3], [w * 3 * h], D, dw * bpp, dw * bpp * dh, n)
            device.sync()
            got = D.cpu().numpy()
        for i in range(n):
            assert np.array_equal(got[i], cl.orc_sws(w, h, dw, dh, FATE, frames[i], frames[i], frames[i], fmt=df, src_fmt=cl.PIX_FMT_RGB24)), (dname, i)
        ctx.free()
    # alpha carried through the scaler (32-bit source and destination): host sws_scale and the batched device entry
    from test_sws_gpu import gpu_sws
    names4 = ["rgba", "bgra", "argb", "abgr"]
    for it, (w, h, dw, dh, fl) in enumerate([(64, 48, 32, 24, FATE), (64, 48, 100, 70, 2), (322, 180, 1280, 720, 4), (1280, 720, 640, 360, 4), (64, 48, 96, 48, 1),
                                             (641, 361, 320, 200, 0x10), (320, 180, 321, 181, 0x20)]):
        sf, df = cl.PACKED_RGB_FORMATS[names4[it % 4]], cl.PACKED_RGB_FORMATS[names4[(it * 3 + 1) % 4]]
        src = cl.rgb_frame(w, h, 3200 + it, 4, "random", pad=it % 3)
        assert np.array_equal(gpu_sws(device, w, h, dw, dh, fl, src, src, src, fmt=df, src_fmt=sf), cl.orc_sws(w, h, dw, dh, fl, src, src, src, fmt=df, src_fmt=sf)), (it, "alpha")
    w, h, dw, dh, n = 320, 180, 200, 100, 3
    frames = [cl.rgb_frame(w, h, 3250 + k, 4) for k in range(n)]
    ctx = sw.sws_getContext(device, w, h, sw.AV_PIX_FMT_RGBA, dw, dh, sw.AV_PIX_FMT_BGRA, 4)
    with torch.cuda.stream(torch.cuda.ExternalStream(device.stream)):
        S = torch.from_numpy(np.stack(frames)).cuda()
        D = torch.zeros((n, dh, dw * 4), dtype=torch.uint8, device="cuda")
        ctx.scale_batch_device([S], [w * 4], [w * 4 * h], D, dw * 4, dw * 4 * dh, n)
        device.sync()
        got = D.cpu().numpy()
    for i in range(n):
        assert np.array_equal(got[i], cl.orc_sws(w, h, dw, dh, 4, frames[i], frames[i], frames[i], fmt=cl.PIX_FMT_BGRA, src_fmt=cl.PIX_FMT_RGBA)), ("alpha batch", i)
    ctx.free()


# ---------------------------------------------------------------------------------------------- swscale: nv12 / nv21 destinations
@isolated
def test_sws_nv_destinations(device):
    """nv12 / nv21 as the destination (the layout NVENC reads) from planar, semi-planar and packed RGB sources, against the oracle;
    then FATE's own md5 sums for these formats (null, copy, vflip, hflip, crop, scale, pixdesc) on the CUDA path's frames"""
    import functools
    import torch
    from ffmpeg_b200 import swscale as sw
    from test_sws_gpu import gpu_sws_planar, gpu_sws
    from cases import SWS_PLANAR_CASES, SWS_RANGE_CASES, SWS_RGBSRC_CASES, FATE
    import test_fate_golden as fg
    for df in (cl.PIX_FMT_NV12, cl.PIX_FMT_NV21):
        for i, (w, h, dw, dh, fl, kind) in enumerate(SWS_PLANAR_CASES):
            y, u, v = cl.yuv_frame(w, h, 2500 + i, kind)
            out = gpu_sws_planar(device, w, h, dw, dh, fl, y, u, v, dst_fmt=df, dst_pad=i % 3)
            exp = cl.orc_sws_planar(w, h, dw, dh, fl, y, u, v, dst_fmt=df, dst_pad=i % 3)
            assert len(out) == 2 and all(np.array_equal(p, q) for p, q in zip(out, exp)), ("planar", i, df)
        for i, (w, h, dw, dh, fl, kind, ranges, det) in enumerate(SWS_RANGE_CASES[:9]):
            y, u, v = cl.yuv_frame(w, h, 2600 + i, kind)
            out = gpu_sws_planar(device, w, h, dw, dh, fl, y, u, v, dst_fmt=df, ranges=ranges)
            exp = cl.orc_sws_planar(w, h, dw, dh, fl, y, u, v, dst_fmt=df, ranges=ranges)
            assert all(np.array_equal(p, q) for p, q in zip(out, exp)), ("range", i, df)
        y, u, v = cl.yuv_frame(640, 360, 2700, "random")
        uv = cl.nv_interleave(u, v, cl.PIX_FMT_NV12)
        for (dw, dh) in ((640, 360), (800, 450)):
            out = gpu_sws_planar(device, 640, 360, dw, dh, FATE, y, uv, uv, src_fmt=cl.PIX_FMT_NV12, dst_fmt=df)
            exp = cl.orc_sws_planar(640, 360, dw, dh, FATE, y, uv, uv, src_fmt=cl.PIX_FMT_NV12, dst_fmt=df)
            assert all(np.array_equal(p, q) for p, q in zip(out, exp)), ("nv12 source", dw, df)
    if cl.have_nut() and os.path.exists(cl.VIDEOGEN):                # FATE's frames and NUT muxer come from the reference build
        fg.check_all(functools.partial(gpu_sws, device), functools.partial(gpu_sws_planar, device), rgb_sources=True, nv_dest=True)     # all 59 FATE sums
    # the encoder feed: bgra 1080p -> nv12 (packed RGB source kernels too), and the batched device entry point with two destination planes
    src = cl.rgb_frame(1920, 1080, 2900, 4)
    out = gpu_sws_planar(device, 1920, 1080, 1920, 1080, FATE, src, src, src, src_fmt=cl.PIX_FMT_BGRA, dst_fmt=cl.PIX_FMT_NV12)
    exp = cl.orc_sws_planar(1920, 1080, 1920, 1080, FATE, src, src, src, src_fmt=cl.PIX_FMT_BGRA, dst_fmt=cl.PIX_FMT_NV12)
    assert all(np.array_equal(p, q) for p, q in zip(out, exp))
    w, h, dw, dh, n = 320, 180, 480, 270, 3
    frames = [cl.yuv_frame(w, h, 2950 + k, "random") for k in range(n)]
    ctx = sw.sws_getContext(device, w, h, 0, dw, dh, sw.AV_PIX_FMT_NV12, FATE)
    with on_stream(device):
        Y, U, V = (torch.from_numpy(np.stack([f[k] for f in frames])).cuda() for k in range(3))
        DY = torch.zeros((n, dh, dw), dtype=torch.uint8, device="cuda")
        DUV = torch.zeros((n, dh // 2, dw), dtype=torch.uint8, device="cuda")
        ctx.scale_batch_device_planar([Y, U, V], [w, w // 2, w // 2], [w * h, w * h // 4, w * h // 4], [DY, DUV], [dw, dw],
                                      [dw * dh, dw * dh // 2], n)
        device.sync()
        gy, guv = DY.cpu().numpy(), DUV.cpu().numpy()
    for i in range(n):
        ey, euv = cl.orc_sws_planar(w, h, dw, dh, FATE, *frames[i], dst_fmt=cl.PIX_FMT_NV12)
        assert np.array_equal(gy[i], ey) and np.array_equal(guv[i], euv), i
    ctx.free()


# ---------------------------------------------------------------------------------------------- tx: AV_TX_FULL_IMDCT
@isolated
def test_tx_full_imdct(device):
    """av_tx_init(AV_TX_FLOAT_MDCT, inverse, flags = AV_TX_FULL_IMDCT): host av_tx_fn against the reference's outputs, batched device
    call against the oracle (power-of-two and compound lengths)"""
    import torch
    import ffmpeg_b200 as fb
    from ffmpeg_b200 import tx
    from test_oracle_more import _tx
    g = np.load(os.path.join(G, "tx_full_imdct.npz"))
    O = cl.oracle()
    for n in (4, 64, 256, 1024, 120, 144):
        for j, sc in enumerate((1.0 / n, -1.0)):
            c = tx.av_tx_init(tx.AV_TX_FLOAT_MDCT, 1, n, scale=sc, flags=tx.AV_TX_FULL_IMDCT)
            x = g[f"in_{n}"]
            out = np.zeros((x.shape[0], 2 * n), np.float32)
            for r in range(x.shape[0]):
                c.fn(out[r], x[r].copy(), 4)
            assert np.array_equal(out.view(np.uint32), g[f"out_{n}_{j}"].view(np.uint32)), (n, j)
            c.uninit()
    rng = np.random.default_rng(23)
    for n in (1024, 2048, 960, 640):
        cnt = 3000
        x = (rng.random((cnt, n), dtype=np.float32) * 2 - 1).astype(np.float32)
        c = tx.av_tx_init(tx.AV_TX_FLOAT_MDCT, 1, n, scale=1.0 / n, flags=tx.AV_TX_FULL_IMDCT, device=device)
        with on_stream(device):
            di, do = torch.from_numpy(x).cuda(), torch.zeros((cnt, 2 * n), dtype=torch.float32, device="cuda")
            c.batch_device(do, di, 4, cnt, 8 * n, 4 * n)
            device.sync()
            got = do.cpu().numpy()
        assert np.array_equal(got.view(np.uint32), _tx(O, "orc", 1, 1, n, 1.0 / n, x, 2 * n, flags=4).view(np.uint32)), n
        with pytest.raises(fb.B200Error):
            c.batch_device(do, di, 8, cnt, 8 * n, 4 * n)                # the mirror step only makes sense with stride == sizeof(float)
        c.uninit()
    for typ, inv in ((tx.AV_TX_FLOAT_MDCT, 0), (tx.AV_TX_FLOAT_FFT, 1), (tx.AV_TX_INT32_MDCT, 1)):
        with pytest.raises(fb.B200Error):
            tx.av_tx_init(typ, inv, 64, scale=1.0, flags=tx.AV_TX_FULL_IMDCT)


@isolated
def test_tx_inplace_fft(device):
    """AV_TX_INPLACE: complex FFT with out == in, batched (several transforms per CTA) and through av_tx_fn; other types refuse the flag"""
    import torch
    import ffmpeg_b200 as fb
    from ffmpeg_b200 import tx
    from test_oracle_more import _tx
    O = cl.oracle()
    rng = np.random.default_rng(29)
    for n in (2, 64, 1024, 4096):
        cnt = 1001
        x = (rng.random((cnt, 2 * n), dtype=np.float32) * 2 - 1).astype(np.float32)
        exp = _tx(O, "orc", 0, 1, n, 1.0, x, 2 * n)
        c = tx.av_tx_init(tx.AV_TX_FLOAT_FFT, 1, n, flags=tx.AV_TX_INPLACE, device=device)
        with on_stream(device):
            d = torch.from_numpy(x).cuda()
            c.batch_device(d, d, 8, cnt, 8 * n, 8 * n)
            device.sync()
            got = d.cpu().numpy()
        assert np.array_equal(got.view(np.uint32), exp.view(np.uint32)), n
        c.uninit()
        c = tx.av_tx_init(tx.AV_TX_FLOAT_FFT, 1, n, flags=tx.AV_TX_INPLACE)
        buf = x[0].copy()
        c.fn(buf, buf, 8)
        assert np.array_equal(buf.view(np.uint32), exp[0].view(np.uint32)), n
        c.uninit()
    for typ in (tx.AV_TX_FLOAT_MDCT, tx.AV_TX_FLOAT_RDFT, tx.AV_TX_FLOAT_DCT):
        with pytest.raises(fb.B200Error):
            tx.av_tx_init(typ, 0, 64, scale=1.0, flags=tx.AV_TX_INPLACE)


# ---------------------------------------------------------------------------------------------- tx: compound 15 x M MDCT (Opus CELT)
@isolated
def test_tx_mdct_pfa15(device):
    """av_tx_init(AV_TX_FLOAT_MDCT, 15 * 2^k): host av_tx_fn against the reference's outputs, batched device call against the oracle"""
    import torch
    import ffmpeg_b200 as fb
    from ffmpeg_b200 import tx
    from test_oracle_more import _tx
    g = np.load(os.path.join(G, "tx_pfa.npz"))
    O = cl.oracle()
    for n in (120, 240, 480, 960, 112, 448, 144, 576):
        for inv in (1, 0):
            for j, sc in enumerate((1.0 / n, -1.0)):
                c = tx.av_tx_init(tx.AV_TX_FLOAT_MDCT, inv, n, scale=sc)
                x = g[f"in_{n}_{inv}"]
                out = np.zeros((x.shape[0], n), np.float32)
                for r in range(x.shape[0]):
                    c.fn(out[r], x[r].copy(), 4)
                assert np.array_equal(out.view(np.uint32), g[f"out_{n}_{inv}_{j}"].view(np.uint32)), (n, inv, j)
                c.uninit()
    rng = np.random.default_rng(21)
    for n in (120, 960, 1920, 96, 640, 224, 1152):                     # 15 x M, 3 x M, 5 x M, 7 x M, 9 x M
        for inv in (1, 0):
            cnt = 3000
            x = (rng.random((cnt, n if inv else 2 * n), dtype=np.float32) * 2 - 1).astype(np.float32)
            c = tx.av_tx_init(tx.AV_TX_FLOAT_MDCT, inv, n, scale=1.0 / n, device=device)
            with on_stream(device):
                di, do = torch.from_numpy(x).cuda(), torch.zeros((cnt, n), dtype=torch.float32, device="cuda")
                c.batch_device(do, di, 4, cnt, 4 * n, x.strides[0])
                device.sync()
                got = do.cpu().numpy()
            assert np.array_equal(got.view(np.uint32), _tx(O, "orc", 1, inv, n, 1.0 / n, x, n).view(np.uint32)), (n, inv)
            c.uninit()
    with pytest.raises(fb.B200Error):
        tx.av_tx_init(tx.AV_TX_FLOAT_MDCT, 1, 84, scale=1.0)            # 7 x 6: the sub-transform would be a compound FFT, not built
    with pytest.raises(fb.B200Error):
        tx.av_tx_init(tx.AV_TX_FLOAT_FFT, 0, 90)                        # 45 x 2: a nested compound tree in the reference, not built


# ---------------------------------------------------------------------------------------------- tx: compound N x 2^k complex FFT
def test_tx_fft_pfa(device):
    """av_tx_init(AV_TX_FLOAT_FFT, N * 2^k), N = 15, 9, 7, 5, 3 (checkasm av_tx.c lengths 120 / 960 / 1920): host av_tx_fn against the
    reference's outputs, batched device call (out of place, in place, strided output) against the oracle"""
    import torch
    import ffmpeg_b200 as fb
    from ffmpeg_b200 import tx
    from test_oracle_more import _tx, PFA_FFT_SIZES
    g = np.load(os.path.join(G, "tx_pfa_fft.npz"))
    O = cl.oracle()
    for n in PFA_FFT_SIZES:
        for inv in (0, 1):
            c = tx.av_tx_init(tx.AV_TX_FLOAT_FFT, inv, n)
            x = g[f"in_{n}"]
            out = np.zeros((x.shape[0], 2 * n), np.float32)
            for r in range(x.shape[0]):
                c.fn(out[r], x[r].copy(), 8)
            assert np.array_equal(out.view(np.uint32), g[f"out_{n}_{inv}"].view(np.uint32)), (n, inv)
            c.uninit()
    rng = np.random.default_rng(22)
    for n in (120, 960, 1920, 7680, 96, 640, 224, 1152):               # 15 x M, 3 x M, 5 x M, 7 x M, 9 x M
        for inv in (0, 1):
            cnt = 2000 if n < 4000 else 300
            x = (rng.random((cnt, 2 * n), dtype=np.float32) * 2 - 1).astype(np.float32)
            exp = _tx(O, "orc", 0, inv, n, 1.0, x, 2 * n)
            c = tx.av_tx_init(tx.AV_TX_FLOAT_FFT, inv, n, device=device)
            with on_stream(device):
                di, do = torch.from_numpy(x).cuda(), torch.zeros((cnt, 2 * n), dtype=torch.float32, device="cuda")
                c.batch_device(do, di, 8, cnt, 8 * n, 8 * n)
                device.sync()
                assert np.array_equal(do.cpu().numpy().view(np.uint32), exp.view(np.uint32)), (n, inv)
                if n in (120, 224):                                     # strided output: out[i * stride] (tx_template.c:1078-1079)
                    d2 = torch.zeros((cnt, 4 * n), dtype=torch.float32, device="cuda")
                    c.batch_device(d2, di, 16, cnt, 16 * n, 8 * n)
                    device.sync()
                    got = d2.cpu().numpy().reshape(cnt, n, 4)
                    assert np.array_equal(got[:, :, :2].reshape(cnt, 2 * n).view(np.uint32), exp.view(np.uint32)) and not got[:, :, 2:].any(), (n, inv, "stride")
            c.uninit()
            if n in (960, 96):                                          # AV_TX_INPLACE
                c = tx.av_tx_init(tx.AV_TX_FLOAT_FFT, inv, n, flags=tx.AV_TX_INPLACE, device=device)
                with on_stream(device):
                    di = torch.from_numpy(x).cuda()
                    c.batch_device(di, di, 8, cnt, 8 * n, 8 * n)
                    device.sync()
                    assert np.array_equal(di.cpu().numpy().view(np.uint32), exp.view(np.uint32)), (n, inv, "inplace")
                c.uninit()


# ---------------------------------------------------------------------------------------------- tx: DCT-II / DCT-III
@isolated
def test_tx_dct(device):
    """AV_TX_FLOAT_DCT: host av_tx_fn against the reference's outputs, batched device call against the oracle"""
    import torch
    import ffmpeg_b200 as fb
    from ffmpeg_b200 import tx
    from test_oracle_more import _dct
    g = np.load(os.path.join(G, "tx_dct.npz"))
    O = cl.oracle()
    for n in (8, 64, 512):
        for inv, asked in ((0, n), (1, n // 2)):
            for j, sc in enumerate((1.0, 0.5 / n)):
                c = tx.av_tx_init(tx.AV_TX_FLOAT_DCT, inv, asked, scale=sc)
                x = g[f"in_{n}"]
                out = np.zeros((x.shape[0], n), np.float32)
                for r in range(x.shape[0]):
                    xin = x[r, :n].copy()
                    c.fn(out[r], xin, 4)
                    assert np.array_equal(xin, x[r, :n])                                 # the input is left alone
                assert np.array_equal(out.view(np.uint32), g[f"out_{n}_{inv}_{j}"].view(np.uint32)), (n, inv, j)
                c.uninit()
    rng = np.random.default_rng(22)
    for n in (16, 1024):
        for inv, asked in ((0, n), (1, n // 2)):
            cnt = 2000
            x = (rng.random((cnt, n + 2), dtype=np.float32) * 2 - 1).astype(np.float32)
            c = tx.av_tx_init(tx.AV_TX_FLOAT_DCT, inv, asked, scale=1.0, device=device)
            with on_stream(device):
                di, do = torch.from_numpy(np.ascontiguousarray(x[:, :n])).cuda(), torch.zeros((cnt, n), dtype=torch.float32, device="cuda")
                c.batch_device(do, di, 4, cnt, 4 * n, 4 * n)
                device.sync()
                got = do.cpu().numpy()
            assert np.array_equal(got.view(np.uint32), _dct(O, "orc", inv, asked, 1.0, x, n).view(np.uint32)), (n, inv)
            c.uninit()
    with pytest.raises(fb.B200Error):
        tx.av_tx_init(tx.AV_TX_FLOAT_DCT, 0, 96, scale=1.0)


# ---------------------------------------------------------------------------------------------- tx: 32-bit fixed point
@isolated
def test_tx_int32(device):
    """AV_TX_INT32_FFT / AV_TX_INT32_MDCT: host av_tx_fn against the reference's outputs, batched device call against the oracle"""
    import torch
    from ffmpeg_b200 import tx
    from test_oracle_more import _txi
    g = np.load(os.path.join(G, "tx_int32.npz"))
    O = cl.oracle()
    for n in (8, 64, 1024):
        x = g[f"in_{n}"]
        xs = (x >> 6).astype(np.int32)
        for inv in (0, 1):
            c = tx.av_tx_init(tx.AV_TX_INT32_FFT, inv, n)
            out = np.zeros_like(x)
            for r in range(2):
                c.fn(out[r], x[r].copy(), 8)
            assert np.array_equal(out, g[f"fft_{n}_{inv}"]), (n, inv)
            c.uninit()
        for j, sc in enumerate((1.0 / n, -1.0 / 32768)):
            for inv in (1, 0):
                xi = np.ascontiguousarray(xs[:, :n]) if inv else xs
                c = tx.av_tx_init(tx.AV_TX_INT32_MDCT, inv, n, scale=sc)
                out = np.zeros((2, n), np.int32)
                for r in range(2):
                    c.fn(out[r], xi[r].copy(), 4)
                assert np.array_equal(out, g[f"mdct_{n}_{inv}_{j}"]), (n, inv, j)
                c.uninit()
    rng = np.random.default_rng(23)
    for n in (16, 1024):
        cnt = 2000
        x = rng.integers(-(1 << 29), 1 << 29, (cnt, 2 * n)).astype(np.int32)
        for typ, inv, xin, outn in ((4, 0, x, 2 * n), (4, 1, x, 2 * n), (5, 1, np.ascontiguousarray(x[:, :n]), n), (5, 0, x, n)):
            c = tx.av_tx_init(typ, inv, n, scale=1.0 / n, device=device)
            with on_stream(device):
                di, do = torch.from_numpy(xin).cuda(), torch.zeros((cnt, outn), dtype=torch.int32, device="cuda")
                c.batch_device(do, di, 8 if typ == 4 else 4, cnt, 4 * outn, xin.strides[0])
                device.sync()
                got = do.cpu().numpy()
            assert np.array_equal(got, _txi(O, "orc", typ, inv, n, 1.0 / n, xin, outn)), (typ, inv, n)
            c.uninit()


# ---------------------------------------------------------------------------------------------- ProresDSPContext
@isolated
def test_prores_idct_put(device):
    """ProresDSPContext.idct_put (dequant + IDCT + bias + clip) at 10 and 12 bit: function table against the reference's pixels,
    batched device call against the oracle"""
    import torch
    from ffmpeg_b200 import idctdsp
    g = np.load(os.path.join(G, "prores.npz"))
    for bits in (10, 12):
        c = idctdsp.ff_proresdsp_init(bits)
        for seed in (0, 1, 2):
            blocks, qmat = cl.prores_case(90 + seed, bits, 60)
            px = np.zeros((8, 60 * 8), np.uint16)
            for i in range(60):
                blk = blocks[i].copy()                                  # kept alive across the call
                c.idct_put(px.ctypes.data + 16 * i, px.strides[0], blk.ctypes.data, qmat.ctypes.data)
            assert np.array_equal(px, g[f"b{bits}_s{seed}"]), (bits, seed)
        n = 20000
        blocks, qmat = cl.prores_case(700 + bits, bits, n)
        dest = np.zeros((8, n * 8 + 4), np.uint16)
        off = np.arange(n, dtype=np.int64) * 16
        with on_stream(device):
            db, dq = torch.from_numpy(blocks).cuda(), torch.from_numpy(qmat).cuda()
            dd, do = torch.from_numpy(dest.view(np.int16).copy()).cuda(), torch.from_numpy(off).cuda()
            idctdsp.prores_idct_put_batch_device(device, bits, db, n, dq, dd, do, None, dest.strides[0])
            device.sync()
            got = dd.cpu().numpy().view(np.uint16)
        assert np.array_equal(got, cl.orc_prores(bits, blocks, qmat, dest, dest.strides[0])[1]), bits


# ---------------------------------------------------------------------------------------------- H.264 deblocking filters
@isolated
def test_h264_loop_filter(device):
    """H264DSPContext loop filters, 8 bit: the function table on host pointers reproduces the reference's fixture picture; the batched
    device call over 65536 independent edges matches the oracle"""
    import hashlib
    import torch
    from ffmpeg_b200 import pel
    from ffmpeg_b200._lib import H264LoopFilterContext
    g = np.load(os.path.join(G, "h264lf.npz"))
    names = [f[0] for f in H264LoopFilterContext._fields_]
    c420, c422 = pel.ff_h264dsp_loop_filter_init(8, 1), pel.ff_h264dsp_loop_filter_init(8, 2)
    member = {k: (c420, names[k]) for k in range(12)}
    member.update({12: (c422, "h_loop_filter_chroma"), 13: (c422, "h_loop_filter_chroma_mbaff"), 14: (c422, "h_loop_filter_chroma_intra"),
                   15: (c422, "h_loop_filter_chroma_mbaff_intra")})
    pic, kinds, off, alpha, beta, tc0 = cl.h264lf_case(40, 512)
    d = pic.copy()
    for e in range(512):
        c, m = member[int(kinds[e])]
        args = (d.ctypes.data + int(off[e]), d.strides[0], int(alpha[e]), int(beta[e]))
        tcc = tc0[e].copy()                                             # kept alive across the call
        getattr(c, m)(*args, tcc.ctypes.data) if "intra" not in m else getattr(c, m)(*args)
    assert np.array_equal(d[:64], g["head_0"])
    assert hashlib.sha256(d.tobytes()).digest() == g["sha_0"].tobytes()
    for seed in (0, 1, 2):
        n = 512 if seed else 65536
        pic, kinds, off, alpha, beta, tc0 = cl.h264lf_case(40 + seed, n) if seed else cl.h264lf_case(77, n, cols=64)
        with on_stream(device):
            dp = torch.from_numpy(pic).cuda()
            dk, do, da, db, dt = (torch.from_numpy(x).cuda() for x in (kinds, off, alpha, beta, tc0))
            pel.h264_loop_filter_batch_device(device, n, dk, dp, do, pic.strides[0], da, db, dt)
            device.sync()
            got = dp.cpu().numpy()
        if seed:
            assert hashlib.sha256(got.tobytes()).digest() == g[f"sha_{seed}"].tobytes(), seed
        else:
            assert np.array_equal(got, cl.orc_h264lf(pic, kinds, off, alpha, beta, tc0))
    assert pel.ff_h264dsp_loop_filter_init(10, 1).v_loop_filter_luma              # the 16-bit members (test_h264_loop_filter_hbd)


# ---------------------------------------------------------------------------------------------- av_pixelutils_get_sad_fn
@isolated
def test_pixelutils_sad(device):
    """av_pixelutils_get_sad_fn: the functions on host pointers reproduce the reference's sums; the batched device call (two strides,
    100000 block pairs) matches the oracle"""
    import torch
    from ffmpeg_b200 import me_cmp
    g = np.load(os.path.join(G, "pixelutils.npz"))
    for bits in range(1, 6):
        f1, f2, o1, o2 = cl.pixelutils_case(50 + bits, bits, 200)
        fn = me_cmp.av_pixelutils_get_sad_fn(bits, bits)
        got = [fn(f1.ctypes.data + int(a), f1.strides[0], f2.ctypes.data + int(b), f2.strides[0]) for a, b in zip(o1[:40], o2[:40])]
        assert got == list(g[f"sad_{bits}"][:40]), bits
        n = 100000
        f1, f2, o1, o2 = cl.pixelutils_case(250 + bits, bits, n)
        with on_stream(device):
            d1, d2, do1, do2 = (torch.from_numpy(x).cuda() for x in (f1, f2, o1, o2))
            out = torch.full((n,), -1, dtype=torch.int32, device="cuda")
            me_cmp.pixelutils_sad_batch_device(device, bits, d1, f1.strides[0], d2, f2.strides[0], do1, do2, n, out)
            device.sync()
            res = out.cpu().numpy()
        O = cl.oracle()
        O.orc_pixelutils_sad.argtypes = [C_int, C_vp, C_ss, C_vp, C_ss]
        idx = np.random.default_rng(bits).integers(0, n, 3000)
        exp = cl.orc_pixelutils(bits, f1, f2, o1[idx], o2[idx])
        assert np.array_equal(res[idx], exp), bits
    assert me_cmp.av_pixelutils_get_sad_fn(3, 4) is None and me_cmp.av_pixelutils_get_sad_fn(6, 6) is None


# ---------------------------------------------------------------------------------------------- h264qpel, 9 / 10 / 12 / 14 bit samples
def test_h264qpel_hbd(device):
    """ff_h264qpel_init(c, depth) for depth 9 / 10 / 12 / 14: the drop-in table functions (host pointers) against the hashes of the compiled
    reference's outputs, and a macroblock stream through the batched device entry against the oracle"""
    import ctypes as C
    import hashlib
    import torch
    import ffmpeg_b200 as fb
    from ffmpeg_b200 import pel
    from ffmpeg_b200._lib import u8p
    O = cl.oracle()
    O.orc_h264qpel_hbd_batch.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_ssize_t]
    tabs, pics, n = {}, {}, 0
    for k, line in enumerate(open(os.path.join(G, "pel_hbd_hashes.txt"))):
        if k % 3:
            continue
        depth, kind, avg, si, pos, h = line.split()
        depth, kind, avg, si, pos = int(depth), int(kind), int(avg), int(si), int(pos)
        if depth not in tabs:
            tabs[depth] = pel.ff_h264qpel_init(depth)
        if (depth, kind) not in pics:
            pics[(depth, kind)] = cl.hbd_picture(depth, kind)
        img, d0 = pics[(depth, kind)]
        d = d0.copy()
        off = (8 * 64 + 8) * 2
        f = (tabs[depth].avg_h264_qpel_pixels_tab if avg else tabs[depth].put_h264_qpel_pixels_tab)[si][pos]
        f(C.cast(d.ctypes.data + off, u8p), C.cast(img.ctypes.data + off, u8p), 128)
        assert hashlib.sha256(d.tobytes()).hexdigest() == h, line
        n += 1
    assert n == 256
    with pytest.raises(fb.B200Error):
        pel.ff_h264qpel_init(11)
    rng = np.random.default_rng(14)
    W, H = 640, 368
    for depth in (9, 10, 12, 14):
        ref_ = rng.integers(0, 1 << depth, (H, W)).astype(np.uint16)
        dst0 = rng.integers(0, 1 << depth, (H, W)).astype(np.uint16)
        ops, doffs, soffs = [], [], []
        for by in range(1, H // 16 - 1):
            for bx in range(1, W // 16 - 1):
                ops.append(pel.qpel_op(int(rng.integers(0, 2)), int(rng.integers(0, 3)), int(rng.integers(0, 16))))
                dx, dy = (int(v) for v in rng.integers(-10, 11, 2))
                doffs.append((by * 16 * W + bx * 16) * 2); soffs.append(((by * 16 + dy) * W + bx * 16 + dx) * 2)
        cnt = len(ops)
        ops_a, do_a, so_a = np.array(ops, np.uint8), np.array(doffs, np.int64), np.array(soffs, np.int64)
        exp = dst0.copy()
        O.orc_h264qpel_hbd_batch(depth, cnt, ops_a.ctypes.data, exp.ctypes.data, do_a.ctypes.data, ref_.ctypes.data, so_a.ctypes.data, W * 2)
        with on_stream(device):
            d_ops, d_do, d_so = torch.from_numpy(ops_a).cuda(), torch.from_numpy(do_a).cuda(), torch.from_numpy(so_a).cuda()
            d_dst, d_src = torch.from_numpy(dst0.view(np.int16)).cuda(), torch.from_numpy(ref_.view(np.int16)).cuda()
            pel.h264qpel_hbd_batch_device(device, depth, cnt, d_ops, d_dst, d_do, d_src, d_so, W * 2)
            device.sync()
            got = d_dst.cpu().numpy().view(np.uint16)
        assert np.array_equal(got, exp), (depth, int((got != exp).sum()))


# ---------------------------------------------------------------------------------------------- swscale: same-size packed RGB -> packed RGB
def test_sws_same_size_rgb_to_rgb(device):
    """rgbToRgbWrapper / packedCopyWrapper (byte shuffles; the scaler where SWS_BITEXACT removes the 24 -> 32 bit shuffle): sws_scale on host
    buffers against the reference's hashes for every ordered pair of formats, then slices, a batch on the device (vector and byte
    paths) and a 4K frame against the oracle"""
    import torch
    from ffmpeg_b200 import swscale as sw
    from test_oracle import rgb2rgb_rows, run_rgb2rgb_row, sha
    from test_sws_gpu import gpu_sws
    import functools
    rows = rgb2rgb_rows()
    assert len(rows) == 288
    for row in rows:
        assert sha(run_rgb2rgb_row(functools.partial(gpu_sws, device), row)) == row[-1], row[:5]
    rng = np.random.default_rng(8)
    names = list(cl.PACKED_RGB_FORMATS)
    for it in range(12):                                                # band by band (convert_unscaled converts exactly the band it is given)
        sn, dn = names[it % 6], names[(it * 5 + 1) % 6]
        sf, df = cl.PACKED_RGB_FORMATS[sn], cl.PACKED_RGB_FORMATS[dn]
        w, h = 50 + it, 33
        src = cl.rgb_frame(w, h, 2800 + it, cl.fmt_bpp(sf), "random", pad=it % 4)
        exp = cl.orc_sws(w, h, w, h, 4, src, src, src, fmt=df, src_fmt=sf)
        ctx = sw.sws_getContext(device, w, h, sf, w, h, df, 4)
        out = np.zeros_like(exp)
        y = 0
        for bh in (5, 1, 16, 11):
            assert ctx.scale([src[y:]], [src.strides[0]], y, bh, [out], [out.strides[0]]) == bh
            y += bh
        assert y == h and np.array_equal(out, exp), (sn, dn)
        ctx.free()
    for (sn, dn, w, h, n, pad) in (("rgba", "bgra", 640, 360, 3, 0), ("rgb24", "bgr24", 640, 360, 3, 0), ("bgr24", "argb", 322, 75, 2, 2),
                                   ("abgr", "rgb24", 641, 33, 2, 0), ("rgb24", "rgb24", 128, 16, 2, 0), ("rgba", "abgr", 3840, 2160, 1, 0)):
        sf, df = cl.PACKED_RGB_FORMATS[sn], cl.PACKED_RGB_FORMATS[dn]
        sb, db = cl.fmt_bpp(sf), cl.fmt_bpp(df)
        frames = [cl.rgb_frame(w, h, 2900 + k, sb, "random", pad=pad) for k in range(n)]
        ctx = sw.sws_getContext(device, w, h, sf, w, h, df, 4)
        with torch.cuda.stream(torch.cuda.ExternalStream(device.stream)):
            S = torch.from_numpy(np.stack(frames)).cuda()
            D = torch.zeros((n, h, w * db + pad), dtype=torch.uint8, device="cuda")
            ctx.scale_batch_device([S], [w * sb + pad], [(w * sb + pad) * h], D, w * db + pad, (w * db + pad) * h, n)
            device.sync()
            got = D.cpu().numpy()
        for i in range(n):
            exp = cl.orc_sws(w, h, w, h, 4, frames[i], frames[i], frames[i], fmt=df, src_fmt=sf)
            assert np.array_equal(got[i][:, :w * db], exp), (sn, dn, i)
        ctx.free()


# ---------------------------------------------------------------------------------------------- swscale: yuv -> yuv with two matrices
def test_sws_yuv_matrix_cascade(device):
    """sws_setColorspaceDetails with different source and destination matrices on a yuv -> yuv context: two cascaded contexts through a
    bgr24 picture like the reference (utils.c:914-989); host sws_scale and the batched device entry against the oracle; a hash of the
    oracle's outputs ties it to the fixture generated from the compiled reference"""
    import torch
    from ffmpeg_b200 import swscale as sw
    from test_sws_gpu import gpu_sws_planar
    from cases import SWS_CASCADE_CASES
    for i, (w, h, dw, dh, fl, sf, df, ranges, det) in enumerate(SWS_CASCADE_CASES + [(1920, 1080, 1280, 720, 4, 0, 0, (0, 0), (1, 0, 9, 0, 0, 1 << 16, 1 << 16))]):
        y, u, v = cl.yuv_frame(w, h, 5200 + i, "random" if i % 2 else "smooth")
        if sf:
            u = v = cl.nv_interleave(u, v, sf)
        out = gpu_sws_planar(device, w, h, dw, dh, fl, y, u, v, src_fmt=sf, dst_fmt=df, ranges=ranges, details=det, dst_pad=i % 3)
        exp = cl.orc_sws_planar(w, h, dw, dh, fl, y, u, v, src_fmt=sf, dst_fmt=df, ranges=ranges, details=det, dst_pad=i % 3)
        assert all(np.array_equal(p, q) for p, q in zip(out, exp)), (i, w, h, dw, dh, hex(fl))
    w, h, dw, dh, fl, det, n = 320, 180, 480, 270, 4, (1, 0, 5, 0, 0, 1 << 16, 1 << 16), 3
    frames = [cl.yuv_frame(w, h, 5400 + k, "random") for k in range(n)]
    ctx = sw.sws_getContext(device, w, h, sw.AV_PIX_FMT_YUV420P, dw, dh, sw.AV_PIX_FMT_YUV420P, fl)
    assert ctx.setColorspaceDetails(cl.COEFFS[det[0]], det[1], cl.COEFFS[det[2]], det[3], *det[4:]) == 0
    with torch.cuda.stream(torch.cuda.ExternalStream(device.stream)):
        S = [torch.from_numpy(np.stack([f[k] for f in frames])).cuda() for k in range(3)]
        DY = torch.zeros((n, dh, dw), dtype=torch.uint8, device="cuda")
        DU = torch.zeros((n, dh // 2, dw // 2), dtype=torch.uint8, device="cuda")
        DV = torch.zeros((n, dh // 2, dw // 2), dtype=torch.uint8, device="cuda")
        ctx.scale_batch_device_planar(S, [w, w // 2, w // 2], [w * h, w * h // 4, w * h // 4], [DY, DU, DV], [dw, dw // 2, dw // 2],
                                      [dw * dh, dw * dh // 4, dw * dh // 4], n)
        device.sync()
        got = [t.cpu().numpy() for t in (DY, DU, DV)]
    for k in range(n):
        exp = cl.orc_sws_planar(w, h, dw, dh, fl, *frames[k], details=det)
        assert all(np.array_equal(got[j][k], exp[j]) for j in range(3)), k
    ctx.free()


# ---------------------------------------------------------------------------------------------- h264chroma + emulated_edge_mc, 16-bit samples
def test_h264chroma_and_edge_hbd(device):
    """ff_h264chroma_init(c, depth > 8) and ff_videodsp_init(ctx, bpc > 8): drop-in table functions against the hashes of the compiled
    reference's outputs; batched device entries against the oracle"""
    import ctypes as C
    import hashlib
    import torch
    from ffmpeg_b200 import pel
    from ffmpeg_b200._lib import u8p
    from test_oracle_more import hbd_chroma_rows
    O = cl.oracle()
    O.orc_h264chroma_hbd.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_ssize_t, C.c_int, C.c_int, C.c_int]
    O.orc_emulated_edge_mc_hbd.argtypes = [C.c_void_p, C.c_void_p, C.c_ssize_t, C.c_ssize_t] + [C.c_int] * 6
    tabs, pics = {}, {}
    vd = pel.ff_videodsp_init(10)
    for k, row in enumerate(hbd_chroma_rows()):
        if row[0] == "c":
            if k % 3:
                continue
            _, depth, avg, idx, x, y, h, hsh = row
            c = tabs.setdefault(depth, pel.ff_h264chroma_init(depth))
            img, d0 = pics.setdefault(depth, cl.hbd_picture(depth, 0))
            d = d0.copy()
            off = (8 * 64 + 8) * 2
            (c.avg_h264_chroma_pixels_tab if avg else c.put_h264_chroma_pixels_tab)[idx](C.cast(d.ctypes.data + off, u8p), C.cast(img.ctypes.data + off, u8p), 128, h, x, y)
            assert hashlib.sha256(d.tobytes()).hexdigest() == hsh, row[:7]
        else:
            _, bw, bh, sx, sy, hsh = row
            pic, _ = pics.setdefault(10, cl.hbd_picture(10, 0))
            out = np.zeros((bh, bw + 3), np.uint16)
            vd.emulated_edge_mc(C.cast(out.ctypes.data, u8p), C.cast(pic.ctypes.data + sy * pic.strides[0] + sx * 2, u8p), out.strides[0], pic.strides[0], bw, bh, sx, sy, 64, 48)
            assert hashlib.sha256(out.tobytes()).hexdigest() == hsh, row[:5]
    assert not tabs[10].put_h264_chroma_pixels_tab[3]
    rng = np.random.default_rng(23)
    W, H = 640, 368
    ref_ = rng.integers(0, 1 << 10, (H, W)).astype(np.uint16)
    dst0 = rng.integers(0, 1 << 10, (H, W)).astype(np.uint16)
    ops, hs, xys, doffs, soffs = [], [], [], [], []
    for by in range(1, H // 16 - 1):
        for bx in range(1, W // 8 - 1):
            idx = int(rng.integers(0, 3))
            ops.append(pel.chroma_op(int(rng.integers(0, 2)), idx)); hs.append(int(rng.choice([2, 4, 8, 16]))); xys.append(int(rng.integers(0, 64)))
            dx, dy = (int(v) for v in rng.integers(-6, 7, 2))
            doffs.append((by * 16 * W + bx * 8) * 2); soffs.append(((by * 16 + dy) * W + bx * 8 + dx) * 2)
    n = len(ops)
    a = [np.array(v, t) for v, t in ((ops, np.uint8), (hs, np.uint8), (xys, np.uint8), (doffs, np.int64), (soffs, np.int64))]
    exp = dst0.copy()
    for j in range(n):
        O.orc_h264chroma_hbd(ops[j] & 1, ops[j] >> 1, exp.ctypes.data + doffs[j], ref_.ctypes.data + soffs[j], W * 2, hs[j], xys[j] & 7, xys[j] >> 3)
    with on_stream(device):
        d = [torch.from_numpy(v).cuda() for v in a]
        d_dst, d_src = torch.from_numpy(dst0.view(np.int16)).cuda(), torch.from_numpy(ref_.view(np.int16)).cuda()
        pel.h264chroma_hbd_batch_device(device, n, d[0], d[1], d[2], d_dst, d[3], d_src, d[4], W * 2)
        device.sync()
        got = d_dst.cpu().numpy().view(np.uint16)
    assert np.array_equal(got, exp), int((got != exp).sum())
    # edge emulation: windows all around a 64 x 48 picture, one call
    pic, _ = cl.hbd_picture(10, 0)
    geoms = [(int(rng.integers(1, 25)), int(rng.integers(1, 25)), int(rng.integers(-30, 80)), int(rng.integers(-30, 70))) for _ in range(500)]
    BW = 32
    g = np.array(geoms, np.int32); og = np.zeros(500, np.int64); bo = (np.arange(500, dtype=np.int64) * 25 * BW * 2)
    with on_stream(device):
        d_pic = torch.from_numpy(pic.view(np.int16)).cuda()
        d_buf = torch.zeros((500 * 25, BW), dtype=torch.int16, device="cuda")
        d_g, d_og, d_bo = torch.from_numpy(g).cuda(), torch.from_numpy(og).cuda(), torch.from_numpy(bo).cuda()
        pel.emulated_edge_mc_hbd_batch_device(device, 500, d_buf, d_bo, BW * 2, d_pic, d_og, pic.strides[0], d_g, 64, 48)
        device.sync()
        buf = d_buf.cpu().numpy().view(np.uint16)
    for it, (bw, bh, sx, sy) in enumerate(geoms):
        e = np.zeros((bh, bw), np.uint16)
        O.orc_emulated_edge_mc_hbd(e.ctypes.data, pic.ctypes.data + sy * pic.strides[0] + sx * 2, e.strides[0], pic.strides[0], bw, bh, sx, sy, 64, 48)
        assert np.array_equal(buf[it * 25:it * 25 + bh, :bw], e), ("edge", it)


# ---------------------------------------------------------------------------------------------- H.264 weighted prediction, 16-bit samples
def test_h264_weight_hbd(device):
    """ff_h264dsp_init(c, 9 / 10 / 12 / 14) weight / biweight tables: table functions against the hashes of the compiled reference's
    outputs, batched device entry against the oracle"""
    import ctypes as C
    import hashlib
    import torch
    import ffmpeg_b200 as fb
    from ffmpeg_b200 import pel
    from ffmpeg_b200._lib import u8p
    from test_oracle_more import run_weight_hbd_case, weight_hbd_hashes
    O = cl.oracle()
    O.orc_h264_weight_hbd.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_ssize_t] + [C.c_int] * 4
    O.orc_h264_biweight_hbd.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_ssize_t] + [C.c_int] * 5
    hs = weight_hbd_hashes()
    for depth in (9, 10, 12, 14):
        t = pel.ff_h264dsp_weight_init(depth)
        wf = lambda dp, idx, blk, st, h, d, wd, off: t.weight_pixels_tab[idx](C.cast(blk, u8p), st, h, d, wd, off)
        bf = lambda dp, idx, blk, src, st, h, d, wd, ws, off: t.biweight_pixels_tab[idx](C.cast(blk, u8p), C.cast(src, u8p), st, h, d, wd, ws, off)
        for k, case in enumerate(cl.hbd_weight_cases(depth)):
            if k % 2:
                continue
            assert hashlib.sha256(run_weight_hbd_case(wf, bf, depth, case).tobytes()).hexdigest() == hs[(depth, k)], (depth, case)
    with pytest.raises(fb.B200Error):
        pel.ff_h264dsp_weight_init(11)
    rng = np.random.default_rng(29)
    W, H, depth = 640, 368, 10
    ref_ = rng.integers(0, 1 << depth, (H, W)).astype(np.uint16)
    dst0 = rng.integers(0, 1 << depth, (H, W)).astype(np.uint16)
    for bi in (0, 1):
        prm, doffs = [], []
        for by in range(H // 16):
            for bx in range(W // 16):
                idx, h, d = int(rng.integers(0, 4)), int(rng.choice([2, 4, 8, 16])), int(rng.integers(0, 8))
                prm.append([idx | (h << 8) | (d << 16), int(rng.integers(-128, 128)), int(rng.integers(-128, 128)), int(rng.integers(-128, 128))])
                doffs.append((by * 16 * W + bx * 16) * 2)
        prm_a, do_a = np.array(prm, np.int32), np.array(doffs, np.int64)
        exp = dst0.copy()
        for p_, o_ in zip(prm, doffs):
            if bi:
                O.orc_h264_biweight_hbd(depth, p_[0] & 3, exp.ctypes.data + o_, ref_.ctypes.data + o_, W * 2, (p_[0] >> 8) & 255, p_[0] >> 16, p_[1], p_[2], p_[3])
            else:
                O.orc_h264_weight_hbd(depth, p_[0] & 3, exp.ctypes.data + o_, W * 2, (p_[0] >> 8) & 255, p_[0] >> 16, p_[1], p_[3])
        with on_stream(device):
            d_p, d_o = torch.from_numpy(prm_a).cuda(), torch.from_numpy(do_a).cuda()
            d_dst, d_src = torch.from_numpy(dst0.view(np.int16)).cuda(), torch.from_numpy(ref_.view(np.int16)).cuda()
            pel.h264_weight_hbd_batch_device(device, depth, len(prm), d_p, d_dst, d_o, d_src if bi else None, d_o if bi else None, W * 2)
            device.sync()
            got = d_dst.cpu().numpy().view(np.uint16)
        assert np.array_equal(got, exp), (bi, int((got != exp).sum()))


# ---------------------------------------------------------------------------------------------- H.264 residual adds, 16-bit samples
def test_h264_idct_hbd(device):
    """ff_h264dsp_init(c, 9 / 10 / 12 / 14) idct_add / idct8_add / idct_dc_add / idct8_dc_add (int32 coefficients): member functions against
    the hashes of the compiled reference's outputs, batched device entry against the oracle"""
    import ctypes as C
    import torch
    import ffmpeg_b200 as fb
    from ffmpeg_b200 import idctdsp
    from ffmpeg_b200._lib import lib, vp, check, H264IDCTContext
    from test_oracle_more import h264_idct_hbd_hashes, run_h264_idct_hbd_case
    O = cl.oracle()
    O.orc_h264_idct_hbd.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_ssize_t]
    hs = h264_idct_hbd_hashes()
    for depth in (9, 10, 12, 14):
        c = H264IDCTContext()
        check(lib().b200_h264_idct_init(C.byref(c), depth, 1), "h264_idct_init")
        members = [c.idct_add, c.idct8_add, c.idct_dc_add, c.idct8_dc_add]
        fn = lambda dp, kind, d, b, st: members[kind](C.cast(d, C.POINTER(C.c_uint8)), C.cast(b, C.POINTER(C.c_int16)), st)
        for kind in range(4):
            for k, case in enumerate(cl.h264_idct_hbd_cases(depth, kind)):
                if k % 3 == 0:
                    assert run_h264_idct_hbd_case(fn, depth, kind, case) == hs[(depth, kind, k)], (depth, kind, k)
    c = H264IDCTContext()
    assert lib().b200_h264_idct_init(C.byref(c), 11, 1) < 0
    rng = np.random.default_rng(37)
    W, H, depth = 640, 368, 10
    for kind in range(4):
        N, B = (64, 8) if kind & 1 else (16, 4)
        nb = (W // B) * (H // B)
        blocks = rng.integers(-3000, 3000, (nb, N)).astype(np.int32)
        pic = rng.integers(0, 1 << depth, (H, W)).astype(np.uint16)
        boff = np.arange(nb, dtype=np.int64) * N
        doff = np.array([((k // (W // B)) * B * W + (k % (W // B)) * B) * 2 for k in range(nb)], np.int64)
        exp, eb = pic.copy(), blocks.copy()
        for k in range(nb):
            O.orc_h264_idct_hbd(depth, kind, exp.ctypes.data + int(doff[k]), eb.ctypes.data + 4 * int(boff[k]), W * 2)
        with on_stream(device):
            d_b, d_bo, d_do = torch.from_numpy(blocks).cuda(), torch.from_numpy(boff).cuda(), torch.from_numpy(doff).cuda()
            d_p = torch.from_numpy(pic.view(np.int16)).cuda()
            check(lib().b200_h264_idct_hbd_batch_device(device.handle, depth, kind, nb, vp(d_b.data_ptr()), vp(d_bo.data_ptr()), vp(d_p.data_ptr()), vp(d_do.data_ptr()), W * 2), "h264_idct_hbd_batch")
            device.sync()
            got, gb = d_p.cpu().numpy().view(np.uint16), d_b.cpu().numpy()
        assert np.array_equal(got, exp) and np.array_equal(gb, eb), kind


# ---------------------------------------------------------------------------------------------- H.264 deblocking, 16-bit samples
def test_h264_loop_filter_hbd(device):
    """ff_h264dsp_init(c, 9 / 10 / 12 / 14, idc) loop-filter members: the batched device entry against the hashes of the compiled reference's
    pictures (1024 edges of all 16 kinds per depth), the member functions edge by edge against the oracle"""
    import ctypes as C
    import hashlib
    import torch
    from ffmpeg_b200._lib import lib, vp, check, H264LoopFilterContext
    from test_oracle_more import h264lf_hbd_hashes
    hs = h264lf_hbd_hashes()
    names = [f[0] for f in H264LoopFilterContext._fields_]
    for depth in (9, 10, 12, 14):
        pic, kinds, off, alpha, beta, tc0 = cl.h264lf_hbd_case(50 + depth, 1024, depth)
        with on_stream(device):
            d = [torch.from_numpy(v).cuda() for v in (kinds, off, alpha, beta, tc0)]
            dp = torch.from_numpy(pic.view(np.int16)).cuda()
            check(lib().b200_h264_loop_filter_hbd_batch_device(device.handle, depth, 1024, vp(d[0].data_ptr()), vp(dp.data_ptr()), vp(d[1].data_ptr()), pic.strides[0],
                                                               vp(d[2].data_ptr()), vp(d[3].data_ptr()), vp(d[4].data_ptr())), "h264_loop_filter_hbd_batch")
            device.sync()
            got = dp.cpu().numpy().view(np.uint16)
        assert hashlib.sha256(got.tobytes()).hexdigest() == hs[depth], depth
        c = H264LoopFilterContext()
        check(lib().b200_h264_loop_filter_init(C.byref(c), depth, 1), "h264_loop_filter_init")
        pic, kinds, off, alpha, beta, tc0 = cl.h264lf_hbd_case(70 + depth, 48, depth)
        members = [names[i % 12] for i in range(48)]
        kinds = np.array([names.index(m) for m in members], np.uint8)
        dd = pic.copy()
        for i, m in enumerate(members):
            t = tc0[i].copy()
            args = (dd.ctypes.data + int(off[i]), dd.strides[0], int(alpha[i]), int(beta[i]))
            getattr(c, m)(*args, t.ctypes.data) if "intra" not in m else getattr(c, m)(*args)
        assert np.array_equal(dd, cl.orc_h264lf_hbd(depth, pic, kinds, off, alpha, beta, tc0)), depth


# ---------------------------------------------------------------------------------------------- swscale: srcFilter / dstFilter
def test_sws_src_dst_filters(device):
    """sws_getContext with srcFilter / dstFilter vectors (blur / sharpen): whole frames against the oracle (itself equal to the compiled
    reference on these cases), plus a 1080p blur"""
    from ffmpeg_b200 import swscale as sw
    from cases import SWS_FILTER_CASES, _gauss
    from test_oracle import run_filter_case

    def dvec(lens):
        return None if not any(lens) else [[1.0 / n] * n if n else None for n in lens]

    def run_rgb(w, h, dw, dh, fl, y, u, v, filters=None, fmt=cl.PIX_FMT_RGB24):
        ctx = sw.sws_getContext(device, w, h, 0, dw, dh, fmt, fl, src_filter=filters[0], dst_filter=dvec(filters[1]))
        try:
            return ctx.convert(y, u, v)
        finally:
            ctx.free()

    def run_planar(w, h, dw, dh, fl, y, u, v, filters=None):
        ctx = sw.sws_getContext(device, w, h, 0, dw, dh, 0, fl, src_filter=filters[0], dst_filter=dvec(filters[1]))
        try:
            return ctx.convert_planar(y, u, v)
        finally:
            ctx.free()
    cases = SWS_FILTER_CASES + [(1920, 1080, 1280, 720, 4, "rgb24", (_gauss(1.2, 7), _gauss(1.2, 7), None, None), (0, 0, 0, 0))]
    for i, case in enumerate(cases):
        got, exp = run_filter_case(run_rgb, run_planar, i, case), run_filter_case(cl.orc_sws, cl.orc_sws_planar, i, case)
        assert all(np.array_equal(p, q) for p, q in zip(got, exp)), (i, case[:6])


# ---------------------------------------------------------------------------------------------- tx: double precision
def test_tx_double(device):
    """AV_TX_DOUBLE_FFT / AV_TX_DOUBLE_MDCT, power-of-two lengths: av_tx_fn on host buffers and the batched device entry against the hashes of
    the compiled reference's outputs; a larger batch against the checker"""
    import hashlib
    import torch
    import ffmpeg_b200 as fb
    from ffmpeg_b200 import tx
    from test_oracle_more import txd_hashes
    from test_cuda_emu import _orc_txd
    hs = txd_hashes()
    for (typ, n, inv, sc) in cl.txd_cases():
        x = cl.txd_input(typ, n, inv)
        oute = 2 * n if typ == 2 else n
        st = 16 if typ == 2 else 8
        c = tx.av_tx_init(typ, inv, n, scale=sc, device=device)
        out = np.zeros((x.shape[0], oute))
        for r in range(x.shape[0]):
            xr = x[r].copy()
            c.fn(out[r], xr, st)
        assert hashlib.sha256(out.tobytes()).hexdigest() == hs[(typ, n, inv, sc)], ("av_tx_fn", typ, n, inv, sc)
        with on_stream(device):
            di, do = torch.from_numpy(x).cuda(), torch.zeros((x.shape[0], oute), dtype=torch.float64, device="cuda")
            c.batch_device(do, di, st, x.shape[0], do.stride(0) * 8, di.stride(0) * 8)
            device.sync()
            assert hashlib.sha256(do.cpu().numpy().tobytes()).hexdigest() == hs[(typ, n, inv, sc)], ("batch", typ, n, inv, sc)
        c.uninit()
    rng = np.random.default_rng(47)
    for (typ, n, inv, sc) in ((2, 1024, 0, 1.0), (3, 2048, 1, 1.0 / 2048), (3, 512, 0, 1.0), (2, 8192, 1, 1.0)):
        cnt = 500 if n < 8192 else 40
        x = rng.random((cnt, 2 * n if typ == 2 else (n if inv else 2 * n))) * 2 - 1
        oute = 2 * n if typ == 2 else n
        c = tx.av_tx_init(typ, inv, n, scale=sc, device=device)
        with on_stream(device):
            di, do = torch.from_numpy(x).cuda(), torch.zeros((cnt, oute), dtype=torch.float64, device="cuda")
            c.batch_device(do, di, 16 if typ == 2 else 8, cnt, oute * 8, x.shape[1] * 8)
            device.sync()
            got = do.cpu().numpy()
        assert np.array_equal(got.view(np.uint64), _orc_txd(typ, inv, n, sc, x, oute).view(np.uint64)), (typ, n, inv)
        c.uninit()
    with pytest.raises(fb.B200Error):
        tx.av_tx_init(tx.AV_TX_DOUBLE_FFT, 0, 96, device=device)


# ---------------------------------------------------------------------------------------------- me_cmp: transform-domain comparisons
def test_mecmp_dct_families(device):
    """dct_sad / dct_max (both integer DCTs, b200_me_cmp_set_dct_algo) and dct264_sad: the drop-in table entries against the committed
    reference values, the batched entry against the checker"""
    import ctypes as C
    import torch
    from ffmpeg_b200 import me_cmp
    from ffmpeg_b200._lib import u8p
    from test_oracle_more import mecmp_dct_pairs
    pairs = mecmp_dct_pairs()
    c = me_cmp.ff_me_cmp_init()
    tabs = {8: c.dct_sad, 9: c.dct_max, 10: c.dct264_sad}
    O = cl.oracle()
    try:
        for fn, idx, algo, pi, x1, y1, x2, y2, h, v in np.load(os.path.join(G, "mecmp_dct.npz"))["cases"][::2]:
            me_cmp.me_cmp_set_dct_algo(int(algo))
            img1, img2 = pairs[int(pi)]
            got = tabs[int(fn)][int(idx)](None, C.cast(img1.ctypes.data + int(y1) * 64 + int(x1), u8p), C.cast(img2.ctypes.data + int(y2) * 64 + int(x2), u8p), 64, int(h))
            assert got == v, (fn, idx, algo, pi, h)
        rng = np.random.default_rng(8)
        W, H, n = 256, 128, 3001
        f1 = rng.integers(0, 256, (H, W), dtype=np.uint8)
        f2 = (f1.astype(int) + rng.integers(-40, 41, f1.shape)).clip(0, 255).astype(np.uint8)
        off1 = (rng.integers(0, H - 16, n) * W + rng.integers(0, W - 16, n)).astype(np.int64)
        off2 = (rng.integers(0, H - 16, n) * W + rng.integers(0, W - 16, n)).astype(np.int64)
        with on_stream(device):
            d1, d2 = torch.from_numpy(f1).cuda(), torch.from_numpy(f2).cuda()
            o1, o2 = torch.from_numpy(off1).cuda(), torch.from_numpy(off2).cuda()
            out = torch.zeros(n, dtype=torch.int32, device="cuda")
            for algo in (0, 1):
                me_cmp.me_cmp_set_dct_algo(algo)
                O.orc_me_cmp_set_dct_algo(algo)
                for fn in (8, 9, 10):
                    for idx, h in ((0, 16), (0, 8), (1, 8)):
                        me_cmp.me_cmp_batch_device(device, fn, idx, d1, d2, W, h, o1, o2, n, out)
                        device.sync()
                        got = out.cpu().numpy()
                        sel = list(range(250)) + [n - 1]
                        exp = np.array([O.orc_me_cmp(fn, idx, C.cast(f1.ctypes.data + int(off1[i]), cl.u8p), C.cast(f2.ctypes.data + int(off2[i]), cl.u8p), W, h) for i in sel])
                        assert np.array_equal(got[sel], exp), (algo, fn, idx, h)
        with pytest.raises(Exception):
            me_cmp.me_cmp_set_dct_algo(me_cmp.FF_DCT_FAAN)
    finally:
        me_cmp.me_cmp_set_dct_algo(0)
        O.orc_me_cmp_set_dct_algo(0)


# ---------------------------------------------------------------------------------------------- fdctdsp
def test_fdctdsp(device):
    """FDCTDSPContext (fdct / fdct248; islow 8 / 10 bit and ifast): the batched device entry against the hashes of the compiled reference's
    outputs, the drop-in table entries (host pointers) against the checker, FF_DCT_FAAN refused"""
    import hashlib
    import torch
    import ffmpeg_b200 as fb
    from ffmpeg_b200 import fdctdsp
    from ffmpeg_b200._lib import i16p
    from test_oracle_more import fdct_hashes
    from test_cuda_emu import fdct_blocks
    O = cl.oracle()
    for (algo, bits, is248), h in fdct_hashes().items():
        x = fdct_blocks(bits, 200, 7000 + 10 * algo + bits + is248)
        with on_stream(device):
            d = torch.from_numpy(x).cuda()
            fdctdsp.fdct_batch_device(device, d, x.shape[0], algo, bits, is248)
            device.sync()
            assert hashlib.sha256(d.cpu().numpy().tobytes()).hexdigest() == h, (algo, bits, is248)
        c = fdctdsp.ff_fdctdsp_init(algo, bits)
        kind = 2 if bits in (9, 10) else 1 if algo == 1 else 0
        for i in range(6):
            got, exp = x[i].copy(), x[i].copy()
            (c.fdct248 if is248 else c.fdct)(got.ctypes.data_as(i16p))
            O.orc_fdct(kind, is248, cl.ptr(exp, cl.i16p))
            assert np.array_equal(got, exp), (algo, bits, is248, i)
    rng = np.random.default_rng(12)
    big = rng.integers(-255, 256, (100003, 64)).astype(np.int16)       # not a multiple of the 32 blocks of a CTA
    with on_stream(device):
        d = torch.from_numpy(big).cuda()
        fdctdsp.fdct_batch_device(device, d, big.shape[0])
        device.sync()
        got = d.cpu().numpy()
    for i in list(range(64)) + [big.shape[0] - 1]:
        e = big[i].copy()
        O.orc_fdct(0, 0, cl.ptr(e, cl.i16p))
        assert np.array_equal(got[i], e), i
    with pytest.raises(fb.B200Error):
        fdctdsp.ff_fdctdsp_init(fdctdsp.FF_DCT_FAAN, 8)
