"""CPU tier: the device code of the kernels that have not run on a GPU yet, executed on the host by a small CUDA emulation
(tests/cuda_emu/emu.h: one CUDA thread after the other, an OS thread per lane for the warp collective) and compared with the
oracle.  The [device-code ...] blocks are cut out of ffmpeg_b200/csrc/*.cu as they are and compiled with g++; the launch geometry
in tests/cuda_emu/emu_kernels.cpp repeats the library's host code.  This checks arithmetic and indexing of the kernels and the
tables the host set-up feeds them — not memory-space rules, races or speed, which need the hardware."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import cpulibs as cl
from cases import FATE

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.path.join(ROOT, "tests", "cuda_emu")


@pytest.fixture(scope="module")
def emu():
    gen = os.path.join(EMU, "_gen")
    os.makedirs(gen, exist_ok=True)
    found = {}
    src_dir = os.path.join(ROOT, "ffmpeg_b200", "csrc")
    for f in sorted(os.listdir(src_dir)):
        if f.endswith(".cu"):
            txt = open(os.path.join(src_dir, f)).read()
            for m in re.finditer(r"// \[device-code (\w+)\][^\n]*\n(.*?)// \[/device-code \1\]", txt, re.S):
                found[m.group(1)] = m.group(2)
    assert sorted(found) == ["fdsp", "h264lf", "idct_hbd", "pixelutils", "sws_new", "sws_nvout", "tx_dct", "tx_int32", "tx_pfa", "unquant"], sorted(found)
    found["tx_pfa"], n_sh = re.subn(r"extern __shared__ float2 pfa_z\[\];", "float2 *pfa_z = (float2 *)emu_smem;", found["tx_pfa"])
    assert n_sh == 3
    found["tx_int32"], n_sh = re.subn(r"extern __shared__ int2 i32_z\[\];", "int2 *i32_z = (int2 *)emu_smem;", found["tx_int32"])
    assert n_sh == 1
    for k, v in found.items():
        open(os.path.join(gen, k + ".inc"), "w").write(v)
    so = os.path.join(gen, "libemu.so")
    cxx = "/opt/gcc/bin/g++" if os.path.exists("/opt/gcc/bin/g++") else "g++"
    r = subprocess.run([cxx, "-std=c++20", "-O1", "-fPIC", "-shared", "-pthread", "-ffp-contract=off", "-w", "-I" + os.path.join(ROOT, "include"),
                        "-I" + EMU, os.path.join(EMU, "emu_kernels.cpp"), "-o", so], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return C.CDLL(so)


def vp(a):
    return C.c_void_p(a.ctypes.data) if a is not None else None


WARP_KERNELS = {"mpv_unquant_kernel"}                   # kernels that use a warp collective: one OS thread per lane
BLOCK_KERNELS = {"sws_mma_plane_kernel", "sws_mma_rgb_kernel", "tx_fft_kernel", "tx_mdct_inv_kernel", "tx_mdct_fwd_kernel", "tx_rdft_r2c_kernel", "tx_rdft_c2r_kernel",
                 "sws_fused_plane_kernel", "sws_fused_rgb_kernel", "tx_mdct_pfa_inv_kernel", "tx_mdct_pfa_fwd_kernel", "tx_fft_pfa_kernel", "tx_i32_kernel",
                 "tx_dbl_fft_kernel", "tx_dbl_mdct_inv_kernel", "tx_dbl_mdct_fwd_kernel", "me_dct_kernel", "fdct_kernel"}    # __syncthreads + dynamic shared memory


def rewrite_launches(txt):
    """`kernel<<<grid, block, smem, stream>>>(args)` -> a call of emu_cfg_launch() (tests/cuda_emu/fake/cuda_runtime.h)"""
    out, i = [], 0
    pat = re.compile(r"([A-Za-z_]\w*(?:<[^;<>()]*>)?)\s*<<<(.*?)>>>\s*\(")
    while True:
        m = pat.search(txt, i)
        if not m:
            out.append(txt[i:])
            break
        out.append(txt[i:m.start()])
        j, depth = m.end(), 1
        while depth:
            depth += (txt[j] == "(") - (txt[j] == ")")
            j += 1
        kern, cfg, args = m.group(1), m.group(2), txt[m.end():j - 1]
        name = re.match(r"\w+", kern).group(0)
        mode = 1 if name in WARP_KERNELS else 2 if name in BLOCK_KERNELS else 0
        out.append(f"emu_cfg_launch({mode}, [&] {{ {kern}({args}); }}, {cfg})")
        i = j
    return "".join(out)


@pytest.fixture(scope="module")
def emuhost():
    """libemuhost.so: the translation units without inline PTX (fdsp, unquant, idct_hbd, tx_pfa, h264lf, pixelutils), HOST CODE INCLUDED, compiled with
    g++ against a stand-in CUDA runtime (tests/cuda_emu/fake/cuda_runtime.h): the library's own entry points run on the CPU"""
    gen = os.path.join(EMU, "_gen")
    os.makedirs(gen, exist_ok=True)
    cs = os.path.join(ROOT, "ffmpeg_b200", "csrc")
    srcs = []
    for f in ("fdsp.cu", "unquant.cu", "idct_hbd.cu", "tx_pfa.cu", "h264lf.cu", "pixelutils.cu", "pel_hbd.cu", "h264idct_hbd.cu", "h264lf_hbd.cu", "mecmp_dct.cu", "fdctdsp.cu"):
        t = rewrite_launches(open(os.path.join(cs, f)).read())
        t = t.replace("extern __shared__ float2 pfa_z[];", "float2 *pfa_z = (float2 *)emu_smem;")
        assert "<<<" not in t
        p = os.path.join(gen, "host_" + f[:-3] + ".cpp")
        open(p, "w").write(t)
        srcs.append(p)
    so = os.path.join(gen, "libemuhost.so")
    cxx = "/opt/gcc/bin/g++" if os.path.exists("/opt/gcc/bin/g++") else "g++"
    r = subprocess.run([cxx, "-std=c++20", "-O1", "-fPIC", "-shared", "-pthread", "-ffp-contract=off", "-w", "-I" + os.path.join(EMU, "fake"), "-I" + cs,
                        "-I" + os.path.join(ROOT, "include"), "-I" + EMU] + srcs + [os.path.join(EMU, "fake_device.cpp"), os.path.join(EMU, "fake_pel_hbd.cpp"), os.path.join(EMU, "fake_h264idct_hbd.cpp"), os.path.join(EMU, "fake_mecmp_dct.cpp"), "-o", so],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return C.CDLL(so)


def plan(cfg, details=None):
    """(info48, [filter banks (coef int16 [n, size], pos int32 [n])]) from the product's host set-up, no GPU"""
    import ffmpeg_b200 as fb
    L = fb.lib()
    c = np.array(cfg, np.int32)
    info = np.zeros(48, np.int32)
    banks = []
    for which in range(4):
        assert L.b200_sws_plan_probe2(cl.ptr(c, cl.i32p), None, which, None, None, 0, cl.ptr(info, cl.i32p)) >= 0
        size, n = int(info[which]), [cfg[4], int(info[6]), cfg[5], int(info[7])][which]
        f, p = np.zeros(max(n * size, 1), np.int16), np.zeros(max(n, 1), np.int32)
        if size:
            L.b200_sws_plan_probe2(cl.ptr(c, cl.i32p), None, which, cl.ptr(f, cl.i16p), cl.ptr(p, cl.i32p), n, None)
        banks.append((f, p, size))
    return info, banks


RGB_OFFSETS = {"rgb24": (3, 0, 1, 2), "bgr24": (3, 2, 1, 0), "rgba": (4, 0, 1, 2), "bgra": (4, 2, 1, 0), "argb": (4, 1, 2, 3), "abgr": (4, 3, 2, 1)}


def test_emu_alpha_through_the_scaler(emu):
    """sws_rgbin_hscale_a_kernel + sws_vscale_alpha_kernel (alpha of a 32-bit source scaled with the luma filters, both writer families)
    with the product's own filter banks: the oracle's picture with its alpha bytes reset to 255 must get exactly the oracle's alpha back"""
    rng = np.random.default_rng(17)
    names = ["rgba", "bgra", "argb", "abgr"]
    AO = {"rgba": 3, "bgra": 3, "argb": 0, "abgr": 0}
    for it, (w, h, dw, dh, fl) in enumerate([(40, 24, 64, 40, 4), (64, 40, 33, 17, 4), (48, 20, 48, 31, 2), (50, 30, 100, 30, 1), (36, 28, 20, 28, 0x10),
                                             (64, 32, 96, 48, 1 | 0x80000), (33, 21, 50, 40, 0x20), (64, 48, 32, 24, 4 | 0x80000 | 0x40000)]):
        sn, dn = names[it % 4], names[(it * 3 + 1) % 4]
        sf, df = cl.PACKED_RGB_FORMATS[sn], cl.PACKED_RGB_FORMATS[dn]
        src = cl.rgb_frame(w, h, 3100 + it, 4, "random", pad=it % 3)
        if it % 2:
            src[:, AO[sn]:w * 4:4] = rng.integers(0, 2, (h, w)) * 255
        exp = cl.orc_sws(w, h, dw, dh, fl, src, src, src, fmt=df, src_fmt=sf)
        info, banks = plan([w, h, sf, 0, dw, dh, df, 0, fl])
        (hl, hlp, hls), _, (vl, vlp, vls), (vc, vcp, vcs) = banks
        full = 0 if info[11] else 1
        A = np.zeros((h, dw), np.int16)
        emu.emu_sws_rgbin_a(vp(src), src.strides[0], 0, vp(A), dw, 0, vp(hl), vp(hlp), hls, AO[sn], h, 1)
        rm = np.zeros((dh, 4), np.int32)                            # packed_vscale's writer choice per line (vscale.c:144-169)
        for dy in range(dh):
            lf, cf = vl[dy * vls:(dy + 1) * vls].astype(np.uint16).astype(int), vc[dy * vcs:(dy + 1) * vcs].astype(np.uint16).astype(int)
            if vls == 1 and vcs == 1:
                rm[dy] = (1, 0, 0, 0)
            elif vls == 1 and vcs == 2 and cf[0] + cf[1] == 4096 and cf[1] <= 4096:
                rm[dy] = (1, 0, cf[1], 0)
            elif vls == 2 and vcs == 2 and lf[0] + lf[1] == 4096 and lf[1] <= 4096 and cf[0] + cf[1] == 4096 and cf[1] <= 4096:
                rm[dy] = (2, lf[1], cf[1], 0)
        got = exp.copy()
        got[:, AO[dn]::4] = 255
        emu.emu_sws_alpha(vp(A), 0, h, vp(got), got.strides[0], 0, dw, dh, 4, AO[dn], vp(vl), vp(vlp), vls, vp(rm), full, 1)
        assert np.array_equal(got, exp), (it, sn, dn, hex(fl), int((got != exp).sum()))
        assert len(np.unique(exp[:, AO[dn]::4])) > 2                 # the alpha plane is not constant: the check means something


def test_emu_rgb_source_horizontal_pass_and_range(emu):
    """sws_rgbin_hscale_{y,uv}_kernel with the filter banks and the rgb -> yuv table of the product's own host set-up, against the
    oracle's reader + 16-bit horizontal pass; then sws_range_kernel on those lines against the oracle's range conversion"""
    O = cl.oracle()
    O.orc_sws_hlines.argtypes = [C.c_void_p] + [C.c_void_p, C.c_int] * 3 + [C.c_void_p] * 3
    O.orc_sws_range_lines.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]
    n = 0
    for (w, h, dw, dh, fl) in [(64, 48, 100, 70, FATE), (64, 48, 33, 21, cl.SWS_BILINEAR), (63, 47, 63, 47, cl.SWS_BICUBIC), (64, 48, 128, 96, cl.SWS_BICUBIC | 0x4000),
                               (64, 48, 40, 30, 1), (352, 288, 200, 100, FATE), (64, 48, 64, 48, FATE)]:
        for name, sf in cl.PACKED_RGB_FORMATS.items():
            for dr in (0, 1):
                bpp, ro, go, bo = RGB_OFFSETS[name]
                src = cl.rgb_frame(w, h, 3000 + n, bpp, "random", pad=(n % 3) * 3)
                n += 1
                info, banks = plan([w, h, sf, 0, dw, dh, 0, dr, fl])
                assert info[27] == bpp and not info[30] and not info[16]
                cw, csh = int(info[6]), int(info[5])                   # chroma: chrDstW samples per line, chrSrcH lines
                rgbin = np.array([bpp, ro, go, bo, int(info[28])] + [int(x) for x in info[32:41]], np.int32)
                L, CU, CV = np.zeros((h, dw), np.int16), np.zeros((csh, cw), np.int16), np.zeros((csh, cw), np.int16)
                emu.emu_sws_rgbin_y(vp(src), C.c_longlong(src.strides[0]), C.c_longlong(0), vp(L), dw, C.c_longlong(0), vp(banks[0][0]), vp(banks[0][1]),
                                    banks[0][2], vp(rgbin), h, 1)
                emu.emu_sws_rgbin_uv(vp(src), C.c_longlong(src.strides[0]), C.c_longlong(0), vp(CU), vp(CV), cw, C.c_longlong(0), vp(banks[1][0]),
                                     vp(banks[1][1]), banks[1][2], vp(rgbin), csh, 1)
                octx = O.orc_sws_open_range(sf, w, h, 0, 0, dw, dh, dr, fl)
                assert octx
                eL, eU, eV = np.zeros_like(L), np.zeros_like(CU), np.zeros_like(CV)
                assert O.orc_sws_hlines(octx, vp(src), src.strides[0], vp(src), 0, vp(src), 0, vp(eL), vp(eU), vp(eV)) == 0
                assert np.array_equal(L, eL) and np.array_equal(CU, eU) and np.array_equal(CV, eV), (w, h, dw, dh, hex(fl), name)
                if dr:                                                  # limited -> full behind an RGB source
                    assert info[17] == 1
                    emu.emu_sws_range(vp(L), dw, h, 1, C.c_longlong(0), int(info[18]), int(info[19]), 1)
                    emu.emu_sws_range(vp(CU), cw, csh, 1, C.c_longlong(0), int(info[20]), int(info[21]), 1)
                    O.orc_sws_range_lines(octx, vp(eL), dw, h, 0)
                    O.orc_sws_range_lines(octx, vp(eU), cw, csh, 1)
                    assert np.array_equal(L, eL) and np.array_equal(CU, eU), ("range", w, h, dw, dh, name)
                O.orc_sws_close(octx)


def test_emu_range_kernel_both_directions(emu):
    O = cl.oracle()
    O.orc_sws_range_lines.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]
    rng = np.random.default_rng(7)
    for (sr, dr) in ((0, 1), (1, 0)):
        info, _ = plan([64, 48, 0, sr, 100, 70, 0, dr, FATE])
        assert info[17] == (1 if dr else 2)
        octx = O.orc_sws_open_range(0, 64, 48, sr, 0, 100, 70, dr, FATE)
        for chroma in (0, 1):
            frames, rows, w = 3, 5, 301
            a = rng.integers(-2000, 32768, (frames, rows + 2, w)).astype(np.int16)      # frame stride larger than rows * w
            e = a.copy()
            emu.emu_sws_range(vp(a), w, rows, frames, C.c_longlong((rows + 2) * w), int(info[18 + 2 * chroma]), int(info[19 + 2 * chroma]), int(dr))
            for f in range(frames):
                O.orc_sws_range_lines(octx, C.c_void_p(e.ctypes.data + f * (rows + 2) * w * 2), w, rows, chroma)
            assert np.array_equal(a, e), (sr, dr, chroma)
            assert not np.array_equal(a[:, :rows], rng.integers(0, 1, 1))              # (something happened)
        O.orc_sws_close(octx)


def test_emu_bgr24_yv12_and_nv_interleave(emu):
    for (w, h) in ((64, 48), (66, 51), (352, 288)):
        src = cl.rgb_frame(w, h, 3100 + w, 3, "random", pad=5)
        info, _ = plan([w, h, cl.PIX_FMT_BGR24, 0, w, h, 0, 0, cl.SWS_BICUBIC])
        assert info[30] == 1
        rgbin = np.array([3, 2, 1, 0, 0] + [int(x) for x in info[32:41]], np.int32)
        cw, ch = w // 2, (h + 1) // 2
        dy, du, dv = np.zeros((h, w + 3), np.uint8), np.zeros((ch, cw + 1), np.uint8), np.zeros((ch, cw + 2), np.uint8)
        emu.emu_sws_bgr24_yv12(vp(src), C.c_longlong(src.strides[0]), vp(dy), C.c_longlong(dy.strides[0]), vp(du), C.c_longlong(du.strides[0]),
                               vp(dv), C.c_longlong(dv.strides[0]), w, h, vp(rgbin))
        ey, eu, ev = cl.orc_sws_planar(w, h, w, h, cl.SWS_BICUBIC, src, src, src, src_fmt=cl.PIX_FMT_BGR24)
        assert np.array_equal(dy[:, :w], ey) and np.array_equal(du[:, :cw], eu) and np.array_equal(dv[:, :cw], ev), (w, h)
        uv = np.zeros((ch, 2 * cw + 4), np.uint8)
        emu.emu_sws_nv_interleave(vp(eu), vp(ev), C.c_longlong(eu.strides[0]), vp(uv), C.c_longlong(uv.strides[0]), cw, ch)
        assert np.array_equal(uv[:, :2 * cw], cl.nv_interleave(eu, ev, cl.PIX_FMT_NV12)) and not uv[:, 2 * cw:].any()


def test_emu_float_dsp(emu):
    emu.emu_fdsp.argtypes = [C.c_int, C.c_longlong, C.c_int, C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong,
                             C.c_void_p, C.c_longlong, C.c_double]
    for op in range(12):
        for length, nvec in ((1024, 3), (77, 9), (8, 40), (1, 2)):
            dt = np.float64 if op in cl.FDSP_DOUBLE else np.float32
            n2 = 2 * length if op == 5 else length
            cases = [cl.fdsp_case(700 + op * 31 + v, op, length) for v in range(nvec)]
            dst, s0, s1 = (np.stack([c[k] for c in cases]) for k in range(3))
            s2, mul = cases[0][3], cases[0][4]
            dot = op in (9, 11)
            d = np.zeros(nvec, dt) if dot else dst.copy()
            a = s0.copy()
            assert emu.emu_fdsp(op, nvec, length, d.ctypes.data, 1 if dot else n2, a.ctypes.data, length, s1.ctypes.data, length, s2.ctypes.data, 0, mul) == 0
            for v in range(nvec):
                e, e0 = cl.orc_fdsp(op, cases[v][0], cases[v][1], cases[v][2], s2, mul, length)
                assert (d[v:v + 1] if dot else d[v]).tobytes() == e.tobytes() and a[v].tobytes() == e0.tobytes(), (cl.FDSP_OPS[op], length, v)


def test_emu_idct_hbd(emu):
    emu.emu_idct_hbd.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_int]
    for depth in (10, 12):
        for kind in (0, 1, 2):
            n = 300
            blocks = cl.idct_hbd_blocks(600 + depth + kind, depth, n)
            dest = np.random.default_rng(kind).integers(0, 1 << depth, (8, n * 8 + 4), dtype=np.uint16)
            b, d = blocks.copy(), dest.copy()
            off = np.arange(n, dtype=np.int64) * 16
            assert emu.emu_idct_hbd(depth, kind, b.ctypes.data, n, d.ctypes.data, off.ctypes.data, dest.strides[0]) == 0
            eb, ed = cl.orc_idct_hbd(depth, kind, blocks, dest, dest.strides[0])
            assert np.array_equal(d, ed) and np.array_equal(b, eb if kind == 0 else blocks), (depth, kind)


def test_emu_unquant(emu):
    from ffmpeg_b200._lib import MpvUnquant
    emu.emu_unquant.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p]
    for variant in range(7):
        for seed in range(3):
            cfg, blocks, blk_n, q, last = cl.unquant_case(800 + seed * 7 + variant, variant, nblocks=50 + seed)
            p = cl.unquant_params(struct=MpvUnquant, **cfg)
            use_n = blk_n if seed != 1 else None
            b = np.ascontiguousarray(blocks).copy()
            assert emu.emu_unquant(variant, C.byref(p), b.ctypes.data, b.shape[0], use_n.ctypes.data if use_n is not None else None,
                                   q.ctypes.data, last.ctypes.data) == 0
            assert np.array_equal(b, cl.orc_unquant(variant, cfg, blocks, use_n, q, last)), (cl.UNQUANT_VARIANTS[variant], seed)


def test_emu_tx_mdct_pfa15(emu):
    """the compound 15 x M MDCT kernels (Opus CELT sizes) with the tables of the library's own host set-up, against the oracle,
    bit for bit; strided input (inverse) and output (forward), several transforms per launch"""
    import ffmpeg_b200 as fb
    from test_oracle_more import _tx
    L, O = fb.lib(), cl.oracle()
    L.b200_tx_pfa_tables.argtypes = [C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_int, C.c_void_p]
    emu.emu_tx_pfa.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong, C.c_longlong,
                               C.c_longlong, C.c_void_p]
    rng = np.random.default_rng(11)
    assert L.b200_tx_pfa_tables(1, 84, 1.0, None, 0, None) < 0 and L.b200_tx_pfa_tables(1, 1024, 1.0, None, 0, None) < 0      # 7 x 6, power of two
    for n in (120, 240, 480, 960, 1920, 60, 12, 96, 1536, 20, 160, 640, 28, 112, 448, 36, 144, 2304):  # 15 x M; 3 x M and 5 x M; 7 x M and 9 x M
        for inv in (1, 0):
            for sc in (1.0 / n, -1.0, -1.0 / 32768):
                lay = np.zeros(8, np.int32)
                nw = L.b200_tx_pfa_tables(inv, n, sc, None, 0, lay.ctypes.data)
                assert nw > 0
                words = np.zeros(nw, np.int32)
                assert L.b200_tx_pfa_tables(inv, n, sc, words.ctypes.data, nw, lay.ctypes.data) == nw
                cnt = 5
                x = (rng.random((cnt, n if inv else 2 * n), dtype=np.float32) * 2 - 1).astype(np.float32)
                exp = _tx(O, "orc", 1, inv, n, sc, x, n)
                out = np.zeros((cnt, n), np.float32)
                scratch = np.zeros((cnt, n // 2, 2), np.float32)
                assert emu.emu_tx_pfa(inv, n, words.ctypes.data, lay.ctypes.data, out.ctypes.data, x.ctypes.data, 1, out.strides[0], x.strides[0],
                                      cnt, scratch.ctypes.data) == 0
                assert np.array_equal(out.view(np.uint32), exp.view(np.uint32)), (n, inv, sc)
        # stride 2 floats: the inverse reads every other input float, the forward writes every other output float
        lay = np.zeros(8, np.int32)
        nw = L.b200_tx_pfa_tables(1, n, 1.0, None, 0, lay.ctypes.data)
        words = np.zeros(nw, np.int32)
        L.b200_tx_pfa_tables(1, n, 1.0, words.ctypes.data, nw, lay.ctypes.data)
        x = (rng.random((2, n), dtype=np.float32) * 2 - 1).astype(np.float32)
        xs = np.zeros((2, 2 * n), np.float32)
        xs[:, ::2] = x
        out, scratch = np.zeros((2, n), np.float32), np.zeros((2, n // 2, 2), np.float32)
        emu.emu_tx_pfa(1, n, words.ctypes.data, lay.ctypes.data, out.ctypes.data, xs.ctypes.data, 2, out.strides[0], xs.strides[0], 2, scratch.ctypes.data)
        assert np.array_equal(out.view(np.uint32), _tx(O, "orc", 1, 1, n, 1.0, x, n).view(np.uint32)), (n, "strided inverse")


# ------------------------------------------------------------------ all of swscale (sws.cu + sws_plan.cpp) on the stand-in runtime
@pytest.fixture(scope="module")
def emusws():
    """libemusws.so: ffmpeg_b200/csrc/sws.cu — every kernel and all host code — plus sws_plan.cpp on the stand-in runtime.  The only
    edit besides the launch rewrite: the bodies of the two inline-PTX helpers (dp2a.lo / dp2a.hi) are replaced by their definition."""
    gen = os.path.join(EMU, "_gen")
    os.makedirs(gen, exist_ok=True)
    cs = os.path.join(ROOT, "ffmpeg_b200", "csrc")
    t = open(os.path.join(cs, "sws.cu")).read()
    # the tensor-core scaler (sws_mma.cuh) joins the translation unit with its three PTX helpers replaced by their definitions:
    # mma.sync.m16n8k32 by the fragment-layout model of emu.h, the 16-byte cp.async by a copy, its wait by nothing
    m = open(os.path.join(cs, "sws_mma.cuh")).read()
    m, k1 = re.subn(r'\{\s*asm volatile\("mma\.sync\.aligned\.m16n8k32\.row\.col\.s32\.u8\.s8\.s32.*?\n\s*:[^\n]*\n\}', "{ emu_mma_m16n8k32(d, a, b0, b1, true); }", m, flags=re.S)
    m, k2 = re.subn(r'\{\s*asm volatile\("mma\.sync\.aligned\.m16n8k32\.row\.col\.s32\.u8\.u8\.s32.*?\n\s*:[^\n]*\n\}', "{ emu_mma_m16n8k32(d, a, b0, b1, false); }", m, flags=re.S)
    m, k3 = re.subn(r'\{\s*asm volatile\("cp\.async\.cg\.shared\.global[^\n]*\n\}', "{ memcpy(smem_dst, gsrc, 16); }", m)
    m, k4 = re.subn(r'\{ asm volatile\("cp\.async\.wait_all;" ::: "memory"\); \}', "{ }", m)
    m, k5 = re.subn(r"extern __shared__ __align__\(16\) uint8_t mt_smem\[\];", "uint8_t *mt_smem = (uint8_t *)emu_smem;", m)
    assert (k1, k2, k3, k4, k5) == (1, 1, 1, 1, 2), (k1, k2, k3, k4, k5)
    assert t.count('#include "sws_mma.cuh"') == 1
    t = t.replace('#include "sws_mma.cuh"', m)
    t, n1 = re.subn(r'\{ int d; asm\("dp2a\.lo\.s32\.u32[^\n]*\n', "{ return emu_dp2a_su(a, b, c, 0); }\n", t)
    t, n2 = re.subn(r'\{ int d; asm\("dp2a\.hi\.s32\.u32[^\n]*\n', "{ return emu_dp2a_su(a, b, c, 1); }\n", t)
    assert n1 == 1 and n2 == 1 and not re.search(r"\basm\b", t)
    t, n3 = re.subn(r"extern __shared__ __align__\(16\) int16_t fused_lines\[\];", "int16_t *fused_lines = (int16_t *)emu_smem;", t)   # fused scaler tiles
    assert n3 == 2 and "__shared__" not in t
    t = rewrite_launches(t)
    assert "<<<" not in t
    open(os.path.join(gen, "host_sws.cpp"), "w").write(t)
    open(os.path.join(gen, "host_tx_pfa.cpp"), "w").write(rewrite_launches(open(os.path.join(cs, "tx_pfa.cu")).read()).replace("extern __shared__ float2 pfa_z[];", "float2 *pfa_z = (float2 *)emu_smem;"))    # fake_device.cpp refers to it
    so = os.path.join(gen, "libemusws.so")
    cxx = "/opt/gcc/bin/g++" if os.path.exists("/opt/gcc/bin/g++") else "g++"
    r = subprocess.run([cxx, "-std=c++20", "-O1", "-fPIC", "-shared", "-pthread", "-ffp-contract=off", "-w", "-I" + os.path.join(EMU, "fake"), "-I" + cs,
                        "-I" + os.path.join(ROOT, "include"), "-I" + EMU, os.path.join(gen, "host_sws.cpp"), os.path.join(cs, "sws_plan.cpp"),
                        os.path.join(EMU, "fake_device.cpp"), os.path.join(gen, "host_tx_pfa.cpp"), "-o", so], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    L = C.CDLL(so)
    L.b200_sws_getContext_range.restype = C.c_void_p
    L.b200_sws_getContext_range.argtypes = [C.c_void_p] + [C.c_int] * 9
    L.b200_sws_freeContext.argtypes = [C.c_void_p]
    L.b200_sws_setColorspaceDetails.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]
    L.b200_sws_scale.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.b200_sws_scale_batch_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int]
    L.b200_sws_scale_batch_device_planar.argtypes = [C.c_void_p] + [C.c_void_p] * 6 + [C.c_int]
    L.b200_last_error.restype = C.c_char_p
    dev = C.c_void_p()
    assert L.b200_device_open(C.byref(dev), 0, None) == 0
    L.dev = dev
    return L


def _emu_filters(filters, keep):
    """(srcFilter address, dstFilter address) for b200_sws_getContext_filters from (four source vectors, four destination lengths)"""
    from ffmpeg_b200._lib import SwsFilter, SwsVector

    def mk(vs):
        f = SwsFilter()
        for name, v in zip(("lumH", "lumV", "chrH", "chrV"), vs):
            if v:
                arr = (C.c_double * len(v))(*v)
                vec = SwsVector(C.cast(arr, C.POINTER(C.c_double)), len(v))
                keep.extend([arr, vec])
                setattr(f, name, C.pointer(vec))
        keep.append(f)
        return C.addressof(f)
    src, dlen = filters
    return mk(src or [None] * 4), mk([[1.0 / n] * n if n else None for n in (dlen or [0] * 4)])


def _emu_ctx(L, w, h, src_fmt, dw, dh, dst_fmt, fl, ranges=(0, 0), details=None, filters=None):
    if filters is not None:
        keep = []
        L.b200_sws_getContext_filters.restype = C.c_void_p
        L.b200_sws_getContext_filters.argtypes = [C.c_void_p] + [C.c_int] * 9 + [C.c_void_p] * 3
        sfp, dfp = _emu_filters(filters, keep)
        ctx = L.b200_sws_getContext_filters(L.dev, w, h, src_fmt, ranges[0], dw, dh, dst_fmt, ranges[1], fl, sfp, dfp, None)
    else:
        ctx = L.b200_sws_getContext_range(L.dev, w, h, src_fmt, ranges[0], dw, dh, dst_fmt, ranges[1], fl)
    if ctx and details is not None:
        ta, tb = (np.array(cl.COEFFS[k], np.int32) for k in (details[0], details[2]))
        assert L.b200_sws_setColorspaceDetails(ctx, ta.ctypes.data, details[1], tb.ctypes.data, details[3], *details[4:]) == 0
    return ctx


def _emu_scale(L, ctx, planes, h, dst):
    sp = (C.c_void_p * 4)(*[a.ctypes.data for a in planes] + [None] * (4 - len(planes)))
    ss = (C.c_int32 * 4)(*[a.strides[0] for a in planes] + [0] * (4 - len(planes)))
    dp = (C.c_void_p * 4)(*[a.ctypes.data for a in dst] + [None] * (4 - len(dst)))
    ds = (C.c_int32 * 4)(*[a.strides[0] for a in dst] + [0] * (4 - len(dst)))
    return L.b200_sws_scale(ctx, sp, ss, 0, h, dp, ds)


def emu_sws(L, w, h, dw, dh, fl, y, u, v, dst_pad=0, colorspace=None, fmt=cl.PIX_FMT_RGB24, src_fmt=0, filters=None):
    """the library's sws_scale() path for a packed RGB destination, on the emulated device (same signature as cpulibs.orc_sws)"""
    det = None if colorspace is None else (colorspace[0], colorspace[1], colorspace[2], colorspace[3], colorspace[4], colorspace[5], colorspace[6])
    ctx = _emu_ctx(L, w, h, src_fmt, dw, dh, fmt, fl, details=det, filters=filters)
    if not ctx:
        return None
    out = np.full((dh, dw * cl.fmt_bpp(fmt) + dst_pad), 0xA5, np.uint8)
    planes = [y] if src_fmt in cl.PACKED_RGB_FORMATS.values() else [y, u] if src_fmt in (cl.PIX_FMT_NV12, cl.PIX_FMT_NV21) else [y, u, v]
    n = _emu_scale(L, ctx, planes, h, [out])
    L.b200_sws_freeContext(ctx)
    assert n == dh, (n, L.b200_last_error())
    return out


def emu_sws_planar(L, w, h, dw, dh, fl, y, u, v, dst_pad=0, src_fmt=0, ranges=(0, 0), details=None, dst_fmt=0, filters=None):
    ctx = _emu_ctx(L, w, h, src_fmt, dw, dh, dst_fmt, fl, ranges, details, filters)
    if not ctx:
        return None
    cw, ch = (dw + 1) // 2, (dh + 1) // 2
    nvd = dst_fmt in (cl.PIX_FMT_NV12, cl.PIX_FMT_NV21)
    dst = [np.full((dh, dw + dst_pad), 0xA5, np.uint8), np.full((ch, (2 * cw if nvd else cw) + dst_pad), 0xA5, np.uint8)]
    if not nvd:
        dst.append(np.full((ch, cw + dst_pad), 0xA5, np.uint8))
    planes = [y] if src_fmt in cl.PACKED_RGB_FORMATS.values() else [y, u] if src_fmt in (cl.PIX_FMT_NV12, cl.PIX_FMT_NV21) else [y, u, v]
    n = _emu_scale(L, ctx, planes, h, dst)
    L.b200_sws_freeContext(ctx)
    assert n == dh, (n, L.b200_last_error())
    return tuple(dst)


def test_sws_emulation_agrees_with_hardware_verified_paths(emusws):
    """calibration of the emulation itself: paths that already passed on a B200 (vector kernels with dp2a / prmt / vimin, LUT converter,
    scaled path, nv12 source, planar scaling) must give the oracle's bytes here too"""
    import functools
    from cases import SWS_FORMAT_CASES, SWS_PLANAR_CASES, SWS_NV_CASES, SWS_FASTBIL_CASES
    er, ep = functools.partial(emu_sws, emusws), functools.partial(emu_sws_planar, emusws)
    for i, (w, h, dw, dh, fl, kind) in enumerate(SWS_FORMAT_CASES):
        y, u, v = cl.yuv_frame(w, h, 3300 + i, kind)
        for name in ("rgb24", "bgra", "argb"):
            f = cl.PACKED_RGB_FORMATS[name]
            assert np.array_equal(er(w, h, dw, dh, fl, y, u, v, fmt=f, dst_pad=i % 3), cl.orc_sws(w, h, dw, dh, fl, y, u, v, fmt=f, dst_pad=i % 3)), (i, name)
    for i, (w, h, dw, dh, fl, kind) in enumerate(SWS_PLANAR_CASES + SWS_FASTBIL_CASES[:6]):
        y, u, v = cl.yuv_frame(w, h, 3400 + i, kind)
        assert all(np.array_equal(a, b) for a, b in zip(ep(w, h, dw, dh, fl, y, u, v), cl.orc_sws_planar(w, h, dw, dh, fl, y, u, v))), ("planar", i)
    for i, (w, h, dw, dh, fl, kind) in enumerate(SWS_NV_CASES[:6]):
        y, u, v = cl.yuv_frame(w, h, 3500 + i, kind)
        uv = cl.nv_interleave(u, v, cl.PIX_FMT_NV12)
        assert np.array_equal(er(w, h, dw, dh, fl, y, uv, uv, src_fmt=cl.PIX_FMT_NV12), cl.orc_sws(w, h, dw, dh, fl, y, uv, uv, src_fmt=cl.PIX_FMT_NV12)), ("nv12", i)
    # odd widths through the unscaled LUT converter: the reference works on pixel pairs and leaves the last column of the
    # destination alone (yuv2rgb.c:137-236) — the host entry point must not copy that column back either
    for (w, h) in ((7, 6), (17, 10), (33, 6), (1, 2)):
        y, u, v = cl.yuv_frame(w, h, 3700 + w, "random")
        for name in ("rgb24", "bgra"):
            f = cl.PACKED_RGB_FORMATS[name]
            got, exp = er(w, h, w, h, cl.SWS_BICUBIC, y, u, v, fmt=f, dst_pad=2), cl.orc_sws(w, h, w, h, cl.SWS_BICUBIC, y, u, v, fmt=f, dst_pad=2)
            assert np.array_equal(got, exp) and (got[:, (w - 1) * cl.fmt_bpp(f):] == 0xA5).all(), (w, h, name)
    y, u, v = cl.yuv_frame(640, 352, 3600, "random")                     # 16-pixel-group vector kernels, FATE flags and LUT path
    for fl in (FATE, cl.SWS_BICUBIC):
        assert np.array_equal(er(640, 352, 640, 352, fl, y, u, v), cl.orc_sws(640, 352, 640, 352, fl, y, u, v)), hex(fl)


def test_sws_range_conversion_whole_path(emusws):
    """the range-conversion GPU tests of tests/test_sws_gpu.py, through the library's real entry points on the emulated device"""
    import functools
    from cases import SWS_RANGE_CASES
    from test_oracle import fate_sws_yuv_range_crc, FATE_SWS_YUV_RANGE, sha
    ep = functools.partial(emu_sws_planar, emusws)
    lines = open(os.path.join(ROOT, "tests", "golden", "sws_range_hashes.txt")).read().split("\n")[:-1]
    for line, (w, h, dw, dh, fl, kind, ranges, details) in zip(lines, SWS_RANGE_CASES):
        i, hout = int(line.split()[0]), line.split()[-1]
        y, u, v = cl.yuv_frame(w, h, 1200 + i, kind)
        out = ep(w, h, dw, dh, fl, y, u, v, ranges=ranges, details=details)
        assert sha(np.concatenate([p.ravel() for p in out])) == hout, (i, ranges, details)
    assert fate_sws_yuv_range_crc(ep) == FATE_SWS_YUV_RANGE
    y, u, v = cl.yuv_frame(351, 287, 1751, "random", pad=5)
    assert all(np.array_equal(a, b) for a, b in zip(ep(351, 287, 351, 287, cl.SWS_BICUBIC, y, u, v, dst_pad=7, ranges=(1, 0)),
                                                    cl.orc_sws_planar(351, 287, 351, 287, cl.SWS_BICUBIC, y, u, v, dst_pad=7, ranges=(1, 0))))
    # batched device entry point with range conversion (host arrays stand in for device memory), and the refused matrix change
    L = emusws
    w, h, dw, dh, n = 320, 180, 480, 270, 3
    frames = [cl.yuv_frame(w, h, 1600 + k, "random") for k in range(n)]
    Y, U, V = (np.ascontiguousarray(np.stack([f[k] for f in frames])) for k in range(3))
    DY, DU, DV = np.zeros((n, dh, dw), np.uint8), np.zeros((n, dh // 2, dw // 2), np.uint8), np.zeros((n, dh // 2, dw // 2), np.uint8)
    ctx = _emu_ctx(L, w, h, 0, dw, dh, 0, FATE, (1, 0))
    arr = lambda t, vals: (t * 3)(*vals)
    assert L.b200_sws_scale_batch_device_planar(ctx, arr(C.c_void_p, [Y.ctypes.data, U.ctypes.data, V.ctypes.data]), arr(C.c_int32, [w, w // 2, w // 2]),
                                                arr(C.c_int64, [w * h, w * h // 4, w * h // 4]), arr(C.c_void_p, [DY.ctypes.data, DU.ctypes.data, DV.ctypes.data]),
                                                arr(C.c_int32, [dw, dw // 2, dw // 2]), arr(C.c_int64, [dw * dh, dw * dh // 4, dw * dh // 4]), n) == 0
    for i in range(n):
        e = cl.orc_sws_planar(w, h, dw, dh, FATE, *frames[i], ranges=(1, 0))
        assert np.array_equal(DY[i], e[0]) and np.array_equal(DU[i], e[1]) and np.array_equal(DV[i], e[2]), i
    ta, tb = np.array(cl.COEFFS[1], np.int32), np.array(cl.COEFFS[5], np.int32)
    assert L.b200_sws_setColorspaceDetails(ctx, ta.ctypes.data, 0, tb.ctypes.data, 1, 0, 1 << 16, 1 << 16) == 0       # two matrices: cascades (its own test)
    L.b200_sws_freeContext(ctx)


def test_sws_rgb_sources_nv_destinations_and_all_fate_sums(emusws):
    """packed RGB sources, nv12 / nv21 destinations and RGB -> RGB scaling through the library's real entry points, against the
    reference's outputs; then all 59 FATE md5 sums from the emulated device's frames"""
    import functools
    from test_oracle import rgbsrc_rows, run_rgbsrc_row, sha
    from cases import SWS_PLANAR_CASES
    import test_fate_golden as fg
    er, ep = functools.partial(emu_sws, emusws), functools.partial(emu_sws_planar, emusws)
    for row in rgbsrc_rows():
        assert sha(run_rgbsrc_row(er, ep, row)) == row[-1], row[:6]
    for df in (cl.PIX_FMT_NV12, cl.PIX_FMT_NV21):
        for i, (w, h, dw, dh, fl, kind) in enumerate(SWS_PLANAR_CASES):
            y, u, v = cl.yuv_frame(w, h, 2500 + i, kind)
            out, exp = ep(w, h, dw, dh, fl, y, u, v, dst_fmt=df, dst_pad=i % 3), cl.orc_sws_planar(w, h, dw, dh, fl, y, u, v, dst_fmt=df, dst_pad=i % 3)
            assert len(out) == 2 and all(np.array_equal(a, b) for a, b in zip(out, exp)), (i, df)
        src = cl.rgb_frame(64, 48, 2990, 4)
        out, exp = (f(64, 48, 100, 70, FATE, src, src, src, src_fmt=cl.PIX_FMT_BGRA, dst_fmt=df, ranges=(0, 1)) for f in (ep, cl.orc_sws_planar))
        assert all(np.array_equal(a, b) for a, b in zip(out, exp)), ("bgra -> nv, full range", df)
    if cl.have_nut() and os.path.exists(cl.VIDEOGEN):
        fg.check_all(er, ep, rgb_sources=True, nv_dest=True)
    # same-size rgb -> rgb (byte shuffles; the scaler for 24 -> bgra under SWS_BITEXACT) and alpha through the scaler, whole host path
    s3 = cl.rgb_frame(64, 48, 2991, 3)
    for (sf, df, a, fl) in ((cl.PIX_FMT_RGB24, cl.PIX_FMT_BGR24, s3, FATE), (cl.PIX_FMT_RGB24, cl.PIX_FMT_BGRA, s3, FATE), (cl.PIX_FMT_RGB24, cl.PIX_FMT_ARGB, s3, 4),
                            (cl.PIX_FMT_RGBA, cl.PIX_FMT_ABGR, src, 4), (cl.PIX_FMT_BGRA, cl.PIX_FMT_RGB24, src, FATE), (cl.PIX_FMT_ARGB, cl.PIX_FMT_ARGB, src, 4)):
        assert np.array_equal(er(64, 48, 64, 48, fl, a, a, a, fmt=df, src_fmt=sf), cl.orc_sws(64, 48, 64, 48, fl, a, a, a, fmt=df, src_fmt=sf)), ("same size", sf, df)
    for (sf, df, dw2, dh2, fl) in ((cl.PIX_FMT_RGBA, cl.PIX_FMT_BGRA, 32, 24, FATE), (cl.PIX_FMT_ARGB, cl.PIX_FMT_RGBA, 100, 70, 2), (cl.PIX_FMT_BGRA, cl.PIX_FMT_ABGR, 96, 48, 1),
                                   (cl.PIX_FMT_ABGR, cl.PIX_FMT_ARGB, 64, 70, 0x10)):
        assert np.array_equal(er(64, 48, dw2, dh2, fl, src, src, src, fmt=df, src_fmt=sf), cl.orc_sws(64, 48, dw2, dh2, fl, src, src, src, fmt=df, src_fmt=sf)), ("alpha", sf, df)
    # batched device entry points: rgba -> nv12 (two destination planes) and rgb24 -> bgra
    L = emusws
    w, h, dw, dh, n = 64, 48, 100, 70, 2
    frames = [cl.rgb_frame(w, h, 2960 + k, 4) for k in range(n)]
    S = np.ascontiguousarray(np.stack(frames))
    DY, DUV = np.zeros((n, dh, dw), np.uint8), np.zeros((n, dh // 2, dw), np.uint8)
    ctx = _emu_ctx(L, w, h, cl.PIX_FMT_RGBA, dw, dh, cl.PIX_FMT_NV12, FATE)
    arr = lambda t, vals: (t * 3)(*vals)
    assert L.b200_sws_scale_batch_device_planar(ctx, arr(C.c_void_p, [S.ctypes.data, None, None]), arr(C.c_int32, [w * 4, 0, 0]), arr(C.c_int64, [w * 4 * h, 0, 0]),
                                                arr(C.c_void_p, [DY.ctypes.data, DUV.ctypes.data, None]), arr(C.c_int32, [dw, dw, 0]),
                                                arr(C.c_int64, [dw * dh, dw * dh // 2, 0]), n) == 0
    L.b200_sws_freeContext(ctx)
    for i in range(n):
        ey, euv = cl.orc_sws_planar(w, h, dw, dh, FATE, frames[i], frames[i], frames[i], src_fmt=cl.PIX_FMT_RGBA, dst_fmt=cl.PIX_FMT_NV12)
        assert np.array_equal(DY[i], ey) and np.array_equal(DUV[i], euv), i
    frames = [cl.rgb_frame(w, h, 2970 + k, 3) for k in range(n)]
    S = np.ascontiguousarray(np.stack(frames))
    D = np.zeros((n, dh, dw * 4), np.uint8)
    ctx = _emu_ctx(L, w, h, cl.PIX_FMT_RGB24, dw, dh, cl.PIX_FMT_BGRA, FATE)
    assert L.b200_sws_scale_batch_device(ctx, arr(C.c_void_p, [S.ctypes.data, None, None]), arr(C.c_int32, [w * 3, 0, 0]), arr(C.c_int64, [w * 3 * h, 0, 0]),
                                         D.ctypes.data, dw * 4, dw * 4 * dh, n) == 0
    L.b200_sws_freeContext(ctx)
    for i in range(n):
        assert np.array_equal(D[i], cl.orc_sws(w, h, dw, dh, FATE, frames[i], frames[i], frames[i], fmt=cl.PIX_FMT_BGRA, src_fmt=cl.PIX_FMT_RGB24)), i


def test_sws_slice_calls_planar_destination(emusws, refrec):
    """sws_scale() band by band into yuv420p / nv12 on the emulated device: per-call return values and the final planes equal the
    compiled reference's (the luma test of ff_swscale's "enough lines" uses the last line of the chroma pair, swscale.c:419-421)"""
    import random
    L, R = emusws, cl.ref() if cl.have_ref() else None
    if R:
        R.ffref_sws_scale_planar.argtypes = [C.c_void_p] + [C.c_void_p, C.c_int] * 3 + [C.c_int, C.c_int] + [C.c_void_p, C.c_int] * 3
    rnd = random.Random(77)
    for it in range(40):
        w, h = rnd.choice([16, 34, 64, 100]), rnd.choice([8, 16, 34, 48, 66])
        dw, dh = (w, h) if it % 4 == 0 else (rnd.choice([8, 18, 32, 64, 100]), rnd.choice([8, 18, 32, 64, 100]))
        if h > 2 * dh:
            dh = (h // 2 + 2) & ~1                                         # steep vertical reductions trip the reference's own assert (swscale.c:474) when sliced
        fl, df, ranges = rnd.choice([cl.SWS_BICUBIC, cl.SWS_BILINEAR, FATE, 0x10]), rnd.choice([0, cl.PIX_FMT_NV12]), rnd.choice([(0, 0), (0, 1), (1, 0)])
        y, u, v = cl.yuv_frame(w, h, 7700 + it, "random")
        cuts = sorted(set([0, h] + [2 * rnd.randrange(1, h // 2) for _ in range(rnd.randrange(1, 4))]))
        bands = [(a, b - a) for a, b in zip(cuts[:-1], cuts[1:])]
        cw, ch = (dw + 1) // 2, (dh + 1) // 2
        mk = lambda: [np.full((dh, dw), 0xA5, np.uint8), np.full((ch, 2 * cw if df else cw), 0xA5, np.uint8), np.full((ch, cw), 0xA5, np.uint8)]
        rp, gp = mk(), mk()

        def ref_returns():
            rc = R.ffref_sws_open_range(0, w, h, ranges[0], df, dw, dh, ranges[1], fl, 1)
            assert rc
            rr = [R.ffref_sws_scale_planar(rc, y[sy:].ctypes.data, y.strides[0], u[sy // 2:].ctypes.data, u.strides[0], v[sy // 2:].ctypes.data, v.strides[0],
                                           sy, sh, rp[0].ctypes.data, rp[0].strides[0], rp[1].ctypes.data, rp[1].strides[0], rp[2].ctypes.data, rp[2].strides[0])
                  for (sy, sh) in bands]
            R.ffref_sws_close(rc)
            return rr
        ctx = _emu_ctx(L, w, h, 0, dw, dh, df, fl, ranges)
        assert ctx
        for rep in range(2):                                              # the library's context is reusable for the next picture
            gr = [L.b200_sws_scale(ctx, (C.c_void_p * 4)(y[sy:].ctypes.data, u[sy // 2:].ctypes.data, v[sy // 2:].ctypes.data, None),
                                   (C.c_int32 * 4)(y.strides[0], u.strides[0], v.strides[0], 0), sy, sh,
                                   (C.c_void_p * 4)(gp[0].ctypes.data, gp[1].ctypes.data, gp[2].ctypes.data, None),
                                   (C.c_int32 * 4)(gp[0].strides[0], gp[1].strides[0], gp[2].strides[0], 0)) for (sy, sh) in bands]
            assert (refrec.same(gr, ref_returns) if rep == 0 else gr == gr0) and sum(gr) == dh, (it, bands, gr)
            gr0 = gr
        L.b200_sws_freeContext(ctx)
        planes = lambda p: np.concatenate([a.ravel() for a in p[:2 if df else 3]])
        assert refrec.same(planes(gp), lambda: planes(rp)), (it, w, h, dw, dh, hex(fl), df, ranges, bands)


def test_sws_scaler_params(emusws):
    """sws_getContext's `param` (bicubic B / C, Gaussian exponent, Lanczos width, the experimental scaler's power) through
    b200_sws_getContext_params on the emulated device, against the checker and the compiled reference; a Lanczos width whose
    filter would exceed the reference's limit of 50 is refused by all three"""
    from cases import SWS_PARAM_CASES
    L = emusws
    L.b200_sws_getContext_params.restype = C.c_void_p
    L.b200_sws_getContext_params.argtypes = [C.c_void_p] + [C.c_int] * 9 + [C.c_void_p]

    def emu(w, h, dw, dh, fl, y, u, v, prm):
        ctx = L.b200_sws_getContext_params(L.dev, w, h, 0, 0, dw, dh, cl.PIX_FMT_RGB24, 0, fl, (C.c_double * 2)(*prm))
        if not ctx:
            return None
        out = np.full((dh, dw * 3), 0xA5, np.uint8)
        assert _emu_scale(L, ctx, [y, u, v], h, [out]) == dh
        L.b200_sws_freeContext(ctx)
        return out
    for i, (fl, prm) in enumerate(SWS_PARAM_CASES):
        for (w, h, dw, dh, extra) in ((64, 48, 100, 30, 0), (352, 288, 200, 100, 0xc0000), (34, 16, 200, 151, 0x2000)):
            y, u, v = cl.yuv_frame(w, h, 4500 + i, "random")
            exp = cl.orc_sws(w, h, dw, dh, fl | extra, y, u, v, param=prm)
            assert np.array_equal(emu(w, h, dw, dh, fl | extra, y, u, v, prm), exp), (hex(fl), prm, w, h)
            if cl.have_ref():
                assert np.array_equal(cl.ref_sws(w, h, dw, dh, fl | extra, y, u, v, param=prm), exp), ("checker != reference", hex(fl), prm, w, h)
    # the parameters change the picture, and the default marker in both slots is the plain context
    y, u, v = cl.yuv_frame(64, 48, 4600, "random")
    base = cl.orc_sws(64, 48, 100, 30, 4, y, u, v)
    assert np.array_equal(emu(64, 48, 100, 30, 4, y, u, v, (123456.0, 123456.0)), base) and not np.array_equal(emu(64, 48, 100, 30, 4, y, u, v, (1.0, 0.0)), base)
    assert emu(64, 48, 100, 30, 0x200, y, u, v, (26.0, 123456.0)) is None and cl.orc_sws(64, 48, 100, 30, 0x200, y, u, v, param=(26.0, 123456.0)) is None


def test_sws_yuv_matrix_cascade_on_emulated_device(emusws):
    """sws_setColorspaceDetails with two different yuv matrices: b200_sws_scale on host pointers and the batched device entry run the
    two cascaded contexts (yuv -> bgr24 -> yuv) like the reference; against the checker"""
    import functools
    from cases import SWS_CASCADE_CASES
    ep = functools.partial(emu_sws_planar, emusws)
    for i, (w, h, dw, dh, fl, sf, df, ranges, det) in enumerate(SWS_CASCADE_CASES):
        y, u, v = cl.yuv_frame(w, h, 5200 + i, "random" if i % 2 else "smooth")
        if sf:
            u = v = cl.nv_interleave(u, v, sf)
        out = ep(w, h, dw, dh, fl, y, u, v, src_fmt=sf, dst_fmt=df, ranges=ranges, details=det, dst_pad=i % 3)
        exp = cl.orc_sws_planar(w, h, dw, dh, fl, y, u, v, src_fmt=sf, dst_fmt=df, ranges=ranges, details=det, dst_pad=i % 3)
        assert out is not None and all(np.array_equal(p, q) for p, q in zip(out, exp)), (i, w, h, dw, dh, hex(fl))
    # the batched device entry (two frames, yuv420p both sides), and slices are refused
    L = emusws
    w, h, dw, dh, fl, det = 64, 48, 100, 70, FATE, (1, 0, 5, 0, 0, 1 << 16, 1 << 16)
    ctx = _emu_ctx(L, w, h, 0, dw, dh, 0, fl, (0, 0), det)
    assert ctx
    frames = [cl.yuv_frame(w, h, 5300 + k, "random") for k in range(2)]
    Y, U, V = (np.stack([f[k] for f in frames]) for k in range(3))
    DY, DU, DV = np.zeros((2, dh, dw), np.uint8), np.zeros((2, dh // 2, dw // 2), np.uint8), np.zeros((2, dh // 2, dw // 2), np.uint8)
    sp = (C.c_void_p * 3)(Y.ctypes.data, U.ctypes.data, V.ctypes.data)
    ss = (C.c_int * 3)(w, w // 2, w // 2)
    sfs = (C.c_int64 * 3)(w * h, w * h // 4, w * h // 4)
    dp = (C.c_void_p * 3)(DY.ctypes.data, DU.ctypes.data, DV.ctypes.data)
    dss = (C.c_int * 3)(dw, dw // 2, dw // 2)
    dfs = (C.c_int64 * 3)(dw * dh, dw * dh // 4, dw * dh // 4)
    L.b200_sws_scale_batch_device_planar.argtypes = [C.c_void_p] * 7 + [C.c_int]
    assert L.b200_sws_scale_batch_device_planar(ctx, sp, ss, sfs, dp, dss, dfs, 2) == 0
    for k in range(2):
        exp = cl.orc_sws_planar(w, h, dw, dh, fl, *frames[k], details=det)
        assert np.array_equal(DY[k], exp[0]) and np.array_equal(DU[k], exp[1]) and np.array_equal(DV[k], exp[2]), k
    sl = (C.c_void_p * 4)(Y.ctypes.data, U.ctypes.data, V.ctypes.data, None)
    sls = (C.c_int * 4)(w, w // 2, w // 2, 0)
    dl = (C.c_void_p * 4)(DY.ctypes.data, DU.ctypes.data, DV.ctypes.data, None)
    dls = (C.c_int * 4)(dw, dw // 2, dw // 2, 0)
    L.b200_sws_scale.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    assert L.b200_sws_scale(ctx, sl, sls, 0, 16, dl, dls) == -38
    L.b200_sws_freeContext(ctx)


def test_sws_src_dst_filters_on_emulated_device(emusws):
    """b200_sws_getContext_filters: source vectors convolved into the banks by the product's own host set-up, the unscaled converters ruled
    out; whole frames through sws_scale on the emulated device against the checker"""
    from ffmpeg_b200._lib import SwsFilter, SwsVector
    from cases import SWS_FILTER_CASES
    from test_oracle import run_filter_case
    L = emusws
    L.b200_sws_getContext_filters.restype = C.c_void_p
    L.b200_sws_getContext_filters.argtypes = [C.c_void_p] + [C.c_int] * 9 + [C.c_void_p] * 3

    def ctx_of(w, h, sf, dw, dh, df, fl, filters):
        keep = []

        def mk(vs, lens=None):
            f = SwsFilter()
            for k, name in enumerate(("lumH", "lumV", "chrH", "chrV")):
                v = vs[k] if vs is not None else None
                if lens is not None:
                    v = [1.0 / lens[k]] * lens[k] if lens[k] else None
                if v:
                    arr = (C.c_double * len(v))(*v)
                    vec = SwsVector(C.cast(arr, C.POINTER(C.c_double)), len(v))
                    keep.extend([arr, vec])
                    setattr(f, name, C.pointer(vec))
            keep.append(f)
            return C.addressof(f)
        return L.b200_sws_getContext_filters(L.dev, w, h, sf, 0, dw, dh, df, 0, fl, mk(filters[0]), mk(None, filters[1]), None), keep

    def run_rgb(w, h, dw, dh, fl, y, u, v, filters=None, fmt=cl.PIX_FMT_RGB24):
        ctx, keep = ctx_of(w, h, 0, dw, dh, fmt, fl, filters)
        assert ctx
        out = np.full((dh, dw * cl.fmt_bpp(fmt)), 0xA5, np.uint8)
        assert _emu_scale(L, ctx, [y, u, v], h, [out]) == dh
        L.b200_sws_freeContext(ctx)
        return out

    def run_planar(w, h, dw, dh, fl, y, u, v, filters=None):
        ctx, keep = ctx_of(w, h, 0, dw, dh, 0, fl, filters)
        assert ctx
        cw, ch = (dw + 1) // 2, (dh + 1) // 2
        dst = [np.full((dh, dw), 0xA5, np.uint8), np.full((ch, cw), 0xA5, np.uint8), np.full((ch, cw), 0xA5, np.uint8)]
        assert _emu_scale(L, ctx, [y, u, v], h, dst) == dh
        L.b200_sws_freeContext(ctx)
        return tuple(dst)
    for i, case in enumerate(SWS_FILTER_CASES):
        got, exp = run_filter_case(run_rgb, run_planar, i, case), run_filter_case(cl.orc_sws, cl.orc_sws_planar, i, case)
        assert all(np.array_equal(p, q) for p, q in zip(got, exp)), (i, case[:6])


def test_sws_differential_fuzz(emusws):
    """seeded random contexts (sizes incl. odd ones, every source / destination format of the library, scaler flags, ranges,
    sws_setColorspaceDetails with other matrices / brightness / contrast / saturation, padded destinations) through the library's
    real entry points on the emulated device, against the checker and — where it is built — the compiled reference.  This is the
    loop that found the odd-column write-back of the unscaled converter and the nv12 <-> nv21 copy shortcut; what the library
    refuses, the checker must refuse too."""
    import functools
    import random
    er, ep = functools.partial(emu_sws, emusws), functools.partial(emu_sws_planar, emusws)
    NIT, SEED = int(os.environ.get("B200_FUZZ_N", "90")), int(os.environ.get("B200_FUZZ_SEED", "20260923"))      # longer / other runs: set these
    rnd = random.Random(SEED)
    flags = [cl.SWS_BICUBIC, cl.SWS_BILINEAR, FATE, cl.SWS_BICUBIC | 0x40000, cl.SWS_BILINEAR | 0x80000, 1, cl.SWS_BICUBIC | 0x2000, FATE | 0x2000,
             cl.SWS_BICUBIC | 0x4000, 0x10, 0x20, 0x40, 0x8, 0x80, 0x100, 0x200, 0x400, 0x200 | 0xc0000]
    fmts = [0, cl.PIX_FMT_NV12, cl.PIX_FMT_NV21] + list(cl.PACKED_RGB_FORMATS.values())
    ran = refused = 0
    for it in range(NIT):
        w, h = rnd.choice([2, 4, 6, 8, 10, 16, 18, 34, 66, 100, 130]), rnd.choice([2, 4, 6, 8, 10, 16, 18, 34, 50])
        w, h = w + (rnd.random() < 0.3), h + (rnd.random() < 0.3)
        dw, dh = (w, h) if rnd.random() < 0.35 else (rnd.choice([2, 3, 8, 17, 32, 64, 100, 200]), rnd.choice([2, 3, 8, 17, 32, 64, 100]))
        fl, sf, df = rnd.choice(flags), rnd.choice(fmts), rnd.choice(fmts)
        rgbsrc, rgbdst = sf in cl.PACKED_RGB_FORMATS.values(), df in cl.PACKED_RGB_FORMATS.values()
        ranges = (0, 0) if rgbdst else rnd.choice([(0, 0), (0, 0), (0, 1), (1, 0), (1, 1)])
        dpad = rnd.choice([0, 0, 1, 5, 13])
        cs = None
        if rnd.random() < 0.4:
            cs = (rnd.choice([1, 2, 4, 5, 6, 7, 9]), rnd.choice([0, 1]), rnd.choice([1, 5, 6, 7, 9]), rnd.choice([0, 1]), rnd.choice([0, 1 << 12, -(1 << 13)]),
                  rnd.choice([1 << 16, 70000, 50000]), rnd.choice([1 << 16, 80000, 40000]))
        if rgbsrc:
            y = u = v = cl.rgb_frame(w, h, 9000 + it, cl.fmt_bpp(sf))
        else:
            y, u, v = cl.yuv_frame(w, h, 9000 + it, rnd.choice(["random", "limited", "smooth"]))
            if sf:
                u = v = cl.nv_interleave(u, v, sf)
        kw = dict(fmt=df, src_fmt=sf, dst_pad=dpad, colorspace=cs) if rgbdst else dict(src_fmt=sf, dst_fmt=df, ranges=ranges, dst_pad=dpad, details=cs)
        filt = None
        if rnd.random() < 0.2:                                            # srcFilter / dstFilter vectors
            vecs = [None, [1.0], [0.25, 0.5, 0.25], [-0.25, 1.5, -0.25], [0.3, 0.7], [0.05, 0.25, 0.4, 0.25, 0.05]]
            filt = ([rnd.choice(vecs) for _ in range(4)], [rnd.choice([0, 0, 1, 3]) for _ in range(4)])
            kw["filters"] = filt
        orc, ref, emu = (cl.orc_sws, cl.ref_sws, er) if rgbdst else (cl.orc_sws_planar, cl.ref_sws_planar, ep)
        desc = (it, w, h, dw, dh, hex(fl), sf, df, ranges, dpad, cs)
        try:
            exp = orc(w, h, dw, dh, fl, y, u, v, **kw)
        except Exception:
            exp = None                                                    # the checker refuses (e.g. other matrices for yuv -> yuv)
        ctx = _emu_ctx(emusws, w, h, sf, dw, dh, df, fl, ranges, None, filt)
        if ctx and cs is not None:
            ta, tb = (np.array(cl.COEFFS[k], np.int32) for k in (cs[0], cs[2]))
            if emusws.b200_sws_setColorspaceDetails(ctx, ta.ctypes.data, cs[1], tb.ctypes.data, cs[3], *cs[4:]) != 0:
                emusws.b200_sws_freeContext(ctx)
                ctx = None
        if not ctx:
            assert exp is None, ("refused by the library only", desc)
            refused += 1
            continue
        emusws.b200_sws_freeContext(ctx)
        assert exp is not None, ("refused by the checker only", desc)
        got = emu(w, h, dw, dh, fl, y, u, v, **kw)
        same = (lambda a, b: np.array_equal(a, b)) if rgbdst else (lambda a, b: all(np.array_equal(p, q) for p, q in zip(a, b)))
        assert same(got, exp), ("library != checker", desc)
        if cl.have_ref():
            r = ref(w, h, dw, dh, fl, y, u, v, **kw)
            if rgbdst and rgbsrc and (w, h) == (dw, dh) and cl.fmt_bpp(sf) == 3 and df in (cl.PIX_FMT_ARGB, cl.PIX_FMT_ABGR):
                # rgbToRgbWrapper writes the alpha of a "next" pixel one byte past every line (swscale_unscaled.c:2030-2042): picture area only
                r, e2 = r[:, :dw * 4], exp[:, :dw * 4]
            else:
                e2 = exp
            casc = not rgbsrc and not rgbdst and cs is not None and cl.COEFFS[cs[0]] != cl.COEFFS[cs[2]]
            tw = dw if w * h > dw * dh else w
            if casc and (tw & 1):
                # two-matrix cascade through an odd-width bgr24 picture: when its first context is the unscaled LUT converter the last
                # column is never written and the reference reads uninitialised memory there (DESIGN.md) -- nothing to compare with
                ran += 1
                continue
            assert same(r, e2), ("checker != reference", desc)
        ran += 1
    assert ran >= NIT * 8 // 9 and ran + refused == NIT, (ran, refused)          # since same-size RGB -> RGB and alpha went in, only other-matrix yuv -> yuv is refused


# ------------------------------------------------------------------ all of libavutil/tx (tx.cu + tx_pfa.cu) on the stand-in runtime
@pytest.fixture(scope="module")
def emutx():
    """libemutx.so: ffmpeg_b200/csrc/tx.cu (shared-memory kernels: one OS thread per CUDA thread of a block, __syncthreads = barrier) and
    tx_pfa.cu with their host code.  Edits besides the launch rewrite: `extern __shared__ float2 z[]` becomes a pointer to the block's buffer."""
    gen = os.path.join(EMU, "_gen")
    os.makedirs(gen, exist_ok=True)
    cs = os.path.join(ROOT, "ffmpeg_b200", "csrc")
    t = open(os.path.join(cs, "tx.cu")).read()
    t, n = re.subn(r"extern __shared__ float2 z\[\];", "float2 *z = (float2 *)emu_smem;", t)
    assert n == 5 and "__shared__" not in t and not re.search(r"\basm\b", t)
    t = rewrite_launches(t)
    assert "<<<" not in t
    open(os.path.join(gen, "host_tx.cpp"), "w").write(t)
    open(os.path.join(gen, "host_tx_pfa.cpp"), "w").write(rewrite_launches(open(os.path.join(cs, "tx_pfa.cu")).read()).replace("extern __shared__ float2 pfa_z[];", "float2 *pfa_z = (float2 *)emu_smem;"))
    open(os.path.join(gen, "host_tx_dct.cpp"), "w").write(rewrite_launches(open(os.path.join(cs, "tx_dct.cu")).read()))
    open(os.path.join(gen, "host_tx_int32.cpp"), "w").write(rewrite_launches(open(os.path.join(cs, "tx_int32.cu")).read()).replace(
        "extern __shared__ int2 i32_z[];", "int2 *i32_z = (int2 *)emu_smem;"))
    open(os.path.join(gen, "host_tx_double.cpp"), "w").write(rewrite_launches(open(os.path.join(cs, "tx_double.cu")).read()).replace(
        "extern __shared__ double2 dbl_z[];", "double2 *dbl_z = (double2 *)emu_smem;"))
    # tx_r16.cu (bulk async copies + mbarriers in inline PTX) cannot run here: the emulated library keeps tx.cu's level-by-level kernels,
    # which stay the fallback of the product; the register-resident schedule is checked by tests/test_tx_r16_plan.py and on the GPU
    open(os.path.join(gen, "host_tx_r16_stub.cpp"), "w").write(
        '#include "tx_r16.h"\nTxR16 *tx_r16_create(int, int, const int *, const float2 *, int) { return nullptr; }\n'
        'void tx_r16_destroy(TxR16 *) {}\nbool tx_r16_accepts(const TxR16 *, const void *, const void *, long long, long long) { return false; }\n'
        'int tx_r16_launch(TxR16 *, cudaStream_t, void *, const void *, long long, long long, long long) { return -38; }\n')
    so = os.path.join(gen, "libemutx.so")
    cxx = "/opt/gcc/bin/g++" if os.path.exists("/opt/gcc/bin/g++") else "g++"
    r = subprocess.run([cxx, "-std=c++20", "-O1", "-fPIC", "-shared", "-pthread", "-ffp-contract=off", "-w", "-I" + os.path.join(EMU, "fake"), "-I" + cs,
                        "-I" + os.path.join(ROOT, "include"), "-I" + EMU, os.path.join(gen, "host_tx.cpp"), os.path.join(gen, "host_tx_pfa.cpp"),
                        os.path.join(gen, "host_tx_dct.cpp"), os.path.join(gen, "host_tx_int32.cpp"), os.path.join(gen, "host_tx_double.cpp"), os.path.join(gen, "host_tx_r16_stub.cpp"),
                        os.path.join(EMU, "fake_device.cpp"), "-o", so],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    L = C.CDLL(so)
    L.b200_tx_init_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_uint64]
    L.b200_tx_batch_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_ssize_t, C.c_int64, C.c_ssize_t, C.c_ssize_t]
    L.b200_tx_uninit.argtypes = [C.c_void_p]
    dev = C.c_void_p()
    assert L.b200_device_open(C.byref(dev), 0, None) == 0
    L.dev = dev
    return L


def orc_txi(typ, inv, n, scale, x, out_words):
    """the int32 oracle (txi_oracle.c): type 4 FFT / 5 MDCT"""
    O = cl.oracle()
    O.orc_txi_open.restype = C.c_void_p
    O.orc_txi_open.argtypes = [C.c_int, C.c_int, C.c_int, C.c_float, C.c_uint]
    O.orc_txi_run.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_ssize_t, C.c_int, C.c_ssize_t, C.c_ssize_t]
    O.orc_txi_close.argtypes = [C.c_void_p]
    h = O.orc_txi_open(typ, inv, n, scale, 0)
    assert h
    out, xin = np.zeros((x.shape[0], out_words), np.int32), x.copy()
    O.orc_txi_run(h, out.ctypes.data, xin.ctypes.data, 8 if typ == 4 else 4, x.shape[0], out.strides[0], xin.strides[0])
    O.orc_txi_close(h)
    return out


def _emu_tx(L, typ, inv, n, scale, x, out_floats, host_fn=False, flags=0):
    """b200_tx_init_device + b200_tx_batch_device (or the av_tx_fn host entry, one transform at a time) on the emulated device"""
    from ffmpeg_b200._lib import TX_FN
    ctx, fn = C.c_void_p(), TX_FN()
    sc = C.c_float(scale)
    ret = L.b200_tx_init_device(L.dev, C.byref(ctx), C.byref(fn), typ, inv, n, C.byref(sc), flags)
    if ret < 0:
        return ret
    out = np.zeros((x.shape[0], out_floats), x.dtype)
    xin = x.copy()
    st = 8 if typ in (0, 4) else 4
    if host_fn:
        for r in range(x.shape[0]):
            fn(ctx, out[r].ctypes.data, xin[r].ctypes.data, st)
    else:
        assert L.b200_tx_batch_device(ctx, out.ctypes.data, xin.ctypes.data, st, x.shape[0], out.strides[0], xin.strides[0]) == 0
    L.b200_tx_uninit(C.byref(ctx))
    return out


def _orc_txd(typ, inv, n, scale, x, out_doubles):
    O = cl.oracle()
    O.orc_txd_open.restype = C.c_void_p
    O.orc_txd_open.argtypes = [C.c_int, C.c_int, C.c_int, C.c_double, C.c_uint]
    O.orc_txd_run.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_ssize_t, C.c_int, C.c_ssize_t, C.c_ssize_t]
    O.orc_txd_close.argtypes = [C.c_void_p]
    h = O.orc_txd_open(typ, inv, n, scale, 0)
    assert h
    out, xin = np.zeros((x.shape[0], out_doubles), np.float64), x.copy()
    O.orc_txd_run(h, out.ctypes.data, xin.ctypes.data, 16 if typ == 2 else 8, x.shape[0], out.strides[0], xin.strides[0])
    O.orc_txd_close(h)
    return out


def test_tx_double_on_emulated_device(emutx):
    """AV_TX_DOUBLE_FFT / AV_TX_DOUBLE_MDCT (tx_double.cu) through b200_tx_init_device: batch and av_tx_fn entries, strided MDCT samples, against the
    double-precision checker (itself bit-identical to the compiled reference)"""
    from ffmpeg_b200._lib import TX_FN
    L = emutx
    rng = np.random.default_rng(43)
    for typ in (2, 3):
        for n in (2, 4, 8, 16, 64, 256, 1024):
            if typ == 3 and n < 4:
                continue
            for inv in (0, 1):
                for sc in ((1.0,) if typ == 2 else (1.0 / n, -1.0)):
                    ine = 2 * n if typ == 2 else (n if inv else 2 * n)
                    oute = 2 * n if typ == 2 else n
                    x = rng.random((5 if n <= 64 else 2, ine)) * 2 - 1
                    exp = _orc_txd(typ, inv, n, sc, x, oute)
                    ctx, fn = C.c_void_p(), TX_FN()
                    scc = C.c_double(sc)
                    assert L.b200_tx_init_device(L.dev, C.byref(ctx), C.byref(fn), typ, inv, n, C.byref(scc), 0) == 0, (typ, n, inv)
                    out, xin = np.zeros((x.shape[0], oute)), x.copy()
                    st = 16 if typ == 2 else 8
                    assert L.b200_tx_batch_device(ctx, out.ctypes.data, xin.ctypes.data, st, x.shape[0], out.strides[0], xin.strides[0]) == 0
                    assert np.array_equal(out.view(np.uint64), exp.view(np.uint64)), ("double batch", typ, n, inv, sc)
                    o1, x0 = np.zeros(oute), x[0].copy()
                    fn(ctx, o1.ctypes.data, x0.ctypes.data, st)
                    assert np.array_equal(o1.view(np.uint64), exp[0].view(np.uint64)), ("double av_tx_fn", typ, n, inv, sc)
                    if typ == 3 and n == 64:                       # strided samples: input of the inverse, output of the forward transform
                        if inv:
                            xs = np.zeros((x.shape[0], 3 * ine)); xs[:, ::3] = x
                            o2 = np.zeros((x.shape[0], oute))
                            assert L.b200_tx_batch_device(ctx, o2.ctypes.data, xs.ctypes.data, 24, x.shape[0], o2.strides[0], xs.strides[0]) == 0
                            assert np.array_equal(o2.view(np.uint64), exp.view(np.uint64)), "strided in"
                        else:
                            o2 = np.zeros((x.shape[0], 3 * oute))
                            assert L.b200_tx_batch_device(ctx, o2.ctypes.data, xin.ctypes.data, 24, x.shape[0], o2.strides[0], xin.strides[0]) == 0
                            assert np.array_equal(o2[:, ::3].view(np.uint64), exp.view(np.uint64)) and not o2[:, 1::3].any(), "strided out"
                    L.b200_tx_uninit(C.byref(ctx))
    ctx, fn, scc = C.c_void_p(), TX_FN(), C.c_double(1.0)
    assert L.b200_tx_init_device(L.dev, C.byref(ctx), C.byref(fn), 2, 0, 96, C.byref(scc), 0) == -38          # compound double lengths: not built
    assert L.b200_tx_init_device(L.dev, C.byref(ctx), C.byref(fn), 3, 1, 64, C.byref(scc), 4) == -38          # AV_TX_FULL_IMDCT: float only here
    assert L.b200_tx_init_device(L.dev, C.byref(ctx), C.byref(fn), 7, 0, 64, C.byref(scc), 0) == -38          # AV_TX_DOUBLE_RDFT: not built


def test_tx_whole_path_on_emulated_device(emutx):
    """calibration on the hardware-verified transforms (power-of-two FFT / MDCT / RDFT: the emulated shared-memory kernels give the
    oracle's bits), then the compound 15 x M MDCT through b200_tx_init_device — the path tx.cu now dispatches to tx_pfa.cu"""
    from test_oracle_more import _tx
    O = cl.oracle()
    rng = np.random.default_rng(41)
    for n in (16, 64, 256, 1024):
        x = (rng.random((5, 2 * n), dtype=np.float32) * 2 - 1).astype(np.float32)
        for inv in (0, 1):
            assert np.array_equal(_emu_tx(emutx, 0, inv, n, 1.0, x, 2 * n).view(np.uint32), _tx(O, "orc", 0, inv, n, 1.0, x, 2 * n).view(np.uint32)), ("fft", n, inv)
        xi = np.ascontiguousarray(x[:, :n])
        assert np.array_equal(_emu_tx(emutx, 1, 1, n, 1.0 / n, xi, n).view(np.uint32), _tx(O, "orc", 1, 1, n, 1.0 / n, xi, n).view(np.uint32)), ("imdct", n)
        assert np.array_equal(_emu_tx(emutx, 1, 0, n, 1.0, x, n).view(np.uint32), _tx(O, "orc", 1, 0, n, 1.0, x, n).view(np.uint32)), ("mdct", n)
        assert np.array_equal(_emu_tx(emutx, 6, 0, n, 1.0, xi, n + 2).view(np.uint32), _tx(O, "orc", 6, 0, n, 1.0, xi.copy(), n + 2).view(np.uint32)), ("r2c", n)
    for n in (120, 240, 960, 24, 384, 40, 320, 56, 72):
        for inv in (1, 0):
            x = (rng.random((70, n if inv else 2 * n), dtype=np.float32) * 2 - 1).astype(np.float32)
            exp = _tx(O, "orc", 1, inv, n, 1.0 / n, x, n)
            assert np.array_equal(_emu_tx(emutx, 1, inv, n, 1.0 / n, x, n).view(np.uint32), exp.view(np.uint32)), ("pfa batch", n, inv)
            assert np.array_equal(_emu_tx(emutx, 1, inv, n, 1.0 / n, x[:3], n, host_fn=True).view(np.uint32), exp[:3].view(np.uint32)), ("pfa av_tx_fn", n, inv)
    # compound complex FFTs (fft_pfa over fftN_ns x 2^k; checkasm lengths 120 / 960 / 1920): batch, av_tx_fn and in-place entries
    for n in (6, 12, 96, 10, 160, 14, 224, 18, 288, 30, 120, 960, 1920):
        for inv in (0, 1):
            x = (rng.random((70 if n == 120 else 3, 2 * n), dtype=np.float32) * 2 - 1).astype(np.float32)
            exp = _tx(O, "orc", 0, inv, n, 1.0, x, 2 * n)
            assert np.array_equal(_emu_tx(emutx, 0, inv, n, 1.0, x, 2 * n).view(np.uint32), exp.view(np.uint32)), ("fft pfa batch", n, inv)
            assert np.array_equal(_emu_tx(emutx, 0, inv, n, 1.0, x[:2], 2 * n, host_fn=True).view(np.uint32), exp[:2].view(np.uint32)), ("fft pfa av_tx_fn", n, inv)
    assert _emu_tx(emutx, 0, 0, 90, 1.0, x, 180) == -38 and _emu_tx(emutx, 0, 0, 75, 1.0, x, 150) == -38 and _emu_tx(emutx, 0, 0, 15, 1.0, x, 30) == -38
    # AV_TX_FULL_IMDCT around the power-of-two and the compound inverse MDCT: batch and av_tx_fn entries; refused elsewhere
    for n in (4, 64, 1024, 120, 144, 96):
        x = (rng.random((70 if n == 64 else 4, n), dtype=np.float32) * 2 - 1).astype(np.float32)
        exp = _tx(O, "orc", 1, 1, n, 1.0 / n, x, 2 * n, flags=4)
        assert np.array_equal(_emu_tx(emutx, 1, 1, n, 1.0 / n, x, 2 * n, flags=4).view(np.uint32), exp.view(np.uint32)), ("full imdct", n)
        assert np.array_equal(_emu_tx(emutx, 1, 1, n, 1.0 / n, x[:2], 2 * n, host_fn=True, flags=6).view(np.uint32), exp[:2].view(np.uint32)), ("full imdct fn", n)
    assert _emu_tx(emutx, 1, 0, 64, 1.0, x, 64, flags=4) == -38 and _emu_tx(emutx, 0, 1, 64, 1.0, x, 128, flags=4) == -38
    assert _emu_tx(emutx, 5, 1, 64, 1.0, x, 128, flags=4) == -38 and _emu_tx(emutx, 1, 1, 64, 1.0, x, 128, flags=1) == -38
    assert _emu_tx(emutx, 1, 1, 2, 1.0, x, 2) == -38                      # 2-point MDCT: the reference's naive fallback, not built
    # AV_TX_INPLACE: complex FFT only, out == in through the batch entry and through av_tx_fn
    from ffmpeg_b200._lib import TX_FN
    for n in (2, 16, 1024):
        x = (rng.random((6, 2 * n), dtype=np.float32) * 2 - 1).astype(np.float32)
        exp = _tx(O, "orc", 0, 0, n, 1.0, x, 2 * n)
        ctx, fn, sc = C.c_void_p(), TX_FN(), C.c_float(1.0)
        assert emutx.b200_tx_init_device(emutx.dev, C.byref(ctx), C.byref(fn), 0, 0, n, C.byref(sc), 1) == 0
        buf = x.copy()
        assert emutx.b200_tx_batch_device(ctx, buf.ctypes.data, buf.ctypes.data, 8, 6, buf.strides[0], buf.strides[0]) == 0
        assert np.array_equal(buf.view(np.uint32), exp.view(np.uint32)), ("in place", n)
        buf = x[:1].copy()
        fn(ctx, buf.ctypes.data, buf.ctypes.data, 8)
        assert np.array_equal(buf.view(np.uint32), exp[:1].view(np.uint32)), ("in place fn", n)
        emutx.b200_tx_uninit(C.byref(ctx))
    assert _emu_tx(emutx, 1, 1, 64, 1.0, x, 64, flags=1) == -38 and _emu_tx(emutx, 6, 0, 64, 1.0, x, 66, flags=1) == -38
    # AV_TX_FLOAT_DCT: DCT-II forward (len points), DCT-III inverse (asked for len, works on 2 * len), batch and av_tx_fn entries;
    # the input is left alone
    for n in (4, 16, 64, 512):
        for sc in (1.0, 0.5 / n):
            x = (rng.random((70 if n == 64 else 3, n), dtype=np.float32) * 2 - 1).astype(np.float32)
            xp = np.concatenate([x, np.zeros((x.shape[0], 2), np.float32)], axis=1)       # the reference wants two floats of padding
            for inv, asked in ((0, n), (1, n // 2)):
                h = O.orc_tx_open(9, inv, asked, sc, 0)
                e, xin = np.zeros((x.shape[0], n + 2), np.float32), xp.copy()
                O.orc_tx_run(h, e.ctypes.data, xin.ctypes.data, 4, x.shape[0], e.strides[0], xin.strides[0])
                O.orc_tx_close(h)
                got = _emu_tx(emutx, 9, inv, asked, sc, x, n)
                assert np.array_equal(got.view(np.uint32), e[:, :n].view(np.uint32)), ("dct batch", n, inv, sc)
                got = _emu_tx(emutx, 9, inv, asked, sc, x[:2], n, host_fn=True)
                assert np.array_equal(got.view(np.uint32), e[:2, :n].view(np.uint32)), ("dct av_tx_fn", n, inv, sc)
    # AV_TX_INT32_FFT / AV_TX_INT32_MDCT (one thread per transform), batch and av_tx_fn entries, full-range inputs (sums wrap)
    for n in (2, 8, 32, 256, 2048):
        xi32 = rng.integers(-(1 << 31), 1 << 31, (70 if n == 32 else 3, 2 * n)).astype(np.int32)
        for inv in (0, 1):
            e = orc_txi(4, inv, n, 1.0, xi32, 2 * n)
            assert np.array_equal(_emu_tx(emutx, 4, inv, n, 1.0, xi32, 2 * n), e), ("int32 fft", n, inv)
            assert np.array_equal(_emu_tx(emutx, 4, inv, n, 1.0, xi32[:2], 2 * n, host_fn=True), e[:2]), ("int32 fft av_tx_fn", n, inv)
        if n >= 8:
            xs = (xi32 >> 6).astype(np.int32)
            for sc in (1.0, 1.0 / n, -1.0 / 32768):
                e = orc_txi(5, 1, n, sc, np.ascontiguousarray(xs[:, :n]), n)
                assert np.array_equal(_emu_tx(emutx, 5, 1, n, sc, np.ascontiguousarray(xs[:, :n]), n), e), ("int32 imdct", n, sc)
                e = orc_txi(5, 0, n, sc, xs, n)
                assert np.array_equal(_emu_tx(emutx, 5, 0, n, sc, xs, n), e), ("int32 mdct", n, sc)
                assert np.array_equal(_emu_tx(emutx, 5, 0, n, sc, xs[:2], n, host_fn=True), e[:2]), ("int32 mdct av_tx_fn", n, sc)
    x = np.zeros((1, 1920), np.float32)
    assert _emu_tx(emutx, 4, 0, 96, 1.0, x, 192) == -38 and _emu_tx(emutx, 5, 1, 960, 1.0, x, 960) == -38 and _emu_tx(emutx, 1, 1, 84, 1.0, x, 84) == -38 and _emu_tx(emutx, 7, 0, 64, 1.0, x, 128) == -38
    assert _emu_tx(emutx, 9, 0, 96, 1.0, x, 96) == -38 and _emu_tx(emutx, 9, 0, 2, 1.0, x, 2) == -38 and _emu_tx(emutx, 9, 1, 1, 1.0, x, 2) == -38
    assert _emu_tx(emutx, 0, 0, 90, 1.0, x, 180) == -38 and _emu_tx(emutx, 6, 0, 96, 1.0, x, 98) == -38


# ------------------------------------------------------------------ the library's own host code on the stand-in runtime
def test_host_float_dsp_entry_points(emuhost):
    """b200_float_dsp_batch_device (strides, shared operand, more vectors than one grid holds, argument checks) and the
    AVFloatDSPContext function table (host pointers: copy in, launch, copy out), all through the library's real code"""
    from ffmpeg_b200._lib import FloatDSPContext
    L = emuhost
    L.b200_float_dsp_batch_device.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64,
                                              C.c_void_p, C.c_int64, C.c_double]
    for op in range(12):
        for length, nvec in ((64, 5), (9, 3), (4, 66000 if op in (0, 9) else 7)):
            dt = np.float64 if op in cl.FDSP_DOUBLE else np.float32
            n2 = 2 * length if op == 5 else length
            cases = [cl.fdsp_case(900 + op * 17 + v, op, length) for v in range(min(nvec, 6))]
            idx = np.arange(nvec) % len(cases)
            dst, s0, s1 = (np.stack([cases[i][k] for i in idx]) for k in range(3))
            s2, mul = cases[0][3], cases[0][4]
            dot = op in (9, 11)
            d = np.zeros(nvec, dt) if dot else dst.copy()
            a = s0.copy()
            assert L.b200_float_dsp_batch_device(None, op, nvec, length, d.ctypes.data, 1 if dot else n2, a.ctypes.data, length, s1.ctypes.data, length,
                                                 s2.ctypes.data, 0, mul) == 0
            exp = [cl.orc_fdsp(op, c[0], c[1], c[2], s2, mul, length) for c in cases]
            for v in range(nvec):
                e, e0 = exp[idx[v]]
                assert (d[v:v + 1] if dot else d[v]).tobytes() == e.tobytes() and a[v].tobytes() == e0.tobytes(), (cl.FDSP_OPS[op], length, v)
    x = np.zeros(8, np.float32)
    assert L.b200_float_dsp_batch_device(None, 12, 1, 8, x.ctypes.data, 8, x.ctypes.data, 8, x.ctypes.data, 8, None, 0, 0.0) < 0       # unknown op
    assert L.b200_float_dsp_batch_device(None, 6, 1, 8, x.ctypes.data, 8, x.ctypes.data, 8, x.ctypes.data, 8, None, 0, 0.0) < 0        # fmul_add needs src2
    assert L.b200_float_dsp_batch_device(None, 0, 1, 8, x.ctypes.data + 2, 8, x.ctypes.data, 8, x.ctypes.data, 8, None, 0, 0.0) < 0    # misaligned
    assert L.b200_float_dsp_batch_device(None, 0, 0, 8, None, 8, None, 8, None, 8, None, 0, 0.0) == 0                                 # nothing to do
    c = FloatDSPContext()
    assert L.b200_float_dsp_init(C.byref(c)) == 0
    F, D = C.POINTER(C.c_float), C.POINTER(C.c_double)
    for op in range(12):
        P = D if op in cl.FDSP_DOUBLE else F
        for length in (16, 100):
            dst, s0, s1, s2, mul = cl.fdsp_case(40 + op, op, length)
            e, e0 = cl.orc_fdsp(op, dst, s0, s1, s2, mul, length)
            p = lambda z: z.ctypes.data_as(P)
            fn = getattr(c, cl.FDSP_OPS[op])
            if op in (0, 7, 10):
                fn(p(dst), p(s0), p(s1), length)
            elif op in (1, 2, 3, 4):
                fn(p(dst), p(s0), mul, length)
            elif op in (5, 6):
                fn(p(dst), p(s0), p(s1), p(s2), length)
            elif op == 8:
                fn(p(dst), p(s0), length)
            else:
                dst = np.array([fn(p(s0), p(s1), length)], dst.dtype)
            assert (dst[:1] if op in (9, 11) else dst).tobytes() == e.tobytes() and s0.tobytes() == e0.tobytes(), (cl.FDSP_OPS[op], length)


def test_host_unquant_entry_point(emuhost):
    from ffmpeg_b200._lib import MpvUnquant
    L = emuhost
    L.b200_mpv_unquantize_batch_device.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
    for variant in range(7):
        cfg, blocks, blk_n, q, last = cl.unquant_case(1100 + variant, variant, nblocks=37)
        p = cl.unquant_params(struct=MpvUnquant, **cfg)
        for use_n in (blk_n, None):
            b = np.ascontiguousarray(blocks).copy()
            assert L.b200_mpv_unquantize_batch_device(None, variant, C.byref(p), b.ctypes.data, b.shape[0], use_n.ctypes.data if use_n is not None else None,
                                                      q.ctypes.data, last.ctypes.data) == 0
            assert np.array_equal(b, cl.orc_unquant(variant, cfg, blocks, use_n, q, last)), (cl.UNQUANT_VARIANTS[variant], use_n is None)
    b = np.ascontiguousarray(blocks).copy()
    assert L.b200_mpv_unquantize_batch_device(None, 7, C.byref(p), b.ctypes.data, 4, None, q.ctypes.data, last.ctypes.data) < 0
    assert L.b200_mpv_unquantize_batch_device(None, 0, C.byref(p), b.ctypes.data, 0, None, q.ctypes.data, last.ctypes.data) == 0
    p.permutated[5] = p.permutated[6]
    assert L.b200_mpv_unquantize_batch_device(None, 0, C.byref(p), b.ctypes.data, 4, None, q.ctypes.data, last.ctypes.data) < 0
    assert np.array_equal(b, blocks)


def test_host_idct_hbd_entry_points(emuhost):
    from ffmpeg_b200._lib import IDCTDSPContext, u8p, i16p
    L = emuhost
    L.b200_idct_hbd_batch_device.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    for depth_arg, depth in ((9, 10), (10, 10), (12, 12)):
        for kind in (0, 1, 2):
            n = 70
            blocks = cl.idct_hbd_blocks(1200 + depth + kind, depth, n)
            dest = np.random.default_rng(kind).integers(0, 1 << depth, (8, n * 8 + 4), dtype=np.uint16)
            b, d = blocks.copy(), dest.copy()
            off = np.arange(n, dtype=np.int64) * 16
            assert L.b200_idct_hbd_batch_device(None, depth_arg, kind, b.ctypes.data, n, d.ctypes.data, off.ctypes.data, None, dest.strides[0]) == 0
            eb, ed = cl.orc_idct_hbd(depth, kind, blocks, dest, dest.strides[0])
            assert np.array_equal(d, ed) and np.array_equal(b, eb if kind == 0 else blocks), (depth_arg, kind)
        c = IDCTDSPContext()
        assert L.b200_idctdsp_init_hbd(C.byref(c), 2, depth_arg, 0) == 0
        blocks = cl.idct_hbd_blocks(depth_arg, depth, 6)
        dest = np.random.default_rng(depth_arg).integers(0, 1 << depth, (8, 6 * 8 + 3), dtype=np.uint16)
        for kind in (0, 1, 2):
            b, d = blocks.copy(), dest.copy()
            for i in range(6):
                blk = b[i].ctypes.data_as(i16p)
                if kind == 0:
                    c.idct(blk)
                else:
                    (c.idct_put if kind == 1 else c.idct_add)(C.cast(d.ctypes.data + 16 * i, u8p), d.strides[0], blk)
            eb, ed = cl.orc_idct_hbd(depth, kind, blocks, dest, dest.strides[0])
            assert np.array_equal(d, ed) and (kind != 0 or np.array_equal(b, eb)), (depth_arg, kind, "table")
    c = IDCTDSPContext()
    assert L.b200_idctdsp_init_hbd(C.byref(c), 2, 8, 0) < 0 and L.b200_idctdsp_init_hbd(C.byref(c), 2, 10, 1) < 0
    x = np.zeros(64, np.int16)
    assert L.b200_idct_hbd_batch_device(None, 11, 0, x.ctypes.data, 1, None, None, None, 0) < 0


def test_host_prores_entry_points(emuhost):
    """b200_prores_idct_put_batch_device and the ProresDSPContext table (dequantise + transform + bias + clip) against the oracle"""
    from ffmpeg_b200._lib import ProresDSPContext
    L = emuhost
    L.b200_prores_idct_put_batch_device.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    for bits in (10, 12):
        n = 150
        blocks, qmat = cl.prores_case(500 + bits, bits, n)
        dest = np.zeros((8, n * 8 + 5), np.uint16)
        d, b = dest.copy(), blocks.copy()
        off = np.arange(n, dtype=np.int64) * 16
        assert L.b200_prores_idct_put_batch_device(None, bits, b.ctypes.data, n, qmat.ctypes.data, d.ctypes.data, off.ctypes.data, None, dest.strides[0]) == 0
        _, e = cl.orc_prores(bits, blocks, qmat, dest, dest.strides[0])
        assert np.array_equal(d, e) and np.array_equal(b, blocks), bits
        c = ProresDSPContext()
        assert L.b200_proresdsp_init(C.byref(c), bits) == 0 and c.idct_permutation_type == 0 and list(c.idct_permutation) == list(range(64))
        d = dest.copy()
        for i in range(8):
            blk = blocks[i].copy()
            c.idct_put(d.ctypes.data + 16 * i, d.strides[0], blk.ctypes.data, qmat.ctypes.data)
            assert np.array_equal(blk, blocks[i])
        assert np.array_equal(d[:, :64], e[:, :64]), (bits, "table")
    c = ProresDSPContext()
    assert L.b200_proresdsp_init(C.byref(c), 8) < 0
    assert L.b200_prores_idct_put_batch_device(None, 11, blocks.ctypes.data, 1, qmat.ctypes.data, dest.ctypes.data, off.ctypes.data, None, 16) < 0


def test_host_h264_loop_filter_entry_points(emuhost):
    """b200_h264_loop_filter_batch_device over 2048 independent edges of all 16 kinds, and the H264DSPContext loop-filter table edge
    by edge (4:2:0 and 4:2:2 selections), against the oracle"""
    from ffmpeg_b200._lib import H264LoopFilterContext
    L = emuhost
    L.b200_h264_loop_filter_batch_device.argtypes = [C.c_void_p, C.c_int64] + [C.c_void_p] * 3 + [C.c_ssize_t] + [C.c_void_p] * 3
    pic, kinds, off, alpha, beta, tc0 = cl.h264lf_case(21, 2048)
    d = pic.copy()
    assert L.b200_h264_loop_filter_batch_device(None, 2048, kinds.ctypes.data, d.ctypes.data, off.ctypes.data, d.strides[0], alpha.ctypes.data,
                                                beta.ctypes.data, tc0.ctypes.data) == 0
    e = cl.orc_h264lf(pic, kinds, off, alpha, beta, tc0)
    assert np.array_equal(d, e) and not np.array_equal(d, pic)
    names = [f[0] for f in H264LoopFilterContext._fields_]
    for idc in (1, 2):
        c = H264LoopFilterContext()
        assert L.b200_h264_loop_filter_init(C.byref(c), 8, idc) == 0
        # member -> kind, as ff_h264dsp_init selects (h264dsp.c:116-132)
        kind_of = dict(zip(names, range(12)))
        if idc == 2:
            kind_of.update(h_loop_filter_chroma=12, h_loop_filter_chroma_mbaff=13, h_loop_filter_chroma_intra=14, h_loop_filter_chroma_mbaff_intra=15)
        pic, kinds, off, alpha, beta, tc0 = cl.h264lf_case(30 + idc, 192)
        members = [names[i % 12] for i in range(192)]
        kinds = np.array([kind_of[m] for m in members], np.uint8)
        d = pic.copy()
        for i, m in enumerate(members):
            t = tc0[i].copy()
            args = (d.ctypes.data + int(off[i]), d.strides[0], int(alpha[i]), int(beta[i]))
            getattr(c, m)(*args, t.ctypes.data) if "intra" not in m else getattr(c, m)(*args)
            assert np.array_equal(t, tc0[i])
        assert np.array_equal(d, cl.orc_h264lf(pic, kinds, off, alpha, beta, tc0)), idc
    c = H264LoopFilterContext()
    assert L.b200_h264_loop_filter_init(C.byref(c), 11, 1) < 0 and L.b200_h264_loop_filter_init(None, 8, 1) < 0
    assert L.b200_h264_loop_filter_batch_device(None, 0, None, None, None, 0, None, None, None) == 0
    assert L.b200_h264_loop_filter_batch_device(None, 1, None, d.ctypes.data, off.ctypes.data, 16, alpha.ctypes.data, beta.ctypes.data, tc0.ctypes.data) < 0


def test_host_h264_loop_filter_hbd(emuhost):
    """h264lf_hbd.cu (deblocking for 9 / 10 / 12 / 14 bit samples) with its host code on the stand-in runtime: the batched device entry against
    the hashes of the compiled reference's pictures, and the H264DSPContext members edge by edge against the checker"""
    import hashlib
    from ffmpeg_b200._lib import H264LoopFilterContext
    from test_oracle_more import h264lf_hbd_hashes
    L = emuhost
    L.b200_h264_loop_filter_hbd_batch_device.argtypes = [C.c_void_p, C.c_int, C.c_int64] + [C.c_void_p] * 3 + [C.c_ssize_t] + [C.c_void_p] * 3
    hs = h264lf_hbd_hashes()
    names = [f[0] for f in H264LoopFilterContext._fields_]
    for depth in (9, 10, 12, 14):
        pic, kinds, off, alpha, beta, tc0 = cl.h264lf_hbd_case(50 + depth, 1024, depth)
        d = pic.copy()
        assert L.b200_h264_loop_filter_hbd_batch_device(None, depth, 1024, kinds.ctypes.data, d.ctypes.data, off.ctypes.data, d.strides[0], alpha.ctypes.data,
                                                        beta.ctypes.data, tc0.ctypes.data) == 0
        assert hashlib.sha256(d.tobytes()).hexdigest() == hs[depth], depth
        for idc in (1, 2):
            c = H264LoopFilterContext()
            assert L.b200_h264_loop_filter_init(C.byref(c), depth, idc) == 0
            kind_of = dict(zip(names, range(12)))
            if idc == 2:
                kind_of.update(h_loop_filter_chroma=12, h_loop_filter_chroma_mbaff=13, h_loop_filter_chroma_intra=14, h_loop_filter_chroma_mbaff_intra=15)
            pic, kinds, off, alpha, beta, tc0 = cl.h264lf_hbd_case(60 + idc, 96, depth)
            members = [names[i % 12] for i in range(96)]
            kinds = np.array([kind_of[m] for m in members], np.uint8)
            d = pic.copy()
            for i, m in enumerate(members):
                t = tc0[i].copy()
                args = (d.ctypes.data + int(off[i]), d.strides[0], int(alpha[i]), int(beta[i]))
                getattr(c, m)(*args, t.ctypes.data) if "intra" not in m else getattr(c, m)(*args)
            assert np.array_equal(d, cl.orc_h264lf_hbd(depth, pic, kinds, off, alpha, beta, tc0)), (depth, idc)
    assert L.b200_h264_loop_filter_hbd_batch_device(None, 11, 1, kinds.ctypes.data, d.ctypes.data, off.ctypes.data, d.strides[0], alpha.ctypes.data, beta.ctypes.data, tc0.ctypes.data) == -38


def test_host_pixelutils_entry_points(emuhost):
    """b200_pixelutils_sad_batch_device (two strides, 2x2 ... 32x32) and the functions av_pixelutils_get_sad_fn hands out, against the oracle"""
    from ffmpeg_b200.me_cmp import PIXELUTILS_SAD_FN
    L = emuhost
    L.b200_pixelutils_sad_batch_device.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_ssize_t, C.c_void_p, C.c_ssize_t, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    L.b200_pixelutils_get_sad_fn.restype = C.c_void_p
    L.b200_pixelutils_get_sad_fn.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p]
    for bits in range(1, 6):
        f1, f2, o1, o2 = cl.pixelutils_case(70 + bits, bits, 700)
        out = np.full(700, -5, np.int32)
        assert L.b200_pixelutils_sad_batch_device(None, bits, f1.ctypes.data, f1.strides[0], f2.ctypes.data, f2.strides[0], o1.ctypes.data, o2.ctypes.data,
                                                  700, out.ctypes.data) == 0
        exp = cl.orc_pixelutils(bits, f1, f2, o1, o2)
        assert np.array_equal(out, exp), bits
        fn = PIXELUTILS_SAD_FN(L.b200_pixelutils_get_sad_fn(bits, bits, 0, None))
        for i in range(6):
            assert fn(f1.ctypes.data + int(o1[i]), f1.strides[0], f2.ctypes.data + int(o2[i]), f2.strides[0]) == exp[i]
    assert not L.b200_pixelutils_get_sad_fn(0, 0, 0, None) and not L.b200_pixelutils_get_sad_fn(6, 6, 0, None) and not L.b200_pixelutils_get_sad_fn(3, 4, 0, None)
    assert L.b200_pixelutils_sad_batch_device(None, 6, f1.ctypes.data, 160, f2.ctypes.data, 203, o1.ctypes.data, o2.ctypes.data, 1, out.ctypes.data) < 0
    assert L.b200_pixelutils_sad_batch_device(None, 3, None, 160, None, 203, None, None, 0, None) == 0


def test_host_h264qpel_hbd(emuhost):
    """pel_hbd.cu (9 / 10 / 12 / 14 bit h264qpel) with its host code on the stand-in runtime: the batched device entry and the drop-in
    table functions against the checker, every position / size / put+avg, extreme sample patterns included"""
    L, O = emuhost, cl.oracle()
    L.b200_h264qpel_hbd_batch_device.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_ssize_t]
    L.emu_host_qpel_hbd_tab.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_longlong]
    O.orc_h264qpel_hbd_batch.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_ssize_t]
    O.orc_h264qpel_hbd.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_ssize_t]
    dev = C.c_void_p()
    assert L.b200_device_open(C.byref(dev), 0, None) == 0
    rng = np.random.default_rng(9)
    Wd, Hd = 96, 80
    for depth in (9, 10, 12, 14):
        mx = (1 << depth) - 1
        for kind in range(2):
            img = rng.integers(0, mx + 1, (Hd, Wd)).astype(np.uint16) if kind == 0 else (rng.integers(0, 2, (Hd, Wd)) * mx).astype(np.uint16)
            ops, doff, soff = [], [], []
            for avg in (0, 1):
                for si in range(3):
                    for pos in range(16):
                        ops.append(avg | (si << 1) | (pos << 3))
            n = len(ops)
            for k in range(n):                                      # destination blocks on a 16 x 16 grid, sources anywhere inside the padding
                doff.append(((k % 4) * 16 * Wd + (k // 4 % 6) * 16) * 2)
                soff.append((int(rng.integers(3, Hd - 19)) * Wd + int(rng.integers(3, Wd - 19))) * 2)
            # 96 operations need 96 disjoint blocks: 4 rows x 6 columns = 24 per picture -> four destination pictures
            ops_a, doff_a, soff_a = np.array(ops, np.uint8), np.array(doff, np.int64), np.array(soff, np.int64)
            for part in range(4):
                sl = slice(part * 24, part * 24 + 24)
                d0 = rng.integers(0, mx + 1, (Hd, Wd)).astype(np.uint16)
                got, exp = d0.copy(), d0.copy()
                assert L.b200_h264qpel_hbd_batch_device(dev, depth, 24, ops_a[sl].ctypes.data, got.ctypes.data, np.ascontiguousarray(doff_a[sl]).ctypes.data,
                                                        img.ctypes.data, np.ascontiguousarray(soff_a[sl]).ctypes.data, Wd * 2) == 0
                O.orc_h264qpel_hbd_batch(depth, 24, np.ascontiguousarray(ops_a[sl]).ctypes.data, exp.ctypes.data, np.ascontiguousarray(doff_a[sl]).ctypes.data,
                                         img.ctypes.data, np.ascontiguousarray(soff_a[sl]).ctypes.data, Wd * 2)
                assert np.array_equal(got, exp), (depth, kind, part)
            for k in range(0, n, 7):                                # the drop-in table functions (host pointers, one block)
                o = ops[k]
                d0 = rng.integers(0, mx + 1, (Hd, Wd)).astype(np.uint16)
                got, exp = d0.copy(), d0.copy()
                off = (20 * Wd + 24) * 2
                assert L.emu_host_qpel_hbd_tab(depth, o & 1, (o >> 1) & 3, o >> 3, got.ctypes.data + off, img.ctypes.data + off, Wd * 2) == 0
                O.orc_h264qpel_hbd(depth, o & 1, (o >> 1) & 3, o >> 3, exp.ctypes.data + off, img.ctypes.data + off, Wd * 2)
                assert np.array_equal(got, exp), (depth, kind, "tab", o)
    assert L.b200_h264qpel_hbd_batch_device(dev, 11, 1, ops_a.ctypes.data, got.ctypes.data, doff_a.ctypes.data, img.ctypes.data, soff_a.ctypes.data, Wd * 2) == -38
    assert L.emu_host_qpel_hbd_tab(8, 0, 0, 0, got.ctypes.data, img.ctypes.data, Wd * 2) == -38


def test_host_chroma_and_edge_hbd(emuhost):
    """pel_hbd.cu: h264chroma and emulated_edge_mc for 16-bit samples, batched device entries and drop-in table functions on the stand-in
    runtime against the checker (every eighth-pel phase, put / avg, widths 8 / 4 / 2; windows on and beyond every picture border)"""
    L, O = emuhost, cl.oracle()
    L.b200_h264chroma_hbd_batch_device.argtypes = [C.c_void_p, C.c_int64] + [C.c_void_p] * 7 + [C.c_ssize_t]
    L.b200_emulated_edge_mc_hbd_batch_device.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_ssize_t, C.c_void_p, C.c_void_p, C.c_ssize_t, C.c_void_p, C.c_int, C.c_int]
    L.emu_host_chroma_hbd_tab.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_int]
    L.emu_host_edge_hbd_tab.argtypes = [C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong] + [C.c_int] * 6
    O.orc_h264chroma_hbd.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_ssize_t, C.c_int, C.c_int, C.c_int]
    O.orc_emulated_edge_mc_hbd.argtypes = [C.c_void_p, C.c_void_p, C.c_ssize_t, C.c_ssize_t] + [C.c_int] * 6
    dev = C.c_void_p()
    assert L.b200_device_open(C.byref(dev), 0, None) == 0
    rng = np.random.default_rng(19)
    Wd, Hd = 96, 80
    for depth in (10, 16):
        img = rng.integers(0, 1 << depth, (Hd, Wd)).astype(np.uint16)
        ops, hs, xys, doff, soff = [], [], [], [], []
        k = 0
        for avg in (0, 1):
            for idx in range(3):
                for x in range(8):
                    for y in range(8):
                        ops.append(avg | (idx << 1)); hs.append([4, 8, 16, 2][(x + y + idx) % 4]); xys.append(x | (y << 3))
                        doff.append(((k % 4) * 16 * Wd + (k // 4 % 10) * 8) * 2); soff.append((int(rng.integers(0, Hd - 18)) * Wd + int(rng.integers(0, Wd - 10))) * 2)
                        k += 1
        n = len(ops)
        ops_a, hs_a, xy_a, do_a, so_a = np.array(ops, np.uint8), np.array(hs, np.uint8), np.array(xys, np.uint8), np.array(doff, np.int64), np.array(soff, np.int64)
        for part in range(0, n, 40):                                # 40 disjoint destination blocks per picture
            sl = slice(part, min(part + 40, n))
            cnt = sl.stop - sl.start
            d0 = rng.integers(0, 1 << depth, (Hd, Wd)).astype(np.uint16)
            got, exp = d0.copy(), d0.copy()
            a = [np.ascontiguousarray(v[sl]) for v in (ops_a, hs_a, xy_a, do_a, so_a)]
            assert L.b200_h264chroma_hbd_batch_device(dev, cnt, a[0].ctypes.data, a[1].ctypes.data, a[2].ctypes.data, got.ctypes.data, a[3].ctypes.data,
                                                      img.ctypes.data, a[4].ctypes.data, Wd * 2) == 0
            for j in range(cnt):
                O.orc_h264chroma_hbd(int(a[0][j]) & 1, int(a[0][j]) >> 1, exp.ctypes.data + int(a[3][j]), img.ctypes.data + int(a[4][j]), Wd * 2, int(a[1][j]), int(a[2][j]) & 7, int(a[2][j]) >> 3)
            assert np.array_equal(got, exp), (depth, part)
        for j in range(0, n, 11):                                   # drop-in table functions
            d0 = rng.integers(0, 1 << depth, (Hd, Wd)).astype(np.uint16)
            got, exp = d0.copy(), d0.copy()
            off = (20 * Wd + 24) * 2
            args = (ops[j] & 1, ops[j] >> 1)
            assert L.emu_host_chroma_hbd_tab(*args, got.ctypes.data + off, img.ctypes.data + off, Wd * 2, hs[j], xys[j] & 7, xys[j] >> 3) == 0
            O.orc_h264chroma_hbd(*args, exp.ctypes.data + off, img.ctypes.data + off, Wd * 2, hs[j], xys[j] & 7, xys[j] >> 3)
            assert np.array_equal(got, exp), (depth, "tab", j)
    pic = rng.integers(0, 1024, (30, 41)).astype(np.uint16)
    geoms, origins, boffs = [], [], []
    BW = 32
    for it in range(60):
        bw, bh = int(rng.integers(1, 25)), int(rng.integers(1, 25))
        sx, sy = int(rng.integers(-30, 60)), int(rng.integers(-30, 50))
        geoms.append((bw, bh, sx, sy)); origins.append(0); boffs.append(it * 25 * BW * 2)
        got, exp = np.zeros((bh, bw + 3), np.uint16), np.zeros((bh, bw + 3), np.uint16)
        src = pic.ctypes.data + sy * pic.strides[0] + sx * 2
        L.emu_host_edge_hbd_tab(got.ctypes.data, src, got.strides[0], pic.strides[0], bw, bh, sx, sy, 41, 30)
        O.orc_emulated_edge_mc_hbd(exp.ctypes.data, src, exp.strides[0], pic.strides[0], bw, bh, sx, sy, 41, 30)
        assert np.array_equal(got, exp), ("edge tab", bw, bh, sx, sy)
    g = np.array(geoms, np.int32); og = np.array(origins, np.int64); bo = np.array(boffs, np.int64)
    buf = np.zeros((60 * 25, BW), np.uint16)
    assert L.b200_emulated_edge_mc_hbd_batch_device(dev, 60, buf.ctypes.data, bo.ctypes.data, BW * 2, pic.ctypes.data, og.ctypes.data, pic.strides[0], g.ctypes.data, 41, 30) == 0
    for it, (bw, bh, sx, sy) in enumerate(geoms):
        exp = np.zeros((bh, bw), np.uint16)
        O.orc_emulated_edge_mc_hbd(exp.ctypes.data, pic.ctypes.data + sy * pic.strides[0] + sx * 2, exp.strides[0], pic.strides[0], bw, bh, sx, sy, 41, 30)
        assert np.array_equal(buf[it * 25:it * 25 + bh, :bw], exp), ("edge batch", it)


def test_host_h264_weight_hbd(emuhost):
    """pel_hbd.cu: explicit weighted prediction for 9 / 10 / 12 / 14 bit samples, table functions and the batched device entry on the
    stand-in runtime against the checker"""
    from test_oracle_more import run_weight_hbd_case
    L, O = emuhost, cl.oracle()
    O.orc_h264_weight_hbd.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_ssize_t] + [C.c_int] * 4
    O.orc_h264_biweight_hbd.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_ssize_t] + [C.c_int] * 5
    L.emu_host_weight_hbd_tab.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_longlong] + [C.c_int] * 5
    L.b200_h264_weight_hbd_batch_device.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_ssize_t]
    dev = C.c_void_p()
    assert L.b200_device_open(C.byref(dev), 0, None) == 0
    for depth in (9, 10, 12, 14):
        cases = cl.hbd_weight_cases(depth)
        for case in cases[:25]:
            exp = run_weight_hbd_case(O.orc_h264_weight_hbd, O.orc_h264_biweight_hbd, depth, case)
            wf = lambda dp, idx, blk, st, h, d, wd, off: L.emu_host_weight_hbd_tab(dp, 0, idx, blk, None, st, h, d, wd, 0, off)
            bf = lambda dp, idx, blk, src, st, h, d, wd, ws, off: L.emu_host_weight_hbd_tab(dp, 1, idx, blk, src, st, h, d, wd, ws, off)
            assert np.array_equal(run_weight_hbd_case(wf, bf, depth, case), exp), (depth, case)
        # batch: the weight cases in place, then the biweight cases, blocks on a 16 x 16 grid of a 64 x 48 picture (12 per call)
        img, d0 = cl.hbd_picture(depth, 0)
        for bi in (0, 1):
            sel = [c for c in cases if c[0] == bi][:12]
            params = np.array([[c[1] | (c[2] << 8) | (c[3] << 16), c[4], c[5], c[6]] for c in sel], np.int32)
            doff = np.array([((k // 4) * 16 * 64 + (k % 4) * 16) * 2 for k in range(len(sel))], np.int64)
            got, exp = d0.copy(), d0.copy()
            assert L.b200_h264_weight_hbd_batch_device(dev, depth, len(sel), params.ctypes.data, got.ctypes.data, doff.ctypes.data,
                                                       img.ctypes.data if bi else None, doff.ctypes.data if bi else None, 128) == 0
            for k, c in enumerate(sel):
                if bi:
                    O.orc_h264_biweight_hbd(depth, c[1], exp.ctypes.data + int(doff[k]), img.ctypes.data + int(doff[k]), 128, c[2], c[3], c[4], c[5], c[6])
                else:
                    O.orc_h264_weight_hbd(depth, c[1], exp.ctypes.data + int(doff[k]), 128, c[2], c[3], c[4], c[6])
            assert np.array_equal(got, exp), (depth, bi)
    assert L.emu_host_weight_hbd_tab(11, 0, 0, None, None, 0, 0, 0, 0, 0, 0) == -38


def test_host_h264_idct_hbd(emuhost):
    """h264idct_hbd.cu (residual adds for 9 / 10 / 12 / 14 bit samples, int32 coefficients) with its host code on the stand-in runtime: the member
    functions and the batched device entry against the hashes of the compiled reference's outputs and the checker"""
    from test_oracle_more import h264_idct_hbd_hashes, run_h264_idct_hbd_case
    L, O = emuhost, cl.oracle()
    L.emu_host_h264_idct_hbd.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_longlong]
    L.b200_h264_idct_hbd_batch_device.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_ssize_t]
    O.orc_h264_idct_hbd.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_ssize_t]
    dev = C.c_void_p()
    assert L.b200_device_open(C.byref(dev), 0, None) == 0
    hs = h264_idct_hbd_hashes()
    for depth in (9, 10, 12, 14):
        for kind in range(4):
            cases = cl.h264_idct_hbd_cases(depth, kind)
            for k, case in enumerate(cases[:10]):
                assert run_h264_idct_hbd_case(L.emu_host_h264_idct_hbd, depth, kind, case) == hs[(depth, kind, k)], (depth, kind, k)
            # batch: all 24 blocks into one 48 x 64 picture (8 x 8 grid cells), coefficient blocks back to back
            N = 64 if kind & 1 else 16
            blocks = np.concatenate([c[0] for c in cases]).astype(np.int32)
            boff = np.arange(len(cases), dtype=np.int64) * N
            doff = np.array([((k // 6) * 8 * 64 + (k % 6) * 8) * 2 for k in range(len(cases))], np.int64)
            pic = np.random.default_rng(depth * 10 + kind).integers(0, 1 << depth, (48, 64)).astype(np.uint16)
            got, exp, gb, eb = pic.copy(), pic.copy(), blocks.copy(), blocks.copy()
            assert L.b200_h264_idct_hbd_batch_device(dev, depth, kind, len(cases), gb.ctypes.data, boff.ctypes.data, got.ctypes.data, doff.ctypes.data, 128) == 0
            for k in range(len(cases)):
                O.orc_h264_idct_hbd(depth, kind, exp.ctypes.data + int(doff[k]), eb.ctypes.data + 4 * int(boff[k]), 128)
            assert np.array_equal(got, exp) and np.array_equal(gb, eb), (depth, kind)
    assert L.emu_host_h264_idct_hbd(11, 0, None, None, 0) == -38


def test_host_tx_pfa_create_and_launch(emuhost):
    from test_oracle_more import _tx
    L, O = emuhost, cl.oracle()
    L.emu_host_tx_pfa.argtypes = [C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong, C.c_longlong, C.c_longlong]
    rng = np.random.default_rng(31)
    for n in (120, 960, 48, 80, 224, 288):
        for inv in (1, 0):
            cnt = 70                                                    # more than one 64-thread block
            x = (rng.random((cnt, n if inv else 2 * n), dtype=np.float32) * 2 - 1).astype(np.float32)
            out = np.zeros((cnt, n), np.float32)
            assert L.emu_host_tx_pfa(inv, n, 1.0 / n, out.ctypes.data, x.ctypes.data, 4, cnt, out.strides[0], x.strides[0]) == 0
            assert np.array_equal(out.view(np.uint32), _tx(O, "orc", 1, inv, n, 1.0 / n, x, n).view(np.uint32)), (n, inv)
    assert L.emu_host_tx_pfa(1, 84, 1.0, None, None, 4, 1, 0, 0) < 0


def _aligned(shape, align=64):
    """uint8 array whose first byte sits on an `align`-byte boundary (the vector / tensor-core paths want 16-byte aligned planes)"""
    n = int(np.prod(shape))
    raw = np.zeros(n + align, np.uint8)
    o = (-raw.ctypes.data) % align
    return raw[o:o + n].reshape(shape)


@pytest.mark.parametrize("case", [(320, 96, 160, 48, FATE), (352, 64, 208, 40, FATE), (192, 48, 384, 96, cl.SWS_BICUBIC), (1024, 64, 96, 16, FATE),
                                  (640, 40, 272, 24, cl.SWS_BILINEAR | 0x40000 | 0x80000)])
def test_sws_tensor_core_scaler_on_the_emulated_device(emusws, case):
    """The fused scaler with the mma.m16n8k32 horizontal pass (csrc/sws_mma.cuh): whole kernels — staging, fragment addressing, hi / lo
    coefficient split, 15-bit lines, vertical pass and writers — through the batched device entry points, against the checker; the
    context must report that the tensor-core kernels ran."""
    L = emusws
    L.b200_sws_last_path.argtypes = [C.c_void_p]
    w, h, dw, dh, fl = case
    n = 2
    frames = [cl.yuv_frame(w, h, 1700 + k, kind) for k, kind in enumerate(("random", "limited"))]
    cw, ch, cdw, cdh = (w + 1) // 2, (h + 1) // 2, (dw + 1) // 2, (dh + 1) // 2
    Y, U, V = _aligned((n, h, w)), _aligned((n, ch, cw)), _aligned((n, ch, cw))
    for k, f in enumerate(frames):
        Y[k], U[k], V[k] = f
    arr = lambda t, vals: (t * 3)(*vals)
    srcp, srcs, srcf = arr(C.c_void_p, [Y.ctypes.data, U.ctypes.data, V.ctypes.data]), arr(C.c_int32, [w, cw, cw]), arr(C.c_int64, [w * h, cw * ch, cw * ch])
    # three-plane destination
    DY, DU, DV = _aligned((n, dh, dw)), _aligned((n, cdh, cdw)), _aligned((n, cdh, cdw))
    ctx = _emu_ctx(L, w, h, 0, dw, dh, 0, fl)
    assert L.b200_sws_scale_batch_device_planar(ctx, srcp, srcs, srcf, arr(C.c_void_p, [DY.ctypes.data, DU.ctypes.data, DV.ctypes.data]),
                                                arr(C.c_int32, [dw, cdw, cdw]), arr(C.c_int64, [dw * dh, cdw * cdh, cdw * cdh]), n) == 0
    assert L.b200_sws_last_path(ctx) == 4
    L.b200_sws_freeContext(ctx)
    for i in range(n):
        e = cl.orc_sws_planar(w, h, dw, dh, fl, *frames[i])
        assert np.array_equal(DY[i], e[0]) and np.array_equal(DU[i], e[1]) and np.array_equal(DV[i], e[2]), (case, i)
    # packed destinations (rgb24 and one 32-bit order)
    if dw % 16 == 0:
        for fmt, bpp in ((cl.PIX_FMT_RGB24, 3), (cl.PIX_FMT_BGRA, 4)):
            D = _aligned((n, dh, dw * bpp))
            ctx = _emu_ctx(L, w, h, 0, dw, dh, fmt, fl)
            assert L.b200_sws_scale_batch_device(ctx, srcp, srcs, srcf, D.ctypes.data, dw * bpp, dw * dh * bpp, n) == 0
            path = L.b200_sws_last_path(ctx)
            assert path == 4 or (w > 4 * dw and path == 1), path     # a 10:1 tile of three planes does not fit in shared memory: two passes
            L.b200_sws_freeContext(ctx)
            for i in range(n):
                assert np.array_equal(D[i], cl.orc_sws(w, h, dw, dh, fl, *frames[i], fmt=fmt)), (case, fmt, i)


def test_sws_bottom_up_slice_sequences(emusws, refrec):
    """sws_scale() fed bottom-up (the band touching the last line first — what the reference flips internally, swscale.c:1096-1159):
    per-call return values and the final picture equal the compiled reference's, planar and packed destinations, scaled and LUT paths."""
    import random
    L, R = emusws, cl.ref() if cl.have_ref() else None
    if R:
        R.ffref_sws_scale_planar.argtypes = [C.c_void_p] + [C.c_void_p, C.c_int] * 3 + [C.c_int, C.c_int] + [C.c_void_p, C.c_int] * 3
        R.ffref_sws_scale.argtypes = [C.c_void_p] + [C.c_void_p, C.c_int] * 3 + [C.c_int, C.c_int, C.c_void_p, C.c_int]
    rnd = random.Random(91)
    for it in range(36):
        w, h = rnd.choice([16, 34, 64, 100]), rnd.choice([8, 16, 34, 48, 66])
        dw, dh = (w, h) if it % 3 == 0 else (rnd.choice([8, 18, 32, 64, 100]), rnd.choice([8, 18, 32, 64]))
        if h > 2 * dh:
            dh = (h // 2 + 2) & ~1
        fl = rnd.choice([cl.SWS_BICUBIC, cl.SWS_BILINEAR, FATE])
        df = rnd.choice([0, cl.PIX_FMT_NV12, cl.PIX_FMT_RGB24, cl.PIX_FMT_BGRA])
        planar = df in (0, cl.PIX_FMT_NV12)
        y, u, v = cl.yuv_frame(w, h, 9100 + it, "random")
        cuts = sorted(set([0, h] + [2 * rnd.randrange(1, h // 2) for _ in range(rnd.randrange(1, 4))]))
        bands = [(a, b - a) for a, b in zip(cuts[:-1], cuts[1:])][::-1]                 # last band first
        cw, ch = (dw + 1) // 2, (dh + 1) // 2
        bpp = 1 if planar else cl.fmt_bpp(df)
        mk = lambda: ([np.full((dh, dw), 0xA5, np.uint8), np.full((ch, 2 * cw if df else cw), 0xA5, np.uint8), np.full((ch, cw), 0xA5, np.uint8)]
                      if planar else [np.full((dh, dw * bpp), 0xA5, np.uint8)])
        rp, gp = mk(), mk()

        def ref_returns():
            rc = R.ffref_sws_open_range(0, w, h, 0, df, dw, dh, 0, fl, 1)
            assert rc
            rr = []
            for (sy, sh) in bands:
                if planar:
                    rr.append(R.ffref_sws_scale_planar(rc, y[sy:].ctypes.data, y.strides[0], u[sy // 2:].ctypes.data, u.strides[0], v[sy // 2:].ctypes.data, v.strides[0],
                                                       sy, sh, rp[0].ctypes.data, rp[0].strides[0], rp[1].ctypes.data, rp[1].strides[0], rp[2].ctypes.data, rp[2].strides[0]))
                else:
                    rr.append(R.ffref_sws_scale(rc, y[sy:].ctypes.data, y.strides[0], u[sy // 2:].ctypes.data, u.strides[0], v[sy // 2:].ctypes.data, v.strides[0],
                                                sy, sh, rp[0].ctypes.data, rp[0].strides[0]))
            R.ffref_sws_close(rc)
            return rr
        ctx = _emu_ctx(L, w, h, 0, dw, dh, df, fl)
        assert ctx
        gr = []
        for (sy, sh) in bands:
            dpl = [a.ctypes.data for a in gp] + [None] * (4 - len(gp))
            dst = [a.strides[0] for a in gp] + [0] * (4 - len(gp))
            gr.append(L.b200_sws_scale(ctx, (C.c_void_p * 4)(y[sy:].ctypes.data, u[sy // 2:].ctypes.data, v[sy // 2:].ctypes.data, None),
                                       (C.c_int32 * 4)(y.strides[0], u.strides[0], v.strides[0], 0), sy, sh, (C.c_void_p * 4)(*dpl), (C.c_int32 * 4)(*dst)))
        L.b200_sws_freeContext(ctx)
        assert refrec.same(gr, ref_returns), (it, w, h, dw, dh, hex(fl), df, bands, gr)
        n = 2 if df == cl.PIX_FMT_NV12 else len(gp)
        planes = lambda p: np.concatenate([a.ravel() for a in p[:n]])
        assert refrec.same(planes(gp), lambda: planes(rp)), (it, w, h, dw, dh, hex(fl), df, bands)


def test_sws_slice_sequences_from_packed_rgb_sources(emusws, refrec):
    """sws_scale() band by band from rgb24 / bgra sources into yuv420p, nv12 and packed RGB destinations on the emulated device: per-call
    return values and the final picture equal the compiled reference's (packed sources have no vertical chroma subsampling on the way
    in, so any band boundary is legal)."""
    import random
    L, R = emusws, cl.ref() if cl.have_ref() else None
    if R:
        R.ffref_sws_scale_planar.argtypes = [C.c_void_p] + [C.c_void_p, C.c_int] * 3 + [C.c_int, C.c_int] + [C.c_void_p, C.c_int] * 3
        R.ffref_sws_scale.argtypes = [C.c_void_p] + [C.c_void_p, C.c_int] * 3 + [C.c_int, C.c_int, C.c_void_p, C.c_int]
    rnd = random.Random(93)
    done = 0
    for it in range(60):
        w, h = rnd.choice([16, 34, 64, 100]), rnd.choice([8, 16, 33, 48, 66])
        dw, dh = rnd.choice([8, 18, 32, 64, 100]), rnd.choice([8, 18, 32, 64])
        if h > 2 * dh:
            dh = (h // 2 + 2) & ~1
        fl = rnd.choice([cl.SWS_BICUBIC, cl.SWS_BILINEAR, FATE])
        sf = rnd.choice([cl.PIX_FMT_RGB24, cl.PIX_FMT_BGRA])
        df = rnd.choice([0, cl.PIX_FMT_NV12, cl.PIX_FMT_BGR24, cl.PIX_FMT_RGBA])
        planar = df in (0, cl.PIX_FMT_NV12)
        sb = cl.fmt_bpp(sf)
        src = cl.rgb_frame(w, h, 9300 + it, sb)
        cuts = sorted(set([0, h] + [rnd.randrange(1, h) for _ in range(rnd.randrange(1, 4))]))
        bands = [(a, b - a) for a, b in zip(cuts[:-1], cuts[1:])]
        cw, ch = (dw + 1) // 2, (dh + 1) // 2
        bpp = 1 if planar else cl.fmt_bpp(df)
        mk = lambda: ([np.full((dh, dw), 0xA5, np.uint8), np.full((ch, 2 * cw if df else cw), 0xA5, np.uint8), np.full((ch, cw), 0xA5, np.uint8)]
                      if planar else [np.full((dh, dw * bpp), 0xA5, np.uint8)])
        rp, gp, rc = mk(), mk(), []

        def ref_opens():
            rc.append(R.ffref_sws_open_range(sf, w, h, 0, df, dw, dh, 0, fl, 1))
            return bool(rc[0])

        def ref_returns():
            rr = []
            for (sy, sh) in bands:
                if planar:
                    rr.append(R.ffref_sws_scale_planar(rc[0], src[sy:].ctypes.data, src.strides[0], None, 0, None, 0,
                                                       sy, sh, rp[0].ctypes.data, rp[0].strides[0], rp[1].ctypes.data, rp[1].strides[0], rp[2].ctypes.data, rp[2].strides[0]))
                else:
                    rr.append(R.ffref_sws_scale(rc[0], src[sy:].ctypes.data, src.strides[0], None, 0, None, 0, sy, sh, rp[0].ctypes.data, rp[0].strides[0]))
            return rr
        opened = refrec.same(True, ref_opens)
        ctx = _emu_ctx(L, w, h, sf, dw, dh, df, fl)
        if not opened or not ctx:
            if rc and rc[0]: R.ffref_sws_close(rc[0])
            if ctx: L.b200_sws_freeContext(ctx)
            continue
        gr = []
        for (sy, sh) in bands:
            dpl = [a.ctypes.data for a in gp] + [None] * (4 - len(gp))
            dst = [a.strides[0] for a in gp] + [0] * (4 - len(gp))
            gr.append(L.b200_sws_scale(ctx, (C.c_void_p * 4)(src[sy:].ctypes.data, None, None, None), (C.c_int32 * 4)(src.strides[0], 0, 0, 0), sy, sh,
                                       (C.c_void_p * 4)(*dpl), (C.c_int32 * 4)(*dst)))
        L.b200_sws_freeContext(ctx)
        if any(v < 0 for v in gr):
            if rc: R.ffref_sws_close(rc[0])
            assert all(v == -38 for v in gr if v < 0), (it, gr)              # the bgr24 -> yv12 line-pair converter refuses odd bands (ENOSYS)
            continue
        assert refrec.same(gr, ref_returns), (it, w, h, dw, dh, hex(fl), sf, df, bands, gr)
        if rc: R.ffref_sws_close(rc[0])
        n = 2 if df == cl.PIX_FMT_NV12 else len(gp)
        planes = lambda p: np.concatenate([a.ravel() for a in p[:n]])
        assert refrec.same(planes(gp), lambda: planes(rp)), (it, w, h, dw, dh, hex(fl), sf, df, bands)
        done += 1
    assert done >= 40, done


def test_me_cmp_dct_family_on_emulated_device(emuhost, refrec):
    """mecmp_dct.cu (dct_sad / dct_max with both integer DCTs, dct264_sad; 8x8 and 16 wide with h = 8 / 16) as the library launches it,
    lane for lane on the CPU, against the checker and the compiled reference: random, near-equal, saturated and checkerboard blocks"""
    L, O, R = emuhost, cl.oracle(), cl.ref() if cl.have_ref() else None
    rng = np.random.default_rng(2309)
    stride, rows = 48, 40
    pics = []
    a = rng.integers(0, 256, (rows, stride), dtype=np.uint8); pics.append((a, rng.integers(0, 256, (rows, stride), dtype=np.uint8)))
    pics.append((a, np.clip(a.astype(int) + rng.integers(-5, 6, a.shape), 0, 255).astype(np.uint8)))
    pics.append((np.full((rows, stride), 255, np.uint8), np.zeros((rows, stride), np.uint8)))
    c = ((np.add.outer(np.arange(rows), np.arange(stride)) & 1) * 255).astype(np.uint8); pics.append((c, (255 - c).astype(np.uint8)))
    pics.append(((rng.integers(0, 2, (rows, stride)) * 255).astype(np.uint8), (rng.integers(0, 2, (rows, stride)) * 255).astype(np.uint8)))
    n = 19                                                        # not a multiple of the 8 comparisons of a CTA
    try:
        for algo in (0, 1, 2):
            assert L.b200_me_cmp_set_dct_algo(algo) == 0
            O.orc_me_cmp_set_dct_algo(1 if algo == 1 else 0)
            if R is not None: R.ffref_me_cmp_set_dct_algo(algo)
            for f1, f2 in pics:
                off1 = (rng.integers(0, rows - 16, n) * stride + rng.integers(0, stride - 16, n)).astype(np.int64)
                off2 = (rng.integers(0, rows - 16, n) * stride + rng.integers(0, stride - 16, n)).astype(np.int64)
                for fn in (8, 9, 10):
                    for w, h in ((16, 16), (16, 8), (8, 8)):
                        out = np.full(n, -7, np.int32)
                        assert L.emu_host_me_dct(fn, w, h, vp(f1), vp(f2), C.c_longlong(stride), vp(off1), vp(off2), C.c_longlong(n), vp(out)) == 0
                        idx = 0 if w == 16 else 1
                        for i in range(n):
                            p1, p2 = f1.reshape(-1)[off1[i]:], f2.reshape(-1)[off2[i]:]
                            e = O.orc_me_cmp(fn, idx, cl.ptr(p1, cl.u8p), cl.ptr(p2, cl.u8p), stride, h)
                            assert out[i] == e, (algo, fn, w, h, i, int(out[i]), e)
                            assert refrec.same(e, lambda: R.ffref_me_cmp(fn, idx, cl.ptr(p1, cl.u8p), cl.ptr(p2, cl.u8p), stride, h))
        assert L.b200_me_cmp_set_dct_algo(6) < 0                  # FF_DCT_FAAN
    finally:
        L.b200_me_cmp_set_dct_algo(0); O.orc_me_cmp_set_dct_algo(0)
        if R is not None: R.ffref_me_cmp_set_dct_algo(0)


def fdct_blocks(bits, n, seed):
    """pixel differences / samples of the given depth, saturated +-max blocks, and anything an int16 block can hold (the products wrap like the
    reference's unsigned multiplies)"""
    rng = np.random.default_rng(seed)
    lim = 256 if bits == 8 else 1 << bits
    b = np.empty((n, 64), np.int16)
    for i in range(n):
        m = i % 4
        b[i] = rng.integers(-lim + 1, lim, 64) if m == 0 else rng.integers(0, lim, 64) if m == 1 else rng.choice([-lim + 1, lim - 1], 64) if m == 2 else rng.integers(-32768, 32768, 64)
    return b


def test_fdctdsp_on_emulated_device(emuhost, refrec):
    """fdctdsp.cu as the library launches it (batched entry, 32 blocks per CTA, a block count that leaves idle lane groups) on the CPU: islow 8 / 10 bit
    and ifast, plain and 2-4-8, against the checker and the compiled reference"""
    L, O, R = emuhost, cl.oracle(), cl.ref() if cl.have_ref() else None
    for algo, bits, kind in ((0, 8, 0), (1, 8, 1), (0, 10, 2), (1, 9, 2), (2, 8, 0)):
        for is248 in (0, 1):
            x = fdct_blocks(bits, 37, 100 * algo + bits + is248)
            got = x.copy()
            assert L.b200_fdct_batch_device(None, algo, bits, is248, vp(got), C.c_int64(37)) == 0
            for i in range(37):
                e, r = x[i].copy(), x[i].copy()
                O.orc_fdct(kind, is248, cl.ptr(e, cl.i16p))
                assert refrec.same(e, lambda: (R.ffref_fdct(algo, bits, is248, cl.ptr(r, cl.i16p)), r)[1]) and np.array_equal(got[i], e), (algo, bits, is248, i)
    assert L.b200_fdct_batch_device(None, 6, 8, 0, vp(got), C.c_int64(1)) < 0          # FF_DCT_FAAN
