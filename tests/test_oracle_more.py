"""CPU tier: pin the me_cmp / h264qpel / hpeldsp / tx oracles against the golden fixtures (always) and the compiled
reference (where oracle/_ref exists)."""
import ctypes as C
import os

import numpy as np
import pytest

import cpulibs as cl

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
needs_ref = pytest.mark.skipif(not cl.have_ref(), reason="oracle/_ref not built (no /root/reference here)")


def test_mecmp_oracle_golden():
    g = np.load(os.path.join(G, "mecmp.npz"))
    O = cl.oracle()
    img1, img2 = g["img1"], g["img2"]
    for fn, idx, x1, y1, x2, y2, h, v in g["cases"]:
        got = O.orc_me_cmp(int(fn), int(idx), C.cast(img1.ctypes.data + int(y1) * 64 + int(x1), cl.u8p),
                           C.cast(img2.ctypes.data + int(y2) * 64 + int(x2), cl.u8p), 64, int(h))
        assert got == v, (fn, idx, h)
    W, H = 96, 64
    cur, ref_ = g["esa_cur"], g["esa_ref"]
    flat = np.full((H, W), 99, np.uint8)
    for name, (a, b) in {"shift": (cur, ref_), "flat": (flat, flat), "same": (cur, cur)}.items():
        for mb, sp in ((16, 7), (8, 4), (16, 32), (4, 3)):
            bw, bh = W // mb, H // mb
            mv, cost = np.zeros((bh * bw, 2), np.int32), np.zeros(bh * bw, np.uint64)
            O.orc_esa_frame(cl.ptr(a), cl.ptr(b), W, W, H, mb, sp, 0, bh, cl.ptr(mv, cl.i32p), cl.ptr(cost, cl.u64p))
            assert np.array_equal(mv, g[f"esa_{name}_{mb}_{sp}_mv"]) and np.array_equal(cost, g[f"esa_{name}_{mb}_{sp}_cost"]), (name, mb, sp)


def test_h264chroma_oracle_golden():
    """All 64 eighth-pel phases x put/avg x widths 8/4/2 x heights against the reference's outputs (chroma.npz)."""
    g = np.load(os.path.join(G, "chroma.npz"))
    O = cl.oracle()
    src, dst0 = g["src"], g["dst0"]
    ps = C.cast(src.ctypes.data + 8 * 48 + 8, cl.u8p)
    n = 0
    for key in g.files:
        if key[0] != "c":
            continue
        avg, idx, h = (int(v) for v in key.split("_")[1:])
        for xy in range(64):
            o = dst0.copy()
            assert O.orc_h264chroma(avg, idx, C.cast(o.ctypes.data + 8 * 48 + 8, cl.u8p), ps, 48, h, xy & 7, xy >> 3) == 0
            assert np.array_equal(o[8:24, 8:16], g[key][xy]), (key, xy)
            assert np.array_equal(o[:8], dst0[:8]) and np.array_equal(o[8 + h:], dst0[8 + h:]) and np.array_equal(o[:, 16:], dst0[:, 16:]), key
            n += 1
    assert n == 2 * 8 * 64
    assert O.orc_h264chroma(0, 3, cl.ptr(dst0.copy()), ps, 48, 8, 0, 0) < 0          # table entry [3] does not exist


def test_h264chroma_oracle_vs_ref(refrec):
    R, O = cl.ref() if cl.have_ref() else None, cl.oracle()
    rng = np.random.default_rng(5)
    for it in range(400):
        src = rng.integers(0, 256, (40, 48), dtype=np.uint8)
        if it % 7 == 0:
            src[:] = rng.choice([0, 255], src.shape)
        d1 = rng.integers(0, 256, (40, 48), dtype=np.uint8)
        d2 = d1.copy()
        avg, idx, x, y = int(rng.integers(0, 2)), int(rng.integers(0, 3)), int(rng.integers(0, 8)), int(rng.integers(0, 8))
        h = int(rng.choice([2, 4, 8, 16]))
        ps = C.cast(src.ctypes.data + 8 * 48 + 8, cl.u8p)

        def ref_out():
            assert R.ffref_h264chroma(avg, idx, C.cast(d1.ctypes.data + 8 * 48 + 8, cl.u8p), ps, 48, h, x, y) == 0
            return d1
        assert O.orc_h264chroma(avg, idx, C.cast(d2.ctypes.data + 8 * 48 + 8, cl.u8p), ps, 48, h, x, y) == 0
        assert refrec.same(d2, ref_out), (avg, idx, x, y, h)


def test_h264chroma_batch_oracle_equals_single_calls():
    """orc_h264chroma_batch (the device entry's operation list) applies each operation as orc_h264chroma does, in list order:
    overlapping destinations, avg on top of earlier results, every phase / width / height, unaligned offsets"""
    O = cl.oracle()
    rng = np.random.default_rng(31)
    W, H, n = 80, 72, 3000
    src = rng.integers(0, 256, (H, W), dtype=np.uint8)
    dst0 = rng.integers(0, 256, (H, W), dtype=np.uint8)
    idx = rng.integers(0, 3, n)
    op = ((idx << 1) | rng.integers(0, 2, n)).astype(np.uint8)
    h = np.array([rng.choice(((2, 4, 8, 16), (2, 4, 8), (2, 4))[i]) for i in idx], np.uint8)
    xy = (np.arange(n) % 64).astype(np.uint8)
    doff = (rng.integers(0, H - 16, n) * W + rng.integers(0, W - 8, n)).astype(np.int64)
    soff = (rng.integers(0, H - 17, n) * W + rng.integers(0, W - 9, n)).astype(np.int64)
    exp = dst0.copy()
    for i in range(n):
        assert O.orc_h264chroma(int(op[i]) & 1, int(op[i]) >> 1, C.cast(exp.ctypes.data + int(doff[i]), cl.u8p),
                                C.cast(src.ctypes.data + int(soff[i]), cl.u8p), W, int(h[i]), int(xy[i]) & 7, int(xy[i]) >> 3) == 0
    got = dst0.copy()
    assert O.orc_h264chroma_batch(n, cl.ptr(op), cl.ptr(h), cl.ptr(xy), cl.ptr(got), cl.ptr(doff, cl.i64p), cl.ptr(src),
                                  cl.ptr(soff, cl.i64p), W) == 0
    assert np.array_equal(got, exp), int((got != exp).sum())
    assert not np.array_equal(got, dst0)
    bad = op.copy()
    bad[5] = 3 << 1                                                # table entry [3] does not exist
    assert O.orc_h264chroma_batch(n, cl.ptr(bad), cl.ptr(h), cl.ptr(xy), cl.ptr(dst0.copy()), cl.ptr(doff, cl.i64p), cl.ptr(src),
                                  cl.ptr(soff, cl.i64p), W) == -1


def test_emulated_edge_mc_oracle_golden():
    from cases import EDGE_PIC, EDGE_CASES
    g = np.load(os.path.join(G, "edge.npz"))
    O = cl.oracle()
    W, H, LS = EDGE_PIC
    pic = g["pic"]
    for i, (bw, bh, sx, sy) in enumerate(EDGE_CASES):
        b = np.full((24, 32), 0x5A, np.uint8)
        O.orc_emulated_edge_mc(cl.ptr(b), pic.ctypes.data + sy * LS + sx, 32, LS, bw, bh, sx, sy, W, H)
        assert np.array_equal(b, g[f"e{i}"]), (i, bw, bh, sx, sy)
    b = np.full((24, 32), 0x5A, np.uint8)
    O.orc_emulated_edge_mc(cl.ptr(b), pic.ctypes.data, 32, LS, 8, 8, 0, 0, 0, H)       # w == 0: nothing written
    assert (b == 0x5A).all()


def test_emulated_edge_mc_oracle_vs_ref(refrec):
    R, O = cl.ref() if cl.have_ref() else None, cl.oracle()
    rng = np.random.default_rng(6)
    W, H, LS = 37, 29, 48
    pic = rng.integers(0, 256, (H, LS), dtype=np.uint8)
    for it in range(3000):
        bw, bh = int(rng.integers(1, 24)), int(rng.integers(1, 24))
        sx, sy = int(rng.integers(-40, W + 40)), int(rng.integers(-40, H + 40))
        b1 = np.full((24, 32), 7, np.uint8)
        b2 = b1.copy()
        src = pic.ctypes.data + sy * LS + sx
        O.orc_emulated_edge_mc(cl.ptr(b2), src, 32, LS, bw, bh, sx, sy, W, H)
        assert refrec.same(b2, lambda: (R.ffref_emulated_edge_mc(cl.ptr(b1), src, 32, LS, bw, bh, sx, sy, W, H), b1)[1]), (bw, bh, sx, sy)


def test_h264_idct_oracle_golden():
    """ff_h264_idct_add / idct8_add / dc adds: oracle against the reference's outputs, incl. the cleared coefficients."""
    g = np.load(os.path.join(G, "h264idct.npz"))
    O = cl.oracle()
    for kind in range(4):
        blk, out = g[f"k{kind}_in"].copy(), g[f"k{kind}_dst"].copy()
        n = blk.shape[0]
        for i in range(n):
            assert O.orc_h264_idct(kind, C.cast(out.ctypes.data + 8 * i, cl.u8p), C.cast(blk.ctypes.data + i * blk.strides[0], cl.i16p), n * 8) == 0
        assert np.array_equal(out, g[f"k{kind}_out"]), kind
        assert np.array_equal(blk, g[f"k{kind}_blk_after"]), kind
    assert O.orc_h264_idct(4, cl.ptr(np.zeros(64, np.uint8)), cl.ptr(np.zeros(64, np.int16), cl.i16p), 8) < 0


def test_h264_idct_oracle_vs_ref(refrec):
    R, O = cl.ref() if cl.have_ref() else None, cl.oracle()
    rng = np.random.default_rng(9)
    for it in range(3000):
        kind = int(rng.integers(0, 4))
        n = 16 if kind in (0, 2) else 64
        blk = (rng.integers(-32768, 32768, n) if it % 2 else rng.integers(-600, 601, n)).astype(np.int16)
        if kind >= 2:
            blk[1:] = 0
        d1 = rng.integers(0, 256, (12, 24), dtype=np.uint8)
        d2, b1, b2 = d1.copy(), blk.copy(), blk.copy()
        O.orc_h264_idct(kind, C.cast(d2.ctypes.data + 2 * 24 + 8, cl.u8p), cl.ptr(b2, cl.i16p), 24)

        def ref_out():
            R.ffref_h264_idct(kind, C.cast(d1.ctypes.data + 2 * 24 + 8, cl.u8p), cl.ptr(b1, cl.i16p), 24)
            return np.concatenate([d1.ravel(), b1.view(np.uint8)])
        assert refrec.same(np.concatenate([d2.ravel(), b2.view(np.uint8)]), ref_out), (kind, it)


def test_h264_weight_oracle_golden():
    g = np.load(os.path.join(G, "h264weight.npz"))
    O = cl.oracle()
    src, dst0 = g["src"], g["dst0"]
    ps = C.cast(src.ctypes.data + 2 * 32 + 8, cl.u8p)
    for k, (idx, h, ld, w1, w2, off) in enumerate(g["cases"].tolist()):
        a, b = dst0.copy(), dst0.copy()
        O.orc_h264_weight(idx, C.cast(a.ctypes.data + 2 * 32 + 8, cl.u8p), 32, h, ld, w1, off)
        O.orc_h264_biweight(idx, C.cast(b.ctypes.data + 2 * 32 + 8, cl.u8p), ps, 32, h, ld, w1, w2, off)
        assert np.array_equal(a, g[f"w{k}"]) and np.array_equal(b, g[f"b{k}"]), k


def test_satd_oracle_golden():
    g, c = np.load(os.path.join(G, "mecmp.npz")), np.load(os.path.join(G, "satd.npz"))["cases"]
    O = cl.oracle()
    img1, img2 = g["img1"], g["img2"]
    for fn, idx, x1, y1, x2, y2, h, v in c:
        got = O.orc_me_cmp(int(fn), int(idx), C.cast(img1.ctypes.data + int(y1) * 64 + int(x1), cl.u8p),
                           C.cast(img2.ctypes.data + int(y2) * 64 + int(x2), cl.u8p), 64, int(h))
        assert got == v, (fn, idx, h)


def test_pel_oracle_golden():
    g = np.load(os.path.join(G, "pel.npz"))
    O = cl.oracle()
    src, dst0 = g["src"], g["dst0"]
    ps = C.cast(src.ctypes.data + 8 * 48 + 8, cl.u8p)
    n = 0
    for key in g.files:
        if key[0] not in "qh" or key in ("src", "dst0"):
            continue
        o = dst0.copy()
        po = C.cast(o.ctypes.data + 8 * 48 + 8, cl.u8p)
        parts = [int(v) for v in key.split("_")[1:]]
        if key[0] == "q":
            O.orc_h264qpel(parts[0], parts[1], parts[2], po, ps, 48)
        else:
            assert O.orc_hpel(parts[0], parts[1], parts[2], po, ps, 48, parts[3]) == 0
        assert np.array_equal(o[8:24, 8:24], g[key]), key
        assert np.array_equal(o[:8], dst0[:8]) and np.array_equal(o[24:], dst0[24:]), key      # guard rows untouched
        n += 1
    assert n > 150


def _tx(L, pre, typ, inv, n, scale, x, out_floats, flags=0):
    h = getattr(L, pre + "_tx_open")(typ, inv, n, scale, flags)
    assert h
    out = np.zeros((x.shape[0], out_floats), np.float32)
    getattr(L, pre + "_tx_run")(h, out.ctypes.data, x.ctypes.data, 8 if typ == 0 else 4, x.shape[0], out.strides[0], x.strides[0])
    getattr(L, pre + "_tx_close")(h)
    return out


def test_tx_oracle_golden_bitexact():
    g = np.load(os.path.join(G, "tx.npz"))
    O = cl.oracle()
    for n in (2, 4, 8, 16, 32, 64, 256, 1024, 2048):
        for inv in (0, 1):
            got = _tx(O, "orc", 0, inv, n, 1.0, g[f"fft_in_{n}"], 2 * n)
            assert np.array_equal(got.view(np.uint32), g[f"fft_{n}_{inv}"].view(np.uint32)), (n, inv)
    for n in (8, 16, 64, 256, 1024, 2048):
        for j, sc in enumerate((1.0 / n, -1.0, 1.0)):
            assert np.array_equal(_tx(O, "orc", 1, 1, n, sc, g[f"imdct_in_{n}"], n).view(np.uint32), g[f"imdct_{n}_{j}"].view(np.uint32)), (n, j)
            assert np.array_equal(_tx(O, "orc", 1, 0, n, sc, g[f"mdct_in_{n}"], n).view(np.uint32), g[f"mdct_{n}_{j}"].view(np.uint32)), (n, j)


RDFT_SIZES = (4, 8, 16, 64, 256, 1024, 2048, 4096)


def test_tx_rdft_oracle_golden_bitexact():
    """AV_TX_FLOAT_RDFT r2c / c2r against the reference's outputs, including what c2r leaves in its input buffer."""
    g = np.load(os.path.join(G, "tx_rdft.npz"))
    O = cl.oracle()
    for n in RDFT_SIZES:
        for j, sc in enumerate((1.0, 1.0 / n)):
            got = _tx(O, "orc", 6, 0, n, sc, g[f"r2c_in_{n}_{j}"].copy(), n + 2)
            assert np.array_equal(got.view(np.uint32), g[f"r2c_{n}_{j}"].view(np.uint32)), (n, j)
            xc = g[f"c2r_in_{n}_{j}"].copy()
            got = _tx(O, "orc", 6, 1, n, sc, xc, n)
            assert np.array_equal(got.view(np.uint32), g[f"c2r_{n}_{j}"].view(np.uint32)), (n, j)
            assert np.array_equal(xc.view(np.uint32), g[f"c2r_in_after_{n}_{j}"].view(np.uint32)), (n, j)


def test_tx_rdft_oracle_is_a_real_dft_and_round_trips():
    O = cl.oracle()
    rng = np.random.default_rng(3)
    for n in (16, 1024):
        x = (rng.random((1, n), dtype=np.float32) * 2 - 1).astype(np.float32)
        spec = _tx(O, "orc", 6, 0, n, 1.0, x.copy(), n + 2)
        ref = np.fft.rfft(x[0].astype(np.float64))
        assert np.abs(spec[0, 0::2] - ref.real).max() < 5e-4 * n and np.abs(spec[0, 1::2] - ref.imag).max() < 5e-4 * n
        back = _tx(O, "orc", 6, 1, n, 1.0 / n, spec.copy(), n)       # r2c(scale 1) then c2r(scale 1/len) is the identity
        assert np.abs(back[0] - x[0]).max() < 1e-4


def test_tx_oracle_is_a_dft():
    """Independent sanity check of the oracle itself: against numpy's double-precision FFT (eps like checkasm av_tx.c:27)."""
    O = cl.oracle()
    rng = np.random.default_rng(1)
    for n in (16, 1024, 2048):
        x = rng.random((1, 2 * n), dtype=np.float32)
        z = x[0, 0::2].astype(np.float64) + 1j * x[0, 1::2].astype(np.float64)
        got = _tx(O, "orc", 0, 0, n, 1.0, x, 2 * n)[0]
        ref = np.fft.fft(z)
        assert np.abs(got[0::2] - ref.real).max() < 5e-4 * n and np.abs(got[1::2] - ref.imag).max() < 5e-4 * n


def test_more_oracles_vs_reference_live(refrec):
    R, O = cl.ref() if cl.have_ref() else None, cl.oracle()
    rng = np.random.default_rng(77)
    img1 = rng.integers(0, 256, (80, 96), dtype=np.uint8)
    img2 = rng.integers(0, 256, (80, 96), dtype=np.uint8)
    for _ in range(100):
        x1, y1, x2, y2 = (int(v) for v in rng.integers(0, 60, 4))
        h = int(rng.choice([4, 8, 16]))
        for fn, idxs in ((0, (0, 1)), (1, (0, 1, 2)), (2, range(8))):
            for idx in idxs:
                p1 = C.cast(img1.ctypes.data + y1 * 96 + x1, cl.u8p)
                p2 = C.cast(img2.ctypes.data + y2 * 96 + x2, cl.u8p)
                assert refrec.same(O.orc_me_cmp(fn, idx, p1, p2, 96, h), lambda: R.ffref_me_cmp(fn, idx, p1, p2, 96, h))
    for n in (32, 128, 512, 4096):
        x = rng.random((3, 2 * n), dtype=np.float32)
        for inv in (0, 1):
            assert refrec.same(_tx(O, "orc", 0, inv, n, 1.0, x, 2 * n).view(np.uint32), lambda: _tx(R, "ffref", 0, inv, n, 1.0, x, 2 * n).view(np.uint32))
        assert refrec.same(_tx(O, "orc", 1, 1, n, 1.0 / n, x[:, :n], n).view(np.uint32), lambda: _tx(R, "ffref", 1, 1, n, 1.0 / n, x[:, :n], n).view(np.uint32))
        xr = np.ascontiguousarray(x[:, :n])
        assert refrec.same(_tx(O, "orc", 6, 0, n, 0.5, xr.copy(), n + 2).view(np.uint32), lambda: _tx(R, "ffref", 6, 0, n, 0.5, xr.copy(), n + 2).view(np.uint32))
        xc = np.ascontiguousarray(x[:, :n + 2])
        assert refrec.same(_tx(O, "orc", 6, 1, n, 0.5, xc.copy(), n).view(np.uint32), lambda: _tx(R, "ffref", 6, 1, n, 0.5, xc.copy(), n).view(np.uint32))
        assert refrec.same(_tx(O, "orc", 1, 0, n, -1.0, x, n).view(np.uint32), lambda: _tx(R, "ffref", 1, 0, n, -1.0, x, n).view(np.uint32))


# ---------------------------------------------------------------------------------------------- mpegvideo inverse quantisers
def test_unquant_oracle_golden():
    """the seven dct_unquantize_* functions (mpegvideo_unquantize.c) against the reference's outputs"""
    g = np.load(os.path.join(G, "unquant.npz"))
    for variant in range(7):
        for seed in (11, 12):
            cfg, blocks, blk_n, q, last = cl.unquant_case(seed * 7 + variant, variant, nblocks=48)
            out = cl.orc_unquant(variant, cfg, blocks, blk_n, q, last)
            assert np.array_equal(out, g[f"v{variant}_s{seed}"]), (cl.UNQUANT_VARIANTS[variant], seed)
            assert not np.array_equal(out, blocks)


def test_unquant_oracle_vs_ref(refrec):
    for variant in range(7):
        for seed in range(30):
            cfg, blocks, blk_n, q, last = cl.unquant_case(100 + seed * 7 + variant, variant)
            if seed % 3:
                a = lambda: cl.ref_unquant(variant, cfg, blocks, blk_n, q, last)
                b = cl.orc_unquant(variant, cfg, blocks, blk_n, q, last)
            else:                                                    # macroblock stream order: n = index % 6
                n6 = (np.arange(blocks.shape[0]) % 6).astype(np.uint8)
                a = lambda: cl.ref_unquant(variant, cfg, blocks, n6, q, last)
                b = cl.orc_unquant(variant, cfg, blocks, None, q, last)
            assert refrec.same(b, a), (cl.UNQUANT_VARIANTS[variant], seed)


def test_unquant_properties():
    """mismatch control leaves an odd coefficient sum (ISO 13818-2 7.4.4); untouched tail; mpeg1 results are odd"""
    for variant in (3, 4):
        cfg, blocks, blk_n, q, last = cl.unquant_case(900 + variant, variant, nblocks=200)
        blocks[:, 63] = 0
        for b in range(blocks.shape[0]):
            if last[b] == 63:
                last[b] = 62
        scan = cl.ALTERNATE_VERTICAL if cfg["alternate_scan"] else cl.ZIGZAG
        out = cl.orc_unquant(variant, cfg, blocks, blk_n, q, last).astype(np.int64)
        for b in range(out.shape[0]):
            coded = scan[:int(last[b]) + 1]
            s = int(out[b, coded].sum()) + int(out[b, 63]) + (int(out[b, 0]) if variant == 3 and 0 not in coded else 0)
            assert s & 1, (variant, b)
    for variant in (0, 1):
        cfg, blocks, blk_n, q, last = cl.unquant_case(950 + variant, variant, nblocks=100)
        out = cl.orc_unquant(variant, cfg, blocks, blk_n, q, last)
        scan = cl.ALTERNATE_VERTICAL if cfg["alternate_scan"] else cl.ZIGZAG
        for b in range(out.shape[0]):
            coded = scan[(1 if variant == 0 else 0):int(last[b]) + 1]
            v = out[b, coded]
            assert np.all((v[v != 0] & 1) == 1)
            rest = scan[int(last[b]) + 1:]
            assert np.array_equal(out[b, rest], blocks[b, rest])


# ---------------------------------------------------------------------------------------------- AVFloatDSPContext
def test_fdsp_oracle_golden():
    """the twelve AVFloatDSPContext C functions against the reference's outputs, bit for bit"""
    g = np.load(os.path.join(G, "fdsp.npz"))
    for op in range(12):
        for length in (16, 100, 1024):
            r, a = cl.orc_fdsp(op, *cl.fdsp_case(40 + op, op, length), length)
            assert r.tobytes() == g[f"op{op}_n{length}"].tobytes(), (cl.FDSP_OPS[op], length)
            if op == 8:
                assert a.tobytes() == g[f"op{op}_n{length}_v2"].tobytes()


def test_fdsp_oracle_vs_ref(refrec):
    raw = lambda r, a: np.frombuffer(r.tobytes() + a.tobytes(), np.uint8)
    for op in range(12):
        for k, length in enumerate((1, 3, 17, 64, 333, 2048)):
            case = cl.fdsp_case(500 + 13 * op + k, op, length)
            assert refrec.same(raw(*cl.orc_fdsp(op, *case, length)), lambda: raw(*cl.ref_fdsp(op, *case, length))), (cl.FDSP_OPS[op], length)


# ---------------------------------------------------------------------------------------------- simple IDCT, 10 / 12 bit
def test_idct_hbd_oracle_golden():
    g = np.load(os.path.join(G, "idct_hbd.npz"))
    for depth in (10, 12):
        blocks = cl.idct_hbd_blocks(70 + depth, depth, 60)
        dest = np.random.default_rng(depth).integers(0, 1 << depth, (8, 60 * 8), dtype=np.uint16)
        for kind in (0, 1, 2):
            b, o = cl.orc_idct_hbd(depth, kind, blocks, dest, dest.strides[0])
            assert np.array_equal(b if kind == 0 else o, g[f"d{depth}_k{kind}"]), (depth, kind)
            assert o.max() < (1 << depth)


def test_idct_hbd_oracle_vs_ref(refrec):
    raw = lambda b, d: np.frombuffer(b.tobytes() + d.tobytes(), np.uint8)
    for depth in (10, 12):
        for kind in (0, 1, 2):
            blocks = cl.idct_hbd_blocks(200 + depth + kind, depth, 300)
            dest = np.random.default_rng(kind).integers(0, 1 << depth, (8, 300 * 8 + 5), dtype=np.uint16)
            got = raw(*cl.orc_idct_hbd(depth, kind, blocks, dest, dest.strides[0]))
            assert refrec.same(got, lambda: raw(*cl.ref_idct_hbd(depth, kind, blocks, dest, dest.strides[0]))), (depth, kind)
    # 9-bit content gets the 10-bit functions (idctdsp.c:248)
    blocks = cl.idct_hbd_blocks(9, 10, 30)
    dest = np.zeros((8, 240), np.uint16)
    assert refrec.same(cl.orc_idct_hbd(10, 1, blocks, dest, 480)[1], lambda: cl.ref_idct_hbd(9, 1, blocks, dest, 480)[1])


# ---------------------------------------------------------------------------------------------- tx: compound 15 x M MDCT
def test_tx_pfa15_oracle_golden_bitexact():
    """ff_tx_mdct_pfa_15xM_{inv,fwd}_float_c at the Opus CELT sizes against the reference's outputs, bit for bit"""
    g = np.load(os.path.join(G, "tx_pfa.npz"))
    O = cl.oracle()
    for n in (120, 240, 480, 960, 112, 448, 144, 576):                # 15 x M, then 7 x M and 9 x M
        for inv in (1, 0):
            for j, sc in enumerate((1.0 / n, -1.0)):
                got = _tx(O, "orc", 1, inv, n, sc, g[f"in_{n}_{inv}"], n)
                assert np.array_equal(got.view(np.uint32), g[f"out_{n}_{inv}_{j}"].view(np.uint32)), (n, inv, j)


def test_tx_pfa15_oracle_vs_ref_and_round_trip():
    O = cl.oracle()
    rng = np.random.default_rng(12)
    if cl.have_ref():
        R = cl.ref()
        for n in (60, 120, 480, 1920, 3840, 28, 56, 1792, 7168, 36, 72, 2304, 9216):    # 15 x M; 7 x M; 9 x M
            for inv in (1, 0):
                x = (rng.random((2, n if inv else 2 * n), dtype=np.float32) * 2 - 1).astype(np.float32)
                for sc in (1.0, -1.0 / 32768):
                    assert np.array_equal(_tx(R, "ffref", 1, inv, n, sc, x, n).view(np.uint32), _tx(O, "orc", 1, inv, n, sc, x, n).view(np.uint32)), (n, inv, sc)
    # forward (scale 1) then inverse (scale 1/n) of a windowless frame gives back x - reversed(x) pattern: check energy relation instead:
    n = 480
    x = (rng.random((1, 2 * n), dtype=np.float32) * 2 - 1).astype(np.float32)
    coef = _tx(O, "orc", 1, 0, n, 1.0, x, n)
    ref = np.zeros(n)
    k = np.arange(n)
    for i in range(2 * n):                                          # direct MDCT definition, float64
        ref += x[0, i] * np.cos(np.pi / n * (i + 0.5 + n / 2) * (k + 0.5))
    assert np.allclose(coef[0], ref, atol=2e-3), float(np.abs(coef[0] - ref).max())


def test_h264qpel_hbd_oracle_golden_and_ref():
    """h264qpel for 9 / 10 / 12 / 14 bit samples: the restatement against the hashes of the compiled reference's outputs (every position,
    size, put / avg, a random and a two-level picture per depth), and live against the compiled reference when it is here"""
    import hashlib
    O = cl.oracle()
    sig = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_ssize_t]
    O.orc_h264qpel_hbd.argtypes = sig
    R = cl.ref() if cl.have_ref() else None
    if R:
        R.ffref_h264qpel_hbd.argtypes = sig
    n = 0
    pics = {}
    for line in open(os.path.join(G, "pel_hbd_hashes.txt")):
        depth, kind, avg, si, pos, h = line.split()
        depth, kind, avg, si, pos = int(depth), int(kind), int(avg), int(si), int(pos)
        if (depth, kind) not in pics:
            pics[(depth, kind)] = cl.hbd_picture(depth, kind)
        img, d0 = pics[(depth, kind)]
        d = d0.copy()
        off = (8 * 64 + 8) * 2
        O.orc_h264qpel_hbd(depth, avg, si, pos, d.ctypes.data + off, img.ctypes.data + off, 128)
        assert hashlib.sha256(d.tobytes()).hexdigest() == h, line
        size = 16 >> si
        assert np.array_equal(d[:8], d0[:8]) and np.array_equal(d[8 + size:], d0[8 + size:]) and np.array_equal(d[:, 8 + size:], d0[:, 8 + size:])
        if R and n % 5 == 0:
            r = d0.copy()
            R.ffref_h264qpel_hbd(depth, avg, si, pos, r.ctypes.data + off, img.ctypes.data + off, 128)
            assert np.array_equal(r, d), line
        n += 1
    assert n == 4 * 2 * 96


def hbd_chroma_rows():
    rows = []
    for line in open(os.path.join(G, "pel_hbd_chroma_hashes.txt")):
        t = line.split()
        rows.append((t[0],) + tuple(int(v) for v in t[1:-1]) + (t[-1],))
    return rows


def test_h264chroma_and_edge_hbd_oracle_golden():
    """h264chroma and emulated_edge_mc for 16-bit samples: the restatement against the hashes of the compiled reference's outputs"""
    import hashlib
    O = cl.oracle()
    O.orc_h264chroma_hbd.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_ssize_t, C.c_int, C.c_int, C.c_int]
    O.orc_emulated_edge_mc_hbd.argtypes = [C.c_void_p, C.c_void_p, C.c_ssize_t, C.c_ssize_t] + [C.c_int] * 6
    pics = {}
    nc = ne = 0
    for row in hbd_chroma_rows():
        if row[0] == "c":
            _, depth, avg, idx, x, y, h, hsh = row
            img, d0 = pics.setdefault(depth, cl.hbd_picture(depth, 0))
            d = d0.copy()
            off = (8 * 64 + 8) * 2
            O.orc_h264chroma_hbd(avg, idx, d.ctypes.data + off, img.ctypes.data + off, 128, h, x, y)
            assert hashlib.sha256(d.tobytes()).hexdigest() == hsh, row[:7]
            nc += 1
        else:
            _, bw, bh, sx, sy, hsh = row
            pic, _ = pics.setdefault(10, cl.hbd_picture(10, 0))
            out = np.zeros((bh, bw + 3), np.uint16)
            O.orc_emulated_edge_mc_hbd(out.ctypes.data, pic.ctypes.data + sy * pic.strides[0] + sx * 2, out.strides[0], pic.strides[0], bw, bh, sx, sy, 64, 48)
            assert hashlib.sha256(out.tobytes()).hexdigest() == hsh, row[:5]
            ne += 1
    assert nc == 2 * 384 and ne == 80


def run_weight_hbd_case(weight_fn, biweight_fn, depth, case):
    bi, idx, h, d, wd, ws, off = case
    img, d0 = cl.hbd_picture(depth, 0)
    blk = d0.copy()
    o = (8 * 64 + 8) * 2
    if bi:
        biweight_fn(depth, idx, blk.ctypes.data + o, img.ctypes.data + o, 128, h, d, wd, ws, off)
    else:
        weight_fn(depth, idx, blk.ctypes.data + o, 128, h, d, wd, off)
    return blk


def weight_hbd_hashes():
    out = {}
    for line in open(os.path.join(G, "h264_weight_hbd_hashes.txt")):
        depth, k, h = line.split()
        out[(int(depth), int(k))] = h
    return out


def test_h264_weight_hbd_oracle_golden():
    """weight / biweight for 9 / 10 / 12 / 14 bit samples against the hashes of the compiled reference's outputs"""
    import hashlib
    O = cl.oracle()
    O.orc_h264_weight_hbd.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_ssize_t] + [C.c_int] * 4
    O.orc_h264_biweight_hbd.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_ssize_t] + [C.c_int] * 5
    hs = weight_hbd_hashes()
    assert len(hs) == 240
    for depth in (9, 10, 12, 14):
        for k, case in enumerate(cl.hbd_weight_cases(depth)):
            blk = run_weight_hbd_case(O.orc_h264_weight_hbd, O.orc_h264_biweight_hbd, depth, case)
            assert hashlib.sha256(blk.tobytes()).hexdigest() == hs[(depth, k)], (depth, case)


def h264_idct_hbd_hashes():
    out = {}
    for line in open(os.path.join(G, "h264_idct_hbd_hashes.txt")):
        depth, kind, k, h = line.split()
        out[(int(depth), int(kind), int(k))] = h
    return out


def run_h264_idct_hbd_case(fn, depth, kind, case):
    """fn(depth, kind, dst address, block address, stride bytes); returns sha256 of (picture, block left behind)"""
    import hashlib
    blk, dst = case
    b, d = blk.copy(), dst.copy()
    fn(depth, kind, d.ctypes.data + (2 * 16 + 4) * 2, b.ctypes.data, 32)
    return hashlib.sha256(np.concatenate([d.view(np.uint8).ravel(), b.view(np.uint8).ravel()]).tobytes()).hexdigest()


def test_h264_idct_hbd_oracle_golden():
    """H.264 residual adds for 9 / 10 / 12 / 14 bit samples (int32 coefficients) against the hashes of the compiled reference's outputs"""
    O = cl.oracle()
    O.orc_h264_idct_hbd.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_ssize_t]
    hs = h264_idct_hbd_hashes()
    assert len(hs) == 4 * 4 * 24
    for depth in (9, 10, 12, 14):
        for kind in range(4):
            for k, case in enumerate(cl.h264_idct_hbd_cases(depth, kind)):
                assert run_h264_idct_hbd_case(O.orc_h264_idct_hbd, depth, kind, case) == hs[(depth, kind, k)], (depth, kind, k)


def h264lf_hbd_hashes():
    return {int(l.split()[0]): l.split()[1] for l in open(os.path.join(G, "h264lf_hbd_hashes.txt"))}


def test_h264_loop_filter_hbd_oracle_golden_and_ref():
    """H.264 deblocking for 9 / 10 / 12 / 14 bit samples: 1024 edges of all 16 kinds per depth against the hash of the compiled reference's
    picture, and live on another seed when the reference is here"""
    import hashlib
    hs = h264lf_hbd_hashes()
    for depth in (9, 10, 12, 14):
        case = cl.h264lf_hbd_case(50 + depth, 1024, depth)
        out = cl.orc_h264lf_hbd(depth, *case)
        assert hashlib.sha256(out.tobytes()).hexdigest() == hs[depth], depth
        assert int((out != case[0]).sum()) > 3000                     # the filters did fire
        if cl.have_ref():
            case = cl.h264lf_hbd_case(90 + depth, 512, depth)
            assert np.array_equal(cl.orc_h264lf_hbd(depth, *case), cl.ref_h264lf_hbd(depth, *case)), depth


def txd_hashes():
    out = {}
    for line in open(os.path.join(G, "tx_double_hashes.txt")):
        typ, n, inv, sc, h = line.split()
        out[(int(typ), int(n), int(inv), float(sc))] = h
    return out


def test_tx_double_oracle_golden_and_ref():
    """AV_TX_DOUBLE_FFT / AV_TX_DOUBLE_MDCT: the double-precision restatement against the hashes of the compiled reference's outputs (and live)"""
    import hashlib
    O = cl.oracle()
    O.orc_txd_open.restype, O.orc_txd_open.argtypes = C.c_void_p, [C.c_int, C.c_int, C.c_int, C.c_double, C.c_uint]
    O.orc_txd_run.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_ssize_t, C.c_int, C.c_ssize_t, C.c_ssize_t]
    O.orc_txd_close.argtypes = [C.c_void_p]
    hs = txd_hashes()
    assert len(hs) == len(cl.txd_cases())
    for (typ, n, inv, sc) in cl.txd_cases():
        x = cl.txd_input(typ, n, inv)
        out = np.zeros((x.shape[0], 2 * n if typ == 2 else n))
        h = O.orc_txd_open(typ, inv, n, sc, 0)
        assert h
        xin = x.copy()
        O.orc_txd_run(h, out.ctypes.data, xin.ctypes.data, 16 if typ == 2 else 8, x.shape[0], out.strides[0], xin.strides[0])
        O.orc_txd_close(h)
        assert hashlib.sha256(out.tobytes()).hexdigest() == hs[(typ, n, inv, sc)], (typ, n, inv, sc)
        if typ == 2 and n >= 16:                                    # it is a DFT
            z = x[0, 0::2] + 1j * x[0, 1::2]
            ref = np.fft.ifft(z) * n if inv else np.fft.fft(z)
            assert np.abs(out[0, 0::2] - ref.real).max() < 1e-9 * n and np.abs(out[0, 1::2] - ref.imag).max() < 1e-9 * n
    assert not O.orc_txd_open(2, 0, 96, 1.0, 0) and not O.orc_txd_open(3, 1, 2, 1.0, 0)


PFA_FFT_SIZES = (6, 12, 96, 10, 160, 14, 224, 18, 288, 30, 120, 960, 1920)


def test_tx_pfa_fft_oracle_golden_bitexact():
    """compound complex FFTs (ff_tx_fft_pfa over fftN_ns x 2^k; checkasm lengths 120 / 960 / 1920) against the reference's outputs, bit
    for bit; the fixture also records the codelet tree the reference chose, which is what the restatement assumes"""
    g = np.load(os.path.join(G, "tx_pfa_fft.npz"))
    O = cl.oracle()
    trees = dict(t.split(": ", 1) for t in g["trees"])
    for n in PFA_FFT_SIZES:
        m = n & -n
        for inv in (0, 1):
            tree = trees[f"{n} {inv}"]
            assert f"fft_pfa_float_c {n} " in tree and f"fft{n // m}_ns_float_c {n // m} " in tree and f"fft{m}_ns_float_c {m} " in tree, tree
            got = _tx(O, "orc", 0, inv, n, 1.0, g[f"in_{n}"], 2 * n)
            assert np.array_equal(got.view(np.uint32), g[f"out_{n}_{inv}"].view(np.uint32)), (n, inv)
    assert not O.orc_tx_open(0, 0, 90, 1.0, 0) and not O.orc_tx_open(0, 0, 75, 1.0, 0) and not O.orc_tx_open(0, 0, 15, 1.0, 0)   # nested / naive trees: not restated


def test_tx_pfa_fft_oracle_vs_ref_and_dft():
    O = cl.oracle()
    rng = np.random.default_rng(13)
    if cl.have_ref():
        R = cl.ref()
        for n in (24, 48, 192, 384, 768, 20, 40, 80, 320, 28, 56, 448, 36, 72, 576, 60, 240, 480, 3840, 7680):
            for inv in (0, 1):
                x = (rng.random((2, 2 * n), dtype=np.float32) * 2 - 1).astype(np.float32)
                assert np.array_equal(_tx(R, "ffref", 0, inv, n, 1.0, x, 2 * n).view(np.uint32), _tx(O, "orc", 0, inv, n, 1.0, x, 2 * n).view(np.uint32)), (n, inv)
    for n in (120, 960, 224):                                       # it is a DFT (eps like checkasm av_tx.c:27), and forward then inverse = len * x
        x = (rng.random((1, 2 * n), dtype=np.float32) * 2 - 1).astype(np.float32)
        z = x[0, 0::2].astype(np.float64) + 1j * x[0, 1::2].astype(np.float64)
        got = _tx(O, "orc", 0, 0, n, 1.0, x, 2 * n)
        ref = np.fft.fft(z)
        assert np.abs(got[0, 0::2] - ref.real).max() < 5e-4 * n and np.abs(got[0, 1::2] - ref.imag).max() < 5e-4 * n
        back = _tx(O, "orc", 0, 1, n, 1.0, got.copy(), 2 * n)
        assert np.abs(back[0] / n - x[0]).max() < 1e-4


def test_tx_full_imdct_oracle_golden_and_ref():
    """AV_TX_FULL_IMDCT (ff_tx_mdct_inv_full: cook, atrac3, atrac3+, dolby_e, dca_lbr ask for it): 2 * len outputs, power-of-two and
    compound lengths, against the reference's outputs; refused for anything but the inverse MDCT, like av_tx_init does"""
    g = np.load(os.path.join(G, "tx_full_imdct.npz"))
    O = cl.oracle()
    for n in (4, 64, 256, 1024, 120, 144):
        for j, sc in enumerate((1.0 / n, -1.0)):
            got = _tx(O, "orc", 1, 1, n, sc, g[f"in_{n}"], 2 * n, flags=4)
            assert np.array_equal(got.view(np.uint32), g[f"out_{n}_{j}"].view(np.uint32)), (n, j)
    assert not O.orc_tx_open(1, 0, 64, 1.0, 4) and not O.orc_tx_open(0, 1, 64, 1.0, 4) and not O.orc_tx_open(6, 1, 64, 1.0, 4)
    if cl.have_ref():
        R = cl.ref()
        rng = np.random.default_rng(19)
        assert not R.ffref_tx_open(1, 0, 64, 1.0, 4) and not R.ffref_tx_open(0, 1, 64, 1.0, 4)
        for n in (8, 128, 2048, 32768, 960, 112, 96, 640):
            x = (rng.random((2, n), dtype=np.float32) * 2 - 1).astype(np.float32)
            for sc in (1.0, -1.0 / 32768):
                a, b = _tx(R, "ffref", 1, 1, n, sc, x, 2 * n, flags=4), _tx(O, "orc", 1, 1, n, sc, x, 2 * n, flags=4)
                assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), (n, sc)
    # the middle half is the plain inverse MDCT
    x = g["in_256"]
    full, half = _tx(O, "orc", 1, 1, 256, 1.0, x, 512, flags=4), _tx(O, "orc", 1, 1, 256, 1.0, x, 256)
    assert np.array_equal(full[:, 128:384].view(np.uint32), half.view(np.uint32))
    assert np.array_equal(full[:, :128], -half[:, 127::-1]) and np.array_equal(full[:, 384:], half[:, :127:-1])


# ---------------------------------------------------------------------------------------------- tx: DCT-II / DCT-III
def _dct(L, pre, inv, asked, sc, x_padded, n):
    h = getattr(L, pre + "_tx_open")(9, inv, asked, sc, 0)
    assert h
    out, xin = np.zeros((x_padded.shape[0], n + 2), np.float32), x_padded.copy()
    getattr(L, pre + "_tx_run")(h, out.ctypes.data, xin.ctypes.data, 4, x_padded.shape[0], out.strides[0], xin.strides[0])
    getattr(L, pre + "_tx_close")(h)
    return out[:, :n]


def test_tx_dct_oracle_golden_and_definition():
    """ff_tx_dctII / ff_tx_dctIII against the reference's outputs bit for bit, and against the textbook DCT-II"""
    g = np.load(os.path.join(G, "tx_dct.npz"))
    O = cl.oracle()
    for n in (8, 64, 512):
        for inv, asked in ((0, n), (1, n // 2)):
            for j, sc in enumerate((1.0, 0.5 / n)):
                got = _dct(O, "orc", inv, asked, sc, g[f"in_{n}"], n)
                assert np.array_equal(got.view(np.uint32), g[f"out_{n}_{inv}_{j}"].view(np.uint32)), (n, inv, j)
    if cl.have_ref():
        R = cl.ref()
        rng = np.random.default_rng(13)
        for n in (4, 16, 256, 2048):
            x = (rng.random((2, n + 2), dtype=np.float32) * 2 - 1).astype(np.float32)
            for inv, asked in ((0, n), (1, n // 2)):
                assert np.array_equal(_dct(R, "ffref", inv, asked, -1.0, x, n).view(np.uint32), _dct(O, "orc", inv, asked, -1.0, x, n).view(np.uint32)), (n, inv)
    n = 64
    x = np.random.default_rng(3).random((1, n + 2)).astype(np.float32)
    k, i = np.arange(n)[:, None], np.arange(n)[None, :]
    ref = (np.cos(np.pi / n * (i + 0.5) * k) * x[0, :n].astype(np.float64)).sum(axis=1)
    got = _dct(O, "orc", 0, n, 1.0, x, n)[0]
    assert np.allclose(got, ref, atol=1e-3) or np.allclose(got, 2 * ref, atol=1e-3) or np.allclose(got, ref / 2, atol=1e-3), float(np.abs(got - ref).max())


# ---------------------------------------------------------------------------------------------- tx: 32-bit fixed point
def _txi(L, pre, typ, inv, n, sc, x, outn):
    if pre == "orc":
        L.orc_txi_open.restype = C.c_void_p
        L.orc_txi_open.argtypes = [C.c_int, C.c_int, C.c_int, C.c_float, C.c_uint]
        L.orc_txi_run.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_ssize_t, C.c_int, C.c_ssize_t, C.c_ssize_t]
        L.orc_txi_close.argtypes = [C.c_void_p]
        op, ru, clo = L.orc_txi_open, L.orc_txi_run, L.orc_txi_close
    else:
        op, ru, clo = L.ffref_tx_open, L.ffref_tx_run, L.ffref_tx_close
    h = op(typ, inv, n, sc, 0)
    assert h
    out, xin = np.zeros((x.shape[0], outn), np.int32), x.copy()
    ru(h, out.ctypes.data, xin.ctypes.data, 8 if typ == 4 else 4, x.shape[0], out.strides[0], xin.strides[0])
    clo(h)
    return out


def test_tx_int32_oracle_golden_and_ref():
    """AV_TX_INT32_FFT / _MDCT (TX_INT32 instantiation of tx_template.c) against the reference's outputs"""
    g = np.load(os.path.join(G, "tx_int32.npz"))
    O = cl.oracle()
    for n in (8, 64, 1024):
        x = g[f"in_{n}"]
        xs = (x >> 6).astype(np.int32)
        for inv in (0, 1):
            assert np.array_equal(_txi(O, "orc", 4, inv, n, 1.0, x, 2 * n), g[f"fft_{n}_{inv}"]), (n, inv)
        for j, sc in enumerate((1.0 / n, -1.0 / 32768)):
            for inv in (1, 0):
                xi = np.ascontiguousarray(xs[:, :n]) if inv else xs
                assert np.array_equal(_txi(O, "orc", 5, inv, n, sc, xi, n), g[f"mdct_{n}_{inv}_{j}"]), (n, inv, j)
    if cl.have_ref():
        R = cl.ref()
        rng = np.random.default_rng(14)
        for n in (2, 4, 16, 32, 256, 2048):
            x = rng.integers(-(1 << 31), 1 << 31, (2, 2 * n)).astype(np.int32)
            for inv in (0, 1):
                assert np.array_equal(_txi(R, "ffref", 4, inv, n, 1.0, x, 2 * n), _txi(O, "orc", 4, inv, n, 1.0, x, 2 * n)), (n, inv)
            if n >= 8:
                for inv in (1, 0):
                    xi = np.ascontiguousarray((x >> 5)[:, :n]) if inv else (x >> 5)
                    assert np.array_equal(_txi(R, "ffref", 5, inv, n, 1.0, xi, n), _txi(O, "orc", 5, inv, n, 1.0, xi, n)), (n, inv)


# ---------------------------------------------------------------------------------------------- ProresDSPContext
def test_prores_idct_put_oracle_golden_and_ref():
    g = np.load(os.path.join(G, "prores.npz"))
    for bits in (10, 12):
        for seed in (0, 1, 2):
            blocks, qmat = cl.prores_case(90 + seed, bits, 60)
            b, px = cl.orc_prores(bits, blocks, qmat, np.zeros((8, 60 * 8), np.uint16), 60 * 16)
            assert np.array_equal(px, g[f"b{bits}_s{seed}"]), (bits, seed)
            assert px.min() >= 4 and px.max() <= (1 << bits) - 5
        if cl.have_ref():
            blocks, qmat = cl.prores_case(300 + bits, bits, 400)
            dest = np.zeros((8, 400 * 8 + 3), np.uint16)
            (b1, d1), (b2, d2) = cl.ref_prores(bits, blocks, qmat, dest, dest.strides[0]), cl.orc_prores(bits, blocks, qmat, dest, dest.strides[0])
            assert np.array_equal(d1, d2) and np.array_equal(b1, b2), bits


# ---------------------------------------------------------------------------------------------- H.264 deblocking filters
def test_h264_loop_filter_oracle_golden_and_ref(refrec):
    """oracle/h264lf_oracle.c against the reference's ff_h264dsp_init(8, 1 / 2) loop filters: fixture hashes, then bit-exact over 16
    kinds x noisy / smooth content x the whole alpha / beta / tc0 range (tc0 = -1 skips a group, 0 filters p0 / q0 only)"""
    import hashlib
    g = np.load(os.path.join(G, "h264lf.npz"))
    for seed in (0, 1, 2):
        case = cl.h264lf_case(40 + seed, 512)
        out = cl.orc_h264lf(*case)
        assert hashlib.sha256(out.tobytes()).digest() == g[f"sha_{seed}"].tobytes(), seed
        if seed == 0:
            assert np.array_equal(out[:64], g["head_0"])
    for seed in (7, 8):
        case = cl.h264lf_case(seed, 2048)
        a = cl.orc_h264lf(*case)
        assert refrec.same(a, lambda: cl.ref_h264lf(*case)) and not np.array_equal(a, case[0])
    # nothing outside p2..q2 of the edge's own lines is ever written
    pic, kinds, off, alpha, beta, tc0 = cl.h264lf_case(9, 256)
    out = cl.orc_h264lf(pic, kinds, off, alpha, beta, tc0)
    keep = np.ones(pic.shape, bool)
    for e in range(256):
        y, x = divmod(int(off[e]), pic.strides[0])
        vert = kinds[e] in (0, 3, 6, 9)
        if vert:
            keep[y - 3:y + 3, x:x + 16] = False
        else:
            keep[y:y + 16, x - 3:x + 3] = False
    assert np.array_equal(out[keep], pic[keep])


# ---------------------------------------------------------------------------------------------- av_pixelutils_get_sad_fn
def test_pixelutils_sad_oracle_golden_and_ref():
    g = np.load(os.path.join(G, "pixelutils.npz"))
    for bits in range(1, 6):
        case = cl.pixelutils_case(50 + bits, bits, 200)
        got = cl.orc_pixelutils(bits, *case)
        assert np.array_equal(got, g[f"sad_{bits}"]) and got.min() >= 0 and got[0] < got[1:].max()
        if cl.have_ref():
            case = cl.pixelutils_case(150 + bits, bits, 500)
            assert np.array_equal(cl.orc_pixelutils(bits, *case), cl.ref_pixelutils(bits, *case)), bits
    f = np.zeros((64, 64), np.uint8)
    for bits in (0, 6):                                                   # no such block size: the reference returns NULL
        assert cl.oracle().orc_pixelutils_sad(bits, f.ctypes.data, 64, f.ctypes.data, 64) == -1
        if cl.have_ref():
            assert cl.ref().ffref_pixelutils_sad(bits, f.ctypes.data, 64, f.ctypes.data, 64) == -1


# ---------------------------------------------------------------------------------------------- IDCT accuracy (libavcodec/tests/dct.c)
def _ref_dct_matrix():
    c = np.zeros((8, 8))
    c[0, :] = np.sqrt(0.125)                                              # ff_ref_dct_init, libavcodec/dctref.c:40-50
    for i in range(1, 8):
        c[i, :] = 0.5 * np.cos(i * (np.arange(8) + 0.5) * np.pi / 8)
    return c


def test_idct_accuracy_like_reference_dct_test():
    """The accuracy criteria of the reference's own IDCT test (libavcodec/tests/dct.c:176-270, 20000 blocks per input class)
    applied to the checker's 8-bit simple IDCT, and — 10 / 12 bit use the same test with more input bits there — to the 10-bit
    one: double-precision reference transform with its rounding (dctref.c:60-125), peak error <= 1, mean square error <= 0.02,
    mean error <= 0.0015 (class 2), per-coefficient square error <= 0.06 and systematic error <= 0.015 (classes 0 and 1)."""
    O = cl.oracle()
    cm = _ref_dct_matrix()
    n = 20000
    for bits, run in ((8, "orc8"), (10, "orc10")):
        vals = 1 << bits
        rng = np.random.default_rng(bits)
        for test in (0, 1, 2):
            blocks = np.zeros((n, 8, 8), np.int64)
            if test == 0:                                                 # spatial noise, forward reference DCT, >> 3
                px = rng.integers(-vals, vals, (n, 8, 8))
                out = np.einsum("ik,nkj->nij", cm, px.astype(np.float64)) * 8
                blocks = np.floor(np.einsum("nik,jk->nij", out, cm) + 0.499999999999).astype(np.int64) >> 3
            elif test == 1:                                               # 1 ... 10 non-zero coefficients
                flat = blocks.reshape(n, 64)
                for b in range(n):
                    k = int(rng.integers(1, 11))
                    flat[b, rng.integers(0, 64, k)] = rng.integers(-vals, vals, k)
            else:                                                         # DC plus the parity coefficient
                blocks[:, 0, 0] = rng.integers(-8 * vals, 8 * vals, n)
                blocks[:, 7, 7] = (blocks[:, 0, 0] & 1) ^ 1
            b16 = np.ascontiguousarray(blocks.reshape(n, 64).astype(np.int16))
            exp = np.floor(np.einsum("ki,nkj->nij", cm, np.einsum("nik,kj->nij", b16.reshape(n, 8, 8).astype(np.float64), cm)) + 0.5)
            got = b16.copy()
            if run == "orc8":
                for b in range(n):
                    O.orc_idct(cl.ptr(got[b], cl.i16p))
            else:
                got, _ = cl.orc_idct_hbd(10, 0, b16, np.zeros((8, 8), np.uint16), 16)
            err = got.reshape(n, 64).astype(np.int64) - exp.reshape(n, 64).astype(np.int64)
            err_inf, omse, ome = int(np.abs(err).max()), float((err ** 2).mean()), float(err.mean())
            per_coef_sq, per_coef_sys = float((err ** 2).sum(0).max()) / n, float(np.abs(err.sum(0)).max()) / n
            if test < 2:
                assert per_coef_sq <= 0.06 and per_coef_sys <= 0.015, (bits, test, per_coef_sq, per_coef_sys)
            else:
                assert err_inf <= 1 and omse <= 0.02 and abs(ome) <= 0.0015, (bits, test, err_inf, omse, ome)


def test_mecmp_round2_families_oracle_vs_fixture_and_reference():
    """vsad / vsse (+ intra), nsse, median_sad, hadamard8_intra, sum_abs_dctelem: the checker against the committed reference values
    (tests/golden/mecmp2.npz, scripts/gen_golden_mecmp2.py) and, where it is built, against the compiled reference on fresh inputs."""
    O = cl.oracle()
    O.orc_sum_abs_dctelem.argtypes = [cl.i16p]
    g = np.load(os.path.join(G, "mecmp2.npz"))
    img1, img2 = g["img1"], g["img2"]
    for fn, idx, x1, y1, x2, y2, h, v in g["cases"]:
        got = O.orc_me_cmp(int(fn), int(idx), C.cast(img1.ctypes.data + int(y1) * 64 + int(x1), cl.u8p),
                           C.cast(img2.ctypes.data + int(y2) * 64 + int(x2), cl.u8p), 64, int(h))
        assert got == v, (fn, idx, h)
    for b, v in zip(g["blocks"], g["sums"]):
        assert O.orc_sum_abs_dctelem(cl.ptr(np.ascontiguousarray(b), cl.i16p)) == v
    if not cl.have_ref():
        return
    R = cl.ref()
    rng = np.random.default_rng(31)
    for trial in range(60):
        a = rng.integers(0, 256, (40, 96), dtype=np.uint8)
        b = rng.integers(0, 256, (40, 96), dtype=np.uint8) if trial % 2 else (a.astype(int) + rng.integers(-2, 3, a.shape)).clip(0, 255).astype(np.uint8)
        p1, p2 = C.cast(a.ctypes.data + 96 * 2 + 8, cl.u8p), C.cast(b.ctypes.data + 96 * 3 + 5, cl.u8p)
        for fn, idxs in ((3, (4, 5)), (4, (0, 1, 4, 5)), (5, (0, 1, 4, 5)), (6, (0, 1)), (7, (0, 1))):
            for idx in idxs:
                for h in (8, 16):
                    assert R.ffref_me_cmp(fn, idx, p1, p2, 96, h) == O.orc_me_cmp(fn, idx, p1, p2, 96, h), (fn, idx, h)


def mecmp_dct_pairs():
    """the image pairs of tests/golden/mecmp_dct.npz (scripts/gen_golden.py mecmp_dct): mecmp.npz's random images, a checkerboard against its
    inverse, white against black"""
    g = np.load(os.path.join(G, "mecmp.npz"))
    chk = ((np.add.outer(np.arange(64), np.arange(64)) & 1) * 255).astype(np.uint8)
    return [(g["img1"], g["img2"]), (chk, np.ascontiguousarray(255 - chk)), (np.full((64, 64), 255, np.uint8), np.zeros((64, 64), np.uint8))]


def test_mecmp_dct_families_oracle_vs_fixture_and_reference():
    """dct_sad / dct_max (islow and ifast DCT) and dct264_sad: the checker against the committed reference values and, where the reference is
    built, against it on fresh inputs (random, near-equal, binary)"""
    O = cl.oracle()
    pairs = mecmp_dct_pairs()
    try:
        for fn, idx, algo, pi, x1, y1, x2, y2, h, v in np.load(os.path.join(G, "mecmp_dct.npz"))["cases"]:
            O.orc_me_cmp_set_dct_algo(int(algo))
            img1, img2 = pairs[int(pi)]
            got = O.orc_me_cmp(int(fn), int(idx), C.cast(img1.ctypes.data + int(y1) * 64 + int(x1), cl.u8p),
                               C.cast(img2.ctypes.data + int(y2) * 64 + int(x2), cl.u8p), 64, int(h))
            assert got == v, (fn, idx, algo, pi, h)
        if not cl.have_ref():
            return
        R = cl.ref()
        rng = np.random.default_rng(77)
        for algo in (0, 1):
            O.orc_me_cmp_set_dct_algo(algo); R.ffref_me_cmp_set_dct_algo(algo)
            for trial in range(300):
                a = rng.integers(0, 256, (24, 40), dtype=np.uint8) if trial % 3 else (rng.integers(0, 2, (24, 40)) * 255).astype(np.uint8)
                b = rng.integers(0, 256, (24, 40), dtype=np.uint8) if trial % 2 else (a.astype(int) + rng.integers(-3, 4, a.shape)).clip(0, 255).astype(np.uint8)
                p1, p2 = C.cast(a.ctypes.data + 40 * 2 + 3, cl.u8p), C.cast(b.ctypes.data + 40 * 5 + 7, cl.u8p)
                for fn in (8, 9, 10):
                    for idx, h in ((0, 16), (0, 8), (1, 8)):
                        assert R.ffref_me_cmp(fn, idx, p1, p2, 40, h) == O.orc_me_cmp(fn, idx, p1, p2, 40, h), (algo, fn, idx, h)
    finally:
        O.orc_me_cmp_set_dct_algo(0)
        if cl.have_ref():
            cl.ref().ffref_me_cmp_set_dct_algo(0)


def fdct_hashes():
    return {tuple(int(v) for v in l.split()[:3]): l.split()[3] for l in open(os.path.join(G, "fdct_hashes.txt"))}


def test_fdct_oracle_vs_fixture_and_reference():
    """FDCTDSPContext.fdct / fdct248 (islow 8 / 10 bit, ifast): the checker against the hashes of the compiled reference's outputs
    (tests/golden/fdct_hashes.txt, scripts/gen_golden.py fdct) and, where the reference is built, block by block on other inputs"""
    import hashlib
    from test_cuda_emu import fdct_blocks
    O = cl.oracle()
    for (algo, bits, is248), h in fdct_hashes().items():
        kind = 2 if bits in (9, 10) else 1 if algo == 1 else 0
        x = fdct_blocks(bits, 200, 7000 + 10 * algo + bits + is248)
        for i in range(x.shape[0]):
            O.orc_fdct(kind, is248, cl.ptr(x[i], cl.i16p))
        assert hashlib.sha256(x.tobytes()).hexdigest() == h, (algo, bits, is248)
    if not cl.have_ref():
        return
    R = cl.ref()
    for algo, bits, kind in ((0, 8, 0), (2, 8, 0), (1, 8, 1), (0, 10, 2), (1, 9, 2)):
        for is248 in (0, 1):
            x = fdct_blocks(bits, 400, 31 + algo + bits + is248)
            for i in range(x.shape[0]):
                e, r = x[i].copy(), x[i].copy()
                O.orc_fdct(kind, is248, cl.ptr(e, cl.i16p)); R.ffref_fdct(algo, bits, is248, cl.ptr(r, cl.i16p))
                assert np.array_equal(e, r), (algo, bits, is248, i)
