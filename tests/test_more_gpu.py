"""GPU tier: me_cmp / ESA, h264qpel / hpeldsp and float tx CUDA paths (through the C ABI) against the oracle and the
golden fixtures generated from the unmodified reference."""
import ctypes as C
import os

import numpy as np
import pytest

import cpulibs as cl

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def on_stream(device):
    import torch
    return torch.cuda.stream(torch.cuda.ExternalStream(device.stream))


# ---------------------------------------------------------------------------------------------- me_cmp
def test_mecmp_pointer_table_golden(device):
    """MECmpContext entries called like checkasm motion.c does (NULL context, random offsets, h in {4,8,16})."""
    from ffmpeg_b200 import me_cmp
    from ffmpeg_b200._lib import u8p
    g = np.load(os.path.join(G, "mecmp.npz"))
    c = me_cmp.ff_me_cmp_init()
    img1, img2 = g["img1"], g["img2"]
    assert not c.quant_psnr[0] and not c.sad[2]                # entries not implemented stay NULL
    for fn, idx, x1, y1, x2, y2, h, v in g["cases"]:
        f = c.sad[idx] if fn == 0 else c.sse[idx] if fn == 1 else c.pix_abs[idx >> 2][idx & 3]
        got = f(None, C.cast(img1.ctypes.data + int(y1) * 64 + int(x1), u8p), C.cast(img2.ctypes.data + int(y2) * 64 + int(x2), u8p), 64, int(h))
        assert got == v, (fn, idx, h)


def test_mecmp_batch_vs_oracle(device):
    import torch
    from ffmpeg_b200 import me_cmp
    O = cl.oracle()
    rng = np.random.default_rng(5)
    W, H, n = 256, 128, 3000
    f1 = rng.integers(0, 256, (H, W), dtype=np.uint8)
    f2 = rng.integers(0, 256, (H, W), dtype=np.uint8)
    xs1, ys1, xs2, ys2 = (rng.integers(0, d - 20, n) for d in (W, H, W, H))
    off1 = (ys1 * W + xs1).astype(np.int64)
    off2 = (ys2 * W + xs2).astype(np.int64)
    with on_stream(device):
        d1, d2 = torch.from_numpy(f1).cuda(), torch.from_numpy(f2).cuda()
        o1, o2 = torch.from_numpy(off1).cuda(), torch.from_numpy(off2).cuda()
        out = torch.zeros(n, dtype=torch.int32, device="cuda")
        for fn, idxs in ((0, (0, 1)), (1, (0, 1, 2)), (2, range(8))):
            for idx in idxs:
                for h in (4, 8, 16):
                    me_cmp.me_cmp_batch_device(device, fn, idx, d1, d2, W, h, o1, o2, n, out)
                    device.sync()
                    got = out.cpu().numpy()
                    exp = np.array([O.orc_me_cmp(fn, idx, C.cast(f1.ctypes.data + int(a), cl.u8p), C.cast(f2.ctypes.data + int(b), cl.u8p), W, h)
                                    for a, b in zip(off1[:400], off2[:400])])
                    assert np.array_equal(got[:400], exp), (fn, idx, h)


def test_mecmp_round2_families(device):
    """vsad / vsse (+ intra), nsse, median_sad, hadamard8_intra, sum_abs_dctelem: drop-in entries against the reference fixture
    (NULL context like checkasm), batched entry against the oracle."""
    import torch
    from ffmpeg_b200 import me_cmp
    from ffmpeg_b200._lib import u8p, i16p
    g = np.load(os.path.join(G, "mecmp2.npz"))
    c = me_cmp.ff_me_cmp_init()
    img1, img2 = g["img1"], g["img2"]
    assert not c.quant_psnr[0] and not c.rd[0] and not c.bit[0] and not c.w53[0] and not c.w97[0]         # these run the encoder's quantiser / VLC tables or the snow wavelets: stay NULL
    tabs = {3: c.hadamard8_diff, 4: c.vsad, 5: c.vsse, 6: c.nsse, 7: c.median_sad}
    for fn, idx, x1, y1, x2, y2, h, v in g["cases"]:
        f = tabs[int(fn)][int(idx)]
        got = f(None, C.cast(img1.ctypes.data + int(y1) * 64 + int(x1), u8p), C.cast(img2.ctypes.data + int(y2) * 64 + int(x2), u8p), 64, int(h))
        assert got == v, (fn, idx, h)
    for b, v in zip(g["blocks"][:8], g["sums"][:8]):
        assert c.sum_abs_dctelem(np.ascontiguousarray(b).ctypes.data_as(i16p)) == v
    O = cl.oracle()
    rng = np.random.default_rng(6)
    W, H, n = 256, 128, 2000
    f1 = rng.integers(0, 256, (H, W), dtype=np.uint8)
    f2 = (f1.astype(int) + rng.integers(-9, 10, f1.shape)).clip(0, 255).astype(np.uint8)
    xs1, ys1, xs2, ys2 = (rng.integers(1, d - 20, n) for d in (W, H, W, H))
    off1 = (ys1 * W + xs1).astype(np.int64)
    off2 = (ys2 * W + xs2).astype(np.int64)
    with on_stream(device):
        d1, d2 = torch.from_numpy(f1).cuda(), torch.from_numpy(f2).cuda()
        o1, o2 = torch.from_numpy(off1).cuda(), torch.from_numpy(off2).cuda()
        out = torch.zeros(n, dtype=torch.int32, device="cuda")
        for fn, idxs in ((3, (4, 5)), (4, (0, 1, 4, 5)), (5, (0, 1, 4, 5)), (6, (0, 1)), (7, (0, 1))):
            for idx in idxs:
                for h in (8, 16):
                    me_cmp.me_cmp_batch_device(device, fn, idx, d1, d2, W, h, o1, o2, n, out)
                    device.sync()
                    got = out.cpu().numpy()
                    exp = np.array([O.orc_me_cmp(fn, idx, C.cast(f1.ctypes.data + int(a), cl.u8p), C.cast(f2.ctypes.data + int(b), cl.u8p), W, h)
                                    for a, b in zip(off1[:300], off2[:300])])
                    assert np.array_equal(got[:300], exp), (fn, idx, h)
        blocks = torch.from_numpy(g["blocks"]).cuda()
        so = torch.zeros(blocks.shape[0], dtype=torch.int32, device="cuda")
        me_cmp.sum_abs_dctelem_batch_device(device, blocks, blocks.shape[0], so)
        device.sync()
        assert np.array_equal(so.cpu().numpy(), g["sums"])


def test_satd_pointer_table_and_batch(device):
    """hadamard8_diff (SATD): drop-in entries against the reference fixture, batched entry against the oracle."""
    import torch
    from ffmpeg_b200 import me_cmp
    from ffmpeg_b200._lib import u8p
    g, cases = np.load(os.path.join(G, "mecmp.npz")), np.load(os.path.join(G, "satd.npz"))["cases"]
    c = me_cmp.ff_me_cmp_init()
    img1, img2 = g["img1"], g["img2"]
    for fn, idx, x1, y1, x2, y2, h, v in cases[::3]:
        got = c.hadamard8_diff[idx](None, C.cast(img1.ctypes.data + int(y1) * 64 + int(x1), u8p), C.cast(img2.ctypes.data + int(y2) * 64 + int(x2), u8p), 64, int(h))
        assert got == v, (idx, h)
    O = cl.oracle()
    rng = np.random.default_rng(6)
    W, H, n = 256, 128, 2000
    f1 = rng.integers(0, 256, (H, W), dtype=np.uint8)
    f2 = np.clip(f1.astype(np.int32) + rng.integers(-20, 21, (H, W)), 0, 255).astype(np.uint8)
    off1 = (rng.integers(0, H - 20, n) * W + rng.integers(0, W - 20, n)).astype(np.int64)
    off2 = (rng.integers(0, H - 20, n) * W + rng.integers(0, W - 20, n)).astype(np.int64)
    with on_stream(device):
        d1, d2 = torch.from_numpy(f1).cuda(), torch.from_numpy(f2).cuda()
        o1, o2 = torch.from_numpy(off1).cuda(), torch.from_numpy(off2).cuda()
        out = torch.zeros(n, dtype=torch.int32, device="cuda")
        for idx in (0, 1):
            for h in (8, 16):
                me_cmp.me_cmp_batch_device(device, me_cmp.HADAMARD8, idx, d1, d2, W, h, o1, o2, n, out)
                device.sync()
                got = out.cpu().numpy()
                exp = np.array([O.orc_me_cmp(3, idx, C.cast(f1.ctypes.data + int(a), cl.u8p), C.cast(f2.ctypes.data + int(b), cl.u8p), W, h)
                                for a, b in zip(off1[:500], off2[:500])])
                assert np.array_equal(got[:500], exp), (idx, h)


def gpu_esa(device, cur, ref_, mb, sp):
    import torch
    from ffmpeg_b200 import me_cmp
    nf, H, W = cur.shape
    bw, bh = W // mb, H // mb
    with on_stream(device):
        dc, dr = torch.from_numpy(cur).cuda(), torch.from_numpy(ref_).cuda()
        mv = torch.zeros((nf, bh * bw, 2), dtype=torch.int32, device="cuda")
        cost = torch.zeros((nf, bh * bw), dtype=torch.int64, device="cuda")
        me_cmp.me_esa_device(device, dc, dr, W, W, H, W * H, nf, mb, sp, mv, cost)
        device.sync()
        return mv.cpu().numpy(), cost.cpu().numpy().astype(np.uint64)


def test_esa_golden(device):
    g = np.load(os.path.join(G, "mecmp.npz"))
    W, H = 96, 64
    cur, ref_ = g["esa_cur"], g["esa_ref"]
    flat = np.full((H, W), 99, np.uint8)
    for name, (a, b) in {"shift": (cur, ref_), "flat": (flat, flat), "same": (cur, cur)}.items():
        for mb, sp in ((16, 7), (8, 4), (16, 32), (4, 3)):
            mv, cost = gpu_esa(device, a[None], b[None], mb, sp)
            assert np.array_equal(mv[0], g[f"esa_{name}_{mb}_{sp}_mv"]), (name, mb, sp)
            assert np.array_equal(cost[0], g[f"esa_{name}_{mb}_{sp}_cost"]), (name, mb, sp)


def test_esa_vs_oracle_multi_frame(device):
    """720p-sized frame pairs, +-32 window (BASELINE config 4 geometry at a size the oracle finishes in seconds is too
    slow; use 320x192 for the oracle and check 4K through the minimum-cost property)."""
    O = cl.oracle()
    rng = np.random.default_rng(9)
    nf, W, H, mb, sp = 2, 320, 192, 16, 32
    cur = rng.integers(0, 256, (nf, H, W), dtype=np.uint8)
    ref_ = np.stack([np.roll(cur[i], (5 - 9 * i, -7 + 3 * i), (0, 1)) for i in range(nf)])
    ref_ = (ref_.astype(np.int16) + rng.integers(-2, 3, ref_.shape)).clip(0, 255).astype(np.uint8)
    mv, cost = gpu_esa(device, cur, ref_, mb, sp)
    bw, bh = W // mb, H // mb
    for i in range(nf):
        emv, ec = np.zeros((bh * bw, 2), np.int32), np.zeros(bh * bw, np.uint64)
        O.orc_esa_frame(cl.ptr(cur[i]), cl.ptr(ref_[i]), W, W, H, mb, sp, 0, bh, cl.ptr(emv, cl.i32p), cl.ptr(ec, cl.u64p))
        assert np.array_equal(mv[i], emv) and np.array_equal(cost[i], ec), i


def test_esa_4k_property(device):
    """Full-size 4K pair: the returned cost must equal the SAD at the returned vector and be <= the zero-vector SAD and
    the SAD at a few probe vectors (size-independent property; the oracle would need minutes here)."""
    rng = np.random.default_rng(10)
    W, H, mb, sp = 3840, 2160, 16, 32
    cur = rng.integers(0, 256, (1, H, W), dtype=np.uint8)
    ref_ = np.roll(cur, (0, 11, -6), (0, 1, 2)).copy()
    mv, cost = gpu_esa(device, cur, ref_, mb, sp)
    bw = W // mb
    for b in rng.integers(0, mv.shape[1], 200):
        by, bx = divmod(int(b), bw)
        x_mb, y_mb = bx * mb, by * mb
        blk = cur[0, y_mb:y_mb + mb, x_mb:x_mb + mb].astype(np.int32)
        x, y = mv[0, b]
        sad = lambda xx, yy: int(np.abs(ref_[0, yy:yy + mb, xx:xx + mb].astype(np.int32) - blk).sum())
        assert sad(x, y) == int(cost[0, b])
        assert int(cost[0, b]) <= sad(x_mb, y_mb)
        if 32 <= y_mb <= H - 48 and 32 <= x_mb <= W - 48:
            assert int(cost[0, b]) == 0 and (x, y) == (x_mb - 6, y_mb + 11)        # the true shift is found exactly


# ---------------------------------------------------------------------------------------------- qpel / hpel
def test_pel_pointer_tables_golden(device):
    from ffmpeg_b200 import pel
    from ffmpeg_b200._lib import u8p
    g = np.load(os.path.join(G, "pel.npz"))
    q, hp = pel.ff_h264qpel_init(8), pel.ff_hpeldsp_init(0)
    src, dst0 = g["src"], g["dst0"]
    ps = C.cast(src.ctypes.data + 8 * 48 + 8, u8p)
    for key in g.files:
        if key in ("src", "dst0"):
            continue
        o = dst0.copy()
        po = C.cast(o.ctypes.data + 8 * 48 + 8, u8p)
        parts = [int(v) for v in key.split("_")[1:]]
        if key[0] == "q":
            (q.avg_h264_qpel_pixels_tab if parts[0] else q.put_h264_qpel_pixels_tab)[parts[1]][parts[2]](po, ps, 48)
        else:
            tab = [hp.put_pixels_tab, hp.avg_pixels_tab, hp.put_no_rnd_pixels_tab, None][parts[0]]
            f = hp.avg_no_rnd_pixels_tab[parts[2]] if parts[0] == 3 else tab[parts[1]][parts[2]]
            f(po, ps, 48, parts[3])
        assert np.array_equal(o[8:24, 8:24], g[key]), key
        assert np.array_equal(o[:8], dst0[:8]) and np.array_equal(o[24:], dst0[24:]) and np.array_equal(o[:, :8], dst0[:, :8]), key
    assert not hp.put_no_rnd_pixels_tab[2][0]                  # sizes the reference leaves empty stay NULL


def test_qpel_batch_vs_oracle(device):
    """A macroblock-stream like BASELINE config 3: random quarter-pel positions, put/avg and sizes over a frame."""
    import torch
    from ffmpeg_b200 import pel
    O = cl.oracle()
    rng = np.random.default_rng(12)
    W, H = 640, 368
    ref_ = rng.integers(0, 256, (H, W), dtype=np.uint8)
    dst0 = rng.integers(0, 256, (H, W), dtype=np.uint8)
    ops, doffs, soffs = [], [], []
    for by in range(1, H // 16 - 1):
        for bx in range(1, W // 16 - 1):
            size_idx = int(rng.integers(0, 3))
            op = pel.qpel_op(int(rng.integers(0, 2)), size_idx, int(rng.integers(0, 16)))
            dx, dy = (int(v) for v in rng.integers(-10, 11, 2))
            ops.append(op); doffs.append(by * 16 * W + bx * 16); soffs.append((by * 16 + dy) * W + bx * 16 + dx)
    n = len(ops)
    ops_a, do_a, so_a = np.array(ops, np.uint8), np.array(doffs, np.int64), np.array(soffs, np.int64)
    exp = dst0.copy()
    for op, do, so in zip(ops, doffs, soffs):
        O.orc_h264qpel(op & 1, (op >> 1) & 3, (op >> 3) & 15, C.cast(exp.ctypes.data + do, cl.u8p), C.cast(ref_.ctypes.data + so, cl.u8p), W)
    with on_stream(device):
        d_ops, d_do, d_so = torch.from_numpy(ops_a).cuda(), torch.from_numpy(do_a).cuda(), torch.from_numpy(so_a).cuda()
        d_dst, d_src = torch.from_numpy(dst0).cuda(), torch.from_numpy(ref_).cuda()
        pel.h264qpel_batch_device(device, n, d_ops, d_dst, d_do, d_src, d_so, W)
        device.sync()
        got = d_dst.cpu().numpy()
    assert np.array_equal(got, exp), int((got != exp).sum())


def test_hpel_batch_vs_oracle(device):
    import torch
    from ffmpeg_b200 import pel
    O = cl.oracle()
    rng = np.random.default_rng(13)
    W, H = 320, 192
    ref_ = rng.integers(0, 256, (H, W), dtype=np.uint8)
    dst0 = rng.integers(0, 256, (H, W), dtype=np.uint8)
    ops, hs, doffs, soffs = [], [], [], []
    for by in range(1, H // 16 - 1):
        for bx in range(1, W // 16 - 1):
            tab = int(rng.integers(0, 4))
            sidx = 0 if tab == 3 else int(rng.integers(0, 2)) if tab == 2 else int(rng.integers(0, 4))
            h = int(rng.choice([4, 8, 16] if sidx < 2 else [2, 4, 8]))
            ops.append(pel.hpel_op(tab, sidx, int(rng.integers(0, 4)))); hs.append(h)
            dx, dy = (int(v) for v in rng.integers(-8, 9, 2))
            doffs.append(by * 16 * W + bx * 16); soffs.append((by * 16 + dy) * W + bx * 16 + dx)
    exp = dst0.copy()
    for op, h, do, so in zip(ops, hs, doffs, soffs):
        assert O.orc_hpel(op & 3, (op >> 2) & 3, (op >> 4) & 3, C.cast(exp.ctypes.data + do, cl.u8p), C.cast(ref_.ctypes.data + so, cl.u8p), W, h) == 0
    with on_stream(device):
        t = lambda a, dt: torch.from_numpy(np.array(a, dt)).cuda()
        d_dst, d_src = torch.from_numpy(dst0).cuda(), torch.from_numpy(ref_).cuda()
        pel.hpel_batch_device(device, len(ops), t(ops, np.uint8), t(hs, np.uint8), d_dst, t(doffs, np.int64), d_src, t(soffs, np.int64), W)
        device.sync()
        got = d_dst.cpu().numpy()
    assert np.array_equal(got, exp), int((got != exp).sum())


def test_h264chroma_pointer_table_golden(device):
    """H264ChromaContext drop-in (host pointers): every phase / width / height of chroma.npz, guard pixels untouched."""
    from ffmpeg_b200 import pel
    from ffmpeg_b200._lib import u8p
    g = np.load(os.path.join(G, "chroma.npz"))
    c = pel.ff_h264chroma_init(8)
    assert not c.put_h264_chroma_pixels_tab[3] and not c.avg_h264_chroma_pixels_tab[3]
    src, dst0 = g["src"], g["dst0"]
    ps = C.cast(src.ctypes.data + 8 * 48 + 8, u8p)
    for key in g.files:
        if key[0] != "c":
            continue
        avg, idx, h = (int(v) for v in key.split("_")[1:])
        f = (c.avg_h264_chroma_pixels_tab if avg else c.put_h264_chroma_pixels_tab)[idx]
        for xy in range(0, 64, 3 if h != 8 else 1):
            o = dst0.copy()
            f(C.cast(o.ctypes.data + 8 * 48 + 8, u8p), ps, 48, h, xy & 7, xy >> 3)
            assert np.array_equal(o[8:24, 8:16], g[key][xy]), (key, xy)
            assert np.array_equal(o[:8], dst0[:8]) and np.array_equal(o[8 + h:], dst0[8 + h:]) and np.array_equal(o[:, 16:], dst0[:, 16:]), key
    assert pel.ff_h264chroma_init(10).put_h264_chroma_pixels_tab[0]        # the 16-bit tables (test_h264chroma_and_edge_hbd)


def test_h264chroma_batch_vs_oracle(device):
    """Chroma half of a 4:2:0 macroblock stream: random eighth-pel phases, widths, heights, unaligned offsets."""
    import torch
    from ffmpeg_b200 import pel
    O = cl.oracle()
    rng = np.random.default_rng(14)
    W, H = 336, 208
    ref_ = rng.integers(0, 256, (H, W), dtype=np.uint8)
    dst0 = rng.integers(0, 256, (H, W), dtype=np.uint8)
    ops, hs, xys, doffs, soffs = [], [], [], [], []
    for by in range(1, H // 16 - 1):
        for bx in range(1, W // 16 - 1):
            idx = int(rng.integers(0, 3))
            ops.append(pel.chroma_op(int(rng.integers(0, 2)), idx))
            hs.append(int(rng.choice(((4, 8, 16), (2, 4, 8), (2, 4))[idx])))
            xys.append(int(rng.integers(0, 64)))
            dx, dy, jx = int(rng.integers(-8, 9)), int(rng.integers(-8, 9)), int(rng.integers(0, 8))
            doffs.append(by * 16 * W + bx * 16 + jx); soffs.append((by * 16 + dy) * W + bx * 16 + dx)
    exp = dst0.copy()
    for op, h, xy, do, so in zip(ops, hs, xys, doffs, soffs):
        assert O.orc_h264chroma(op & 1, op >> 1, C.cast(exp.ctypes.data + do, cl.u8p), C.cast(ref_.ctypes.data + so, cl.u8p), W, h, xy & 7, xy >> 3) == 0
    with on_stream(device):
        t = lambda a, dt: torch.from_numpy(np.array(a, dt)).cuda()
        d_dst, d_src = torch.from_numpy(dst0).cuda(), torch.from_numpy(ref_).cuda()
        pel.h264chroma_batch_device(device, len(ops), t(ops, np.uint8), t(hs, np.uint8), t(xys, np.uint8), d_dst, t(doffs, np.int64),
                                    d_src, t(soffs, np.int64), W)
        device.sync()
        got = d_dst.cpu().numpy()
    assert np.array_equal(got, exp), int((got != exp).sum())


def test_h264chroma_no_reads_past_block_when_phase_zero(device):
    """x == 0 / y == 0 must not touch the column right of / the row below the block (h264chroma_template.c D == 0 branches):
    blocks that end exactly at the end of the device allocation, checked under the allocation's own bounds."""
    import torch
    from ffmpeg_b200 import pel
    O = cl.oracle()
    rng = np.random.default_rng(15)
    W = 64
    for (x, y) in ((0, 0), (0, 5), (3, 0)):
        rows = 8 + (1 if y else 0)
        src = rng.integers(0, 256, rows * W, dtype=np.uint8)
        if x == 0:
            src = src[: (rows - 1) * W + 56 + 8]                   # block is the last 8 columns of the buffer: nothing after it
        dst0 = rng.integers(0, 256, 8 * W, dtype=np.uint8)
        so = 56 if x == 0 else 40
        exp = dst0.copy()
        pad = np.concatenate([src, np.zeros(2 * W, np.uint8)])
        assert O.orc_h264chroma(0, 0, cl.ptr(exp), C.cast(pad.ctypes.data + so, cl.u8p), W, 8, x, y) == 0
        with on_stream(device):
            t = lambda a, dt: torch.from_numpy(np.array(a, dt)).cuda()
            d_dst, d_src = torch.from_numpy(dst0).cuda(), torch.from_numpy(src).cuda()
            pel.h264chroma_batch_device(device, 1, t([0], np.uint8), t([8], np.uint8), t([x | y << 3], np.uint8), d_dst, t([0], np.int64),
                                        d_src, t([so], np.int64), W)
            device.sync()
            assert np.array_equal(d_dst.cpu().numpy(), exp), (x, y)


def test_emulated_edge_mc_pointer_table_golden(device):
    from cases import EDGE_PIC, EDGE_CASES
    from ffmpeg_b200 import pel
    g = np.load(os.path.join(G, "edge.npz"))
    v = pel.ff_videodsp_init(8)
    W, H, LS = EDGE_PIC
    pic = g["pic"]
    for i, (bw, bh, sx, sy) in enumerate(EDGE_CASES):
        b = np.full((24, 32), 0x5A, np.uint8)
        v.emulated_edge_mc(b.ctypes.data, pic.ctypes.data + sy * LS + sx, 32, LS, bw, bh, sx, sy, W, H)
        assert np.array_equal(b, g[f"e{i}"]), (i, bw, bh, sx, sy)
    b = np.full((24, 32), 0x5A, np.uint8)
    v.emulated_edge_mc(b.ctypes.data, pic.ctypes.data, 32, LS, 8, 8, 0, 0, 0, H)
    assert (b == 0x5A).all()
    v.prefetch(pic.ctypes.data, LS, 4)
    assert pel.ff_videodsp_init(10).emulated_edge_mc                         # the 16-bit template (test_h264chroma_and_edge_hbd)


def test_emulated_edge_mc_batch_vs_oracle(device):
    """Windows hanging over every border of several frames in one call (the mc_dir_part case: 21x21 luma, 9x9 chroma)."""
    import torch
    from ffmpeg_b200 import pel
    O = cl.oracle()
    rng = np.random.default_rng(16)
    NF, W, H, LS = 3, 100, 60, 112
    pics = rng.integers(0, 256, (NF, H, LS), dtype=np.uint8)
    n = 600
    geom = np.zeros((n, 4), np.int32)
    geom[:, 0] = rng.choice([9, 21, 5, 16], n); geom[:, 1] = rng.choice([9, 21, 5, 16], n)
    geom[:, 2] = rng.integers(-30, W + 10, n); geom[:, 3] = rng.integers(-30, H + 10, n)
    fr = rng.integers(0, NF, n)
    origin = (fr * H * LS).astype(np.int64)
    BLS = 32
    boff = (np.arange(n) * 24 * BLS).astype(np.int64)
    exp = np.full((n * 24, BLS), 0x33, np.uint8)
    for i in range(n):
        bw, bh, sx, sy = (int(v) for v in geom[i])
        O.orc_emulated_edge_mc(C.cast(exp.ctypes.data + int(boff[i]), cl.u8p), pics[fr[i]].ctypes.data + sy * LS + sx, BLS, LS, bw, bh, sx, sy, W, H)
    with on_stream(device):
        d_buf = torch.full((n * 24, BLS), 0x33, dtype=torch.uint8, device="cuda")
        pel.emulated_edge_mc_batch_device(device, n, d_buf, torch.from_numpy(boff).cuda(), BLS, torch.from_numpy(pics).cuda(),
                                          torch.from_numpy(origin).cuda(), LS, torch.from_numpy(geom).cuda(), W, H)
        device.sync()
        got = d_buf.cpu().numpy()
    assert np.array_equal(got, exp), int((got != exp).sum())


def test_h264_weight_pointer_table_golden(device):
    from ffmpeg_b200 import pel
    g = np.load(os.path.join(G, "h264weight.npz"))
    t = pel.ff_h264dsp_weight_init(8)
    src, dst0 = g["src"], g["dst0"]
    for k, (idx, h, ld, w1, w2, off) in enumerate(g["cases"].tolist()):
        a, b = dst0.copy(), dst0.copy()
        t.weight_pixels_tab[idx](a.ctypes.data + 2 * 32 + 8, 32, h, ld, w1, off)
        t.biweight_pixels_tab[idx](b.ctypes.data + 2 * 32 + 8, src.ctypes.data + 2 * 32 + 8, 32, h, ld, w1, w2, off)
        assert np.array_equal(a, g[f"w{k}"]), ("weight", k)
        assert np.array_equal(b, g[f"b{k}"]), ("biweight", k)
    assert pel.ff_h264dsp_weight_init(10).weight_pixels_tab[0]               # the 16-bit tables (test_h264_weight_hbd)


def test_h264_weight_batch_vs_oracle(device):
    """Weighted and bi-weighted prediction over a frame of partitions (all widths, heights, denominators, unaligned x)."""
    import torch
    from ffmpeg_b200 import pel
    O = cl.oracle()
    rng = np.random.default_rng(17)
    W, H = 352, 208
    src = rng.integers(0, 256, (H, W), dtype=np.uint8)
    dst0 = rng.integers(0, 256, (H, W), dtype=np.uint8)
    params, doffs, soffs = [], [], []
    for by in range(H // 16):
        for bx in range(W // 16 - 1):
            idx = int(rng.integers(0, 4))
            h = int(rng.choice([2, 4, 8, 16]))
            ld = int(rng.integers(0, 8))
            w1, w2, off = (int(v) for v in rng.integers(-128, 128, 3))
            params.append(pel.weight_params(idx, h, ld, w1, w2, off))
            jx = 0 if idx == 0 else int(rng.integers(0, 4)) * (1 if idx < 3 else 2)      # destinations of one call must not overlap
            doffs.append(by * 16 * W + bx * 16 + jx); soffs.append(by * 16 * W + bx * 16 + int(rng.integers(0, 8)))
    n = len(params)
    pa = np.array(params, np.int32)
    for bi in (False, True):
        exp = dst0.copy()
        for (p0, w1, w2, off), do, so in zip(params, doffs, soffs):
            idx, h, ld = p0 & 3, (p0 >> 8) & 255, (p0 >> 16) & 31
            if bi:
                O.orc_h264_biweight(idx, C.cast(exp.ctypes.data + do, cl.u8p), C.cast(src.ctypes.data + so, cl.u8p), W, h, ld, w1, w2, off)
            else:
                O.orc_h264_weight(idx, C.cast(exp.ctypes.data + do, cl.u8p), W, h, ld, w1, off)
        with on_stream(device):
            t = lambda a, dt: torch.from_numpy(np.array(a, dt)).cuda()
            d_dst, d_src = torch.from_numpy(dst0).cuda(), torch.from_numpy(src).cuda()
            pel.h264_weight_batch_device(device, n, torch.from_numpy(pa).cuda(), d_dst, t(doffs, np.int64), d_src if bi else None,
                                         t(soffs, np.int64) if bi else None, W)
            device.sync()
            got = d_dst.cpu().numpy()
        assert np.array_equal(got, exp), (bi, int((got != exp).sum()))


# ---------------------------------------------------------------------------------------------- tx
def ulp_diff(a, b):
    ai, bi = a.view(np.int32).astype(np.int64), b.view(np.int32).astype(np.int64)
    ai = np.where(ai < 0, -(ai & 0x7fffffff), ai)
    bi = np.where(bi < 0, -(bi & 0x7fffffff), bi)
    return np.abs(ai - bi).max()


def test_tx_host_fn_golden(device):
    """av_tx_fn on host buffers: north_star bar is 1 ULP against the reference's *_float_c; we expect 0."""
    from ffmpeg_b200 import tx
    g = np.load(os.path.join(G, "tx.npz"))
    for n in (2, 4, 8, 16, 32, 64, 256, 1024, 2048):
        for inv in (0, 1):
            c = tx.av_tx_init(tx.AV_TX_FLOAT_FFT, inv, n)
            x = g[f"fft_in_{n}"]
            out = np.zeros_like(x)
            for r in range(x.shape[0]):
                c.fn(out[r], x[r].copy(), 8)
            assert ulp_diff(out, g[f"fft_{n}_{inv}"]) <= 1, (n, inv)
            assert np.array_equal(out, g[f"fft_{n}_{inv}"]), (n, inv)
            c.uninit()
    for n in (8, 16, 64, 256, 1024, 2048):
        for j, sc in enumerate((1.0 / n, -1.0, 1.0)):
            c = tx.av_tx_init(tx.AV_TX_FLOAT_MDCT, 1, n, scale=sc)
            x = g[f"imdct_in_{n}"]
            out = np.zeros((x.shape[0], n), np.float32)
            for r in range(x.shape[0]):
                c.fn(out[r], x[r].copy(), 4)
            assert np.array_equal(out, g[f"imdct_{n}_{j}"]), (n, j)
            c.uninit()
            c = tx.av_tx_init(tx.AV_TX_FLOAT_MDCT, 0, n, scale=sc)
            x = g[f"mdct_in_{n}"]
            out = np.zeros((x.shape[0], n), np.float32)
            for r in range(x.shape[0]):
                c.fn(out[r], x[r].copy(), 4)
            assert np.array_equal(out, g[f"mdct_{n}_{j}"]), (n, j)
            c.uninit()


@pytest.mark.parametrize("n", [512, 1024, 2048, 4096])
def test_tx_batch_vs_oracle(device, n):
    import torch
    from ffmpeg_b200 import tx
    O = cl.oracle()
    rng = np.random.default_rng(n)
    cnt = 300

    def orc(typ, inv, scale, x, of):
        h = O.orc_tx_open(typ, inv, n, scale, 0)
        out = np.zeros((x.shape[0], of), np.float32)
        O.orc_tx_run(h, out.ctypes.data, x.ctypes.data, 8 if typ == 0 else 4, x.shape[0], out.strides[0], x.strides[0])
        O.orc_tx_close(h)
        return out
    with on_stream(device):
        x = rng.random((cnt, 2 * n), dtype=np.float32)
        dx = torch.from_numpy(x).cuda()
        for inv in (0, 1):
            c = tx.av_tx_init(tx.AV_TX_FLOAT_FFT, inv, n, device=device)
            do = torch.zeros_like(dx)
            c.batch_device(do, dx, 8, cnt, 8 * n, 8 * n)
            device.sync()
            assert np.array_equal(do.cpu().numpy(), orc(0, inv, 1.0, x, 2 * n)), ("fft", inv)
            c.uninit()
        xi = np.ascontiguousarray(x[:, :n])
        c = tx.av_tx_init(tx.AV_TX_FLOAT_MDCT, 1, n, scale=1.0 / n, device=device)
        di, do = torch.from_numpy(xi).cuda(), torch.zeros((cnt, n), dtype=torch.float32, device="cuda")
        c.batch_device(do, di, 4, cnt, 4 * n, 4 * n)
        device.sync()
        assert np.array_equal(do.cpu().numpy(), orc(1, 1, 1.0 / n, xi, n)), "imdct"
        c.uninit()
        c = tx.av_tx_init(tx.AV_TX_FLOAT_MDCT, 0, n, scale=-1.0, device=device)
        do = torch.zeros((cnt, n), dtype=torch.float32, device="cuda")
        c.batch_device(do, dx, 4, cnt, 4 * n, 8 * n)
        device.sync()
        assert np.array_equal(do.cpu().numpy(), orc(1, 0, -1.0, x, n)), "mdct"
        c.uninit()


def test_tx_rdft_host_fn_golden(device):
    """AV_TX_FLOAT_RDFT through av_tx_fn on host buffers: bit-identical to the reference, and the inverse leaves the same
    values in its input buffer as ff_tx_rdft_c2r does."""
    from ffmpeg_b200 import tx
    g = np.load(os.path.join(G, "tx_rdft.npz"))
    for n in (4, 8, 16, 64, 256, 1024, 2048, 4096):
        for j, sc in enumerate((1.0, 1.0 / n)):
            c = tx.av_tx_init(tx.AV_TX_FLOAT_RDFT, 0, n, scale=sc)
            x = g[f"r2c_in_{n}_{j}"].copy()
            out = np.zeros((2, n + 2), np.float32)
            for r in range(2):
                c.fn(out[r], x[r], 4)
            assert np.array_equal(out.view(np.uint32), g[f"r2c_{n}_{j}"].view(np.uint32)), ("r2c", n, j)
            c.uninit()
            c = tx.av_tx_init(tx.AV_TX_FLOAT_RDFT, 1, n, scale=sc)
            xc = g[f"c2r_in_{n}_{j}"].copy()
            out = np.zeros((2, n), np.float32)
            for r in range(2):
                c.fn(out[r], xc[r], 8)
            assert np.array_equal(out.view(np.uint32), g[f"c2r_{n}_{j}"].view(np.uint32)), ("c2r", n, j)
            assert np.array_equal(xc.view(np.uint32), g[f"c2r_in_after_{n}_{j}"].view(np.uint32)), ("c2r input", n, j)
            c.uninit()
    with pytest.raises(Exception):
        tx.av_tx_init(tx.AV_TX_FLOAT_RDFT, 0, 2, scale=1.0)            # min_len 4
    with pytest.raises(Exception):
        tx.av_tx_init(tx.AV_TX_FLOAT_RDFT, 0, 96, scale=1.0)           # 3 x 2^n: PFA lengths are not implemented


@pytest.mark.parametrize("n", [512, 2048, 8192])
def test_tx_rdft_batch_vs_oracle(device, n):
    import torch
    from ffmpeg_b200 import tx
    O = cl.oracle()
    rng = np.random.default_rng(n + 1)
    cnt = 203

    def orc(inv, scale, x, of):
        h = O.orc_tx_open(6, inv, n, scale, 0)
        out = np.zeros((x.shape[0], of), np.float32)
        O.orc_tx_run(h, out.ctypes.data, x.ctypes.data, 4, x.shape[0], out.strides[0], x.strides[0])
        O.orc_tx_close(h)
        return out
    with on_stream(device):
        x = (rng.random((cnt, n), dtype=np.float32) * 2 - 1).astype(np.float32)
        c = tx.av_tx_init(tx.AV_TX_FLOAT_RDFT, 0, n, scale=1.0, device=device)
        dx, do = torch.from_numpy(x).cuda(), torch.zeros((cnt, n + 2), dtype=torch.float32, device="cuda")
        c.batch_device(do, dx, 4, cnt, 4 * (n + 2), 4 * n)
        device.sync()
        spec = do.cpu().numpy()
        assert np.array_equal(spec.view(np.uint32), orc(0, 1.0, x.copy(), n + 2).view(np.uint32)), "r2c"
        c.uninit()
        c = tx.av_tx_init(tx.AV_TX_FLOAT_RDFT, 1, n, scale=1.0 / n, device=device)
        di, do = torch.from_numpy(spec).cuda(), torch.zeros((cnt, n), dtype=torch.float32, device="cuda")
        c.batch_device(do, di, 8, cnt, 4 * n, 4 * (n + 2))
        device.sync()
        back = do.cpu().numpy()
        assert np.array_equal(di.cpu().numpy().view(np.uint32), spec.view(np.uint32)), "batched c2r must not touch its input"
        assert np.array_equal(back.view(np.uint32), orc(1, 1.0 / n, spec.copy(), n).view(np.uint32)), "c2r"
        assert np.abs(back - x).max() < 1e-4                      # r2c (scale 1) then c2r (scale 1/len) is the identity
        c.uninit()


def test_tx_linearity_1m_batch(device):
    """BASELINE config 5 size (a large batch of len-1024 transforms): FFT(a) + FFT(b) ~= FFT(a + b) and Parseval,
    size-independent properties of a 200 000-transform batch; plus unsupported configurations are refused loudly.  The bit-exact
    comparison with the oracle over several rounds of the persistent grid, for every tx_r16 size, is test_batch_rounds_gpu.py's."""
    import torch
    import ffmpeg_b200 as fb
    from ffmpeg_b200 import tx
    n, cnt = 1024, 200_000
    with on_stream(device):
        a = torch.rand((cnt, 2 * n), device="cuda")
        b = torch.rand((cnt, 2 * n), device="cuda")
        c = tx.av_tx_init(tx.AV_TX_FLOAT_FFT, 0, n, device=device)
        fa, fb_, fab = torch.empty_like(a), torch.empty_like(a), torch.empty_like(a)
        c.batch_device(fa, a, 8, cnt, 8 * n, 8 * n)
        c.batch_device(fb_, b, 8, cnt, 8 * n, 8 * n)
        c.batch_device(fab, a + b, 8, cnt, 8 * n, 8 * n)
        device.sync()
        assert float((fa + fb_ - fab).abs().max()) < 2e-2
        e_t = (a[:1000].double() ** 2).sum(1)
        e_f = (fa[:1000].double() ** 2).sum(1) / n
        assert float(((e_t - e_f).abs() / e_t).max()) < 1e-5
        c.uninit()
    with pytest.raises(fb.B200Error):
        tx.av_tx_init(tx.AV_TX_FLOAT_FFT, 0, 90, device=device)             # 45 x 2: nested compound tree, not implemented
    with pytest.raises(fb.B200Error):
        tx.av_tx_init(7, 0, 1024, device=device)                            # other transform types (AV_TX_DOUBLE_RDFT)
