"""GPU tier: the persistent kernels past their first round.  tx_r16_kernel, chroma_kernel_p (the default h264chroma path),
mpv_unquant_kernel and the tx_double kernels launch a capped grid and let each thread group, warp or CTA loop over the batch; the
code that only runs from the second round on (tx_r16's refetch into its two-slot TMA input ring, the descriptors chroma_kernel_p
prefetches for its next batch, the grid-stride loops) is only reached by batches larger than one round of the grid.

Sizing: S is the device's SM count and no occupancy is assumed.  Where the grid cap depends on occupancy, 8 CTAs of 256 threads per
SM (2048 threads) bound one round from above; every multi-round count is k such rounds plus a small odd remainder that is not a
multiple of a CTA's work unit, so the batch takes at least k rounds on any part and the last CTA's groups or warps finish on
different rounds.  Every element of every batch is compared with the oracle bit for bit; a failure reports how many transforms,
operations or blocks differ, the first of them, and the share of them that lie past one round of the widest possible grid."""
import os

import numpy as np
import pytest

import cpulibs as cl

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CTAS_PER_SM = 8                          # upper bound of resident 256-thread CTAs per SM


def on_stream(device):
    import torch
    return torch.cuda.stream(torch.cuda.ExternalStream(device.stream))


@pytest.fixture(scope="module")
def sms(device):
    import torch
    return torch.cuda.get_device_properties(device.ordinal).multi_processor_count


def mismatch(bad, round_size, what):
    """failure message for a per-unit mismatch mask: how many units differ, the first few, and how many of them lie at or past
    one round of the widest grid (a fault of the code that only runs from the second round on shows up there only)"""
    idx = np.flatnonzero(bad)
    late = int((idx >= round_size).sum())
    return (f"{what}: {idx.size} of {bad.size} differ, first {idx[:8].tolist()}; "
            f"{late} of them ({late / max(idx.size, 1):.0%}) at index >= {round_size} (one round of the widest grid)")


# ---------------------------------------------------------------------------------------------- tx_r16: FFT 512-4096, iMDCT 1024-8192
def tx_groups(points):
    """transforms per CTA of tx_r16_kernel: points / 16 threads per transform, 256 threads per CTA"""
    return 256 // (points // 16)


def tx_init(monkeypatch, env, *args, **kw):
    """av_tx_init with exactly the A/B switches in `env` set (tx_r16_create reads them once per context); the process
    environment is restored before this returns"""
    from ffmpeg_b200 import tx
    with monkeypatch.context() as m:
        for k in ("B200_TX_LEAF", "B200_TX_OLD"):
            m.delenv(k, raising=False)
        for k, v in env.items():
            m.setenv(k, v)
        return tx.av_tx_init(*args, **kw)


def np_fft(z, inv):
    """float64 numpy FFT with av_tx's conventions (unscaled both ways); which numpy direction av_tx's forward transform is comes
    from the reference's 8-point outputs in tx.npz"""
    g = np.load(os.path.join(G, "tx.npz"))
    cplx = lambda a: a[:, 0::2].astype(np.float64) + 1j * a[:, 1::2]
    x8, y8 = cplx(g["fft_in_8"]), cplx(g["fft_8_0"])
    fwd_is_fft = np.abs(np.fft.fft(x8) - y8).max() < np.abs(np.fft.ifft(x8) * 8 - y8).max()
    return np.fft.fft(z) if fwd_is_fft != bool(inv) else np.fft.ifft(z) * z.shape[-1]


class TxCheck:
    """one oracle output, against which every variant of a case must come out bit-identical"""

    def __init__(self, what, exp, round_size, x=None, inv=None):
        self.what, self.exp, self.round_size, self.x, self.inv = what, exp, round_size, x, inv

    def __call__(self, got, variant, cnt=None):
        exp = self.exp[:cnt] if cnt is not None else self.exp
        assert got.shape == exp.shape, (self.what, variant, got.shape)
        bad = (got.view(np.uint32) != exp.view(np.uint32)).any(axis=1)
        if not bad.any():
            return
        msg = mismatch(bad, self.round_size, f"{self.what}, {variant}: transforms")
        if self.x is not None:                                    # FFT: a one-ULP drift or a garbage transform?
            rows = np.flatnonzero(bad)
            x = self.x[rows].astype(np.float64)
            ref = np_fft(x[:, 0::2] + 1j * x[:, 1::2], self.inv)
            g = got[rows].astype(np.float64)
            err = np.linalg.norm(g[:, 0::2] + 1j * g[:, 1::2] - ref, axis=1) / np.maximum(np.linalg.norm(ref, axis=1), 1e-30)
            msg += f"; worst relative L2 error of those against a float64 numpy.fft: {err.max():.3g}"
        pytest.fail(msg)


def tx_run(c, dx, cnt, row_out, stride, in_pad=0, out_off=0, inplace=False):
    """one batched call on the first cnt rows of dx (device, float32 [rows, row_in]); in_pad floats after every input row,
    output base moved by out_off floats (the floats before it must stay untouched); returns the output rows on the host"""
    import torch
    row_in = dx.shape[1]
    if inplace:
        d = dx[:cnt].clone()
        c.batch_device(d, d, stride, cnt, 4 * row_in, 4 * row_in)
        return d.cpu().numpy()
    if in_pad:
        di = torch.zeros((cnt, row_in + in_pad), dtype=torch.float32, device="cuda")
        di[:, :row_in] = dx[:cnt]
    else:
        di = dx[:cnt]
    flat = torch.zeros(cnt * row_out + out_off, dtype=torch.float32, device="cuda")
    do = flat[out_off:].view(cnt, row_out)
    c.batch_device(do, di, stride, cnt, 4 * row_out, 4 * di.shape[1])
    if out_off:
        assert not flat[:out_off].any(), "a store before the output base"
    return do.cpu().numpy()


def tx_variants(monkeypatch, device, check, dx, cnt, row_out, stride, init_args, init_kw, groups, inplace):
    """every route a batch of this transform can take, all against one oracle output"""
    with on_stream(device):
        for leaf in ("0", "1"):                                    # both leaf-chunk orders of tx_r16_kernel
            c = tx_init(monkeypatch, {"B200_TX_LEAF": leaf}, *init_args, **init_kw)
            check(tx_run(c, dx, cnt, row_out, stride), f"B200_TX_LEAF={leaf}")
            for t in sorted({1, groups - 1, groups, groups + 1} - {0}):     # some groups of the only CTA never enter the loop
                check(tx_run(c, dx, t, row_out, stride), f"B200_TX_LEAF={leaf}, count {t}", t)
            c.uninit()
        c = tx_init(monkeypatch, {"B200_TX_OLD": "1"}, *init_args, **init_kw)              # the level-by-level kernels of tx.cu
        check(tx_run(c, dx, cnt, row_out, stride), "B200_TX_OLD=1")
        c.uninit()
        c = tx_init(monkeypatch, {}, *init_args, **init_kw)
        # an input step that is not a multiple of 16 bytes: tx_r16_accepts refuses it and the batch runs on tx.cu's kernels
        check(tx_run(c, dx, cnt, row_out, stride, in_pad=2 if stride == 8 else 1), "input step + 8 / + 4 bytes")
        check(tx_run(c, dx, cnt, row_out, stride, out_off=2), "output base + 8 bytes")        # still tx_r16: 8-byte stores
        c.uninit()
        if inplace:
            from ffmpeg_b200 import tx
            c = tx_init(monkeypatch, {}, *init_args, flags=tx.AV_TX_INPLACE, **init_kw)
            check(tx_run(c, dx, cnt, row_out, stride, inplace=True), "AV_TX_INPLACE, out == in")
            c.uninit()


@pytest.mark.parametrize("n", [512, 1024, 2048, 4096])
def test_tx_r16_fft_multi_round(device, monkeypatch, sms, n):
    """complex FFT, both directions, three rounds of the widest grid: both leaf orders, tx.cu's kernels (by switch and by an
    input step tx_r16 refuses), an 8-byte-aligned output base, in place, and the tail counts of a single CTA"""
    import torch
    from ffmpeg_b200 import tx
    from test_oracle_more import _tx
    O = cl.oracle()
    groups = tx_groups(n)
    rnd = sms * CTAS_PER_SM * groups
    cnt = 3 * rnd + 5
    rng = np.random.default_rng(7000 + n)
    x = (rng.random((cnt, 2 * n), dtype=np.float32) * 2 - 1).astype(np.float32)
    with on_stream(device):
        dx = torch.from_numpy(x).cuda()
    for inv in (0, 1):
        check = TxCheck(f"fft {n} inv {inv}", _tx(O, "orc", 0, inv, n, 1.0, x, 2 * n), rnd, x=x, inv=inv)
        tx_variants(monkeypatch, device, check, dx, cnt, 2 * n, 8, (tx.AV_TX_FLOAT_FFT, inv, n), {"device": device}, groups, True)


@pytest.mark.parametrize("length", [1024, 2048, 4096, 8192])
def test_tx_r16_imdct_multi_round(device, monkeypatch, sms, length):
    """inverse MDCT (length / 2 complex points), scales 1 / length and -1, three rounds of the widest grid: the same routes as the FFT
    except in place, which the MDCT refuses"""
    import torch
    from ffmpeg_b200 import tx
    from test_oracle_more import _tx
    O = cl.oracle()
    groups = tx_groups(length // 2)
    rnd = sms * CTAS_PER_SM * groups
    cnt = 3 * rnd + 5
    rng = np.random.default_rng(7100 + length)
    x = (rng.random((cnt, length), dtype=np.float32) * 2 - 1).astype(np.float32)
    with on_stream(device):
        dx = torch.from_numpy(x).cuda()
    for sc in (1.0 / length, -1.0):
        check = TxCheck(f"imdct {length} scale {sc}", _tx(O, "orc", 1, 1, length, sc, x, length), rnd)
        tx_variants(monkeypatch, device, check, dx, cnt, length, 4, (tx.AV_TX_FLOAT_MDCT, 1, length), {"scale": sc, "device": device},
                    groups, False)


# ---------------------------------------------------------------------------------------------- chroma_kernel_p (h264chroma, default)
CHROMA_ROUND_OPS = CTAS_PER_SM * 4 * 8          # per SM: the grid cap (8 CTAs), 4 warps per CTA, 8 operations per warp batch


def chroma_case(n, seed, planes=4):
    """n operations, each writing its own 16 x 16 cell of `planes` destination planes (cells in shuffled order, 16 guard rows
    below every plane), reading a window at +-8 pixels around a block of a padded reference plane; stride 1024 for both"""
    from ffmpeg_b200 import pel
    rng = np.random.default_rng(seed)
    W, HR = 1024, 512
    rows = -(-n // (64 * planes))                                  # cell rows per plane, 64 cells per row
    ph = rows * 16 + 16
    ref_ = rng.integers(0, 256, (HR, W), dtype=np.uint8)
    dst0 = rng.integers(0, 256, (planes, ph, W), dtype=np.uint8)
    idx = rng.integers(0, 3, n)
    op = np.array([pel.chroma_op(int(a), int(i)) for a, i in zip(rng.integers(0, 2, n), idx)], np.uint8)
    hs = np.array([rng.choice(((4, 8, 16), (2, 4, 8), (2, 4))[i]) for i in idx], np.uint8)
    xy = rng.permutation(np.arange(n) % 64).astype(np.uint8)          # every phase, so both x == 0 and y == 0 branches
    cell = rng.permutation(planes * rows * 64)[:n]
    doff = (cell // (rows * 64)) * ph * W + ((cell // 64) % rows) * 16 * W + (cell % 64) * 16 + rng.integers(0, 8, n)
    by, bx = rng.integers(1, HR // 16 - 1, n), rng.integers(1, W // 16 - 1, n)
    soff = (by * 16 + rng.integers(-8, 9, n)) * W + bx * 16 + rng.integers(-8, 9, n)
    return dict(W=W, ref=ref_, dst0=dst0, op=op, h=hs, xy=xy, doff=doff.astype(np.int64), soff=soff.astype(np.int64), cell=cell, rows=rows)


def chroma_oracle(case, n):
    O = cl.oracle()
    exp = case["dst0"].copy()
    assert O.orc_h264chroma_batch(n, cl.ptr(case["op"]), cl.ptr(case["h"]), cl.ptr(case["xy"]), cl.ptr(exp), cl.ptr(case["doff"], cl.i64p),
                                  cl.ptr(case["ref"]), cl.ptr(case["soff"], cl.i64p), case["W"]) == 0
    return exp


def chroma_gpu(device, case, n):
    import torch
    from ffmpeg_b200 import pel
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    with on_stream(device):
        d_dst = t(case["dst0"])
        pel.h264chroma_batch_device(device, n, t(case["op"]), t(case["h"]), t(case["xy"]), d_dst, t(case["doff"]), t(case["ref"]),
                                    t(case["soff"]), case["W"])
        device.sync()
        return d_dst.cpu().numpy()


def chroma_check(case, n, got, exp, round_size):
    if np.array_equal(got, exp):
        return
    planes, rows = got.shape[0], case["rows"]
    cells = lambda a: a[:, : rows * 16].reshape(planes, rows, 16, 64, 16)
    cell_bad = (cells(got) != cells(exp)).any(axis=(2, 4)).ravel()
    guard = int((got[:, rows * 16:] != exp[:, rows * 16:]).sum())
    pytest.fail(mismatch(cell_bad[case["cell"][:n]], round_size, f"h264chroma, {n} ops: operations") + f"; guard-row bytes changed: {guard}")


def test_h264chroma_multi_round(device, sms):
    """chroma_kernel_p: three rounds of its widest grid (each warp works on several batches, with the next batch's descriptors
    prefetched), and the small counts around one warp batch (8 operations) and one CTA (32)"""
    n = 3 * CHROMA_ROUND_OPS * sms + 13
    case = chroma_case(n, 71)
    chroma_check(case, n, chroma_gpu(device, case, n), chroma_oracle(case, n), CHROMA_ROUND_OPS * sms)
    for k in (1, 7, 8, 9, 31, 32, 33):
        chroma_check(case, k, chroma_gpu(device, case, k), chroma_oracle(case, k), CHROMA_ROUND_OPS * sms)


# ---------------------------------------------------------------------------------------------- mpv_unquant_kernel
UNQUANT_ROUND_BLOCKS = 128 * 4                  # per SM: the grid cap (128 CTAs), one block per warp, 4 warps per CTA


@pytest.mark.parametrize("variant", range(7))
def test_mpv_unquant_multi_round(device, sms, variant):
    """every inverse quantiser, two rounds of the grid-stride loop, with the block numbers given and with n = index % 6"""
    from test_zz_next_gpu import gpu_unquant
    cnt = 2 * UNQUANT_ROUND_BLOCKS * sms + 11
    cfg, blocks, blk_n, q, last = cl.unquant_case(5100 + 2 * variant, variant, nblocks=cnt)      # even seed: random block numbers
    for use_n in (blk_n, None):
        got = gpu_unquant(device, variant, cfg, blocks, use_n, q, last)
        exp = cl.orc_unquant(variant, cfg, blocks, use_n, q, last)
        if not np.array_equal(got, exp):
            pytest.fail(mismatch((got != exp).any(axis=1), UNQUANT_ROUND_BLOCKS * sms,
                                 f"{cl.UNQUANT_VARIANTS[variant]}, blk_n {'given' if use_n is not None else 'None'}: blocks"))


# ---------------------------------------------------------------------------------------------- tx_double
@pytest.mark.parametrize("n", [1024, 4096])
def test_tx_double_multi_round(device, sms, n):
    """AV_TX_DOUBLE_FFT / AV_TX_DOUBLE_MDCT, both directions: two rounds of the grid-stride loop (one transform per CTA, 8 CTAs
    per SM) against the double-precision oracle"""
    import torch
    from ffmpeg_b200 import tx
    from test_cuda_emu import _orc_txd
    rnd = 8 * sms
    cnt = 2 * rnd + 3
    rng = np.random.default_rng(7200 + n)
    for typ, inv, sc in ((tx.AV_TX_DOUBLE_FFT, 0, 1.0), (tx.AV_TX_DOUBLE_FFT, 1, 1.0), (tx.AV_TX_DOUBLE_MDCT, 0, 1.0),
                         (tx.AV_TX_DOUBLE_MDCT, 1, 1.0 / n)):
        fft = typ == tx.AV_TX_DOUBLE_FFT
        x = rng.random((cnt, n if (not fft and inv) else 2 * n)) * 2 - 1
        oute = 2 * n if fft else n
        c = tx.av_tx_init(typ, inv, n, scale=sc, device=device)
        with on_stream(device):
            di, do = torch.from_numpy(x).cuda(), torch.zeros((cnt, oute), dtype=torch.float64, device="cuda")
            c.batch_device(do, di, 16 if fft else 8, cnt, oute * 8, x.shape[1] * 8)
            device.sync()
            got = do.cpu().numpy()
        c.uninit()
        exp = _orc_txd(typ, inv, n, sc, x, oute)
        bad = (got.view(np.uint64) != exp.view(np.uint64)).any(axis=1)
        if bad.any():
            pytest.fail(mismatch(bad, rnd, f"{'fft' if fft else 'mdct'} {n} inv {inv}: transforms"))
