/*
 * oracle.h — TEST INFRASTRUCTURE ONLY (CPU restatement of the reference algorithms).
 *
 * Plain-C restatements of the five FFmpeg DSP hot paths, written from the reference's behaviour
 * (each function cites the reference file:line it follows).  They are the checker for the CUDA path:
 * only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may load liboracle.so.
 * The product (ffmpeg_b200/, libb200dsp.so) never links or calls anything declared here.
 *
 * Parity pinning: every function below is checked bit-for-bit (tx: bit-for-bit too, same float op order)
 * against the unmodified reference compiled in oracle/_ref (tests/test_oracle_vs_ref.py, run wherever
 * oracle/_ref/libffref.so exists) and against the committed fixtures in tests/golden/ (generated from
 * oracle/_ref by scripts/gen_golden.py).
 */
#ifndef B200_ORACLE_H
#define B200_ORACLE_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------ swscale: yuv420p -> rgb24 */
/* flag values identical to libswscale/swscale.h:88-118 */
#define ORC_SWS_FAST_BILINEAR 0x1
#define ORC_SWS_BILINEAR      0x2
#define ORC_SWS_BICUBIC       0x4
#define ORC_SWS_X             0x8
#define ORC_SWS_POINT         0x10
#define ORC_SWS_AREA          0x20
#define ORC_SWS_BICUBLIN      0x40
#define ORC_SWS_GAUSS         0x80
#define ORC_SWS_SINC          0x100
#define ORC_SWS_LANCZOS       0x200
#define ORC_SWS_SPLINE        0x400
#define ORC_SWS_FULL_CHR_H_INT 0x2000
#define ORC_SWS_FULL_CHR_H_INP 0x4000
#define ORC_SWS_ACCURATE_RND  0x40000
#define ORC_SWS_BITEXACT      0x80000

typedef struct OrcSws OrcSws;

/* AVPixelFormat values, libavutil/pixfmt.h */
#define ORC_PIX_FMT_YUV420P 0
#define ORC_PIX_FMT_RGB24 2
#define ORC_PIX_FMT_NV12  23
#define ORC_PIX_FMT_NV21  24
#define ORC_PIX_FMT_BGR24 3
#define ORC_PIX_FMT_ARGB  25
#define ORC_PIX_FMT_RGBA  26
#define ORC_PIX_FMT_ABGR  27
#define ORC_PIX_FMT_BGRA  28
OrcSws *orc_sws_open(int srcW, int srcH, int dstW, int dstH, int flags);                      /* rgb24 */
OrcSws *orc_sws_open_fmt(int srcW, int srcH, int dstW, int dstH, int dstFormat, int flags);                 /* yuv420p source */
/* srcFormat yuv420p, nv12 or nv21: for the semi-planar sources the scale calls take the interleaved plane as `u` (`v` unused).
 * srcFormat rgb24 / bgr24 / rgba / bgra / argb / abgr (packed RGB source, the input readers of libswscale/input.c): the scale calls
 * take the packed picture as `y` (`u`, `v` unused).  Not restated (open returns NULL): same-size RGB -> RGB (the reference's
 * rgb2rgb shuffles) and a source with alpha scaled to a destination with alpha (the alpha plane then goes through the scaler). */
OrcSws *orc_sws_open_io(int srcFormat, int srcW, int srcH, int dstFormat, int dstW, int dstH, int flags);
/* src_range / dst_range (0 = limited "mpeg", 1 = full "jpeg") given before initialisation, like SwsContext.src_range /
 * .dst_range set ahead of sws_init_context; only a yuv destination converts ranges (swscale.c:626-660) */
/* with SwsContext.scaler_params (sws_getContext's `param`; NULL or 123456 = default) */
OrcSws *orc_sws_open_params(int srcFormat, int srcW, int srcH, int srcRange, int dstFormat, int dstW, int dstH, int dstRange, int flags,
                            const double *param);
OrcSws *orc_sws_open_filters(int srcFormat, int srcW, int srcH, int srcRange, int dstFormat, int dstW, int dstH, int dstRange, int flags,
                             const double *const srcCoef[4], const int srcLen[4], const int dstLen[4], const double *param);
OrcSws *orc_sws_open_range(int srcFormat, int srcW, int srcH, int srcRange, int dstFormat, int dstW, int dstH, int dstRange, int flags);
void    orc_sws_close(OrcSws *s);
/* inv_table = 4 coefficients as ff_yuv2rgb_coeffs rows; contrast/saturation 16.16 */
int     orc_sws_set_colorspace(OrcSws *s, const int inv_table[4], int srcRange,
                               int brightness, int contrast, int saturation);
/* the full sws_setColorspaceDetails(): for a yuv destination the ranges are kept and the range conversion between the two
 * passes is re-selected; different matrices for yuv -> yuv (the reference cascades through bgr24) are not restated: -1 */
int     orc_sws_set_colorspace_details(OrcSws *s, const int inv_table[4], int srcRange, const int table[4], int dstRange,
                                       int brightness, int contrast, int saturation);
/* whole-frame conversion; returns number of output lines or <0 */
int     orc_sws_scale(OrcSws *s, const uint8_t *y, int ys, const uint8_t *u, int us,
                      const uint8_t *v, int vs, uint8_t *dst, int ds);
/* planar destination (context opened with ORC_PIX_FMT_YUV420P, or ORC_PIX_FMT_NV12 / NV21: then `du` receives the interleaved
 * chroma plane of 2 * chrDstW bytes per line and `dv` is unused) */
int     orc_sws_scale_planar(OrcSws *s, const uint8_t *y, int ys, const uint8_t *u, int us, const uint8_t *v, int vs,
                             uint8_t *dy, int dys, uint8_t *du, int dus, uint8_t *dv, int dvs);
/* single stages, for checking single kernels: the horizontal pass over a whole picture (L: srcH x dstW, CU / CV: chrSrcH x chrDstW
 * int16; a packed RGB source goes through the input readers first) and the range conversion of n lines of width w in place */
int     orc_sws_hlines(const OrcSws *s, const uint8_t *y, int ys, const uint8_t *u, int us, const uint8_t *v, int vs,
                       int16_t *L, int16_t *CU, int16_t *CV);
void    orc_sws_range_lines(const OrcSws *s, int16_t *lines, int w, int n, int chroma);
/* 16 ints, same layout as ffref_sws_info */
int     orc_sws_info(const OrcSws *s, int *out);
/* 6 ints, same layout as ffref_sws_range_info: conversion kind (0 none, 1 limited->full, 2 full->limited), luma coefficient
 * and offset, chroma coefficient and offset, unscaled converter installed */
int     orc_sws_range_info(const OrcSws *s, int *out);
/* 13 ints, same layout as ffref_sws_rgb_info: bytes per pixel of a packed RGB source (0 = yuv source), horizontal / vertical chroma
 * shift of the source as scaled, bgr24 -> yv12 converter installed, input_rgb2yuv_table[9] */
int     orc_sws_rgb_info(const OrcSws *s, int *out);
/* which: 0 hLum 1 hChr 2 vLum 3 vChr; returns n entries copied */
int     orc_sws_get_filter(const OrcSws *s, int which, int16_t *filter, int32_t *pos, int cap);
/* the bare horizontal FIR */
void    orc_hscale8to15(int16_t *dst, int dstW, const uint8_t *src, const int16_t *filter,
                        const int32_t *filterPos, int filterSize);

/* ------------------------------------------------------------------ idctdsp (simple_idct 8 bit) */
void orc_idct(int16_t *block);                                            /* in place */
void orc_idct_put(uint8_t *dest, ptrdiff_t line_size, int16_t *block);
void orc_idct_add(uint8_t *dest, ptrdiff_t line_size, int16_t *block);
void orc_idct_batch(int kind, int16_t *blocks, int nblocks, uint8_t *dest, ptrdiff_t line_size,
                    const int64_t *dest_off);
/* simple IDCT at 10 / 12 bit (ff_simple_idct_{,put_,add_}int16_{10,12}bit): kind 0 in place, 1 put, 2 add; dest = uint16 pixels,
 * line_size in bytes; the block is clobbered like the reference's */
int  orc_idct_hbd(int depth, int kind, uint8_t *dest, ptrdiff_t line_size, int16_t *block);
/* ProresDSPContext.idct_put for bits_per_raw_sample 10 / 12 (libavcodec/proresdsp.c): dequantise by qmat, inverse transform, bias,
 * clip to [4, 2^bits - 5]; out = uint16 pixels, linesize in bytes; the block is left holding the transformed values like the reference's */
int  orc_prores_idct_put(int bits, uint8_t *out, ptrdiff_t linesize, int16_t *block, const int16_t *qmat);
/* H.264 deblocking, 8 bit: kind 0 v_luma, 1 h_luma, 2 h_luma_mbaff, 3-5 the same three _intra (tc0 unused), 6 v_chroma, 7 h_chroma,
 * 8 h_chroma_mbaff, 9-11 their _intra forms, 12 / 13 h_chroma / h_chroma_mbaff of 4:2:2 content, 14 / 15 their _intra forms.
 * pix points at q0 of the first line (the first pixel on the far side of the edge), as in H264DSPContext */
int  orc_h264_loop_filter(int kind, uint8_t *pix, ptrdiff_t stride, int alpha, int beta, const int8_t *tc0);
int  orc_h264_loop_filter_hbd(int depth, int kind, uint8_t *pix, ptrdiff_t stride_bytes, int alpha, int beta, const int8_t *tc0);   /* 9 / 10 / 12 / 14 bit */
/* inverse quantisers of libavcodec/mpegvideo_unquantize.c (MPVUnquantDSPContext), in place on int16[64] blocks */
enum { ORC_UNQUANT_MPEG1_INTRA, ORC_UNQUANT_MPEG1_INTER, ORC_UNQUANT_MPEG2_INTRA, ORC_UNQUANT_MPEG2_INTRA_BITEXACT,
       ORC_UNQUANT_MPEG2_INTER, ORC_UNQUANT_H263_INTRA, ORC_UNQUANT_H263_INTER };
typedef struct OrcMpvUnquant {            /* what the functions read from MPVContext (libavcodec/mpegvideo.h:70-77,201-203,258) */
    uint16_t intra_matrix[64], inter_matrix[64];
    uint8_t  permutated[64], raster_end[64];      /* ScanTable of the scan in use (intra and inter tables are the same scan) */
    int32_t  y_dc_scale, c_dc_scale, q_scale_type, h263_aic, ac_pred;
} OrcMpvUnquant;
/* ff_init_scantable: permutation = IDCTDSPContext.idct_permutation, scan = ff_zigzag_direct / ff_alternate_vertical_scan */
void orc_mpv_init_scantable(const uint8_t permutation[64], const uint8_t scan[64], uint8_t permutated[64], uint8_t raster_end[64]);
/* n = block number inside the macroblock (0-3 luma, 4+ chroma: picks the DC scale), last_index = block_last_index[n] */
void orc_mpv_unquantize(int variant, const OrcMpvUnquant *p, int16_t *block, int n, int qscale, int last_index);
/* blk_n NULL: blocks come in macroblock order, n = index % 6 */
void orc_mpv_unquantize_batch(int variant, const OrcMpvUnquant *p, int16_t *blocks, int64_t nblocks, const uint8_t *blk_n,
                              const uint8_t *qscale, const int8_t *last_index);
/* AVFloatDSPContext (libavutil/float_dsp.h:24-210), ops numbered in the struct's member order.  dst/src are float (double for
 * the D ops); vector_fmul_window: src2 = the 2*len window, dst has 2*len elements; butterflies: dst = v1, src0 = v2, both
 * written; the scalar products leave their result in dst[0]. */
enum { ORC_FDSP_VECTOR_FMUL, ORC_FDSP_VECTOR_FMAC_SCALAR, ORC_FDSP_VECTOR_DMAC_SCALAR, ORC_FDSP_VECTOR_FMUL_SCALAR,
       ORC_FDSP_VECTOR_DMUL_SCALAR, ORC_FDSP_VECTOR_FMUL_WINDOW, ORC_FDSP_VECTOR_FMUL_ADD, ORC_FDSP_VECTOR_FMUL_REVERSE,
       ORC_FDSP_BUTTERFLIES_FLOAT, ORC_FDSP_SCALARPRODUCT_FLOAT, ORC_FDSP_VECTOR_DMUL, ORC_FDSP_SCALARPRODUCT_DOUBLE };
int  orc_float_dsp(int op, void *dst, const void *src0, const void *src1, const void *src2, double mul, int len);
/* H.264 residual add, 8 bit: kind 0 idct_add (4x4), 1 idct8_add, 2 idct_dc_add, 3 idct8_dc_add; clears the coefficients */
int  orc_h264_idct(int kind, uint8_t *dst, int16_t *block, ptrdiff_t stride);
int  orc_h264_idct_hbd(int depth, int kind, uint8_t *dst, int32_t *block, ptrdiff_t stride_bytes);   /* 9 / 10 / 12 / 14 bit: int32 coefficients, uint16 samples */
void orc_pixels_clamped(int kind, const int16_t *block, uint8_t *pixels, ptrdiff_t line_size);

/* ------------------------------------------------------------------ me_cmp */
/* fn: 0 sad, 1 sse, 2 pix_abs[idx>>2][idx&3]; idx for sad/sse: 0=16 wide,1=8,2=4 (sse only) */
int  orc_me_cmp(int fn, int idx, const uint8_t *blk1, const uint8_t *blk2, ptrdiff_t stride, int h);
int  orc_sum_abs_dctelem(const int16_t *block);
void orc_fdct(int kind, int is248, int16_t *block);   /* FDCTDSPContext.fdct / fdct248: kind 0 islow_8, 1 ifast, 2 islow_10 */
void orc_me_cmp_set_dct_algo(int algo);   /* fn 8 / 9 (dct_sad, dct_max): 0 = ff_jpeg_fdct_islow_8, 1 = ff_fdct_ifast */
int  orc_pixelutils_sad(int bits, const uint8_t *src1, ptrdiff_t stride1, const uint8_t *src2, ptrdiff_t stride2);
void orc_esa_frame(const uint8_t *cur, const uint8_t *ref, int linesize, int width, int height,
                   int mb_size, int search_param, int mb_row0, int mb_row1, int32_t *out_mv, uint64_t *out_cost);

/* ------------------------------------------------------------------ h264qpel / hpeldsp (8 bit) */
void orc_h264qpel(int avg, int size_idx, int pos, uint8_t *dst, const uint8_t *src, ptrdiff_t stride);
void orc_h264_weight_hbd(int depth, int idx, uint8_t *block, ptrdiff_t stride_bytes, int height, int log2_denom, int weight, int offset);
void orc_h264_biweight_hbd(int depth, int idx, uint8_t *dst, const uint8_t *src, ptrdiff_t stride_bytes, int height, int log2_denom,
                           int weightd, int weights, int offset);
int  orc_h264chroma_hbd(int avg, int idx, uint8_t *dst, const uint8_t *src, ptrdiff_t stride_bytes, int h, int x, int y);
void orc_emulated_edge_mc_hbd(uint8_t *buf, const uint8_t *src, ptrdiff_t buf_linesize, ptrdiff_t src_linesize,
                              int block_w, int block_h, int src_x, int src_y, int w, int h);
void orc_h264qpel_hbd(int depth /* 9, 10, 12, 14 */, int avg, int size_idx, int pos, uint8_t *dst, const uint8_t *src, ptrdiff_t stride_bytes);
void orc_h264qpel_hbd_batch(int depth, int n, const uint8_t *op, uint8_t *dstbase, const int64_t *dst_off, const uint8_t *srcbase,
                            const int64_t *src_off, ptrdiff_t stride_bytes);
void orc_h264qpel_batch(int n, const uint8_t *op, uint8_t *dstbase, const int64_t *dst_off, const uint8_t *srcbase,
                        const int64_t *src_off, ptrdiff_t stride);
int  orc_hpel(int tab, int size_idx, int xy, uint8_t *block, const uint8_t *pixels, ptrdiff_t line_size, int h);
void orc_emulated_edge_mc(uint8_t *buf, const uint8_t *src, ptrdiff_t buf_linesize, ptrdiff_t src_linesize,
                          int block_w, int block_h, int src_x, int src_y, int w, int h);
void orc_h264_weight(int idx, uint8_t *block, ptrdiff_t stride, int height, int log2_denom, int weight, int offset);
void orc_h264_biweight(int idx, uint8_t *dst, const uint8_t *src, ptrdiff_t stride, int height, int log2_denom,
                       int weightd, int weights, int offset);
int  orc_h264chroma(int avg, int idx, uint8_t *dst, const uint8_t *src, ptrdiff_t stride, int h, int x, int y);
/* b200_h264chroma_batch_device's operation list (op byte: bit0 avg, bits1-2 width index; xy byte: x | y << 3); -1 at an invalid op */
int  orc_h264chroma_batch(int64_t n, const uint8_t *op, const uint8_t *h, const uint8_t *xy, uint8_t *dstbase, const int64_t *dst_off,
                          const uint8_t *srcbase, const int64_t *src_off, ptrdiff_t stride);

/* ------------------------------------------------------------------ tx (float FFT / MDCT, power-of-two) */
typedef struct OrcTx OrcTx;
OrcTx *orc_tx_open(int type /*0 FFT, 1 MDCT, 6 RDFT (r2c forward, c2r inverse)*/, int inv, int len, float scale, unsigned flags);
void   orc_tx_close(OrcTx *t);
void   orc_tx_run(OrcTx *t, void *out, void *in, ptrdiff_t stride, int count, ptrdiff_t out_step, ptrdiff_t in_step);
/* the 32-bit fixed-point transforms (txi_oracle.c): type 4 AV_TX_INT32_FFT, 5 AV_TX_INT32_MDCT, power-of-two lengths */
typedef struct OrcTxD OrcTxD;
/* AV_TX_DOUBLE_FFT (2) / AV_TX_DOUBLE_MDCT (3), power-of-two lengths */
OrcTxD *orc_txd_open(int type, int inv, int len, double scale, unsigned flags);
void    orc_txd_close(OrcTxD *t);
void    orc_txd_run(OrcTxD *t, void *out, void *in, ptrdiff_t stride, int count, ptrdiff_t out_step, ptrdiff_t in_step);
typedef struct OrcTxI OrcTxI;
OrcTxI *orc_txi_open(int type, int inv, int len, float scale, unsigned flags);
void    orc_txi_close(OrcTxI *t);
void    orc_txi_run(OrcTxI *t, void *out, void *in, ptrdiff_t stride, int count, ptrdiff_t out_step, ptrdiff_t in_step);

#ifdef __cplusplus
}
#endif
#endif
