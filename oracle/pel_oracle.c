/*
 * pel_oracle.c — TEST INFRASTRUCTURE ONLY.  CPU restatement of libavcodec's 8-bit H.264 quarter-pel and MPEG half-pel
 * motion-compensation interpolators.
 *
 * Follows (behaviour, not text):
 *   H264_LOWPASS h/v/hv .... libavcodec/h264qpel_template.c:77-305   taps (1,-5,20,20,-5,1); h and v: clip((t+16)>>5);
 *                                                                    hv: unrounded 16-bit horizontal sums over size+5 rows,
 *                                                                    then the vertical taps and clip((t+512)>>10)
 *   H264_MC mc00..mc33 ..... libavcodec/h264qpel_template.c:313-456  which of {full, h-half, v-half, hv-half} each
 *                                                                    quarter position averages ((a+b+1)>>1, pixelsN_l2)
 *   put / avg ops .......... libavcodec/h264qpel_template.c:461-465  avg: dst = (dst + value + 1) >> 1
 *   table index ............ libavcodec/h264qpel.c:50-104            [0:16,1:8,2:4][x + 4*y]
 *   hpeldsp PIXOP2 ......... libavcodec/hpeldsp.c:38-325             x2/y2: (a+b+1)>>1 (rnd) or (a+b)>>1 (no_rnd);
 *                                                                    xy2: (a+b+c+d+2)>>2 (rnd) or +1 (no_rnd);
 *                                                                    avg tables: dst = (dst + value + 1) >> 1 (rnd_avg32, rnd_avg.h:31-39)
 *   hpel table layout ...... libavcodec/hpeldsp.c:337-352            put[4 sizes 16,8,4,2], avg[4], put_no_rnd[2: 16,8], avg_no_rnd[16 only]
 *   h264chroma ............. libavcodec/h264chroma_template.c:27-176  bilinear eighth-pel: (A*p00 + B*p01 + C*p10 + D*p11 + 32) >> 6 with
 *                                                                    A=(8-x)(8-y), B=x(8-y), C=(8-x)y, D=xy; the reference's D==0 / B+C==0
 *                                                                    branches are the same value but skip the unused row / column reads;
 *                                                                    table libavcodec/h264chroma.c:36-44: [0]=8 wide, [1]=4, [2]=2
 *   emulated_edge_mc ....... libavcodec/videodsp_template.c:24-101   block_w x block_h window whose top-left sample is picture position
 *                                                                    (src_x, src_y); samples outside the w x h picture replicate the
 *                                                                    nearest border sample (the reference clamps the window so at least
 *                                                                    one row and column is inside, then copies and smears the edges)
 *   h264 weight / biweight . libavcodec/h264dsp_template.c:30-99        explicit weighted prediction on the motion-compensated block:
 *                                                                    clip((p*w + o') >> d) with o' = (o << d) + (d ? 1 << (d-1) : 0); and
 *                                                                    clip((s*ws + p*wd + o'') >> (d+1)) with o'' = ((o + 1) | 1) << d
 */
#include "oracle.h"

static int clip8(int v) { return v < 0 ? 0 : v > 255 ? 255 : v; }
static int tap6(int a, int b, int c, int d, int e, int f) { return a - 5 * b + 20 * c + 20 * d - 5 * e + f; }

/* the four sample planes at integer position (x,y) of the block: F full, H horizontal half (between x and x+1),
 * V vertical half (between y and y+1), J centre */
static int sF(const uint8_t *s, ptrdiff_t st, int x, int y) { return s[y * st + x]; }
static int sH(const uint8_t *s, ptrdiff_t st, int x, int y)
{
    const uint8_t *p = s + y * st + x;
    return clip8((tap6(p[-2], p[-1], p[0], p[1], p[2], p[3]) + 16) >> 5);
}
static int sV(const uint8_t *s, ptrdiff_t st, int x, int y)
{
    const uint8_t *p = s + y * st + x;
    return clip8((tap6(p[-2 * st], p[-st], p[0], p[st], p[2 * st], p[3 * st]) + 16) >> 5);
}
static int hraw(const uint8_t *s, ptrdiff_t st, int x, int y)
{
    const uint8_t *p = s + y * st + x;
    return tap6(p[-2], p[-1], p[0], p[1], p[2], p[3]);
}
static int sJ(const uint8_t *s, ptrdiff_t st, int x, int y)
{
    return clip8((tap6(hraw(s, st, x, y - 2), hraw(s, st, x, y - 1), hraw(s, st, x, y), hraw(s, st, x, y + 1),
                       hraw(s, st, x, y + 2), hraw(s, st, x, y + 3)) + 512) >> 10);
}

void orc_h264qpel(int avg, int size_idx, int pos, uint8_t *dst, const uint8_t *src, ptrdiff_t stride)
{
    const int size = 16 >> size_idx, qx = pos & 3, qy = pos >> 2;
    uint8_t out[16 * 16];
    for (int y = 0; y < size; y++)
        for (int x = 0; x < size; x++) {
            int v;
            if (qy == 0) {
                v = qx == 0 ? sF(src, stride, x, y) : qx == 2 ? sH(src, stride, x, y)
                  : (sF(src, stride, x + (qx == 3), y) + sH(src, stride, x, y) + 1) >> 1;
            } else if (qx == 0) {
                v = qy == 2 ? sV(src, stride, x, y) : (sF(src, stride, x, y + (qy == 3)) + sV(src, stride, x, y) + 1) >> 1;
            } else if (qx == 2 && qy == 2) {
                v = sJ(src, stride, x, y);
            } else if (qx == 2) {                   /* mc21, mc23 */
                v = (sH(src, stride, x, y + (qy == 3)) + sJ(src, stride, x, y) + 1) >> 1;
            } else if (qy == 2) {                   /* mc12, mc32 */
                v = (sV(src, stride, x + (qx == 3), y) + sJ(src, stride, x, y) + 1) >> 1;
            } else {                                /* mc11, mc31, mc13, mc33 */
                v = (sH(src, stride, x, y + (qy == 3)) + sV(src, stride, x + (qx == 3), y) + 1) >> 1;
            }
            out[y * 16 + x] = (uint8_t)v;
        }
    for (int y = 0; y < size; y++)
        for (int x = 0; x < size; x++)
            dst[y * stride + x] = avg ? (uint8_t)((dst[y * stride + x] + out[y * 16 + x] + 1) >> 1) : out[y * 16 + x];
}

/* ---- the same for 9 / 10 / 12 / 14 bit samples (h264qpel_template.c with BIT_DEPTH > 8, h264qpel.c:30-46; tables :87-103): uint16
 * pixels, clip = av_clip_uintp2(v, depth).  The 10-bit build biases its int16 horizontal sums by -10 * 1023 and removes the bias in
 * the vertical taps (h264qpel_template.c:131, :146-160): the sums never leave int16 either way, so no value changes.  stride in BYTES. */
typedef struct { const uint16_t *s; ptrdiff_t st; int maxv; } HbSrc;
static int hb_clip(const HbSrc *c, int v) { return v < 0 ? 0 : v > c->maxv ? c->maxv : v; }
static int hbF(const HbSrc *c, int x, int y) { return c->s[y * c->st + x]; }
static int hb_hraw(const HbSrc *c, int x, int y)
{
    const uint16_t *p = c->s + y * c->st + x;
    return tap6(p[-2], p[-1], p[0], p[1], p[2], p[3]);
}
static int hbH(const HbSrc *c, int x, int y) { return hb_clip(c, (hb_hraw(c, x, y) + 16) >> 5); }
static int hbV(const HbSrc *c, int x, int y)
{
    const uint16_t *p = c->s + y * c->st + x;
    const ptrdiff_t st = c->st;
    return hb_clip(c, (tap6(p[-2 * st], p[-st], p[0], p[st], p[2 * st], p[3 * st]) + 16) >> 5);
}
static int hbJ(const HbSrc *c, int x, int y)
{
    return hb_clip(c, (tap6(hb_hraw(c, x, y - 2), hb_hraw(c, x, y - 1), hb_hraw(c, x, y), hb_hraw(c, x, y + 1),
                            hb_hraw(c, x, y + 2), hb_hraw(c, x, y + 3)) + 512) >> 10);
}

void orc_h264qpel_hbd(int depth, int avg, int size_idx, int pos, uint8_t *dst8, const uint8_t *src8, ptrdiff_t stride)
{
    const int size = 16 >> size_idx, qx = pos & 3, qy = pos >> 2;
    const HbSrc c = { (const uint16_t *)src8, stride / 2, (1 << depth) - 1 };
    uint16_t *dst = (uint16_t *)dst8, out[16 * 16];
    for (int y = 0; y < size; y++)
        for (int x = 0; x < size; x++) {
            int v;
            if (qy == 0)
                v = qx == 0 ? hbF(&c, x, y) : qx == 2 ? hbH(&c, x, y) : (hbF(&c, x + (qx == 3), y) + hbH(&c, x, y) + 1) >> 1;
            else if (qx == 0)
                v = qy == 2 ? hbV(&c, x, y) : (hbF(&c, x, y + (qy == 3)) + hbV(&c, x, y) + 1) >> 1;
            else if (qx == 2 && qy == 2)
                v = hbJ(&c, x, y);
            else if (qx == 2)
                v = (hbH(&c, x, y + (qy == 3)) + hbJ(&c, x, y) + 1) >> 1;
            else if (qy == 2)
                v = (hbV(&c, x + (qx == 3), y) + hbJ(&c, x, y) + 1) >> 1;
            else
                v = (hbH(&c, x, y + (qy == 3)) + hbV(&c, x + (qx == 3), y) + 1) >> 1;
            out[y * 16 + x] = (uint16_t)v;
        }
    for (int y = 0; y < size; y++)
        for (int x = 0; x < size; x++) {
            uint16_t *d = dst + y * c.st + x;
            *d = avg ? (uint16_t)((*d + out[y * 16 + x] + 1) >> 1) : out[y * 16 + x];
        }
}

void orc_h264qpel_hbd_batch(int depth, int n, const uint8_t *op, uint8_t *dstbase, const int64_t *dst_off, const uint8_t *srcbase,
                            const int64_t *src_off, ptrdiff_t stride)
{
    for (int i = 0; i < n; i++)
        orc_h264qpel_hbd(depth, op[i] & 1, (op[i] >> 1) & 3, (op[i] >> 3) & 15, dstbase + dst_off[i], srcbase + src_off[i], stride);
}

/* h264chroma for 16-bit samples (h264chroma_template.c:27-176 with BIT_DEPTH 16; ff_h264chroma_init installs it for every depth above 8,
 * h264chroma.c:45-50): same weights, (sum + 32) >> 6, avg (a + b + 1) >> 1; the D == 0 and B + C == 0 forms skip the unused reads */
int orc_h264chroma_hbd(int avg, int idx, uint8_t *dst8, const uint8_t *src8, ptrdiff_t stride, int h, int x, int y)
{
    if (idx < 0 || idx > 2) return -1;
    const int w = 8 >> idx;
    const int A = (8 - x) * (8 - y), B = x * (8 - y), C = (8 - x) * y, D = x * y;
    const ptrdiff_t st = stride / 2;
    uint16_t *dst = (uint16_t *)dst8;
    const uint16_t *src = (const uint16_t *)src8;
    for (int j = 0; j < h; j++)
        for (int i = 0; i < w; i++) {
            const uint16_t *s = src + j * st + i;
            int v;
            if (D) v = A * s[0] + B * s[1] + C * s[st] + D * s[st + 1];
            else if (B + C) v = A * s[0] + (B + C) * s[C ? st : 1];
            else v = A * s[0];
            v = (v + 32) >> 6;
            uint16_t *d = dst + j * st + i;
            *d = (uint16_t)(avg ? (*d + v + 1) >> 1 : v);
        }
    return 0;
}

/* emulated_edge_mc for 16-bit samples (videodsp_template.c:24-101 with BIT_DEPTH 16): geometry in pixels, line sizes in bytes */
void orc_emulated_edge_mc_hbd(uint8_t *buf, const uint8_t *src, ptrdiff_t buf_linesize, ptrdiff_t src_linesize,
                              int block_w, int block_h, int src_x, int src_y, int w, int h)
{
    if (!w || !h) return;
    const uint8_t *origin = src - (ptrdiff_t)src_y * src_linesize - (ptrdiff_t)src_x * 2;
    for (int y = 0; y < block_h; y++) {
        int py = src_y + y;
        py = py < 0 ? 0 : py > h - 1 ? h - 1 : py;
        for (int x = 0; x < block_w; x++) {
            int px = src_x + x;
            px = px < 0 ? 0 : px > w - 1 ? w - 1 : px;
            *(uint16_t *)(buf + y * buf_linesize + 2 * x) = *(const uint16_t *)(origin + py * src_linesize + 2 * px);
        }
    }
}

/* weight / biweight for 9 / 10 / 12 / 14 bit samples (h264dsp_template.c:30-99 instantiated per depth): the offset is scaled to the
 * sample depth, the clip is av_clip_uintp2(v, depth) */
void orc_h264_weight_hbd(int depth, int idx, uint8_t *block8, ptrdiff_t stride, int height, int log2_denom, int weight, int offset)
{
    const int w = 16 >> idx, maxv = (1 << depth) - 1;
    uint16_t *block = (uint16_t *)block8;
    const ptrdiff_t st = stride / 2;
    offset = (int)((unsigned)offset << (log2_denom + (depth - 8)));
    if (log2_denom) offset += 1 << (log2_denom - 1);
    for (int y = 0; y < height; y++, block += st)
        for (int x = 0; x < w; x++) {
            const int v = (block[x] * weight + offset) >> log2_denom;
            block[x] = (uint16_t)(v < 0 ? 0 : v > maxv ? maxv : v);
        }
}

void orc_h264_biweight_hbd(int depth, int idx, uint8_t *dst8, const uint8_t *src8, ptrdiff_t stride, int height, int log2_denom,
                           int weightd, int weights, int offset)
{
    const int w = 16 >> idx, maxv = (1 << depth) - 1;
    uint16_t *dst = (uint16_t *)dst8;
    const uint16_t *src = (const uint16_t *)src8;
    const ptrdiff_t st = stride / 2;
    offset = (int)((unsigned)offset << (depth - 8));
    offset = (int)((unsigned)((offset + 1) | 1) << log2_denom);
    for (int y = 0; y < height; y++, dst += st, src += st)
        for (int x = 0; x < w; x++) {
            const int v = (src[x] * weights + dst[x] * weightd + offset) >> (log2_denom + 1);
            dst[x] = (uint16_t)(v < 0 ? 0 : v > maxv ? maxv : v);
        }
}

/* a list of operations, as ffref_h264qpel_batch / b200_h264qpel_batch_device take it (op byte: bit0 avg, bits1-2 size index, bits3-6 position) */
void orc_h264qpel_batch(int n, const uint8_t *op, uint8_t *dstbase, const int64_t *dst_off, const uint8_t *srcbase,
                        const int64_t *src_off, ptrdiff_t stride)
{
    for (int i = 0; i < n; i++)
        orc_h264qpel(op[i] & 1, (op[i] >> 1) & 3, (op[i] >> 3) & 15, dstbase + dst_off[i], srcbase + src_off[i], stride);
}

int orc_hpel(int tab, int size_idx, int xy, uint8_t *block, const uint8_t *pixels, ptrdiff_t ls, int h)
{
    const int w = 16 >> size_idx, no_rnd = tab >= 2;
    /* quirk kept from the reference: avg_pixels2_xy2 stores without averaging ("FIXME non put", hpeldsp.c:134-166) */
    const int avg = (tab & 1) && !(size_idx == 3 && xy == 3);
    if (tab == 2 && size_idx > 1) return -1;
    if (tab == 3 && size_idx != 0) return -1;
    uint8_t out[16 * 64];
    if (h > 64) return -1;
    for (int y = 0; y < h; y++)
        for (int x = 0; x < w; x++) {
            const uint8_t *p = pixels + y * ls + x;
            int v;
            switch (xy) {
            case 0:  v = p[0]; break;
            case 1:  v = (p[0] + p[1] + 1 - no_rnd) >> 1; break;
            case 2:  v = (p[0] + p[ls] + 1 - no_rnd) >> 1; break;
            default: v = (p[0] + p[1] + p[ls] + p[ls + 1] + 2 - no_rnd) >> 2; break;
            }
            out[y * 16 + x] = (uint8_t)v;
        }
    for (int y = 0; y < h; y++)
        for (int x = 0; x < w; x++)
            block[y * ls + x] = avg ? (uint8_t)((block[y * ls + x] + out[y * 16 + x] + 1) >> 1) : out[y * 16 + x];
    return 0;
}

int orc_h264chroma(int avg, int idx, uint8_t *dst, const uint8_t *src, ptrdiff_t stride, int h, int x, int y)
{
    if (idx < 0 || idx > 2 || x < 0 || x > 7 || y < 0 || y > 7) return -1;
    const int w = 8 >> idx;
    const int A = (8 - x) * (8 - y), B = x * (8 - y), C = (8 - x) * y, D = x * y;
    for (int i = 0; i < h; i++)
        for (int j = 0; j < w; j++) {
            const uint8_t *p = src + i * stride + j;
            int v = A * p[0];
            if (B) v += B * p[1];                 /* only touch the neighbours the reference touches */
            if (C) v += C * p[stride];
            if (D) v += D * p[stride + 1];
            v = (v + 32) >> 6;
            uint8_t *d = dst + i * stride + j;
            *d = (uint8_t)(avg ? (*d + v + 1) >> 1 : v);
        }
    return 0;
}

/* a list of operations, as b200_h264chroma_batch_device takes it (op byte: bit0 avg, bits1-2 width index; xy byte: x | y << 3),
 * applied in list order; -1 at the first invalid operation (the ones before it are done), else 0 */
int orc_h264chroma_batch(int64_t n, const uint8_t *op, const uint8_t *h, const uint8_t *xy, uint8_t *dstbase, const int64_t *dst_off,
                         const uint8_t *srcbase, const int64_t *src_off, ptrdiff_t stride)
{
    for (int64_t i = 0; i < n; i++)
        if (orc_h264chroma(op[i] & 1, (op[i] >> 1) & 3, dstbase + dst_off[i], srcbase + src_off[i], stride, h[i], xy[i] & 7, (xy[i] >> 3) & 7) < 0)
            return -1;
    return 0;
}

void orc_emulated_edge_mc(uint8_t *buf, const uint8_t *src, ptrdiff_t buf_linesize, ptrdiff_t src_linesize,
                          int block_w, int block_h, int src_x, int src_y, int w, int h)
{
    if (!w || !h) return;
    const uint8_t *origin = src - (ptrdiff_t)src_y * src_linesize - src_x;       /* picture sample (0, 0) */
    for (int y = 0; y < block_h; y++) {
        int py = src_y + y;
        py = py < 0 ? 0 : py > h - 1 ? h - 1 : py;
        for (int x = 0; x < block_w; x++) {
            int px = src_x + x;
            px = px < 0 ? 0 : px > w - 1 ? w - 1 : px;
            buf[y * buf_linesize + x] = origin[py * src_linesize + px];
        }
    }
}

static int clip255(int a) { return a < 0 ? 0 : a > 255 ? 255 : a; }

void orc_h264_weight(int idx, uint8_t *block, ptrdiff_t stride, int height, int log2_denom, int weight, int offset)
{
    const int w = 16 >> idx;
    offset = (int)((unsigned)offset << log2_denom);
    if (log2_denom) offset += 1 << (log2_denom - 1);
    for (int y = 0; y < height; y++, block += stride)
        for (int x = 0; x < w; x++) block[x] = (uint8_t)clip255((block[x] * weight + offset) >> log2_denom);
}

void orc_h264_biweight(int idx, uint8_t *dst, const uint8_t *src, ptrdiff_t stride, int height, int log2_denom,
                       int weightd, int weights, int offset)
{
    const int w = 16 >> idx;
    offset = (int)((unsigned)((offset + 1) | 1) << log2_denom);
    for (int y = 0; y < height; y++, dst += stride, src += stride)
        for (int x = 0; x < w; x++) dst[x] = (uint8_t)clip255((src[x] * weights + dst[x] * weightd + offset) >> (log2_denom + 1));
}
