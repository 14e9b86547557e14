/*
 * b2enc_types.h -- plain-C data layouts shared by the CUDA encode stage, the
 * host entropy stage and the CPU oracle.  No CUDA / torch types.
 *
 * The reference (arkanis/video-encoder, av_encode.c) never sees these: they are
 * the hand-off between the pixel-parallel stage (device) and the serial
 * entropy/NAL stage (host), i.e. what lives *inside* x264_encoder_encode()
 * (av_encode.c:970).
 */
#ifndef B2ENC_TYPES_H
#define B2ENC_TYPES_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Replicated border kept around every luma plane held on the device (chroma: half).
 * >= merange(32) + 16 + 3 (6-tap) so that no search/interpolation read, and no TMA
 * box, ever leaves the allocation (SURVEY.md 7.2 item 4). */
#define B2_PAD   64
#define B2_PADC  32

enum { B2_MB_P16x16 = 0, B2_MB_I16x16 = 1, B2_MB_I4x4 = 2, B2_MB_I8x8 = 3 };   /* P16x16 = any inter MB, see `part` */
enum { B2_FRAME_I = 0, B2_FRAME_P = 1 };
/* raw input layouts accepted by the conversion kernel (the sws_scale source formats, av_encode.c:427) */
enum { B2_FMT_YUV420P = 0, B2_FMT_NV12 = 1, B2_FMT_YUYV422 = 2, B2_FMT_UYVY422 = 3,
       /* SURVEY.md 8f row N4: bgr24 is bit-exact against libswscale's dedicated converter; the other three go through
        * libswscale's fast-bilinear scaler, whose x86 code drifts along the row -- they are implemented drift-free and
        * pinned with a tolerance (oracle/b2o_convert.c) */
       B2_FMT_BGR24 = 4, B2_FMT_RGB24 = 5, B2_FMT_YUV422P = 6, B2_FMT_YUV411P = 7, B2_FMT_COUNT = 8 };

/* tight layout of one raw picture of format fmt: returns the number of planes (0: unknown format) and, per plane,
 * the bytes per row and the number of rows */
static inline int b2_fmt_layout(int fmt, int w, int h, int rowbytes[3], int rows[3])
{
    const int cw = (w + 1) / 2, ch = (h + 1) / 2;
    switch (fmt) {
    case B2_FMT_YUV420P: rowbytes[0] = w; rows[0] = h; rowbytes[1] = rowbytes[2] = cw; rows[1] = rows[2] = ch; return 3;
    case B2_FMT_NV12: rowbytes[0] = w; rows[0] = h; rowbytes[1] = 2 * cw; rows[1] = ch; rowbytes[2] = rows[2] = 0; return 2;
    case B2_FMT_YUYV422: case B2_FMT_UYVY422: rowbytes[0] = 2 * w; rows[0] = h; rowbytes[1] = rowbytes[2] = rows[1] = rows[2] = 0; return 1;
    case B2_FMT_BGR24: case B2_FMT_RGB24: rowbytes[0] = 3 * w; rows[0] = h; rowbytes[1] = rowbytes[2] = rows[1] = rows[2] = 0; return 1;
    case B2_FMT_YUV422P: rowbytes[0] = w; rows[0] = h; rowbytes[1] = rowbytes[2] = cw; rows[1] = rows[2] = h; return 3;
    case B2_FMT_YUV411P: rowbytes[0] = w; rows[0] = h; rowbytes[1] = rowbytes[2] = (w + 3) / 4; rows[1] = rows[2] = h; return 3;
    default: return 0;
    }
}
/* sizes for which the conversion is the closed form of oracle/b2o_convert.c (beyond them libswscale resamples the
 * chroma with a varying phase): packed 4:2:2 and rgb24 need even width and height, bgr24 an even width, planar 4:2:2 an
 * even height, planar 4:1:1 a width that is a multiple of 4 and an even height */
static inline int b2_fmt_size_ok(int fmt, int w, int h)
{
    switch (fmt) {
    case B2_FMT_YUYV422: case B2_FMT_UYVY422: case B2_FMT_RGB24: return !((w | h) & 1);
    case B2_FMT_BGR24: return !(w & 1);
    case B2_FMT_YUV422P: return !(h & 1);
    case B2_FMT_YUV411P: return !(w & 3) && !(h & 1);
    default: return 1;
    }
}

/* Slices (x264 i_slice_count).  A picture of mbh macroblock rows is cut into n = b2_slice_count(i_slice_count, mbh) row-aligned
 * slices; slice k covers rows [b2_slice_row(k, n, mbh), b2_slice_row(k + 1, n, mbh)).  Because slices are whole rows, the left
 * neighbour is always in the macroblock's own slice, and the top, top-left and top-right neighbours are unavailable exactly when
 * the row is the first of its slice (b2_slice_row0(mby, n, mbh) == mby).  0 or 1 means one slice. */
#if defined(__CUDACC__)
__host__ __device__
#endif
static inline int b2_slice_count(int slices, int mbh) { return slices < 1 ? 1 : (slices > mbh ? mbh : slices); }
#if defined(__CUDACC__)
__host__ __device__
#endif
static inline int b2_slice_row(int k, int n, int mbh) { return (k * mbh + n / 2) / n; }
/* first row of the slice that holds row r: slice k = max{k : b2_slice_row(k) <= r} = ((r + 1) n - n/2 - 1) / mbh */
#if defined(__CUDACC__)
__host__ __device__
#endif
static inline int b2_slice_row0(int r, int n, int mbh) { return b2_slice_row(((r + 1) * n - n / 2 - 1) / mbh, n, mbh); }

/* intra 16x16 modes (H.264 Table 8-4) */
enum { B2_I16_V = 0, B2_I16_H = 1, B2_I16_DC = 2, B2_I16_PLANE = 3 };
/* intra chroma modes (H.264 Table 8-5) */
enum { B2_IC_DC = 0, B2_IC_H = 1, B2_IC_V = 2, B2_IC_PLANE = 3 };
/* intra 4x4 modes (H.264 Table 8-2) */
enum { B2_I4_V = 0, B2_I4_H, B2_I4_DC, B2_I4_DDL, B2_I4_DDR, B2_I4_VR, B2_I4_HD, B2_I4_VL, B2_I4_HU };

typedef struct { int16_t x, y; } b2_mv_t;

enum { B2_PART_16x16 = 0, B2_PART_16x8 = 1, B2_PART_8x16 = 2, B2_PART_8x8 = 3 };

/* One macroblock's decisions: 48 bytes. */
typedef struct {
    int16_t  mvx, mvy;      /* quarter-pel motion vector of 8x8 quadrant 0 (= the MB's MV for      */
                            /* P16x16); 0 for intra                                                */
    uint8_t  mb_type;       /* B2_MB_*                                                             */
    uint8_t  i16_mode;      /* B2_I16_*  (mb_type == I16x16)                                       */
    uint8_t  chroma_mode;   /* B2_IC_*   (intra MBs)                                               */
    uint8_t  cbp;           /* bits 0-3: luma 8x8 quadrants, bits 4-5: chroma 0/1/2                */
    uint8_t  i4_mode[16];   /* B2_I4_* per 4x4 block, H.264 block-index (z) order; I8x8: the mode  */
                            /* of 8x8 block k in all of i4_mode[4k..4k+3]                          */
    uint32_t cost;          /* cost of the chosen mode (SATD + lambda*bits model)                  */
    uint32_t nnz_mask;      /* bit b (0-15 luma, 16-19 U AC, 20-23 V AC): block has a non-zero     */
                            /* level; bit 24 luma DC, bit 25 U DC, bit 26 V DC.  With the 8x8      */
                            /* transform bit 4q+k is the k-th interleaved quarter of 8x8 block q   */
    b2_mv_t  mv8[3];        /* quarter-pel MVs of 8x8 quadrants 1..3 when part != B2_PART_16x16    */
                            /* (zero otherwise: the whole MB moves by {mvx,mvy})                   */
    uint8_t  part;          /* B2_PART_* partition shape of an inter MB                            */
    uint8_t  transform8x8;  /* 1: the luma residual uses the 8x8 transform (transform_size_8x8_flag) */
    uint16_t i8_modes;      /* intra analysis with the 8x8 transform enabled: best B2_I4_* mode of 8x8 block k in    */
                            /* bits 4k..4k+3 (kept for every MB the analysis ran on, whatever type was chosen)     */
} b2_mbinfo_t;

/* What the serial stage needs of a b2_mbinfo_t, in 24 bytes: the record that crosses PCIe when the engine packs its results
 * (cfg.pack_levels).  Not shipped: `cost`, `i8_modes` (analysis by-products) and the intra analysis modes of macroblocks that
 * ended up inter.  w[0] = mvx | mvy << 16; w[1] = mb_type | i16_mode << 2 | chroma_mode << 4 | part << 6 | transform8x8 << 8 |
 * cbp << 16; w[2] = nnz_mask; w[3..5] = inter: mv8[0..2]; intra: i4_mode[16] as nibbles (w[3], w[4]). */
typedef struct { uint32_t w[6]; } b2_mbinfo_packed_t;

#if defined(__CUDACC__)
__host__ __device__
#endif
static inline b2_mbinfo_packed_t b2_mbinfo_pack(const b2_mbinfo_t *m)
{
    b2_mbinfo_packed_t p;
    const int intra = m->mb_type != B2_MB_P16x16;
    p.w[0] = (uint32_t)(uint16_t)m->mvx | (uint32_t)(uint16_t)m->mvy << 16;
    p.w[1] = (uint32_t)m->mb_type | (intra ? (uint32_t)m->i16_mode << 2 | (uint32_t)m->chroma_mode << 4 : 0u) | (uint32_t)m->part << 6 |
             (uint32_t)(m->transform8x8 != 0) << 8 | (uint32_t)m->cbp << 16;
    p.w[2] = m->nnz_mask;
    if (intra) {
        uint32_t a = 0, b = 0;
        for (int i = 0; i < 8; i++) { a |= (uint32_t)(m->i4_mode[i] & 15) << (4 * i); b |= (uint32_t)(m->i4_mode[8 + i] & 15) << (4 * i); }
        p.w[3] = a; p.w[4] = b; p.w[5] = 0;
    } else {
        for (int q = 0; q < 3; q++) p.w[3 + q] = (uint32_t)(uint16_t)m->mv8[q].x | (uint32_t)(uint16_t)m->mv8[q].y << 16;
    }
    return p;
}
static inline void b2_mbinfo_unpack(const b2_mbinfo_packed_t *p, b2_mbinfo_t *m)
{
    const uint32_t f = p->w[1];
    const int intra = (int)(f & 3u) != B2_MB_P16x16;
    m->mvx = (int16_t)(p->w[0] & 0xffffu); m->mvy = (int16_t)(p->w[0] >> 16);
    m->mb_type = (uint8_t)(f & 3u); m->i16_mode = (uint8_t)((f >> 2) & 3u); m->chroma_mode = (uint8_t)((f >> 4) & 3u);
    m->part = (uint8_t)((f >> 6) & 3u); m->transform8x8 = (uint8_t)((f >> 8) & 1u); m->cbp = (uint8_t)(f >> 16);
    m->cost = 0; m->nnz_mask = p->w[2]; m->i8_modes = 0;
    for (int i = 0; i < 16; i++) m->i4_mode[i] = intra ? (uint8_t)((p->w[3 + (i >> 3)] >> (4 * (i & 7))) & 15u) : 0;
    for (int q = 0; q < 3; q++) {
        m->mv8[q].x = intra ? 0 : (int16_t)(p->w[3 + q] & 0xffffu);
        m->mv8[q].y = intra ? 0 : (int16_t)(p->w[3 + q] >> 16);
    }
}

/* Quantised levels of one macroblock, each block in zig-zag scan order.
 *   blk 0..15  luma 4x4 (z order).  I16x16: index 0 is 0, DC lives in blk 24.
 *              With the 8x8 transform, blk[4q..4q+3] hold the 64 levels of 8x8 block q in 8x8 zig-zag order.
 *   blk 16..19 U AC, 20..23 V AC (index 0 is 0, DC lives in blk 25)
 *   blk 24     luma DC of an I16x16 MB (16 levels, zig-zag)
 *   blk 25     chroma DC: [0..3] U, [4..7] V (raster 2x2)                               */
#define B2_COEF_BLOCKS 26
typedef struct { int16_t blk[B2_COEF_BLOCKS][16]; } b2_mbcoef_t;   /* 832 bytes */

/* Packed levels (engine option pack_levels): per frame, macroblocks in raster order, and for every macroblock the
 * 32-byte blocks blk[b], b ascending, for which bit b of b2_coef_present() is set; absent blocks are all zero.
 * Blocks of an 8x8-transformed quadrant travel together (64 contiguous levels). */
#if defined(__CUDACC__)
__host__ __device__
#endif
static inline uint32_t b2_coef_present(const b2_mbinfo_t *m)
{
    uint32_t luma = m->nnz_mask & 0xffffu;
    if (m->transform8x8)
        for (int q = 0; q < 4; q++)
            if ((luma >> (4 * q)) & 15u) luma |= 15u << (4 * q);
    return luma | (m->nnz_mask & 0x01ff0000u) | ((m->nnz_mask & 0x06000000u) ? 1u << 25 : 0u);
}

#ifdef __cplusplus
}
#endif
#endif
