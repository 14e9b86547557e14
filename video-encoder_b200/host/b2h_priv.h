/*
 * b2h_priv.h -- state shared by the host slice writers (b2h_cavlc.c: CAVLC, parameter sets, slice header;
 * b2h_cabac.c: CABAC).  Internal to the host stage; not part of the C-ABI.
 */
#ifndef B2H_PRIV_H
#define B2H_PRIV_H
#include <string.h>
#include "b2h_bits.h"
#include "b2h_entropy.h"

/* per-encoder scratch: neighbour maps of the picture being written (raster order).  Slices are whole macroblock rows
 * (b2_slice_row, b2enc_types.h): a slice reads nothing above its first row, row0, so writers with their own scratch may code the
 * slices of one picture at the same time. */
struct b2h_entropy {
    int mbw, mbh;
    int row0;                /* first macroblock row of the slice being written                   */
    uint8_t *nnz_y;          /* [4mbh][4mbw] total_coeff of each luma 4x4                         */
    uint8_t *nnz_c[2];       /* [2mbh][2mbw] total_coeff of each chroma AC 4x4                    */
    int8_t *i4;              /* [4mbh][4mbw] intra4x4 pred mode (2 for non-I4x4 MBs)              */
    int8_t *ref4;            /* [4mbh][4mbw] reference index per 4x4: 0 inter, -1 intra           */
    b2_mv_t *mv4;            /* [4mbh][4mbw] motion vector per 4x4                                */
    uint8_t cbp_code_intra[48], cbp_code_inter[48];
    uint8_t *rbsp;
    size_t rbsp_cap;
    /* CABAC only (9.3.3.1.1: context increments read the left / top neighbours) */
    uint8_t *mbf;            /* [mbh][mbw] B2H_MBF_* flags                                        */
    uint8_t *cbp;            /* [mbh][mbw] coded_block_pattern (bits 0-3 luma, 4-5 chroma)        */
    uint8_t *cmode;          /* [mbh][mbw] intra_chroma_pred_mode (0 for inter MBs)               */
    uint8_t *mvd[2];         /* [4mbh][4mbw] |mvd_l0| per 4x4, x and y, saturated at 255          */
};
enum { B2H_MBF_SKIP = 1, B2H_MBF_INTRA = 2, B2H_MBF_I16 = 4, B2H_MBF_T8 = 8,
       B2H_MBF_DC_Y = 16, B2H_MBF_DC_U = 32, B2H_MBF_DC_V = 64 };      /* DC_*: coded_block_flag of that DC block */

/* where a slice writer reads the quantised levels of macroblock mi from: the dense array (832 B/MB) or the packed
 * stream of include/b2enc_types.h (b2_coef_present), which is walked in macroblock order */
typedef struct {
    const b2_mbcoef_t *dense;
    const uint8_t *packed;
    size_t pos, size;
} b2h_levels_t;
extern const int16_t b2h_zero_levels[64];
static inline void b2h_levels_mb(b2h_levels_t *lv, const b2_mbinfo_t *m, int mi, const int16_t *blk[B2_COEF_BLOCKS])
{
    if (lv->dense) {
        for (int b = 0; b < B2_COEF_BLOCKS; b++) blk[b] = lv->dense[mi].blk[b];
        return;
    }
    uint32_t pm = b2_coef_present(m);
    if (!pm && !m->cbp && m->mb_type != B2_MB_I16x16) return;     /* nothing coded: residual() does not look at blk[] */
    for (int b = 0; b < B2_COEF_BLOCKS; b++) blk[b] = b2h_zero_levels;
    while (pm) {                                          /* the few present blocks, in block order = stream order */
        const int b = __builtin_ctz(pm);
        pm &= pm - 1;
        if (lv->pos + 32 > lv->size) break;               /* truncated stream: the remaining blocks read as zero */
        blk[b] = (const int16_t *)(lv->packed + lv->pos);
        lv->pos += 32;
    }
}

/* Motion-vector prediction 8.4.1.3 (single reference frame) for the partition whose top-left 4x4 block is (x4,y4) in
 * picture coordinates and that is w4 blocks wide.  dir: B2H_PRED_MEDIAN, or the directional rule of 16x8 / 8x16
 * partitions (prefer neighbour A, B or C when it is inter).  The partitions of the macroblock being written must
 * already be in the maps (b2h_fill_mv) in coding order. */
enum { B2H_PRED_MEDIAN = 0, B2H_PRED_A = 1, B2H_PRED_B = 2, B2H_PRED_C = 3 };
static inline int b2h_median3(int a, int b, int c)
{
    int mn = a < b ? a : b, mx = a < b ? b : a;
    return c < mn ? mn : (c > mx ? mx : c);
}
/* (inline: the slice writers call these once or twice per macroblock with constant shapes) */
static inline b2_mv_t b2h_mv_pred(const b2h_entropy_t *e, int x4, int y4, int w4, int dir)
{
    const int st = 4 * e->mbw;
    b2_mv_t z = {0, 0}, mvA = z, mvB = z, mvC = z;
    int refA = -1, refB = -1, refC = -1;
    const int top = 4 * e->row0;                          /* first 4x4 row of the slice */
    const int hasA = x4 > 0, hasB = y4 > top;
    /* C = block above and to the right of the partition; it must lie inside the slice and precede the partition in
     * decoding order: always true in the macroblock row above, inside the current row only left of the MB's right edge */
    int hasC = y4 > top && x4 + w4 < st && ((y4 & 3) == 0 || (x4 & 3) + w4 < 4);
    if (hasA) { refA = e->ref4[y4 * st + x4 - 1]; mvA = e->mv4[y4 * st + x4 - 1]; }
    if (hasB) { refB = e->ref4[(y4 - 1) * st + x4]; mvB = e->mv4[(y4 - 1) * st + x4]; }
    if (hasC) { refC = e->ref4[(y4 - 1) * st + x4 + w4]; mvC = e->mv4[(y4 - 1) * st + x4 + w4]; }
    else if (x4 > 0 && y4 > top) { hasC = 1; refC = e->ref4[(y4 - 1) * st + x4 - 1]; mvC = e->mv4[(y4 - 1) * st + x4 - 1]; }   /* D */
    if (dir == B2H_PRED_A && refA == 0) return mvA;
    if (dir == B2H_PRED_B && refB == 0) return mvB;
    if (dir == B2H_PRED_C && refC == 0) return mvC;
    if (!hasB && !hasC && hasA) { mvB = mvA; mvC = mvA; refB = refA; refC = refA; }
    const int n = (refA == 0) + (refB == 0) + (refC == 0);
    if (n == 1) return refA == 0 ? mvA : (refB == 0 ? mvB : mvC);
    b2_mv_t p;
    p.x = (int16_t)b2h_median3(mvA.x, mvB.x, mvC.x);
    p.y = (int16_t)b2h_median3(mvA.y, mvB.y, mvC.y);
    return p;
}
/* inferred motion vector of P_Skip (8.4.1.1) for macroblock (mbx,mby) */
static inline b2_mv_t b2h_skip_mv(const b2h_entropy_t *e, int mbx, int mby)
{
    const int st = 4 * e->mbw, x4 = 4 * mbx, y4 = 4 * mby;
    b2_mv_t z = {0, 0};
    if (mbx == 0 || mby == e->row0) return z;
    const int iA = y4 * st + x4 - 1, iB = (y4 - 1) * st + x4;
    if (e->ref4[iA] == 0 && e->mv4[iA].x == 0 && e->mv4[iA].y == 0) return z;
    if (e->ref4[iB] == 0 && e->mv4[iB].x == 0 && e->mv4[iB].y == 0) return z;
    return b2h_mv_pred(e, x4, y4, 4, B2H_PRED_MEDIAN);
}
static inline void b2h_fill_mv(b2h_entropy_t *e, int x4, int y4, int w4, int h4, b2_mv_t mv, int ref)
{
    const int st = 4 * e->mbw;
    if (w4 == 4) {                                        /* whole rows of a macroblock: 16 + 4 bytes each */
        const b2_mv_t row[4] = {mv, mv, mv, mv};
        for (int y = y4; y < y4 + h4; y++) { memcpy(&e->mv4[y * st + x4], row, sizeof(row)); memset(&e->ref4[y * st + x4], ref, 4); }
        return;
    }
    for (int y = y4; y < y4 + h4; y++)
        for (int x = x4; x < x4 + w4; x++) { e->mv4[y * st + x] = mv; e->ref4[y * st + x] = (int8_t)ref; }
}
/* geometry of partition `idx` of shape `part` (B2_PART_*) inside the macroblock, in 4x4 units, and its prediction rule;
 * returns the number of partitions of the shape */
static inline int b2h_part_geom(int part, int idx, int *x, int *y, int *w, int *h, int *dir)
{
    switch (part) {
    case B2_PART_16x8: *x = 0; *y = 2 * idx; *w = 4; *h = 2; *dir = idx ? B2H_PRED_A : B2H_PRED_B; return 2;
    case B2_PART_8x16: *x = 2 * idx; *y = 0; *w = 2; *h = 4; *dir = idx ? B2H_PRED_C : B2H_PRED_A; return 2;
    case B2_PART_8x8: *x = 2 * (idx & 1); *y = 2 * (idx >> 1); *w = 2; *h = 2; *dir = B2H_PRED_MEDIAN; return 4;
    default: *x = 0; *y = 0; *w = 4; *h = 4; *dir = B2H_PRED_MEDIAN; return 1;
    }
}
/* motion vector of the 8x8 quadrant that contains 4x4 block (x,y) of macroblock m */
static inline b2_mv_t b2h_mb_mv(const b2_mbinfo_t *m, int x, int y)
{
    const int q = (x >> 1) | ((y >> 1) << 1);
    b2_mv_t mv = {m->mvx, m->mvy};
    if (q && m->part != B2_PART_16x16) mv = m->mv8[q - 1];
    return mv;
}
/* slice_header() 7.3.3 up to and including the deblocking fields */
void b2h_slice_header(bs_t *b, const b2h_seq_t *s, int is_p, int frame_num, int idr_pic_id, int first_mb);
/* rows [e->row0, e->row0 + nrows) */
size_t b2h_write_slice_cabac(b2h_entropy_t *e, const b2h_seq_t *s, int frame_type, int frame_num, int idr_pic_id, int nrows,
                             const b2_mbinfo_t *info, b2h_levels_t *lv, uint8_t *out, size_t cap);
extern const uint8_t b2h_blk_x[16], b2h_blk_y[16];

#endif
