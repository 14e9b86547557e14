/*
 * b2h_cabac.c -- H.264 CABAC slice writer (Main / High profile entropy coding): the serial host stage that
 * follows the CUDA encode stage when b_cabac is set (x264's default, as the reference opens it: preset
 * "medium", av_encode.c:102-105, :384).  Stands where the entropy-coding tail of x264_encoder_encode
 * (av_encode.c:970) stands in the reference; SURVEY.md 8f row N3.
 *
 * ITU-T H.264 9.3: context initialisation (9.3.1.1, Tables 9-12..9-23 -> b2h_cabac_ctx.h), binarisations
 * (9.3.2), context index derivation (9.3.3.1) and the arithmetic encoder (9.3.4.2: Figures 9-7..9-12).
 * Row-aligned slices (contexts initialised per slice), one reference frame, frame macroblocks only, constant QP (mb_qp_delta = 0).
 * Pinned by decoding the stream with libavcodec's H.264 decoder (tests/test_cabac.py).
 */
#include <pthread.h>
#include <stdlib.h>
#include <string.h>
#include "b2h_priv.h"
#include "b2h_cabac_ctx.h"

/* Table 9-44: rangeTabLPS[pStateIdx][qCodIRangeIdx] */
static const uint8_t range_lps[64][4] = {
    {128, 176, 208, 240}, {128, 167, 197, 227}, {128, 158, 187, 216}, {123, 150, 178, 205}, {116, 142, 169, 195},
    {111, 135, 160, 185}, {105, 128, 152, 175}, {100, 122, 144, 166}, {95, 116, 137, 158},  {90, 110, 130, 150},
    {85, 104, 123, 142},  {81, 99, 117, 135},   {77, 94, 111, 128},   {73, 89, 105, 122},   {69, 85, 100, 116},
    {66, 80, 95, 110},    {62, 76, 90, 104},    {59, 72, 86, 99},     {56, 69, 81, 94},     {53, 65, 77, 89},
    {51, 62, 73, 85},     {48, 59, 69, 80},     {46, 56, 66, 76},     {43, 53, 63, 72},     {41, 50, 59, 69},
    {39, 48, 56, 65},     {37, 45, 54, 62},     {35, 43, 51, 59},     {33, 41, 48, 56},     {32, 39, 46, 53},
    {30, 37, 43, 50},     {29, 35, 41, 48},     {27, 33, 39, 45},     {26, 31, 37, 43},     {24, 30, 35, 41},
    {23, 28, 33, 39},     {22, 27, 32, 37},     {21, 26, 30, 35},     {20, 24, 29, 33},     {19, 23, 27, 31},
    {18, 22, 26, 30},     {17, 21, 25, 28},     {16, 20, 23, 27},     {15, 19, 22, 25},     {14, 18, 21, 24},
    {14, 17, 20, 23},     {13, 16, 19, 22},     {12, 15, 18, 21},     {12, 14, 17, 20},     {11, 14, 16, 19},
    {11, 13, 15, 18},     {10, 12, 15, 17},     {10, 12, 14, 16},     {9, 11, 13, 15},      {9, 11, 12, 14},
    {8, 10, 12, 14},      {8, 9, 11, 13},       {7, 9, 11, 12},       {7, 9, 10, 12},       {7, 8, 10, 11},
    {6, 8, 9, 11},        {6, 7, 9, 10},        {6, 7, 8, 9},         {2, 2, 2, 2}};
/* Table 9-45: transIdxLPS (transIdxMPS = min(pStateIdx + 1, 62)) */
static const uint8_t trans_lps[64] = {0,  0,  1,  2,  2,  4,  4,  5,  6,  7,  8,  9,  9,  11, 11, 12, 13, 13, 15, 15, 16, 16,
                                      18, 18, 19, 19, 21, 21, 22, 22, 23, 24, 24, 25, 26, 26, 27, 27, 28, 29, 29, 30, 30, 30,
                                      31, 32, 32, 33, 33, 33, 34, 34, 35, 35, 35, 36, 36, 36, 37, 37, 37, 38, 38, 63};

/* ctxIdxOffset per ctxBlockCat 0..4 (Table 9-34, frame coded); cat 5 = luma 8x8 (ctxIdx 402 / 417 / 426) */
static const uint16_t cbf_base[5] = {85 + 0, 85 + 4, 85 + 8, 85 + 12, 85 + 16};
static const uint16_t sig_base[6] = {105 + 0, 105 + 15, 105 + 29, 105 + 44, 105 + 47, 402};
static const uint16_t last_base[6] = {166 + 0, 166 + 15, 166 + 29, 166 + 44, 166 + 47, 417};
static const uint16_t abs_base[6] = {227 + 0, 227 + 10, 227 + 20, 227 + 30, 227 + 39, 426};
/* Table 9-43, frame coded: ctxIdxInc of significant_coeff_flag / last_significant_coeff_flag for 8x8 blocks */
static const uint8_t sig8_inc[63] = {0,  1,  2,  3,  4,  5,  5,  4,  4,  3,  3,  4,  4,  4,  5,  5,  4,  4,  4,  4,  3,
                                     3,  6,  7,  7,  7,  8,  9,  10, 9,  8,  7,  7,  6,  11, 12, 13, 11, 6,  7,  8,  9,
                                     14, 10, 9,  8,  6,  11, 12, 13, 11, 6,  9,  14, 10, 9,  11, 12, 13, 11, 14, 10, 12};
static const uint8_t last8_inc[63] = {0, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2,
                                      3, 3, 3, 3, 3, 3, 3, 3, 4, 4, 4, 4, 4, 4, 4, 4, 5, 5, 5, 5, 6, 6, 6, 6, 7, 7, 7, 7, 8, 8, 8};

/* ---- arithmetic encoder (9.3.4.2) --------------------------------------------------------------------*/
/* Same interval arithmetic as Figures 9-7..9-12, organised for speed (this stage is what bounds a single stream on the host:
 * one bin is one link of a serial dependency chain):
 *  - the interval (low, range) and the count of pending bits live in a small struct of their own that never leaves the
 *    always-inlined coding functions, so the compiler keeps them in registers across a whole slice;
 *  - instead of one PutBit per renormalisation shift (with its outstanding-bit loop) the low end of the interval is kept in a
 *    64-bit register together with `queue + 18` not-yet-written bits; FOUR whole bytes leave at once (one hard-to-predict
 *    branch and one call per 32 bits of output instead of per 8), and a carry is added to the bytes already in the buffer
 *    (the whole RBSP is in memory, so no count of outstanding 0xff bytes is needed; a carry never leaves the first byte);
 *  - the chain through `range` is short: an MPS renormalises by 0 or 1 bit (range - rLPS >= 128), which is an add and a
 *    select; for an LPS the renormalised range and its shift depend on (state, range quarter) only and come from tables. */
typedef struct {
    uint8_t *p, *start, *end;   /* output cursor inside the RBSP buffer */
    int overflow;
    uint16_t state[1024];       /* (pStateIdx << 1) | valMPS.  Not a byte type on purpose: a store through a character type may alias
                                 * everything else, which would force the compiler to reload pointers and tables after every bin */
} cabac_t;
typedef struct {
    uint64_t low;
    uint32_t range;
    int queue;                  /* bits pending in `low` beyond the last byte boundary, minus 18 */
} cabac_reg_t;
#define CABAC_INLINE static inline __attribute__((always_inline))

static uint8_t cabac_next[128][2];          /* state after coding bin b in state s                          */
static uint8_t cabac_lps[128][4];           /* rangeTabLPS by (state, range quarter)                        */
static uint16_t cabac_lps_norm[128][4];     /* the same, renormalised (<< cabac_lps_shift)                  */
static uint8_t cabac_lps_shift[128][4];
static pthread_once_t cabac_tables_once = PTHREAD_ONCE_INIT;      /* slices are written by several entropy workers */

static void cabac_tables(void)
{
    for (int st = 0; st < 128; st++) {
        const int ps = st >> 1, mps = st & 1;
        cabac_next[st][mps] = (uint8_t)(((ps < 62 ? ps + 1 : 62) << 1) | mps);
        cabac_next[st][1 - mps] = (uint8_t)((trans_lps[ps] << 1) | (ps == 0 ? 1 - mps : mps));
        for (int q = 0; q < 4; q++) {
            int r = range_lps[ps][q], sh = 0;
            while ((r << sh) < 256) sh++;
            cabac_lps[st][q] = (uint8_t)r; cabac_lps_norm[st][q] = (uint16_t)(r << sh); cabac_lps_shift[st][q] = (uint8_t)sh;
        }
    }
}

static void cabac_init(cabac_t *c, cabac_reg_t *r, bs_t *bs, int table, int qp)
{
    pthread_once(&cabac_tables_once, cabac_tables);
    c->p = c->start = bs->buf + bs->pos; c->end = bs->buf + bs->cap; c->overflow = 0;
    r->low = 0; r->range = 510; r->queue = -9;                                           /* the first bit is not written */
    for (int i = 0; i < 1024; i++) {
        int pre = ((b2h_cabac_ctx_init[table][i][0] * qp) >> 4) + b2h_cabac_ctx_init[table][i][1];
        pre = pre < 1 ? 1 : (pre > 126 ? 126 : pre);
        c->state[i] = pre <= 63 ? (uint16_t)((63 - pre) << 1) : (uint16_t)(((pre - 64) << 1) | 1);
    }
}
/* a carry out of the pending bits goes into the bytes already written */
static inline void cabac_carry(cabac_t *c)
{
    uint8_t *q = c->p;
    while (q > c->start && ++*--q == 0) ;
}
/* four finished bytes (plus a possible carry in bit 32) leave the register */
static __attribute__((noinline)) void cabac_flush4(cabac_t *c, uint64_t out)
{
    if (c->p + 4 > c->end) { c->overflow = 1; return; }
    if (out >> 32) cabac_carry(c);
    c->p[0] = (uint8_t)(out >> 24); c->p[1] = (uint8_t)(out >> 16); c->p[2] = (uint8_t)(out >> 8); c->p[3] = (uint8_t)out;
    c->p += 4;
}
CABAC_INLINE void cabac_put(cabac_t *c, cabac_reg_t *r)
{
    if (__builtin_expect(r->queue >= 24, 0)) {
        const int keep = r->queue - 24 + 10;                 /* bits that stay: the 10-bit window and the pending bits below 32 */
        const uint64_t out = r->low >> keep;
        r->low &= ((uint64_t)1 << keep) - 1;
        r->queue -= 32;
        cabac_flush4(c, out);
    }
}
CABAC_INLINE void cabac_encode_r(cabac_t *c, cabac_reg_t *r, int ctx, int bin)
{
    const unsigned st = c->state[ctx];
    const unsigned idx = st * 4 + (r->range >> 6) - 4;                 /* range is in [256, 510]: range >> 6 = 4..7 */
    const uint32_t rlps = (&cabac_lps[0][0])[idx];
    const uint32_t lps = 0u - (uint32_t)((bin ^ st) & 1);              /* all ones when the bin is the less probable symbol: */
    const uint32_t range_l = (&cabac_lps_norm[0][0])[idx] & lps;       /* no branch on a value that is hard to predict     */
    const unsigned sh_l = (&cabac_lps_shift[0][0])[idx];
    c->state[ctx] = cabac_next[st][bin];
    const uint32_t rmps = r->range - rlps;                             /* in [128, 510): an MPS shifts by one bit at most */
    const unsigned sh_m = (rmps >> 8) ^ 1;
    const uint32_t range_m = (rmps & 0x100) ? rmps : rmps + rmps;
    const unsigned sh = sh_m ^ ((sh_m ^ sh_l) & lps);
    r->range = (range_m & ~lps) | range_l;
    r->low = (r->low + (rmps & lps)) << sh;
    r->queue += (int)sh;
    cabac_put(c, r);
}
CABAC_INLINE void cabac_bypass_r(cabac_t *c, cabac_reg_t *r, int bin)
{
    r->low <<= 1;
    if (bin) r->low += r->range;
    r->queue += 1;
    cabac_put(c, r);
}
/* end_of_slice_flag / I_PCM flag.  bin = 1 also flushes (9.3.4.5): all pending bits of `low` are written, the lowest one
 * forced to 1 -- it is the rbsp_stop_one_bit -- and the last byte is padded with zeros */
CABAC_INLINE void cabac_terminate_r(cabac_t *c, cabac_reg_t *r, int bin)
{
    r->range -= 2;
    if (!bin) {
        const int sh = __builtin_clz(r->range) - 23;         /* range >= 254 here: 0 or 1 */
        r->range <<= sh; r->low <<= sh; r->queue += sh;
        cabac_put(c, r);
        return;
    }
    r->low += r->range;
    r->low |= 1;
    int nb = r->queue + 18;                                  /* pending bits (a carry may sit above them); at most 49 */
    const int pad = (8 - (nb & 7)) & 7;
    const uint64_t v = r->low << pad;
    nb += pad;
    if (c->p + nb / 8 > c->end) { c->overflow = 1; return; }
    if (v >> nb) cabac_carry(c);
    while (nb > 0) { nb -= 8; *c->p++ = (uint8_t)(v >> nb); }
}
/* k-th order Exp-Golomb suffix in bypass mode (9.3.2.3) */
CABAC_INLINE void cabac_egk_r(cabac_t *c, cabac_reg_t *r, unsigned v, int k)
{
    for (;;) {
        if (v >= (1u << k)) { cabac_bypass_r(c, r, 1); v -= 1u << k; k++; }
        else {
            cabac_bypass_r(c, r, 0);
            while (k--) cabac_bypass_r(c, r, (int)((v >> k) & 1));
            break;
        }
    }
}
/* every coding function below has the coder `c` and the interval registers `r` in scope under these names */
#define cabac_encode(c, ctx, bin) cabac_encode_r(c, r, ctx, bin)
#define cabac_bypass(c, bin) cabac_bypass_r(c, r, bin)
#define cabac_terminate(c, bin) cabac_terminate_r(c, r, bin)
#define cabac_egk(c, v, k) cabac_egk_r(c, r, v, k)

/* Test hooks (tests/test_cabac_coder.py; not part of the C-ABI): the arithmetic coder alone on a caller-made list of bins,
 * compared there with a literal transcription of Figures 9-7..9-12.  op = ctxIdx << 2 | bin, ctxIdx 1024 = bypass,
 * 1025 = terminate; state[] = (pStateIdx << 1) | valMPS per context.  Returns the bytes written (0 on overflow). */
size_t b2h_cabac_code_bins(const uint32_t *ops, size_t n, const uint8_t *state, uint8_t *out, size_t cap)
{
    cabac_t cb, *c = &cb;
    cabac_reg_t rg = {0, 510, -9}, *r = &rg;
    pthread_once(&cabac_tables_once, cabac_tables);
    c->p = c->start = out; c->end = out + cap; c->overflow = 0;
    for (int i = 0; i < 1024; i++) c->state[i] = state[i];
    for (size_t i = 0; i < n; i++) {
        const unsigned ctx = ops[i] >> 2;
        const int bin = (int)(ops[i] & 1);
        if (ctx < 1024) cabac_encode(c, (int)ctx, bin);
        else if (ctx == 1024) cabac_bypass(c, bin);
        else cabac_terminate(c, bin);
    }
    return c->overflow ? 0 : (size_t)(c->p - c->start);
}
const uint8_t *b2h_cabac_table(int which) { return which == 0 ? &range_lps[0][0] : trans_lps; }      /* 64 x 4, 64 */

/* ---- residual_block_cabac (7.3.5.3.3) -----------------------------------------------------------------*/
/* l[0..maxn) in scan order.  cbf_inc < 0: coded_block_flag is not sent (cat 5).  Returns the number of non-zero levels. */
/* any non-zero level among l[0..n)?  (most blocks of a coded 8x8 quadrant are empty: word-wise test, no per-level branch) */
static inline int levels_any(const int16_t *l, int n)
{
    uint64_t acc = 0, w;
    int i = 0;
    for (; i + 4 <= n; i += 4) { memcpy(&w, l + i, 8); acc |= w; }
    for (; i < n; i++) acc |= (uint16_t)l[i];
    return acc != 0;
}

/* always inlined: `cat` and `maxn` are constants at every call site, so the context selection folds away */
CABAC_INLINE int cabac_residual(cabac_t *c, cabac_reg_t *r, int cat, const int16_t *l, int maxn, int cbf_inc)
{
    int last = -1;
    if (levels_any(l, maxn)) { last = maxn - 1; while (!l[last]) last--; }
    if (cbf_inc >= 0) {
        cabac_encode(c, cbf_base[cat] + cbf_inc, last >= 0);
        if (last < 0) return 0;
    }
    /* significance map: positions before `last` carry (sig, last = 0), `last` itself (1, 1) unless it is the final position
     * of the block, whose significance is inferred; the non-zero levels are collected on the way for the level pass */
    int16_t nzv[64];
    int nnz = 0;
    for (int i = 0; i < last; i++) {
        const int inc_s = cat == 5 ? sig8_inc[i] : cat == 3 ? (i < 2 ? i : 2) : i;
        const int v = l[i];
        cabac_encode(c, sig_base[cat] + inc_s, v != 0);
        if (v) {
            const int inc_l = cat == 5 ? last8_inc[i] : cat == 3 ? (i < 2 ? i : 2) : i;
            cabac_encode(c, last_base[cat] + inc_l, 0);
            nzv[nnz++] = (int16_t)v;
        }
    }
    if (last < maxn - 1) {
        const int inc_s = cat == 5 ? sig8_inc[last] : cat == 3 ? (last < 2 ? last : 2) : last;
        const int inc_l = cat == 5 ? last8_inc[last] : cat == 3 ? (last < 2 ? last : 2) : last;
        cabac_encode(c, sig_base[cat] + inc_s, 1);
        cabac_encode(c, last_base[cat] + inc_l, 1);
    }
    nzv[nnz++] = l[last];
    int gt1 = 0, eq1 = 0;
    for (int j = nnz - 1; j >= 0; j--) {                               /* levels in reverse scan order */
        const int lv = nzv[j];
        const unsigned a = (unsigned)abs(lv) - 1;
        const int inc0 = gt1 ? 0 : (1 + eq1 < 4 ? 1 + eq1 : 4);
        cabac_encode(c, abs_base[cat] + inc0, a > 0);
        if (a > 0) {
            const int cap = 4 - (cat == 3);
            const int ctx = abs_base[cat] + 5 + (gt1 < cap ? gt1 : cap);
            const unsigned pre = a < 14 ? a : 14;
            for (unsigned k = 1; k < pre; k++) cabac_encode(c, ctx, 1);
            if (a < 14) cabac_encode(c, ctx, 0);
            else cabac_egk(c, a - 14, 0);
            gt1++;
        } else {
            eq1++;
        }
        cabac_bypass(c, lv < 0);
    }
    return gt1 + eq1;                                                  /* every non-zero level counted exactly once */
}

/* ---- neighbour helpers ------------------------------------------------------------------------------------*/
typedef struct {
    int availA, availB;         /* left / top macroblock inside the picture                       */
    int fA, fB;                 /* their B2H_MBF_* flags (0 when unavailable)                     */
    int cbpA, cbpB;             /* their coded_block_pattern (0 when unavailable)                 */
} nb_t;

/* coded_block_flag increment (9.3.3.1.1.9) from the neighbouring blocks' flags; flagN < 0: block "not available"
 * inside an available macroblock (-> 0), availN == 0: macroblock unavailable (-> 1 for intra, 0 for inter) */
static inline int cbf_term(int availN, int flagN, int cur_intra)
{
    if (!availN) return cur_intra;
    return flagN > 0;
}

CABAC_INLINE void cabac_mvd(cabac_t *c, cabac_reg_t *r, int base, int sum, int v)
{
    const unsigned a = (unsigned)abs(v);
    const unsigned pre = a < 9 ? a : 9;
    int ctx = base + (sum < 3 ? 0 : (sum > 32 ? 2 : 1));
    for (unsigned k = 0; k < pre; k++) {
        cabac_encode(c, ctx, 1);
        ctx = base + (k < 3 ? 3 + (int)k : 6);
    }
    if (a < 9) cabac_encode(c, ctx, 0);
    else cabac_egk(c, a - 9, 3);
    if (a) cabac_bypass(c, v < 0);
}

/* mb_type of an intra macroblock: I-slice binarisation (Table 9-36) with the context layout of I slices
 * (base 3, first bin with neighbour increment) or of the intra suffix in P slices (base 17) */
CABAC_INLINE void cabac_mb_type_intra(cabac_t *c, cabac_reg_t *r, const b2_mbinfo_t *m, int is_p, int inc0)
{
    const int i16 = m->mb_type == B2_MB_I16x16;
    const int b0 = is_p ? 17 : 3 + inc0;
    cabac_encode(c, b0, i16);
    if (!i16) return;
    cabac_terminate(c, 0);                                         /* not I_PCM */
    const int s = is_p ? 17 : 3 + 2;                                /* context of bin k >= 2: s + ... */
    const int cbp_l = m->cbp & 15, cbp_c = m->cbp >> 4;
    cabac_encode(c, s + 1, cbp_l != 0);
    cabac_encode(c, s + 2, cbp_c != 0);
    if (cbp_c) cabac_encode(c, s + 2 + (is_p ? 0 : 1), cbp_c == 2);
    cabac_encode(c, s + 3 + (is_p ? 0 : 1), (m->i16_mode >> 1) & 1);
    cabac_encode(c, s + 3 + (is_p ? 0 : 2), m->i16_mode & 1);
}

/* ---- slice ---------------------------------------------------------------------------------------------------*/
size_t b2h_write_slice_cabac(b2h_entropy_t *e, const b2h_seq_t *s, int frame_type, int frame_num, int idr_pic_id, int nrows,
                             const b2_mbinfo_t *info, b2h_levels_t *lv, uint8_t *out, size_t cap)
{
    bs_t bs, *b = &bs;
    cabac_t cb, *c = &cb;
    cabac_reg_t rg, *r = &rg;
    const int mbw = e->mbw, row0 = e->row0, is_p = frame_type == B2_FRAME_P;
    const int last = (row0 + nrows) * mbw - 1;                                 /* the slice's last macroblock */
    const int ys = 4 * mbw, cs = 2 * mbw, y4top = 4 * row0, y2top = 2 * row0;
    const uint8_t *blk_x = b2h_blk_x, *blk_y = b2h_blk_y;
    bs_init(b, e->rbsp, e->rbsp_cap);
    b2h_slice_header(b, s, is_p, frame_num, idr_pic_id, row0 * mbw);
    if (b->nbits) bs_put(b, 8 - b->nbits, (1u << (8 - b->nbits)) - 1);    /* cabac_alignment_one_bit */
    cabac_init(c, r, b, is_p ? 1 : 0, s->qp);                                  /* cabac_init_idc 0 */

    for (int mby = row0; mby < row0 + nrows; mby++)
        for (int mbx = 0; mbx < mbw; mbx++) {
            const int mi = mby * mbw + mbx;
            const b2_mbinfo_t *m = &info[mi];
            const int16_t *cblk[B2_COEF_BLOCKS];
            b2h_levels_mb(lv, m, mi, cblk);
            const int cbp_l = m->cbp & 15, cbp_c = m->cbp >> 4;
            const int intra = m->mb_type != B2_MB_P16x16;
            nb_t nb;
            nb.availA = mbx > 0; nb.availB = mby > row0;
            nb.fA = nb.availA ? e->mbf[mi - 1] : 0; nb.fB = nb.availB ? e->mbf[mi - mbw] : 0;
            nb.cbpA = nb.availA ? e->cbp[mi - 1] : 0; nb.cbpB = nb.availB ? e->cbp[mi - mbw] : 0;
            /* reset this MB's neighbour state; filled in below as syntax elements are coded */
            for (int r = 0; r < 4; r++) {
                memset(e->nnz_y + (mby * 4 + r) * ys + mbx * 4, 0, 4); memset(e->i4 + (mby * 4 + r) * ys + mbx * 4, 2, 4);
                memset(e->mvd[0] + (mby * 4 + r) * ys + mbx * 4, 0, 4); memset(e->mvd[1] + (mby * 4 + r) * ys + mbx * 4, 0, 4);
            }
            for (int p = 0; p < 2; p++)
                for (int r = 0; r < 2; r++) memset(e->nnz_c[p] + (mby * 2 + r) * cs + mbx * 2, 0, 2);
            e->mbf[mi] = 0; e->cbp[mi] = 0; e->cmode[mi] = 0;
            int flags = intra ? B2H_MBF_INTRA : 0;
            if (m->mb_type == B2_MB_I16x16) flags |= B2H_MBF_I16;
            const int t8 = m->transform8x8 && s->transform8x8 && m->mb_type != B2_MB_I16x16 && (intra || cbp_l);
            if (t8) flags |= B2H_MBF_T8;

            if (!intra) {
                int skip = 0;
                if (m->part == B2_PART_16x16 && m->cbp == 0) {
                    const b2_mv_t skipmv = b2h_skip_mv(e, mbx, mby);
                    skip = m->mvx == skipmv.x && m->mvy == skipmv.y;
                    if (skip) b2h_fill_mv(e, mbx * 4, mby * 4, 4, 4, skipmv, 0);
                }
                cabac_encode(c, 11 + (nb.availA && !(nb.fA & B2H_MBF_SKIP)) + (nb.availB && !(nb.fB & B2H_MBF_SKIP)), skip);
                if (skip) {
                    e->mbf[mi] = B2H_MBF_SKIP;
                    cabac_terminate(c, mi == last);                     /* end_of_slice_flag */
                    continue;
                }
                /* mb_type (Table 9-36, P slices): 16x16 "000", 8x8 "001", 16x8 "011", 8x16 "010" */
                cabac_encode(c, 14, 0);
                if (m->part == B2_PART_16x16 || m->part == B2_PART_8x8) { cabac_encode(c, 15, 0); cabac_encode(c, 16, m->part == B2_PART_8x8); }
                else { cabac_encode(c, 15, 1); cabac_encode(c, 17, m->part == B2_PART_16x8); }
                if (m->part == B2_PART_8x8)
                    for (int k = 0; k < 4; k++) cabac_encode(c, 21, 1);                      /* sub_mb_type P_L0_8x8 */
                {
                    int px, py, pw, ph, dir;
                    const int np = b2h_part_geom(m->part, 0, &px, &py, &pw, &ph, &dir);
                    for (int a = 0; a < np; a++) {
                        b2h_part_geom(m->part, a, &px, &py, &pw, &ph, &dir);
                        const int x4 = mbx * 4 + px, y4 = mby * 4 + py;
                        const b2_mv_t mv = b2h_mb_mv(m, px, py);
                        const b2_mv_t mvp = b2h_mv_pred(e, x4, y4, pw, dir);
                        const int d[2] = {mv.x - mvp.x, mv.y - mvp.y};
                        for (int k = 0; k < 2; k++) {
                            /* |mvd| of the 4x4 blocks left of / above the partition (0 outside the slice, in intra and skipped MBs) */
                            const int sum = (x4 > 0 ? e->mvd[k][y4 * ys + x4 - 1] : 0) + (y4 > y4top ? e->mvd[k][(y4 - 1) * ys + x4] : 0);
                            cabac_mvd(c, r, k ? 47 : 40, sum, d[k]);
                        }
                        const int ax = abs(d[0]) > 255 ? 255 : abs(d[0]), ay = abs(d[1]) > 255 ? 255 : abs(d[1]);
                        for (int r = 0; r < ph; r++) { memset(e->mvd[0] + (y4 + r) * ys + x4, ax, (size_t)pw); memset(e->mvd[1] + (y4 + r) * ys + x4, ay, (size_t)pw); }
                        b2h_fill_mv(e, x4, y4, pw, ph, mv, 0);
                    }
                }
            } else {
                { b2_mv_t z = {0, 0}; b2h_fill_mv(e, mbx * 4, mby * 4, 4, 4, z, -1); }   /* inter MBs fill their blocks partition by partition */
                if (is_p) {
                    cabac_encode(c, 11 + (nb.availA && !(nb.fA & B2H_MBF_SKIP)) + (nb.availB && !(nb.fB & B2H_MBF_SKIP)), 0);
                    cabac_encode(c, 14, 1);                            /* prefix: intra macroblock in a P slice */
                }
                /* ctxIdxInc of the first mb_type bin in I slices: neighbour is available and not I_NxN */
                const int nxnA = (nb.fA & B2H_MBF_INTRA) && !(nb.fA & B2H_MBF_I16), nxnB = (nb.fB & B2H_MBF_INTRA) && !(nb.fB & B2H_MBF_I16);
                cabac_mb_type_intra(c, r, m, is_p, (nb.availA && !nxnA) + (nb.availB && !nxnB));
                if (m->mb_type != B2_MB_I16x16) {
                    if (s->transform8x8) cabac_encode(c, 399 + ((nb.fA & B2H_MBF_T8) != 0) + ((nb.fB & B2H_MBF_T8) != 0), t8);
                    const int step = t8 ? 4 : 1;
                    for (int k = 0; k < 16; k += step) {
                        const int x = mbx * 4 + blk_x[k], y = mby * 4 + blk_y[k];
                        int pred = 2;
                        if (x > 0 && y > y4top) {
                            const int a = e->i4[y * ys + x - 1], bb = e->i4[(y - 1) * ys + x];
                            pred = a < bb ? a : bb;
                        }
                        const int mode = m->i4_mode[k];
                        cabac_encode(c, 68, mode == pred);
                        if (mode != pred) {
                            const int rem = mode < pred ? mode : mode - 1;
                            cabac_encode(c, 69, rem & 1); cabac_encode(c, 69, (rem >> 1) & 1); cabac_encode(c, 69, (rem >> 2) & 1);
                        }
                        for (int yy = 0; yy < (t8 ? 2 : 1); yy++)
                            for (int xx = 0; xx < (t8 ? 2 : 1); xx++) e->i4[(y + yy) * ys + x + xx] = (int8_t)mode;
                    }
                }
                {   /* intra_chroma_pred_mode: TU, cMax 3 */
                    const int inc = (nb.availA && (nb.fA & B2H_MBF_INTRA) && e->cmode[mi - 1] != 0) +
                                    (nb.availB && (nb.fB & B2H_MBF_INTRA) && e->cmode[mi - mbw] != 0);
                    const int cm = m->chroma_mode;
                    cabac_encode(c, 64 + inc, cm > 0);
                    if (cm > 0) {
                        cabac_encode(c, 64 + 3, cm > 1);
                        if (cm > 1) cabac_encode(c, 64 + 3, cm > 2);
                    }
                    e->cmode[mi] = (uint8_t)cm;
                }
            }
            if (m->mb_type != B2_MB_I16x16) {
                /* coded_block_pattern: prefix = 4 luma bins (ctx 73 + condTermA + 2 condTermB, condTerm = neighbouring
                 * 8x8 has its cbp bit CLEAR; unavailable -> 0), suffix = chroma TU cMax 2 (ctx 77) */
                const int la = nb.availA ? nb.cbpA : 15, lb = nb.availB ? nb.cbpB : 15;
                const int a0 = !((la >> 1) & 1), b0 = !((lb >> 2) & 1);
                cabac_encode(c, 73 + a0 + 2 * b0, cbp_l & 1);
                const int a1 = !(cbp_l & 1), b1 = !((lb >> 3) & 1);
                cabac_encode(c, 73 + a1 + 2 * b1, (cbp_l >> 1) & 1);
                const int a2 = !((la >> 3) & 1), b2 = !(cbp_l & 1);
                cabac_encode(c, 73 + a2 + 2 * b2, (cbp_l >> 2) & 1);
                const int a3 = !((cbp_l >> 2) & 1), b3 = !((cbp_l >> 1) & 1);
                cabac_encode(c, 73 + a3 + 2 * b3, (cbp_l >> 3) & 1);
                const int ca = nb.availA ? nb.cbpA >> 4 : 0, cbb = nb.availB ? nb.cbpB >> 4 : 0;
                cabac_encode(c, 77 + (ca != 0) + 2 * (cbb != 0), cbp_c != 0);
                if (cbp_c) cabac_encode(c, 77 + 4 + (ca == 2) + 2 * (cbb == 2), cbp_c == 2);
                if (!intra && cbp_l && s->transform8x8)
                    cabac_encode(c, 399 + ((nb.fA & B2H_MBF_T8) != 0) + ((nb.fB & B2H_MBF_T8) != 0), t8);
            }
            e->cbp[mi] = m->cbp;
            if (m->cbp || m->mb_type == B2_MB_I16x16) cabac_encode(c, 60, 0);      /* mb_qp_delta = 0 (previous delta is 0 too) */

            /* residual(): coded_block_flag increments read the left / top block of the same kind */
            if (m->mb_type == B2_MB_I16x16) {
                const int fa = nb.availA ? ((nb.fA & B2H_MBF_I16) ? ((nb.fA & B2H_MBF_DC_Y) != 0) : -1) : 0;
                const int fb = nb.availB ? ((nb.fB & B2H_MBF_I16) ? ((nb.fB & B2H_MBF_DC_Y) != 0) : -1) : 0;
                if (cabac_residual(c, r, 0, cblk[24], 16, cbf_term(nb.availA, fa, 1) + 2 * cbf_term(nb.availB, fb, 1))) flags |= B2H_MBF_DC_Y;
            }
            if (cbp_l) {
                for (int k = 0; k < 16; k++) {
                    if (!(cbp_l & (1 << (k >> 2)))) continue;
                    const int x = mbx * 4 + blk_x[k], y = mby * 4 + blk_y[k];
                    if (t8) {
                        if (k & 3) continue;
                        const int n = cabac_residual(c, r, 5, cblk[k], 64, -1);
                        const uint8_t v = (uint8_t)(n > 16 ? 16 : (n ? n : 1));        /* cbp bit set: coded_block_flag inferred 1 */
                        e->nnz_y[y * ys + x] = e->nnz_y[y * ys + x + 1] = e->nnz_y[(y + 1) * ys + x] = e->nnz_y[(y + 1) * ys + x + 1] = v;
                        continue;
                    }
                    /* neighbouring 4x4 blocks: inside the picture the map holds 0 for every block that was not coded */
                    const int ta = cbf_term(x > 0, x > 0 ? e->nnz_y[y * ys + x - 1] : 0, intra);
                    const int tb = cbf_term(y > y4top, y > y4top ? e->nnz_y[(y - 1) * ys + x] : 0, intra);
                    if (m->mb_type == B2_MB_I16x16)
                        e->nnz_y[y * ys + x] = (uint8_t)cabac_residual(c, r, 1, cblk[k] + 1, 15, ta + 2 * tb);
                    else
                        e->nnz_y[y * ys + x] = (uint8_t)cabac_residual(c, r, 2, cblk[k], 16, ta + 2 * tb);
                }
            }
            if (cbp_c) {
                for (int p = 0; p < 2; p++) {
                    const int bit = p ? B2H_MBF_DC_V : B2H_MBF_DC_U;
                    const int fa = nb.availA ? ((nb.cbpA >> 4) ? ((nb.fA & bit) != 0) : -1) : 0;
                    const int fb = nb.availB ? ((nb.cbpB >> 4) ? ((nb.fB & bit) != 0) : -1) : 0;
                    if (cabac_residual(c, r, 3, cblk[25] + 4 * p, 4, cbf_term(nb.availA, fa, intra) + 2 * cbf_term(nb.availB, fb, intra)))
                        flags |= bit;
                }
                if (cbp_c == 2)
                    for (int p = 0; p < 2; p++)
                        for (int k = 0; k < 4; k++) {
                            const int x = mbx * 2 + (k & 1), y = mby * 2 + (k >> 1);
                            const int ta = cbf_term(x > 0, x > 0 ? e->nnz_c[p][y * cs + x - 1] : 0, intra);
                            const int tb = cbf_term(y > y2top, y > y2top ? e->nnz_c[p][(y - 1) * cs + x] : 0, intra);
                            e->nnz_c[p][y * cs + x] = (uint8_t)cabac_residual(c, r, 4, cblk[16 + 4 * p + k] + 1, 15, ta + 2 * tb);
                        }
            }
            e->mbf[mi] = (uint8_t)flags;
            cabac_terminate(c, mi == last);                                 /* end_of_slice_flag */
        }
    b->pos = (size_t)(c->p - b->buf);                                       /* the flush already byte-aligned the RBSP */
    if (b->overflow || c->overflow) return 0;
    return nal_pack(is_p ? 2 : 3, is_p ? B2H_NAL_SLICE : B2H_NAL_IDR, e->rbsp, b->pos, out, cap);
}
