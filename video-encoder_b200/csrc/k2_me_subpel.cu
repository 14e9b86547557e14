// k2_me_subpel.cu -- K2: half- then quarter-pel refinement of the full-pel motion vector by SATD.
//
// Replaces the sub-pel half of x264's motion estimation (behind x264_encoder_encode,
// av_encode.c:970); bit-exact against oracle/b2o_me.c:b2o_me_subpel (9 half-pel candidates,
// centre first, then the 8 quarter-pel neighbours of the winner; cost = SATD16x16 +
// lambda*mvbits(mv - pmv); first minimum in scan order wins).
//
// One warp per macroblock, K2_MBS macroblocks per CTA.  The 22x22 reference patch around the full-pel
// winner is staged in shared memory once; the three half-sample planes b (horizontal), h (vertical)
// and j (centre, from the UNROUNDED horizontal intermediates, as 8.4.2.2.1 requires) are built once
// and every one of the 17 candidates is then a two-plane average -- the 6-tap filter runs ~1,300
// times per MB instead of ~50,000 times if each candidate were interpolated on its own.
// Bound: integer ALU; algorithmic work = 17 candidates x 16 SATD4x4 per MB (~10x below K1).
#include "b2_h264.cuh"

namespace {

constexpr int K2_THREADS = 160;                          // wide partition kernel: one CTA per macroblock
// Macroblocks (one warp each) per CTA of k2_me_subpel_kernel.  K2 alone, 64 frames of 1080p on a B200: 2 -> 1.242 ms,
// 4 -> 1.240 ms, 8 -> 1.223 ms (profiles/r3_k2_warp_per_mb.txt); 16 would exceed the 48 KB of static shared memory.
#ifndef B2_K2_MBS
#define B2_K2_MBS 8
#endif
constexpr int K2_MBS = B2_K2_MBS;

// All four sample planes live in ONE shared byte array with a common row pitch, so that a candidate is
// "average of two byte planes" with two base offsets chosen once per thread -- no per-pixel switch.
constexpr int KP = 28;                                    // common row pitch (bytes): 7 words = a 22-byte patch row at any alignment
constexpr int OFF_G = 0;                                  // G : 22 rows, origin (X,Y) = (-3,-3)
constexpr int OFF_B = OFF_G + 22 * KP;                    // b : 18 rows, origin (-1,-1)
constexpr int OFF_H = OFF_B + 18 * KP;                    // h : 17 rows, origin (-1,-1)
constexpr int OFF_J = OFF_H + 17 * KP;                    // j : 17 rows, origin (-1,-1)
constexpr int PLANES_BYTES = OFF_J + 17 * KP;

struct __align__(16) K2Smem {
    uint8_t cur[16][16];      // source macroblock (16-byte rows)
    uint8_t P[PLANES_BYTES];  // G | b | h | j
    int16_t B1[22][18];       // unrounded horizontal half samples: rows -3..18, cols -1..15
    uint32_t cost[9];
    int best;
    // inter partitions (row N1): SATD per candidate and 8x8 quadrant, winners per shape part, final quadrant vectors
    uint32_t costq[9][4];
    uint32_t pcost[9];        // best stage-1 cost of part p: 0 16x16 | 1,2 16x8 top,bottom | 3,4 8x16 left,right | 5..8 quadrants
    int pk[9];                // its half-pel candidate
    int shape;
    int qk[4];                // half-pel winner (candidate index) of the chosen shape's part that owns quadrant q
    int qmv[4];               // final displacement of quadrant q from the full-pel position: (dx & 0xff) | (dy & 0xff) << 8
};

// quadrant masks of the nine shape parts and the parts of each shape
__device__ __constant__ uint8_t c_part_mask[9] = {0xf, 0x3, 0xc, 0x5, 0xa, 0x1, 0x2, 0x4, 0x8};
__device__ __constant__ uint8_t c_shape_first[4] = {0, 1, 3, 5};
__device__ __constant__ uint8_t c_shape_n[4] = {1, 2, 2, 4};
__device__ __constant__ uint8_t c_shape_bits[4] = {0, 2, 2, 8};

// byte offset inside K2Smem::P of sample (X,Y) of plane p (0 G, 1 b, 2 h, 3 j)
// ga: byte alignment the G rows were staged with (the patch is copied as aligned words, so G's columns start at byte ga)
__device__ __forceinline__ int plane_off(int p, int X, int Y, int ga)
{
    return p == 0 ? OFF_G + (Y + 3) * KP + X + 3 + ga
         : (p == 1 ? OFF_B : p == 2 ? OFF_H : OFF_J) + (Y + 1) * KP + X + 1;
}

// The two planes (and their integer displacements) whose rounded average is the quarter-pel sample with
// fraction (fx,fy) -- Table of 8.4.2.2.1; single-plane positions use the same plane twice ((a+a+1)>>1 = a).
// Packed per entry: planeA | dxA<<2 | dyA<<3 | planeB<<4 | dxB<<6 | dyB<<7
__device__ __constant__ uint8_t c_qpel_pair[16] = {
    /* 0 G,G        */ 0 | (0 << 4),
    /* 1 G,b        */ 0 | (1 << 4),
    /* 2 b,b        */ 1 | (1 << 4),
    /* 3 G(1,0),b   */ 0 | (1 << 2) | (1 << 4),
    /* 4 G,h        */ 0 | (2 << 4),
    /* 5 b,h        */ 1 | (2 << 4),
    /* 6 b,j        */ 1 | (3 << 4),
    /* 7 b,h(1,0)   */ 1 | (2 << 4) | (1 << 6),
    /* 8 h,h        */ 2 | (2 << 4),
    /* 9 h,j        */ 2 | (3 << 4),
    /* 10 j,j       */ 3 | (3 << 4),
    /* 11 j,h(1,0)  */ 3 | (2 << 4) | (1 << 6),
    /* 12 G(0,1),h  */ 0 | (1 << 3) | (2 << 4),
    /* 13 h,b(0,1)  */ 2 | (1 << 4) | (1 << 7),
    /* 14 j,b(0,1)  */ 3 | (1 << 4) | (1 << 7),
    /* 15 h(1,0),b(0,1) */ 2 | (1 << 2) | (1 << 4) | (1 << 7)};

__device__ __constant__ int8_t c_subpel_off[9][2] = {{0, 0}, {-1, -1}, {0, -1}, {1, -1}, {-1, 0}, {1, 0}, {-1, 1}, {0, 1}, {1, 1}};

// ---- SATD of one 4x4 block of one candidate, on the dot-product unit ---------------------------------------------------------
// The horizontal Hadamard pass of the residual row (c - p) is linear, so it splits into H.c - H.p: four IDP.4A (u8 x s8) per
// row against the rows of H4, with H.c of the SOURCE block computed once per thread (a thread keeps its block for all of
// its candidates) and passed in as the accumulator.  No byte is ever extracted: the prediction row is fetched as one
// unaligned 32-bit word (two LDS + funnel shift; KP % 4 == 0 keeps the alignment the same on every row) and quarter-sample
// positions average two such words with the SIMD byte average.  The vertical pass folds its last butterfly stage into
// |a+c| + |a-c| = 2 max(|a|,|c|), which also absorbs SATD's final halving.  ~2.3x fewer instructions than the scalar form.
__device__ __forceinline__ int dp4a_us(uint32_t u8x4, uint32_t s8x4, int acc)
{
    int d;
    asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(u8x4), "r"(s8x4), "r"(acc));
    return d;
}

// rows of H4 as s8x4 (byte x = column x): (1,1,1,1) (1,1,-1,-1) (1,-1,-1,1) (1,-1,1,-1), and their negatives
constexpr uint32_t H4P0 = 0x01010101u, H4P1 = 0xffff0101u, H4P2 = 0x01ffff01u, H4P3 = 0xff01ff01u;
constexpr uint32_t H4N0 = 0xffffffffu, H4N1 = 0x0101ffffu, H4N2 = 0xff0101ffu, H4N3 = 0x01ff01ffu;

// H4 applied to the four rows of the source block whose top-left pixel is (px,py) of the macroblock
__device__ __forceinline__ void cur_block_rows(const K2Smem &s, int px, int py, int (&ch)[16])
{
#pragma unroll
    for (int y = 0; y < 4; y++) {
        const uint32_t cw = *(const uint32_t *)&s.cur[py + y][px];
        ch[4 * y + 0] = dp4a_us(cw, H4P0, 0); ch[4 * y + 1] = dp4a_us(cw, H4P1, 0);
        ch[4 * y + 2] = dp4a_us(cw, H4P2, 0); ch[4 * y + 3] = dp4a_us(cw, H4P3, 0);
    }
}

// the two plane offsets of the candidate displaced by (cx,cy) quarter-pels, for the block at part-local pixel (bx,by)
__device__ __forceinline__ void cand_planes(int bx, int by, int cx, int cy, int ga, int &offA, int &offB)
{
    const int ix = cx >> 2, iy = cy >> 2;
    const int e = c_qpel_pair[(cy & 3) * 4 + (cx & 3)];
    offA = plane_off(e & 3, bx + ix + ((e >> 2) & 1), by + iy + ((e >> 3) & 1), ga);
    offB = plane_off((e >> 4) & 3, bx + ix + ((e >> 6) & 1), by + iy + ((e >> 7) & 1), ga);
}

// A plane offset (>= 0) as word index | funnel shift << 16.  Blocks and prediction words start at multiples of 4 bytes in every
// plane (KP % 4 == 0), so a candidate's packed offsets for the block at (0,0) serve every block: add the block's word index.
__device__ __forceinline__ uint32_t pack_off(int off) { return (uint32_t)(off >> 2) | ((uint32_t)(off & 3) << 19); }

// four consecutive bytes of row y below the packed offset po, displaced by wbase words
__device__ __forceinline__ uint32_t plane_word(const K2Smem &s, int wbase, uint32_t po, int y)
{
    const uint32_t *w = (const uint32_t *)s.P + wbase + (po & 0xffffu) + y * (KP / 4);
    return __funnelshift_r(w[0], w[1], po >> 16);
}

// SATD of one 4x4 block (word index wbase = (by * KP + bx) / 4) against the prediction at packed plane offsets pa / pb of the
// block at (0,0); ch = cur_block_rows of the same block.  TWO = false: half-sample grid positions (one plane, stage 1); true:
// average of two planes (stage 2).
template <bool TWO>
__device__ __forceinline__ uint32_t block_satd(const K2Smem &s, const int (&ch)[16], int wbase, uint32_t pa, uint32_t pb)
{
    int t[16];
#pragma unroll
    for (int y = 0; y < 4; y++) {
        uint32_t p = plane_word(s, wbase, pa, y);
        if (TWO) p = __vavgu4(p, plane_word(s, wbase, pb, y));
        t[4 * y + 0] = dp4a_us(p, H4N0, ch[4 * y + 0]); t[4 * y + 1] = dp4a_us(p, H4N1, ch[4 * y + 1]);
        t[4 * y + 2] = dp4a_us(p, H4N2, ch[4 * y + 2]); t[4 * y + 3] = dp4a_us(p, H4N3, ch[4 * y + 3]);
    }
    int sum = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int a = t[k] + t[4 + k], b = t[k] - t[4 + k], c = t[8 + k] + t[12 + k], d = t[8 + k] - t[12 + k];
        sum += max(abs(a), abs(c)) + max(abs(b), abs(d));
    }
    return (uint32_t)sum;
}

// the same for the block at part-local pixel (bx,by) and the candidate displaced by (cx,cy) quarter-pels
template <bool TWO>
__device__ __forceinline__ uint32_t cand_block_satd(const K2Smem &s, const int (&ch)[16], int bx, int by, int cx, int cy, int ga)
{
    int offA, offB;
    cand_planes(0, 0, cx, cy, ga, offA, offB);
    return block_satd<TWO>(s, ch, (by * KP + bx) >> 2, pack_off(offA), pack_off(offB));
}

// quarter-pel offsets of the nine candidates (c_subpel_off) as 2-bit fields (offset + 1), so that a lane can take the offset of
// ITS candidate with a shift instead of a per-lane constant-bank load
constexpr uint32_t SUB_DX = 0x24891u, SUB_DY = 0x2a501u;
__device__ __forceinline__ int sub_dx(int k) { return (int)((SUB_DX >> (2 * k)) & 3u) - 1; }
__device__ __forceinline__ int sub_dy(int k) { return (int)((SUB_DY >> (2 * k)) & 3u) - 1; }

// sum over the 16 lanes of each half-warp: (half 0, half 1), both in every lane
__device__ __forceinline__ void half_sums(uint32_t v, bool upper, uint32_t &lo, uint32_t &hi)
{
    lo = __reduce_add_sync(0xffffffffu, upper ? 0u : v);
    hi = __reduce_add_sync(0xffffffffu, upper ? v : 0u);
}

// sum over the four lanes of one 8x8 quadrant (block bits 0 and 2); the lanes with blk & 5 == 0 write it
__device__ __forceinline__ uint32_t quad_sum(uint32_t v)
{
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    return v + __shfl_xor_sync(0xffffffffu, v, 4);
}

// Refinement of ONE macroblock around the full-pel vector mvf by ONE warp; PART: also the local partition refinement.
// Lane l keeps 4x4 block l & 15 for every candidate it prices; the two half-warps take different candidates (stage 1: 0..4 and
// 5..8, stage 2: 1..4 and 5..8), so the source block's H4 rows are computed twice per macroblock and a candidate's SATD is a
// 16-lane reduction.  Only __syncwarp orders the shared-memory phases.
template <bool PART>
__device__ __forceinline__ void k2_body(K2Smem &s, const uint8_t *__restrict__ cur, const uint8_t *__restrict__ ref, int pitch, size_t plane_stride,
                                        int mbx, int mby, int frame, size_t mbi, const b2_mv_t mvf, const b2_mv_t pm, int lambda, int subpel,
                                        b2_mv_t *__restrict__ mv_out, uint32_t *__restrict__ cost_out, uint8_t *__restrict__ pred_out,
                                        uint8_t *__restrict__ part_out, b2_mv_t *__restrict__ mv8_out)
{
    const int lane = threadIdx.x & 31;
    const uint8_t *cplane = cur + frame * plane_stride + (size_t)(B2_PAD + mby * 16) * pitch + B2_PAD + mbx * 16;
    const uint8_t *rplane = ref + frame * plane_stride + (size_t)(B2_PAD + mby * 16 + mvf.y - 3) * pitch + B2_PAD +
                            mbx * 16 + mvf.x - 3;
    uint8_t *PG = s.P + OFF_G, *PB = s.P + OFF_B, *PH = s.P + OFF_H, *PJ = s.P + OFF_J;
    // 22x22 reference patch as ALIGNED words: 7 words cover a 22-byte row at any of the four alignments, 22 x 7 = 154 loads, all
    // in flight at once.  The row keeps its alignment in shared memory: G's column X sits at byte X + 3 + ga.  pitch, plane_stride
    // and B2_PAD are multiples of 16 and the 64-pixel frame border covers the extra bytes.
    const int ga = (mvf.x + 1) & 3;                          // (mvf.x - 3) mod 4
    {
        const uint32_t *src = (const uint32_t *)(rplane - ga);
#pragma unroll
        for (int k = 0; k < 5; k++) {
            const int i = lane + 32 * k;
            if (i < 154) {
                const int r = i / 7, wi = i - r * 7;
                ((uint32_t *)PG)[r * (KP / 4) + wi] = src[(size_t)r * (pitch >> 2) + wi];
            }
        }
        if (lane < 16) *(uint4 *)&s.cur[lane][0] = *(const uint4 *)(cplane + (size_t)lane * pitch);
    }
    __syncwarp();

    // Half-sample planes with SLIDING WINDOWS: one lane walks a whole row (b1, and b from it) or column (h, j), so that every sample
    // is loaded once and feeds six outputs.  b1: unrounded horizontal half samples, 22 rows x 17 cols (lane = row), rows 2..19
    // also give b; h: vertical half samples, 17 rows x 18 cols (lane = column); j from the unrounded b1 (lane = column).
    if (lane < 22) {
        const uint32_t *row = (const uint32_t *)(PG + lane * KP);                 // 24-byte rows: word aligned
        int g[24];
#pragma unroll
        for (int i = 0; i < 6; i++) {
            const uint32_t wv = __funnelshift_r(row[i], row[i + 1], 8 * ga);
            g[4 * i] = wv & 255; g[4 * i + 1] = (wv >> 8) & 255; g[4 * i + 2] = (wv >> 16) & 255; g[4 * i + 3] = wv >> 24;
        }
        const bool has_b = lane >= 2 && lane < 20;                                // b: Y = r-1 -> B1 row r+2
#pragma unroll
        for (int c = 0; c < 17; c++) {
            const int v = b2::tap6(g[c], g[c + 1], g[c + 2], g[c + 3], g[c + 4], g[c + 5]);
            s.B1[lane][c] = (int16_t)v;
            if (has_b) PB[(lane - 2) * KP + c] = (uint8_t)b2_clip255((v + 16) >> 5);
        }
    }
    if (lane < 18) {
        const uint8_t *q = PG + lane + 2 + ga;                                      // column X = lane - 1
        int g[22];
#pragma unroll
        for (int r = 0; r < 22; r++) g[r] = q[r * KP];
#pragma unroll
        for (int r = 0; r < 17; r++)
            PH[r * KP + lane] = (uint8_t)b2_clip255((b2::tap6(g[r], g[r + 1], g[r + 2], g[r + 3], g[r + 4], g[r + 5]) + 16) >> 5);
    }
    __syncwarp();
    if (lane < 17) {
        int g[22];
#pragma unroll
        for (int r = 0; r < 22; r++) g[r] = s.B1[r][lane];
#pragma unroll
        for (int r = 0; r < 17; r++)
            PJ[r * KP + lane] = (uint8_t)b2_clip255((b2::tap6(g[r], g[r + 1], g[r + 2], g[r + 3], g[r + 4], g[r + 5]) + 512) >> 10);
    }
    __syncwarp();

    const int blk = lane & 15, bx = (blk & 3) * 4, by = (blk >> 2) * 4, wb = (by * KP + bx) >> 2;
    const bool upper = lane >= 16;
    int ch[16];
    cur_block_rows(s, bx, by, ch);
    // Plane offsets are computed once per macroblock, one candidate per lane, and fetched by shuffle: lane k < 9 holds half-pel
    // candidate k's (a single plane)
    uint32_t po1;
    {
        const int k = lane < 9 ? lane : 0;
        int oa, ob;
        cand_planes(0, 0, 2 * sub_dx(k), 2 * sub_dy(k), ga, oa, ob);
        po1 = pack_off(oa);
    }

    uint32_t qm_all = 0;                                     // winner relative to the full-pel position (single-vector path)
    if (PART) {
        // ---- partitions: SATD per (candidate, quadrant); every shape part picks its half-pel winner, the cheapest shape
        // is kept and each of its parts tries the 8 quarter-pel neighbours of ITS winner (oracle: b2o_me_subpel_part) ----
        const int q = ((blk >> 1) & 1) | ((blk >> 3) << 1);
        const bool qlead = (blk & 5) == 0;
#pragma unroll
        for (int i = 0; i < 5; i++) {
            const int cand = i + (upper ? 5 : 0);
            const uint32_t pa = __shfl_sync(0xffffffffu, po1, cand);
            uint32_t v = 0;
            if (cand < 9) v = block_satd<false>(s, ch, wb, pa, 0);
            v = quad_sum(v);
            if (qlead && cand < 9) s.costq[cand][q] = v;
        }
        __syncwarp();
        if (lane < 9) {                                  // one lane per shape part
            const int mask = c_part_mask[lane];
            uint32_t best = 0xffffffffu; int bk = 0;
            for (int k = 0; k < 9; k++) {
                const int mx = mvf.x * 4 + 2 * c_subpel_off[k][0], my = mvf.y * 4 + 2 * c_subpel_off[k][1];
                uint32_t c = (uint32_t)(lambda * (b2_mvbits(mx - pm.x) + b2_mvbits(my - pm.y)));
#pragma unroll
                for (int qq = 0; qq < 4; qq++)
                    if (mask & (1 << qq)) c += s.costq[k][qq];
                if (c < best) { best = c; bk = k; }
            }
            s.pcost[lane] = best; s.pk[lane] = bk;
        }
        __syncwarp();
        if (lane == 0) {
            uint32_t bc = 0xffffffffu; int shape = 0;
            for (int sh = 0; sh < 4; sh++) {
                uint32_t c = (uint32_t)(lambda * c_shape_bits[sh]);
                for (int a = 0; a < c_shape_n[sh]; a++) c += s.pcost[c_shape_first[sh] + a];
                if (c < bc) { bc = c; shape = sh; }
            }
            s.shape = shape;
            for (int a = 0; a < c_shape_n[shape]; a++) {
                const int p = c_shape_first[shape] + a;
                for (int qq = 0; qq < 4; qq++)
                    if (c_part_mask[p] & (1 << qq)) s.qk[qq] = s.pk[p];
            }
        }
        __syncwarp();
        {   // stage 2: entries 1..8 of costq are overwritten; the stage-1 sums are folded into pcost.  Lane 8q + k - 1 holds the
            // plane offsets of quarter-pel candidate k around quadrant q's half-pel winner.
            uint32_t pa2, pb2;
            {
                const int hk = s.qk[lane >> 3], k = (lane & 7) + 1;
                int oa, ob;
                cand_planes(0, 0, 2 * sub_dx(hk) + sub_dx(k), 2 * sub_dy(hk) + sub_dy(k), ga, oa, ob);
                pa2 = pack_off(oa); pb2 = pack_off(ob);
            }
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const int cand = 1 + i + (upper ? 4 : 0), src = 8 * q + cand - 1;
                const uint32_t pa = __shfl_sync(0xffffffffu, pa2, src), pb = __shfl_sync(0xffffffffu, pb2, src);
                const uint32_t v = quad_sum(block_satd<true>(s, ch, wb, pa, pb));
                if (qlead) s.costq[cand][q] = v;
            }
        }
        __syncwarp();
        const int shape = s.shape;
        if (lane < c_shape_n[shape]) {                   // one lane per part of the chosen shape
            const int p = c_shape_first[shape] + lane, mask = c_part_mask[p], hk = s.pk[p];
            const int hx = 2 * c_subpel_off[hk][0], hy = 2 * c_subpel_off[hk][1];
            uint32_t best = s.pcost[p]; int wx = hx, wy = hy;
            for (int k = 1; k < 9; k++) {
                const int dx = hx + c_subpel_off[k][0], dy = hy + c_subpel_off[k][1];
                uint32_t c = (uint32_t)(lambda * (b2_mvbits(mvf.x * 4 + dx - pm.x) + b2_mvbits(mvf.y * 4 + dy - pm.y)));
#pragma unroll
                for (int qq = 0; qq < 4; qq++)
                    if (mask & (1 << qq)) c += s.costq[k][qq];
                if (c < best) { best = c; wx = dx; wy = dy; }
            }
            s.pcost[p] = best;
#pragma unroll
            for (int qq = 0; qq < 4; qq++)
                if (mask & (1 << qq)) s.qmv[qq] = (wx & 0xff) | ((wy & 0xff) << 8);
        }
        __syncwarp();
        if (lane == 0) {
            uint32_t total = (uint32_t)(lambda * c_shape_bits[shape]);
            for (int a = 0; a < c_shape_n[shape]; a++) total += s.pcost[c_shape_first[shape] + a];
            cost_out[mbi] = total;
            part_out[mbi] = (uint8_t)shape;
            for (int qq = 0; qq < 4; qq++) {
                b2_mv_t o;
                o.x = (int16_t)(mvf.x * 4 + (int)(int8_t)(s.qmv[qq] & 0xff));
                o.y = (int16_t)(mvf.y * 4 + (int)(int8_t)((s.qmv[qq] >> 8) & 0xff));
                if (qq == 0) mv_out[mbi] = o;
                else mv8_out[mbi * 3 + qq - 1] = o;
            }
        }
    } else {
        // stage 1: centre + 8 half-pel neighbours (offsets x2 quarter units); without sub-pel: centre only.  Lane k < 9 ends up
        // holding candidate k's SATD, prices it, and a warp minimum picks the first best.
        const int n1 = subpel ? 9 : 1;
        uint32_t mine = 0;
#pragma unroll
        for (int i = 0; i < 5; i++) {
            if (i >= n1) break;
            const int cand = i + (upper ? 5 : 0);
            const uint32_t pa = __shfl_sync(0xffffffffu, po1, cand);
            uint32_t v = 0, lo, hi;
            if (cand < n1) v = block_satd<false>(s, ch, wb, pa, 0);
            half_sums(v, upper, lo, hi);
            if (lane == i) mine = lo;
            if (lane == i + 5) mine = hi;
        }
        uint32_t key = 0xffffffffu;
        if (lane < n1) {
            const int mx = mvf.x * 4 + 2 * sub_dx(lane), my = mvf.y * 4 + 2 * sub_dy(lane);
            const uint32_t c = mine + (uint32_t)(lambda * (b2_mvbits(mx - pm.x) + b2_mvbits(my - pm.y)));
            key = (c << 4) | (uint32_t)lane;             // costs stay far below 2^28; ties go to the lower candidate index
        }
        key = __reduce_min_sync(0xffffffffu, key);
        const int h1 = (int)(key & 15u);
        const int hx = 2 * sub_dx(h1), hy = 2 * sub_dy(h1);
        // candidate 0 = the half-pel winner itself (already priced); 1..8 its quarter-pel neighbours; first minimum wins.  Without
        // sub-pel the centre (candidate 0 of stage 1) is final.
        uint32_t key2 = key;
        if (subpel) {
            key2 = lane == 0 ? (key >> 4) << 4 : 0xffffffffu;
            mine = 0;
            uint32_t pa2, pb2;                           // lane k - 1 (mod 8): plane offsets of quarter-pel candidate k
            {
                const int k = (lane & 7) + 1;
                int oa, ob;
                cand_planes(0, 0, hx + sub_dx(k), hy + sub_dy(k), ga, oa, ob);
                pa2 = pack_off(oa); pb2 = pack_off(ob);
            }
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const int cand = 1 + i + (upper ? 4 : 0);
                const uint32_t pa = __shfl_sync(0xffffffffu, pa2, cand - 1), pb = __shfl_sync(0xffffffffu, pb2, cand - 1);
                uint32_t lo, hi;
                half_sums(block_satd<true>(s, ch, wb, pa, pb), upper, lo, hi);
                if (lane == 1 + i) mine = lo;
                if (lane == 5 + i) mine = hi;
            }
            if (lane >= 1 && lane < 9) {
                const int mx = mvf.x * 4 + hx + sub_dx(lane), my = mvf.y * 4 + hy + sub_dy(lane);
                const uint32_t c = mine + (uint32_t)(lambda * (b2_mvbits(mx - pm.x) + b2_mvbits(my - pm.y)));
                key2 = (c << 4) | (uint32_t)lane;
            }
            key2 = __reduce_min_sync(0xffffffffu, key2);
        }
        const int k = (int)(key2 & 15u);
        const int dx = hx + (k ? sub_dx(k) : 0), dy = hy + (k ? sub_dy(k) : 0);
        if (lane == 0) {
            b2_mv_t o;
            o.x = (int16_t)(mvf.x * 4 + dx); o.y = (int16_t)(mvf.y * 4 + dy);
            mv_out[mbi] = o;
            cost_out[mbi] = key2 >> 4;
        }
        qm_all = (uint32_t)((dx & 0xff) | ((dy & 0xff) << 8));
    }
    // the winner's motion-compensated luma block (K5 subtracts it from the source instead of interpolating again)
    if (pred_out != nullptr) {
        uint32_t pa, pb;                                               // lane q (mod 4): plane offsets of quadrant q's winner
        {
            const int qm = PART ? s.qmv[lane & 3] : (int)qm_all;
            int oa, ob;
            cand_planes(0, 0, (int)(int8_t)(qm & 0xff), (int)(int8_t)((qm >> 8) & 0xff), ga, oa, ob);
            pa = pack_off(oa); pb = pack_off(ob);
        }
#pragma unroll
        for (int k = 0; k < 2; k++) {                                  // 4 pixels per lane and step: row r, columns 4c..4c+3
            const int i = lane + 32 * k, r = i >> 2, c = (i & 3) * 4;
            const int q = (c >> 3) | ((r >> 3) << 1);                  // the quadrant the word lies in
            const uint32_t qa = __shfl_sync(0xffffffffu, pa, q), qb = __shfl_sync(0xffffffffu, pb, q);
            const int w = (r * KP + c) >> 2;
            *(uint32_t *)(pred_out + mbi * 256 + r * 16 + c) = __vavgu4(plane_word(s, w, qa, 0), plane_word(s, w, qb, 0));
        }
    }
}

// one warp per macroblock, K2_MBS consecutive macroblocks of a row per CTA (the tail CTA of a row has idle warps)
template <bool PART>
__global__ void __launch_bounds__(32 * K2_MBS)
k2_me_subpel_kernel(const uint8_t *__restrict__ cur, const uint8_t *__restrict__ ref, int pitch, size_t plane_stride,
                    int mbw, int mbh, const b2_mv_t *__restrict__ mv_full, const b2_mv_t *__restrict__ pmv,
                    int lambda, int subpel, b2_mv_t *__restrict__ mv_out, uint32_t *__restrict__ cost_out,
                    uint8_t *__restrict__ pred_out, uint8_t *__restrict__ part_out, b2_mv_t *__restrict__ mv8_out)
{
    __shared__ K2Smem sm[K2_MBS];
    const int warp = threadIdx.x >> 5;
    const int mbx = blockIdx.x * K2_MBS + warp;
    if (mbx >= mbw) return;                                  // whole warps only: nothing below synchronises the CTA
    const size_t mbi = ((size_t)blockIdx.z * mbh + blockIdx.y) * mbw + mbx;
    b2_mv_t pm = {0, 0};
    if (pmv) pm = pmv[mbi];
    k2_body<PART>(sm[warp], cur, ref, pitch, plane_stride, mbx, blockIdx.y, blockIdx.z, mbi, mv_full[mbi], pm, lambda, subpel, mv_out,
                  cost_out, pred_out, part_out, mv8_out);
}

// ---- wide partition search (row N1, partitions = 2) --------------------------------------------------------------------
// K1<PART> delivered the best full-pel vector and cost of each of the nine shape parts.  This kernel picks the shape on those
// costs (oracle: b2o_me_parts_wide) and refines every part of it on its own: patch around the part's vector, half-sample
// planes for the part's area, 9 half-pel + 8 quarter-pel candidates with SATD over the part.  Geometry in pixels:
__device__ __constant__ uint8_t c_part_geo[9][4] = {{0, 0, 16, 16}, {0, 0, 16, 8}, {0, 8, 16, 8}, {0, 0, 8, 16}, {8, 0, 8, 16},
                                                    {0, 0, 8, 8},   {8, 0, 8, 8},  {0, 8, 8, 8},  {8, 8, 8, 8}};

__global__ void __launch_bounds__(K2_THREADS)
k2_me_subpel_wide_kernel(const uint8_t *__restrict__ cur, const uint8_t *__restrict__ ref, int pitch, size_t plane_stride,
                         int mbw, int mbh, const b2_mv_t *__restrict__ mv9, const uint32_t *__restrict__ cost9,
                         const b2_mv_t *__restrict__ pmv, int lambda, b2_mv_t *__restrict__ mv_out, uint32_t *__restrict__ cost_out,
                         uint8_t *__restrict__ pred_out, uint8_t *__restrict__ part_out, b2_mv_t *__restrict__ mv8_out)
{
    __shared__ __align__(16) K2Smem s;
    __shared__ uint32_t s_total;
    const int tid = threadIdx.x;
    const int mbx = blockIdx.x, mby = blockIdx.y, frame = blockIdx.z;
    const size_t mbi = ((size_t)frame * mbh + mby) * mbw + mbx;
    b2_mv_t pm = {0, 0};
    if (pmv) pm = pmv[mbi];
    const uint8_t *cplane = cur + frame * plane_stride + (size_t)(B2_PAD + mby * 16) * pitch + B2_PAD + mbx * 16;
    uint8_t *PG = s.P + OFF_G, *PB = s.P + OFF_B, *PH = s.P + OFF_H, *PJ = s.P + OFF_J;
    if (tid < 64) {
        const int r = tid >> 2, c = tid & 3;
        *(uint32_t *)&s.cur[r][c * 4] = *(const uint32_t *)(cplane + (size_t)r * pitch + c * 4);
    }
    if (tid == 0) {                                          // shape on the full-pel costs
        uint32_t bc = 0xffffffffu; int shape = 0;
        for (int sh = 0; sh < 4; sh++) {
            uint32_t c = (uint32_t)(lambda * c_shape_bits[sh]);
            for (int a = 0; a < c_shape_n[sh]; a++) c += cost9[mbi * 9 + c_shape_first[sh] + a];
            if (c < bc) { bc = c; shape = sh; }
        }
        s.shape = shape;
        s_total = (uint32_t)(lambda * c_shape_bits[shape]);
    }
    __syncthreads();
    const int shape = s.shape;
    if (shape == B2_PART_16x16) {                            // the common case: the tuned single-vector path around part 0's vector
        const b2_mv_t mv16 = mv9[mbi * 9];
        __syncthreads();                                     // everyone has read s.shape before the body reuses the shared struct
        if (tid >= 32) return;                               // the single-vector body is one warp's work
        k2_body<false>(s, cur, ref, pitch, plane_stride, mbx, mby, frame, mbi, mv16, pm, lambda, 1, mv_out, cost_out, pred_out, nullptr,
                       nullptr);
        if (tid == 0) part_out[mbi] = B2_PART_16x16;
        return;
    }
    for (int a = 0; a < c_shape_n[shape]; a++) {
        const int p = c_shape_first[shape] + a;
        const int ox = c_part_geo[p][0], oy = c_part_geo[p][1], pw = c_part_geo[p][2], ph = c_part_geo[p][3];
        const b2_mv_t mvf = mv9[mbi * 9 + p];
        const uint8_t *rplane = ref + frame * plane_stride + (size_t)(B2_PAD + mby * 16 + oy + mvf.y - 3) * pitch + B2_PAD +
                                mbx * 16 + ox + mvf.x - 3;
        const int gw = pw + 6, gh = ph + 6;
        for (int i = tid; i < gw * gh; i += K2_THREADS) { const int r = i / gw, c = i - r * gw; PG[r * KP + c] = rplane[(size_t)r * pitch + c]; }
        if (tid < 9) s.cost[tid] = 0;
        __syncthreads();
        // unrounded horizontal half samples b1: gh rows x (pw+1) cols; vertical half samples h: (ph+1) rows x (pw+2) cols
        for (int i = tid; i < gh * (pw + 1); i += K2_THREADS) {
            const int r = i / (pw + 1), c = i - r * (pw + 1);
            const uint8_t *q = PG + r * KP + c + 2;
            s.B1[r][c] = (int16_t)b2::tap6(q[-2], q[-1], q[0], q[1], q[2], q[3]);
        }
        for (int i = tid; i < (ph + 1) * (pw + 2); i += K2_THREADS) {
            const int r = i / (pw + 2), c = i - r * (pw + 2);
            const uint8_t *q = PG + r * KP + c + 2;
            const int v = b2::tap6(q[0], q[KP], q[2 * KP], q[3 * KP], q[4 * KP], q[5 * KP]);
            PH[r * KP + c] = (uint8_t)b2_clip255((v + 16) >> 5);
        }
        __syncthreads();
        for (int i = tid; i < (ph + 2) * (pw + 1); i += K2_THREADS) {     // b: Y = r-1 -> B1 row r+2
            const int r = i / (pw + 1), c = i - r * (pw + 1);
            PB[r * KP + c] = (uint8_t)b2_clip255((s.B1[r + 2][c] + 16) >> 5);
        }
        for (int i = tid; i < (ph + 1) * (pw + 1); i += K2_THREADS) {     // j: Y = r-1 -> B1 rows r..r+5
            const int r = i / (pw + 1), c = i - r * (pw + 1);
            const int v = b2::tap6(s.B1[r][c], s.B1[r + 1][c], s.B1[r + 2][c], s.B1[r + 3][c], s.B1[r + 4][c], s.B1[r + 5][c]);
            PJ[r * KP + c] = (uint8_t)b2_clip255((v + 512) >> 10);
        }
        __syncthreads();
        const int nbx = pw >> 2, nb = nbx * (ph >> 2);       // 4x4 blocks of the part
        const int j = tid % nb, lx = (j % nbx) * 4, ly = (j / nbx) * 4;   // a thread keeps its block through both stages
        int ch[16];
        cur_block_rows(s, ox + lx, oy + ly, ch);
        if (tid < 9 * nb) {
            const int cand = tid / nb;
            const uint32_t v = cand_block_satd<false>(s, ch, lx, ly, 2 * c_subpel_off[cand][0], 2 * c_subpel_off[cand][1], 0);
            atomicAdd(&s.cost[cand], v);
        }
        __syncthreads();
        if (tid == 0) {
            uint32_t best = 0xffffffffu; int bi = 0;
            for (int k = 0; k < 9; k++) {
                const int mx = mvf.x * 4 + 2 * c_subpel_off[k][0], my = mvf.y * 4 + 2 * c_subpel_off[k][1];
                const uint32_t c = s.cost[k] + (uint32_t)(lambda * (b2_mvbits(mx - pm.x) + b2_mvbits(my - pm.y)));
                if (c < best) { best = c; bi = k; }
            }
            s.best = bi;
            s.cost[0] = best;
            for (int k = 1; k < 9; k++) s.cost[k] = 0;
        }
        __syncthreads();
        const int hx = 2 * c_subpel_off[s.best][0], hy = 2 * c_subpel_off[s.best][1];
        if (tid < 8 * nb) {
            const int cand = 1 + tid / nb;
            const uint32_t v = cand_block_satd<true>(s, ch, lx, ly, hx + c_subpel_off[cand][0], hy + c_subpel_off[cand][1], 0);
            atomicAdd(&s.cost[cand], v);
        }
        __syncthreads();
        if (tid == 0) {
            uint32_t best = s.cost[0];
            int bx = hx, by = hy;
            for (int k = 1; k < 9; k++) {
                const int dx = hx + c_subpel_off[k][0], dy = hy + c_subpel_off[k][1];
                const uint32_t c = s.cost[k] + (uint32_t)(lambda * (b2_mvbits(mvf.x * 4 + dx - pm.x) + b2_mvbits(mvf.y * 4 + dy - pm.y)));
                if (c < best) { best = c; bx = dx; by = dy; }
            }
            s_total += best;
            s.best = (bx & 0xff) | ((by & 0xff) << 8);
            b2_mv_t o;
            o.x = (int16_t)(mvf.x * 4 + bx); o.y = (int16_t)(mvf.y * 4 + by);
            for (int q = 0; q < 4; q++) {                    // quadrants covered by this part
                const int qx = (q & 1) * 8, qy = (q >> 1) * 8;
                if (qx >= ox && qx < ox + pw && qy >= oy && qy < oy + ph) {
                    if (q == 0) mv_out[mbi] = o;
                    else mv8_out[mbi * 3 + q - 1] = o;
                }
            }
        }
        __syncthreads();
        {   // the part's motion-compensated prediction -> K5
            const int cx = (int)(int8_t)(s.best & 0xff), cy = (int)(int8_t)((s.best >> 8) & 0xff);
            const int wq = pw >> 2;                          // 4-pixel words per row
            if (tid < wq * ph) {
                const int r = tid / wq, c = (tid - r * wq) * 4;
                int offA, offB;
                cand_planes(0, 0, cx, cy, 0, offA, offB);
                const int w = (r * KP + c) >> 2;
                *(uint32_t *)(pred_out + mbi * 256 + (oy + r) * 16 + ox + c) =
                    __vavgu4(plane_word(s, w, pack_off(offA), 0), plane_word(s, w, pack_off(offB), 0));
            }
        }
        __syncthreads();                                     // planes are rebuilt for the next part
    }
    if (tid == 0) { cost_out[mbi] = s_total; part_out[mbi] = (uint8_t)shape; }
}

}  // namespace

int b2_launch_me_subpel(const uint8_t *d_cur, const uint8_t *d_ref, int pitch, size_t plane_stride, int mbw, int mbh,
                        int nframes, const b2_mv_t *d_mv_full, const b2_mv_t *d_pmv, int lambda, int subpel,
                        b2_mv_t *d_mv_out, uint32_t *d_cost_out, uint8_t *d_pred_out, uint8_t *d_part_out, b2_mv_t *d_mv8_out,
                        const b2_mv_t *d_mv9, const uint32_t *d_cost9, cudaStream_t st)
{
    if (d_mv9 && d_part_out && subpel) {
        const dim3 grid(mbw, mbh, nframes);
        k2_me_subpel_wide_kernel<<<grid, K2_THREADS, 0, st>>>(d_cur, d_ref, pitch, plane_stride, mbw, mbh, d_mv9, d_cost9, d_pmv, lambda,
                                                               d_mv_out, d_cost_out, d_pred_out, d_part_out, d_mv8_out);
        B2_CUDA_OK(cudaGetLastError());
        return 0;
    }
    const dim3 grid((mbw + K2_MBS - 1) / K2_MBS, mbh, nframes);
    if (d_part_out && subpel)
        k2_me_subpel_kernel<true><<<grid, 32 * K2_MBS, 0, st>>>(d_cur, d_ref, pitch, plane_stride, mbw, mbh, d_mv_full, d_pmv,
                                                               lambda, subpel, d_mv_out, d_cost_out, d_pred_out, d_part_out, d_mv8_out);
    else
        k2_me_subpel_kernel<false><<<grid, 32 * K2_MBS, 0, st>>>(d_cur, d_ref, pitch, plane_stride, mbw, mbh, d_mv_full, d_pmv,
                                                                lambda, subpel, d_mv_out, d_cost_out, d_pred_out, nullptr, nullptr);
    B2_CUDA_OK(cudaGetLastError());
    return 0;
}
