// k8_deblock.cu -- K8: in-loop deblocking filter (ITU-T H.264 8.7) on the reconstructed frame.
//
// SURVEY.md 8f row N2: x264 runs the loop filter by default inside x264_encoder_encode (av_encode.c:970).
// Bit-exact against oracle/b2o_deblock.c and, through the decoder drift test, against libavcodec.
//
// The filter is defined in macroblock raster order and every macroblock reads samples its left, top and
// top-right neighbours have already modified: MB (x, y) may run once (x-1, y) and (x+1, y-1) are done.
//
// Two schedules; b2_launch_deblock picks one by the number of frames a launch covers.
//
// ROW PIPELINE (fewer than 4 frames).  One warp owns one macroblock row and walks it left to right; row r trails row r-1 by two
// macroblocks.  The CTAs of a frame (8 warps each; up to 16 CTAs for 4K's 135 rows) form a thread-block cluster.  A row hands
// the bottom samples of every macroblock and a progress counter ("x+1 macroblocks done") to the row below through shared
// memory -- distributed shared memory (st.shared::cluster + fence.acq_rel.cluster) when the row below sits in the next CTA --
// and the row below reports back what it has read.  The dependency depth is the same mbw + 2*mbh steps as the wavefront, but
// a step is one warp's macroblock (no cluster-wide barrier: 7 us per diagonal in the wavefront) and the loads are off the
// chain: a warp prefetches the next macroblock's own samples and decision records while it filters the current one, carries
// the four left columns in shared memory, and only fetches the four rows above after the counter.
//
// ANTI-DIAGONAL WAVEFRONT (4 frames and more).  Macroblocks of one diagonal mbx + 2*mby are independent; a cluster of up to
// 8 CTAs x 16 warps per frame takes them, with a cluster barrier between diagonals.  Its chain is longer, its footprint
// smaller: when many frames' chains overlap the other stream groups' kernels, it is the faster one.
//
// Per macroblock (both forms): the 20x20 luma and two 12x12 chroma neighbourhoods live in a per-warp shared-memory tile, lanes
// 0-15 filter the luma lines (rows for vertical edges, columns for horizontal edges), lanes 16-31 the U and V lines;
// the four edges of a line are filtered by the same lane in order.
// Bound: latency of the dependency chain; algorithmic bytes 1.5*W*H read + written.
#include <stddef.h>
#include "b2_mbcode.cuh"

namespace {

using namespace b2;

// measured: 8 instead of 16 warps per CTA (smaller register footprint beside other groups' K1 CTAs) changes nothing at 1080p
// (3,850 frames/s with deblocking either way) and halves the warps available to 4K's 120-MB diagonals
constexpr int K8_WARPS = 16;
constexpr int LP = 24;      // luma tile pitch: rows -4..15, cols -4..15 -> tile[(y+4)*LP + x + 4]
constexpr int CP = 16;      // chroma tile pitch: rows -2..7, cols -4..7 -> tile[(y+2)*CP + x + 4]

__device__ __constant__ uint8_t c_alpha[52] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 4, 4, 5, 6, 7, 8, 9, 10, 12, 13,
                                               15, 17, 20, 22, 25, 28, 32, 36, 40, 45, 50, 56, 63, 71, 80, 90, 101, 113, 127, 144,
                                               162, 182, 203, 226, 255, 255};
__device__ __constant__ uint8_t c_beta[52] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4,
                                              6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13, 14, 14, 15, 15, 16, 16, 17, 17, 18, 18};
__device__ __constant__ uint8_t c_tc0[52][3] = {
    {0, 0, 0}, {0, 0, 0}, {0, 0, 0}, {0, 0, 0}, {0, 0, 0}, {0, 0, 0}, {0, 0, 0}, {0, 0, 0}, {0, 0, 0}, {0, 0, 0}, {0, 0, 0},
    {0, 0, 0}, {0, 0, 0}, {0, 0, 0}, {0, 0, 0}, {0, 0, 0}, {0, 0, 0}, {0, 0, 1}, {0, 0, 1}, {0, 0, 1}, {0, 0, 1}, {0, 1, 1},
    {0, 1, 1}, {1, 1, 1}, {1, 1, 1}, {1, 1, 1}, {1, 1, 1}, {1, 1, 2}, {1, 1, 2}, {1, 1, 2}, {1, 1, 2}, {1, 2, 3}, {1, 2, 3},
    {2, 2, 3}, {2, 2, 4}, {2, 3, 4}, {2, 3, 4}, {3, 3, 5}, {3, 4, 6}, {3, 4, 6}, {4, 5, 7}, {4, 5, 8}, {4, 6, 9}, {5, 7, 10},
    {6, 8, 11}, {6, 8, 13}, {7, 10, 14}, {8, 11, 16}, {9, 12, 18}, {10, 13, 20}, {11, 15, 23}, {13, 17, 25}};

struct K8Warp {
    __align__(16) uint8_t y[20 * LP];
    __align__(16) uint8_t c[2][10 * CP];
    int8_t bs[2][4][4];                  // [0 vertical | 1 horizontal][edge][4-sample segment]
};

__device__ __forceinline__ void cluster_barrier()
{
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ unsigned cluster_ctarank() { unsigned r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ unsigned cluster_nctarank() { unsigned r; asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r)); return r; }

__device__ __forceinline__ int clip3(int lo, int hi, int v) { return min(max(v, lo), hi); }

struct FiltConst { int alpha, beta, tc0[3]; };

// one line of samples across an edge; pix -> q0, step = distance between successive samples across the edge
__device__ __forceinline__ void filter_line(uint8_t *pix, int step, int bs, const FiltConst &fc, bool chroma)
{
    if (bs == 0) return;
    const int p0 = pix[-step], p1 = pix[-2 * step], q0 = pix[0], q1 = pix[step];
    if (!(abs(p0 - q0) < fc.alpha && abs(p1 - p0) < fc.beta && abs(q1 - q0) < fc.beta)) return;
    if (chroma) {
        if (bs < 4) {
            const int tc = fc.tc0[bs - 1] + 1;
            const int d = clip3(-tc, tc, (((q0 - p0) * 4) + (p1 - q1) + 4) >> 3);
            pix[-step] = (uint8_t)b2_clip255(p0 + d); pix[0] = (uint8_t)b2_clip255(q0 - d);
        } else {
            pix[-step] = (uint8_t)((2 * p1 + p0 + q1 + 2) >> 2);
            pix[0] = (uint8_t)((2 * q1 + q0 + p1 + 2) >> 2);
        }
        return;
    }
    const int p2 = pix[-3 * step], q2 = pix[2 * step];
    const int ap = abs(p2 - p0), aq = abs(q2 - q0);
    if (bs < 4) {
        const int tc0 = fc.tc0[bs - 1];
        const int tc = tc0 + (ap < fc.beta) + (aq < fc.beta);
        const int d = clip3(-tc, tc, (((q0 - p0) * 4) + (p1 - q1) + 4) >> 3);
        pix[-step] = (uint8_t)b2_clip255(p0 + d); pix[0] = (uint8_t)b2_clip255(q0 - d);
        if (ap < fc.beta) pix[-2 * step] = (uint8_t)(p1 + clip3(-tc0, tc0, (p2 + ((p0 + q0 + 1) >> 1) - (p1 << 1)) >> 1));
        if (aq < fc.beta) pix[step] = (uint8_t)(q1 + clip3(-tc0, tc0, (q2 + ((p0 + q0 + 1) >> 1) - (q1 << 1)) >> 1));
    } else {
        const int p3 = pix[-4 * step], q3 = pix[3 * step];
        const bool strong = abs(p0 - q0) < ((fc.alpha >> 2) + 2);
        if (ap < fc.beta && strong) {
            pix[-step] = (uint8_t)((p2 + 2 * p1 + 2 * p0 + 2 * q0 + q1 + 4) >> 3);
            pix[-2 * step] = (uint8_t)((p2 + p1 + p0 + q0 + 2) >> 2);
            pix[-3 * step] = (uint8_t)((2 * p3 + 3 * p2 + p1 + p0 + q0 + 4) >> 3);
        } else {
            pix[-step] = (uint8_t)((2 * p1 + p0 + q1 + 2) >> 2);
        }
        if (aq < fc.beta && strong) {
            pix[0] = (uint8_t)((p1 + 2 * p0 + 2 * q0 + 2 * q1 + q2 + 4) >> 3);
            pix[step] = (uint8_t)((p0 + q0 + q1 + q2 + 2) >> 2);
            pix[2 * step] = (uint8_t)((2 * q3 + 3 * q2 + q1 + q0 + p0 + 4) >> 3);
        } else {
            pix[0] = (uint8_t)((2 * q1 + q0 + p1 + 2) >> 2);
        }
    }
}

__device__ __forceinline__ int zidx(int x, int y) { return (x & 1) | ((y & 1) << 1) | ((x >> 1) << 2) | ((y >> 1) << 3); }

// does the transform block containing 4x4 block (bx,by) hold non-zero coefficients?  With the 8x8 transform that is the
// whole 8x8 block (nnz_mask bits 4q..4q+3 = its interleaved quarters)
__device__ __forceinline__ bool blk_coded(const b2_mbinfo_t *m, int bx, int by)
{
    if (m->transform8x8) return ((m->nnz_mask >> (4 * ((bx >> 1) | ((by >> 1) << 1)))) & 15u) != 0;
    return (m->nnz_mask >> zidx(bx, by)) & 1u;
}

// boundary strength (8.7.2.1) between 4x4 block (pbx,pby) of MB p and block (qbx,qby) of MB q
__device__ __forceinline__ int bs_of(const b2_mbinfo_t *mp, int pbx, int pby, const b2_mbinfo_t *mq, int qbx, int qby, bool mb_edge)
{
    if (mp->mb_type != B2_MB_P16x16 || mq->mb_type != B2_MB_P16x16) return mb_edge ? 4 : 3;
    if (blk_coded(mp, pbx, pby) || blk_coded(mq, qbx, qby)) return 2;
    const int pq = (pbx >> 1) | ((pby >> 1) << 1), qq = (qbx >> 1) | ((qby >> 1) << 1);      // 8x8 quadrants: one vector each
    const b2_mv_t a = (pq && mp->part != B2_PART_16x16) ? mp->mv8[pq - 1] : b2_mv_t{mp->mvx, mp->mvy};
    const b2_mv_t b = (qq && mq->part != B2_PART_16x16) ? mq->mv8[qq - 1] : b2_mv_t{mq->mvx, mq->mvy};
    if (abs(a.x - b.x) >= 4 || abs(a.y - b.y) >= 4) return 1;
    return 0;
}

__device__ void k8_mb_task(int lane, K8Warp &ws, uint8_t *const rec[3], int pitch, int pitchc, size_t offy, size_t offc,
                           int mbx, int mby, int mbw, const b2_mbinfo_t *mi, const FiltConst &fy, const FiltConst &fcc)
{
    uint8_t *gy = rec[0] + offy + (size_t)(B2_PAD + mby * 16) * pitch + B2_PAD + mbx * 16;
    // ---- stage the neighbourhood: luma rows -4..15 x cols -4..15 (5 words per row), chroma rows -2..7 x cols -4..7 ----
    for (int i = lane; i < 100; i += 32) {
        const int r = i / 5, w = i - r * 5;
        *(uint32_t *)&ws.y[r * LP + w * 4] = *(const uint32_t *)(gy + (ptrdiff_t)(r - 4) * pitch + (w - 1) * 4);
    }
    for (int i = lane; i < 60; i += 32) {
        const int p = i / 30, k = i - p * 30, r = k / 3, w = k - r * 3;
        const uint8_t *gc = rec[1 + p] + offc + (size_t)(B2_PADC + mby * 8) * pitchc + B2_PADC + mbx * 8;
        *(uint32_t *)&ws.c[p][r * CP + w * 4] = *(const uint32_t *)(gc + (ptrdiff_t)(r - 2) * pitchc + (w - 1) * 4);
    }
    // ---- boundary strengths: lanes 0-15 vertical edges, 16-31 horizontal edges; lane -> (edge e, segment k) ----
    {
        const int dir = lane >> 4, e = (lane >> 2) & 3, k = lane & 3;
        // picture border; with the 8x8 transform only the 8-pel edges are transform-block edges (8.7)
        const bool edge_ok = !(e == 0 && (dir == 0 ? mbx == 0 : mby == 0)) && !((e & 1) && mi->transform8x8);
        int bs = 0;
        if (edge_ok) {
            const b2_mbinfo_t *mp = e == 0 ? (dir == 0 ? mi - 1 : mi - mbw) : mi;
            const int pbx = dir == 0 ? (e == 0 ? 3 : e - 1) : k, pby = dir == 0 ? k : (e == 0 ? 3 : e - 1);
            const int qbx = dir == 0 ? e : k, qby = dir == 0 ? k : e;
            bs = bs_of(mp, pbx, pby, mi, qbx, qby, e == 0);
        }
        ws.bs[dir][e][k] = (int8_t)bs;
    }
    __syncwarp();
    // ---- vertical edges: luma lane = row, chroma lane-16 = (plane, row) ----
    if (lane < 16) {
        uint8_t *row = &ws.y[(lane + 4) * LP + 4];
#pragma unroll
        for (int e = 0; e < 4; e++) filter_line(row + 4 * e, 1, ws.bs[0][e][lane >> 2], fy, false);
    } else {
        const int l = lane - 16, p = l >> 3, r = l & 7;
        uint8_t *row = &ws.c[p][(r + 2) * CP + 4];
#pragma unroll
        for (int e = 0; e < 2; e++) filter_line(row + 4 * e, 1, ws.bs[0][2 * e][r >> 1], fcc, true);
    }
    __syncwarp();
    // ---- horizontal edges: luma lane = column, chroma lane-16 = (plane, column) ----
    if (lane < 16) {
        uint8_t *col = &ws.y[4 * LP + lane + 4];
#pragma unroll
        for (int e = 0; e < 4; e++) filter_line(col + 4 * e * LP, LP, ws.bs[1][e][lane >> 2], fy, false);
    } else {
        const int l = lane - 16, p = l >> 3, x = l & 7;
        uint8_t *col = &ws.c[p][2 * CP + x + 4];
#pragma unroll
        for (int e = 0; e < 2; e++) filter_line(col + 4 * e * CP, CP, ws.bs[1][2 * e][x >> 1], fcc, true);
    }
    __syncwarp();
    // ---- write back what can have changed: own MB, 3 (luma) / 1 (chroma) lines into the top MB, one word into the left MB ----
    for (int i = lane; i < 95; i += 32) {                  // luma rows -3..15 (19 rows) x 5 words
        const int r = i / 5 + 1, w = i - (i / 5) * 5;       // tile row r = y + 4, y = -3..15
        const int y = r - 4;
        if (w == 0 && (mbx == 0 || y < 0)) continue;        // nothing left of the picture; corner block is never modified
        if (y < 0 && mby == 0) continue;
        *(uint32_t *)(gy + (ptrdiff_t)y * pitch + (w - 1) * 4) = *(const uint32_t *)&ws.y[r * LP + w * 4];
    }
    for (int i = lane; i < 54; i += 32) {                  // chroma rows -1..7 (9 rows) x 3 words x 2 planes
        const int p = i / 27, k = i - p * 27, r = k / 3 + 1, w = k - (k / 3) * 3;
        const int y = r - 2;
        if (w == 0 && (mbx == 0 || y < 0)) continue;
        if (y < 0 && mby == 0) continue;
        uint8_t *gc = rec[1 + p] + offc + (size_t)(B2_PADC + mby * 8) * pitchc + B2_PADC + mbx * 8;
        *(uint32_t *)(gc + (ptrdiff_t)y * pitchc + (w - 1) * 4) = *(const uint32_t *)&ws.c[p][r * CP + w * 4];
    }
}

__global__ void __launch_bounds__(K8_WARPS * 32)
k8_deblock_kernel(uint8_t *ry, uint8_t *ru, uint8_t *rv, int pitch, int pitchc, size_t stride_y, size_t stride_c, int mbw, int mbh,
                  int qp, int alpha_off, int beta_off, const b2_mbinfo_t *__restrict__ info)
{
    __shared__ K8Warp s_warp[K8_WARPS];
    const int frame = blockIdx.y;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int ncta = (int)cluster_nctarank(), crank = (int)cluster_ctarank();
    const int gwarp = crank * K8_WARPS + warp, nwarps = ncta * K8_WARPS;
    const int ndiag = mbw + 2 * (mbh - 1);
    const b2_mbinfo_t *finfo = info + (size_t)frame * mbw * mbh;
    uint8_t *const rec[3] = {ry, ru, rv};
    const int qpc = chroma_qp(qp);
    FiltConst fy, fcc;
    // 8.7.2.2: indexA = qPav + 2 * slice_alpha_c0_offset_div2, indexB = qPav + 2 * slice_beta_offset_div2, clipped to 0..51
    const int ia = clip3(0, 51, qp + 2 * alpha_off), ib = clip3(0, 51, qp + 2 * beta_off);
    const int iac = clip3(0, 51, qpc + 2 * alpha_off), ibc = clip3(0, 51, qpc + 2 * beta_off);
    fy.alpha = c_alpha[ia]; fy.beta = c_beta[ib]; fcc.alpha = c_alpha[iac]; fcc.beta = c_beta[ibc];
#pragma unroll
    for (int i = 0; i < 3; i++) { fy.tc0[i] = c_tc0[ia][i]; fcc.tc0[i] = c_tc0[iac][i]; }
    for (int d = 0; d < ndiag; d++) {
        const int y_lo = max(0, (d - mbw + 2) >> 1), y_hi = min(mbh - 1, d >> 1);
        for (int t = y_lo + gwarp; t <= y_hi; t += nwarps) {
            const int mby = t, mbx = d - 2 * mby;
            k8_mb_task(lane, s_warp[warp], rec, pitch, pitchc, frame * stride_y, frame * stride_c, mbx, mby, mbw,
                       &finfo[mby * mbw + mbx], fy, fcc);
        }
        if (ncta > 1) cluster_barrier();
        else __syncthreads();
    }
}


// ---- register-resident line filter (row-pipelined form) ------------------------------------------------------------
// One edge on samples held in registers.  Luma and chroma lanes run the SAME instruction stream: chroma is luma with the
// p1/q1 updates and the strong filter switched off and tc = tc0 + 1 (8.7.2.3 / 8.7.2.4), so a warp filters its sixteen luma
// lines and sixteen chroma lines in one pass instead of one after the other.
__device__ __forceinline__ void filter_edge(int &p3, int &p2, int &p1, int &p0, int &q0, int &q1, int &q2, int &q3, int bs,
                                            int alpha, int beta, int tcpack, bool chroma)
{
    if (bs == 0) return;
    const int d0 = abs(p0 - q0);
    if (!(d0 < alpha && abs(p1 - p0) < beta && abs(q1 - q0) < beta)) return;
    const bool apb = !chroma && abs(p2 - p0) < beta, aqb = !chroma && abs(q2 - q0) < beta;
    if (bs < 4) {
        const int tc0 = (tcpack >> (8 * (bs - 1))) & 255;
        const int tc = tc0 + (chroma ? 1 : (int)apb + (int)aqb);
        const int d = clip3(-tc, tc, (((q0 - p0) * 4) + (p1 - q1) + 4) >> 3);
        const int avg = (p0 + q0 + 1) >> 1;
        if (apb) p1 += clip3(-tc0, tc0, (p2 + avg - (p1 << 1)) >> 1);
        if (aqb) q1 += clip3(-tc0, tc0, (q2 + avg - (q1 << 1)) >> 1);
        p0 = b2_clip255(p0 + d); q0 = b2_clip255(q0 - d);
    } else {
        const bool strong = d0 < ((alpha >> 2) + 2);
        const int P0 = p0, P1 = p1, P2 = p2, Q0 = q0, Q1 = q1, Q2 = q2;
        if (apb && strong) {
            p0 = (P2 + 2 * P1 + 2 * P0 + 2 * Q0 + Q1 + 4) >> 3; p1 = (P2 + P1 + P0 + Q0 + 2) >> 2; p2 = (2 * p3 + 3 * P2 + P1 + P0 + Q0 + 4) >> 3;
        } else {
            p0 = (2 * P1 + P0 + Q1 + 2) >> 2;
        }
        if (aqb && strong) {
            q0 = (P1 + 2 * P0 + 2 * Q0 + 2 * Q1 + Q2 + 4) >> 3; q1 = (P0 + Q0 + Q1 + Q2 + 2) >> 2; q2 = (2 * q3 + 3 * Q2 + Q1 + Q0 + P0 + 4) >> 3;
        } else {
            q0 = (2 * Q1 + Q0 + P1 + 2) >> 2;
        }
    }
}
// the four edges of one line of twenty samples (positions -4..15 across the macroblock; chroma lines use -4..7 and two edges)
__device__ __forceinline__ void filter_line20(int (&px)[20], const int (&bsl)[4], int alpha, int beta, int tcpack, bool chroma)
{
#pragma unroll
    for (int e = 0; e < 4; e++)
        filter_edge(px[4 * e], px[4 * e + 1], px[4 * e + 2], px[4 * e + 3], px[4 * e + 4], px[4 * e + 5], px[4 * e + 6], px[4 * e + 7], bsl[e],
                    alpha, beta, tcpack, chroma);
}

// ---- row-pipelined form -------------------------------------------------------------------------------------------
// what the boundary-strength rule needs of one b2_mbinfo_t (48 bytes = three 16-byte words: {mv, type.., i4_mode[0..7]},
// {i4_mode[8..15], cost, nnz_mask}, {mv8[3], part | transform8x8 << 8 | i8_modes << 16})
struct MbLite { uint32_t mv, typ, nnz, m8a, m8b, m8c, pt; };

__device__ __forceinline__ MbLite load_lite(const b2_mbinfo_t *m)
{
    const uint4 *q = reinterpret_cast<const uint4 *>(m);
    const uint4 a = __ldg(q), b = __ldg(q + 1), c = __ldg(q + 2);
    MbLite l;
    l.mv = a.x; l.typ = a.y & 255u; l.nnz = b.w; l.m8a = c.x; l.m8b = c.y; l.m8c = c.z; l.pt = c.w;
    return l;
}
__device__ __forceinline__ bool lite_coded(const MbLite &m, int bx, int by)
{
    if ((m.pt >> 8) & 255u) return ((m.nnz >> (4 * ((bx >> 1) | ((by >> 1) << 1)))) & 15u) != 0;
    return (m.nnz >> zidx(bx, by)) & 1u;
}
__device__ __forceinline__ uint32_t lite_mv(const MbLite &m, int q)
{
    if (q == 0 || (m.pt & 255u) == B2_PART_16x16) return m.mv;
    return q == 1 ? m.m8a : (q == 2 ? m.m8b : m.m8c);
}
__device__ __forceinline__ int lite_bs(const MbLite &mp, int pbx, int pby, const MbLite &mq, int qbx, int qby, bool mb_edge)
{
    if (mp.typ != B2_MB_P16x16 || mq.typ != B2_MB_P16x16) return mb_edge ? 4 : 3;
    if (lite_coded(mp, pbx, pby) || lite_coded(mq, qbx, qby)) return 2;
    const uint32_t a = lite_mv(mp, (pbx >> 1) | ((pby >> 1) << 1)), b = lite_mv(mq, (qbx >> 1) | ((qby >> 1) << 1));
    const int ax = (int16_t)(a & 0xffffu), ay = (int16_t)(a >> 16), bx = (int16_t)(b & 0xffffu), by = (int16_t)(b >> 16);
    return (abs(ax - bx) >= 4 || abs(ay - by) >= 4) ? 1 : 0;
}

// distributed shared memory: address of a shared-memory object of CTA `cta` of the cluster, plain stores to it, and the
// cluster-scope fence that orders them ahead of the progress counter
__device__ __forceinline__ uint32_t dsmem_addr(const void *local, unsigned cta)
{
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(local)), "r"(cta));
    return r;
}
__device__ __forceinline__ void dsmem_st(uint32_t addr, uint32_t v) { asm volatile("st.shared::cluster.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory"); }
__device__ __forceinline__ void dsmem_st_relaxed(uint32_t addr, int v) { asm volatile("st.relaxed.cluster.shared::cluster.s32 [%0], %1;" ::"r"(addr), "r"(v) : "memory"); }
__device__ __forceinline__ void fence_cluster() { asm volatile("fence.acq_rel.cluster;" ::: "memory"); }

// bottom rows of the macroblocks of one row, handed to the row below through shared memory: entry g % K8_RING belongs to the
// row's g-th macroblock (counted over all rows the warp has walked): y[r * 4 + w] = luma row 12 + r, word w;
// c[p * 4 + r * 2 + w] = chroma plane p, row 6 + r, word w
constexpr int K8_RING = 8;
// warps (macroblock rows) per CTA of the row pipeline: the register-resident lines need ~120 registers; 16 warps per CTA squeeze them
// into 64 and spill
constexpr int K8_ROW_WARPS = 8;
struct K8Ring { uint32_t y[K8_RING][16]; uint32_t c[K8_RING][8]; };      // c directly behind y: word index K8_RING * 16 + ...
static_assert(offsetof(K8Ring, c) == K8_RING * 16 * 4, "K8Ring layout");

__global__ void __launch_bounds__(K8_ROW_WARPS * 32, 2)
k8_deblock_rows_kernel(uint8_t *ry, uint8_t *ru, uint8_t *rv, int pitch, int pitchc, size_t stride_y, size_t stride_c, int mbw, int mbh,
                       int qp, int alpha_off, int beta_off, const b2_mbinfo_t *__restrict__ info)
{
    __shared__ K8Warp s_warp[K8_ROW_WARPS];
    // s_ring[w] / s_done[w]: bottom rows and progress of the producer OF warp w, i.e. of the row above warp w's row.  Warp w - 1
    // of this CTA writes them for w > 0; the last warp of the previous CTA of the cluster writes s_ring[0] / s_done[0] through
    // distributed shared memory.  s_back[w]: progress of the consumer of warp w (next warp, or warp 0 of the next CTA), for the
    // ring's back-pressure.  Every warp only ever POLLS its own CTA's shared memory.
    __shared__ K8Ring s_ring[K8_ROW_WARPS];
    __shared__ int s_done[K8_ROW_WARPS];
    __shared__ int s_back[K8_ROW_WARPS];
    const int frame = blockIdx.y;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int ncta = (int)cluster_nctarank(), crank = (int)cluster_ctarank();
    const int gwarp = crank * K8_ROW_WARPS + warp, nwarps = ncta * K8_ROW_WARPS;
    const b2_mbinfo_t *finfo = info + (size_t)frame * mbw * mbh;
    uint8_t *const py = ry + frame * stride_y, *const pu = ru + frame * stride_c, *const pv = rv + frame * stride_c;
    // per-lane filter constants: lanes 0-15 carry luma lines, 16-31 chroma lines.  8.7.2.2: indexA = qPav + 2 * slice_alpha_c0_offset_div2,
    // indexB = qPav + 2 * slice_beta_offset_div2, clipped to 0..51
    const bool is_c = lane >= 16;
    const int l_qp = is_c ? chroma_qp(qp) : qp;
    const int l_ia = clip3(0, 51, l_qp + 2 * alpha_off), l_ib = clip3(0, 51, l_qp + 2 * beta_off);
    const int l_alpha = c_alpha[l_ia], l_beta = c_beta[l_ib];
    const int l_tc = c_tc0[l_ia][0] | c_tc0[l_ia][1] << 8 | c_tc0[l_ia][2] << 16;
    const int cl = lane - 16, c_pl = (cl >> 3) & 1, c_i = cl & 7;             // chroma lanes: plane, row (vertical pass) / column (horizontal)
    if (threadIdx.x < K8_ROW_WARPS) { s_done[threadIdx.x] = 0; s_back[threadIdx.x] = 0; }
    if (ncta > 1) cluster_barrier();      // nobody stores into a neighbour's counters before they are cleared
    else __syncthreads();

    K8Warp &ws = s_warp[warp];
    // The row below belongs to the next warp of this CTA or, for the last warp, to warp 0 of the next CTA of the cluster: the
    // bottom rows go into THAT warp's ring (s_ring[consumer warp] of the consumer's CTA) with st.shared::cluster, then the
    // progress counter; the consumer reports back into s_back[] of this CTA the same way.  No global round trip and no
    // GPU-scope fence anywhere on the chain.
    const bool cons_remote = warp == K8_ROW_WARPS - 1, prod_remote = warp == 0;
    const unsigned cons_cta = cons_remote ? (unsigned)((crank + 1) % ncta) : (unsigned)crank;
    const unsigned prod_cta = prod_remote ? (unsigned)((crank + ncta - 1) % ncta) : (unsigned)crank;
    const int cons_w = cons_remote ? 0 : warp + 1, prod_w = prod_remote ? K8_ROW_WARPS - 1 : warp - 1;
    const uint32_t out_ring = dsmem_addr(&s_ring[cons_w], cons_cta);             // where this warp's bottom rows go
    const uint32_t out_done = dsmem_addr(&s_done[cons_w], cons_cta);
    const uint32_t out_back = dsmem_addr(&s_back[prod_w], prod_cta);             // where this warp reports what it has consumed
    const volatile int *const prod_done = &s_done[warp];
    const volatile int *const cons_done = &s_back[warp];
    const K8Ring &prod_ring = s_ring[warp];
    // this lane's boundary-strength job: lanes 0-15 vertical edges, 16-31 horizontal edges; lane -> (edge e, segment k)
    const int dir = lane >> 4, e = (lane >> 2) & 3, k = lane & 3;
    // own-sample words: lane -> luma words (row l>>1, words 2*(l&1), 2*(l&1)+1), chroma word (plane l>>4, row (l>>1)&7, word l&1)
    const int oy_row = lane >> 1, oy_w = (lane & 1) * 2;
    const int oc_p = lane >> 4, oc_row = (lane >> 1) & 7, oc_w = lane & 1;

    // Write-back roles, fixed per lane: the tile words that can have changed are luma rows -3..15 x 5 words (95 items, lane takes
    // items lane, lane + 32, lane + 64) and chroma rows -1..7 x 3 words x 2 planes (54 items, lane and lane + 32).  Per item:
    // tile byte offset, offset from the macroblock's first sample in the plane, and what kind of neighbour it touches.
    int wb_t[5], wb_g[5], wb_k[5];        // kind bits: 1 = left neighbour's word, 2 = rows above, 4 = rows the row below rewrites
#pragma unroll
    for (int j = 0; j < 3; j++) {
        const int i = lane + 32 * j, r = i / 5 + 1, w = i - (i / 5) * 5, y = r - 4;
        wb_t[j] = r * LP + w * 4; wb_g[j] = y * pitch + (w - 1) * 4;
        wb_k[j] = i < 95 ? ((w == 0 ? 1 : 0) | (y < 0 ? 2 : 0) | (y >= 13 ? 4 : 0)) : 8;
    }
#pragma unroll
    for (int j = 0; j < 2; j++) {
        const int i = lane + 32 * j, p = i / 27, kk = i - p * 27, r = kk / 3 + 1, w = kk - (kk / 3) * 3, y = r - 2;
        wb_t[3 + j] = (int)(&ws.c[p & 1][r * CP + w * 4] - &ws.y[0]); wb_g[3 + j] = y * pitchc + (w - 1) * 4;
        wb_k[3 + j] = i < 54 ? ((w == 0 ? 1 : 0) | (y < 0 ? 2 : 0) | (y >= 7 ? 4 : 0) | (p ? 16 : 0)) : 8;
    }

    int round = 0;
    for (int mby = gwarp; mby < mbh; mby += nwarps, round++) {
        const int prod_base = ((mby - 1) / nwarps) * mbw;      // what the producer had finished before it started row mby-1
        const int my_base = round * mbw;
        const bool has_cons = mby + 1 < mbh;
        // rows 13..15 (chroma: row 7) of a macroblock are last written by the row below (its top-edge filter); this warp only
        // stores them when nobody below will, or when the row below reads them from global memory
        const bool own_bottom = !has_cons;
        uint8_t *const rowy = py + (size_t)(B2_PAD + mby * 16) * pitch + B2_PAD;
        uint8_t *const rowu = pu + (size_t)(B2_PADC + mby * 8) * pitchc + B2_PADC;
        uint8_t *const rowv = pv + (size_t)(B2_PADC + mby * 8) * pitchc + B2_PADC;
        // ---- prologue: own samples and decision records of macroblock 0 ----
        uint32_t n0, n1, n2;
        MbLite lq, lp;
        {
            const uint32_t *g = (const uint32_t *)(rowy + (size_t)oy_row * pitch) + oy_w;
            n0 = g[0]; n1 = g[1];
            n2 = *((const uint32_t *)((oc_p ? rowv : rowu) + (size_t)oc_row * pitchc) + oc_w);
            const b2_mbinfo_t *mq = &finfo[mby * mbw];
            lq = load_lite(mq);
            lp = (e == 0 && dir == 1 && mby > 0) ? load_lite(mq - mbw) : lq;
        }
        for (int mbx = 0; mbx < mbw; mbx++) {
            const int g_me = my_base + mbx;                       // this macroblock's running number in this warp
            // ---- own samples (prefetched) -> tile; boundary strengths from the prefetched records ----
            *(uint32_t *)&ws.y[(oy_row + 4) * LP + 4 + oy_w * 4] = n0;
            *(uint32_t *)&ws.y[(oy_row + 4) * LP + 8 + oy_w * 4] = n1;
            *(uint32_t *)&ws.c[oc_p][(oc_row + 2) * CP + 4 + oc_w * 4] = n2;
            {
                const bool edge_ok = !(e == 0 && (dir == 0 ? mbx == 0 : mby == 0)) && !((e & 1) && ((lq.pt >> 8) & 255u));
                int bs = 0;
                if (edge_ok) {
                    const int pbx = dir == 0 ? (e == 0 ? 3 : e - 1) : k, pby = dir == 0 ? k : (e == 0 ? 3 : e - 1);
                    const int qbx = dir == 0 ? e : k, qby = dir == 0 ? k : e;
                    bs = lite_bs(lp, pbx, pby, lq, qbx, qby, e == 0);
                }
                ws.bs[dir][e][k] = (int8_t)bs;
            }
            // ---- prefetch the next macroblock: own samples + decision records (nothing in this kernel writes them before) ----
            if (mbx + 1 < mbw) {
                const uint32_t *g = (const uint32_t *)(rowy + (size_t)oy_row * pitch + (mbx + 1) * 16) + oy_w;
                n0 = g[0]; n1 = g[1];
                n2 = *((const uint32_t *)((oc_p ? rowv : rowu) + (size_t)oc_row * pitchc + (mbx + 1) * 8) + oc_w);
                const b2_mbinfo_t *mq = &finfo[mby * mbw + mbx + 1];
                const MbLite cur = lq;                           // becomes the left neighbour
                lq = load_lite(mq);
                lp = e != 0 ? lq : (dir == 0 ? cur : (mby > 0 ? load_lite(mq - mbw) : lq));
            }
            // ---- the four rows above: final once row mby-1 has finished macroblock mbx+1.  Fetched now, written into the
            //      tile after the vertical pass (which only touches rows 0..15) ----
            uint32_t top = 0;
            if (mby > 0) {
                const int need = prod_base + min(mbx + 2, mbw);
                while (*prod_done < need) { }
                if (prod_remote) fence_cluster();                 // the ring entry came through distributed shared memory
                else __threadfence_block();
                const int slot = (prod_base + mbx) % K8_RING;
                if (lane < 16) top = prod_ring.y[slot][lane];
                else if (lane < 24) top = prod_ring.c[slot][lane - 16];
            }
            __syncwarp();
            // ---- vertical edges: luma lane = row, chroma lane-16 = (plane, row); the line lives in registers ----
            {
                uint8_t *rowp = is_c ? &ws.c[c_pl][(c_i + 2) * CP] : &ws.y[(lane + 4) * LP];
                int px[20], bsl[4];
#pragma unroll
                for (int w = 0; w < 5; w++) {
                    const uint32_t v = *(const uint32_t *)(rowp + 4 * w);      // chroma: words 3, 4 belong to the next row and are not used
                    px[4 * w] = v & 255; px[4 * w + 1] = (v >> 8) & 255; px[4 * w + 2] = (v >> 16) & 255; px[4 * w + 3] = v >> 24;
                }
                const int seg = is_c ? c_i >> 1 : lane >> 2;
#pragma unroll
                for (int ee = 0; ee < 4; ee++) bsl[ee] = is_c ? (ee < 2 ? ws.bs[0][2 * ee][seg] : 0) : ws.bs[0][ee][seg];
                filter_line20(px, bsl, l_alpha, l_beta, l_tc, is_c);
#pragma unroll
                for (int w = 0; w < 5; w++)
                    if (!is_c || w < 3)
                        *(uint32_t *)(rowp + 4 * w) = (uint32_t)px[4 * w] | (uint32_t)px[4 * w + 1] << 8 | (uint32_t)px[4 * w + 2] << 16 | (uint32_t)px[4 * w + 3] << 24;
            }
            if (mby > 0) {
                if (lane < 16) *(uint32_t *)&ws.y[(lane >> 2) * LP + 4 + (lane & 3) * 4] = top;          // rows -4..-1, words 0..3
                else if (lane < 24) { const int l = lane - 16; *(uint32_t *)&ws.c[l >> 2][((l >> 1) & 1) * CP + 4 + (l & 1) * 4] = top; }
            }
            __syncwarp();
            // ---- horizontal edges: luma lane = column, chroma lane-16 = (plane, column) ----
            {
                // sample i of the line sits `stride` bytes after sample i-1; chroma columns only exist for i = 2..11 (rows -2..7)
                uint8_t *colp = is_c ? &ws.c[c_pl][4 + c_i] - 2 * CP : &ws.y[4 + lane];
                const int stride = is_c ? CP : LP;
                int px[20], bsl[4];
#pragma unroll
                for (int i = 0; i < 20; i++) px[i] = (!is_c || (i >= 2 && i < 12)) ? colp[i * stride] : 0;
                const int seg = is_c ? c_i >> 1 : lane >> 2;
#pragma unroll
                for (int ee = 0; ee < 4; ee++) bsl[ee] = is_c ? (ee < 2 ? ws.bs[1][2 * ee][seg] : 0) : ws.bs[1][ee][seg];
                filter_line20(px, bsl, l_alpha, l_beta, l_tc, is_c);
#pragma unroll
                for (int i = 1; i < 19; i++)                                       // p2 of the first edge .. q2 of the last
                    if (!is_c || (i >= 2 && i < 12)) colp[i * stride] = (uint8_t)px[i];
            }
            __syncwarp();
            // ---- hand the bottom rows to the row below: this macroblock's entry, and the four rightmost columns of the previous
            //      entry, which this macroblock's left edge has just finished ----
            if (has_cons) {
                while (*cons_done < g_me - K8_RING + 1) { }                         // the entry about to be overwritten has been read
                const int slot = g_me % K8_RING, pslot = (g_me + K8_RING - 1) % K8_RING;
                // which word of the consumer's ring this lane writes, and from where in the tile
                int widx = -1; uint32_t wval = 0;
                if (lane < 16) { widx = slot * 16 + lane; wval = *(const uint32_t *)&ws.y[(16 + (lane >> 2)) * LP + 4 + (lane & 3) * 4]; }
                else if (lane < 24) { const int l = lane - 16; widx = K8_RING * 16 + slot * 8 + l; wval = *(const uint32_t *)&ws.c[l >> 2][(8 + ((l >> 1) & 1)) * CP + 4 + (l & 1) * 4]; }
                else if (mbx > 0) {
                    const int l = lane - 24;                                      // 0..3 luma rows 12..15, 4..7 chroma (plane, row 6..7)
                    if (l < 4) { widx = pslot * 16 + l * 4 + 3; wval = *(const uint32_t *)&ws.y[(16 + l) * LP]; }
                    else { widx = K8_RING * 16 + pslot * 8 + ((l - 4) >> 1) * 4 + ((l - 4) & 1) * 2 + 1; wval = *(const uint32_t *)&ws.c[(l - 4) >> 1][(8 + ((l - 4) & 1)) * CP]; }
                }
                if (widx >= 0) {
                    if (cons_remote) dsmem_st(out_ring + widx * 4, wval);          // into the next CTA of the cluster
                    else ((uint32_t *)&s_ring[warp + 1])[widx] = wval;
                }
            }
            // ---- write back what can have changed: own MB, 3 (luma) / 1 (chroma) lines into the top MB, one word into the left MB ----
            {
                // an item is skipped when it is a corner (left AND above: never modified), lies outside the picture, or belongs to
                // the rows the row below stores after its own top-edge filter
                const int skip = 8 | (mbx == 0 ? 1 : 0) | (mby == 0 ? 2 : 0) | (own_bottom ? 0 : 4);
                uint8_t *gy = rowy + mbx * 16, *gu = rowu + mbx * 8, *gv = rowv + mbx * 8;
#pragma unroll
                for (int j = 0; j < 5; j++) {
                    const int kd = wb_k[j];
                    if ((kd & skip) || (kd & 3) == 3) continue;
                    uint8_t *g = j < 3 ? gy : ((kd & 16) ? gv : gu);
                    *(uint32_t *)(g + wb_g[j]) = *(const uint32_t *)(&ws.y[0] + wb_t[j]);
                }
            }
            // ---- publish: the ring stores of every lane are ordered ahead of the counter; tell the row above what has been read ----
            if (cons_remote || prod_remote) fence_cluster();
            else __threadfence_block();
            __syncwarp();
            if (lane == 0) {
                if (has_cons) {
                    if (cons_remote) dsmem_st_relaxed(out_done, g_me + 1);
                    else *(volatile int *)&s_done[warp + 1] = g_me + 1;
                }
                if (mby > 0) {                                                    // in the producer's numbering
                    if (prod_remote) dsmem_st_relaxed(out_back, prod_base + mbx + 1);
                    else *(volatile int *)&s_back[warp - 1] = prod_base + mbx + 1;
                }
            }
            // ---- carry the four rightmost columns over as the next macroblock's left neighbour ----
            if (lane < 16) *(uint32_t *)&ws.y[(lane + 4) * LP] = *(const uint32_t *)&ws.y[(lane + 4) * LP + 16];
            else *(uint32_t *)&ws.c[(lane - 16) >> 3][(((lane - 16) & 7) + 2) * CP] = *(const uint32_t *)&ws.c[(lane - 16) >> 3][(((lane - 16) & 7) + 2) * CP + 8];
            __syncwarp();
        }
    }
    if (ncta > 1) cluster_barrier();      // no CTA leaves while a neighbour may still store into its shared memory
}

}  // namespace

void b2_deblock_shape(int mbw, int mbh, int nframes, int *wavefront, int *ncta, int *rounds)
{
    // Two schedules.  The row pipeline has the shorter chain (0.87 vs 1.59 ms for one 1080p frame) and is what a launch of few
    // frames wants -- the drop-in's one-GOP-per-stream shape, live streams.  A launch that covers many frames (bench.py: 8 per
    // stream group, 8 groups) is throughput-bound, its chains hide behind the other groups' K1, and there the anti-diagonal
    // wavefront's smaller footprint (40 registers, nothing spinning) is worth ~3 % of the step: 4 frames and up take it.
    if (nframes < 4) {
        // One warp per macroblock row (beyond 8 CTAs of rows, warps take several); the CTAs of a frame form a cluster so that
        // the hand-off between the last row of one CTA and the first row of the next stays in (distributed) shared memory.
        int n = (mbh + K8_ROW_WARPS - 1) / K8_ROW_WARPS;
        if (n > 8) {
            // tall pictures (4K: 135 rows): a cluster of up to 16 CTAs (non-portable size, supported on B200) keeps one warp per row;
            // with 8 CTAs the rows beyond the 64th would have to wait for a warp of the first rows to finish its whole row
            // (the attribute is per device; engines may live on several devices of one process, so it is set on every such launch)
            const bool np_ok = cudaFuncSetAttribute(k8_deblock_rows_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess;
            n = np_ok ? (n > 16 ? 16 : n) : 8;
            cudaGetLastError();
        }
        *wavefront = 0; *ncta = n;
        *rounds = (mbh + n * K8_ROW_WARPS - 1) / (n * K8_ROW_WARPS);
        return;
    }
    int n = 1;
    const int maxdiag = mbh < (mbw + 1) / 2 ? mbh : (mbw + 1) / 2;
    while (n < 8 && n * K8_WARPS < maxdiag) n *= 2;
    *wavefront = 1; *ncta = n;
    *rounds = (maxdiag + n * K8_WARPS - 1) / (n * K8_WARPS);
}

int b2_launch_deblock(uint8_t *const rec[3], int pitch, int pitchc, size_t stride_y, size_t stride_c, int mbw, int mbh,
                      int nframes, int qp, int alpha_off, int beta_off, const b2_mbinfo_t *d_info, int *d_flags, cudaStream_t st)
{
    (void)d_flags;
    int wavefront, ncta, rounds;
    b2_deblock_shape(mbw, mbh, nframes, &wavefront, &ncta, &rounds);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(ncta, nframes, 1);
    cfg.blockDim = dim3((wavefront ? K8_WARPS : K8_ROW_WARPS) * 32, 1, 1);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = ncta; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    if (wavefront)
        B2_CUDA_OK(cudaLaunchKernelEx(&cfg, k8_deblock_kernel, rec[0], rec[1], rec[2], pitch, pitchc, stride_y, stride_c, mbw, mbh, qp,
                                      alpha_off, beta_off, d_info));
    else
        B2_CUDA_OK(cudaLaunchKernelEx(&cfg, k8_deblock_rows_kernel, rec[0], rec[1], rec[2], pitch, pitchc, stride_y, stride_c, mbw, mbh, qp,
                                      alpha_off, beta_off, d_info));
    return 0;
}
