// k1_me_fullpel.cu -- K1: exhaustive full-pel SAD motion search, one MV per 16x16 macroblock.
//
// Replaces the full-pel half of the motion estimation that the reference reaches through
// x264_encoder_encode() (av_encode.c:970); bit-exact against oracle/b2o_me.c:b2o_me_fullpel.
//
// Bound: integer ALU (VABSDIFF4.U8.ACC issue rate).  Algorithmic work per macroblock:
// (2R+1)^2 candidates x 256 pixel-SADs = (2R+1)^2 x 64 VABSDIFF4 lane-instructions.
//
// Design (SURVEY.md 7.2 items 3-5):
//  * One CTA searches a strip of NMB = 6 horizontally adjacent macroblocks of one frame.  The
//    (16 NMB + 2R) x (16+2R) search window of the *padded* reference plane and the 16 NMB x 16 current
//    tile are fetched by TMA (cp.async.bulk.tensor.3d), never leaving the allocation because
//    every plane carries a 64-px replicated border.
//  * Operand supply, not the ALU, is the first limiter (32 shared-memory words/clk/SM vs 64
//    VABSDIFF4 lanes/clk/SM).  Two reuse tricks remove it:
//      - the window is expanded once into "one 32-bit word per pixel position"
//        (word x = pixels x..x+3), so every byte alignment is a plain conflict-free LDS.32;
//      - register tiling: a lane owns one dx and K consecutive dy; the current macroblock sits
//        in 64 registers, each reference row is loaded once (4 LDS.32) and applied to up to K
//        current rows (K accumulators) -> (16+K-1)*4 loads per 64*K VABSDIFF4.
//  * Lanes of a warp are 32 consecutive LANE-TASKS (mb, dy-group, dx).  Inside one (mb, dy-group) segment that is 32 consecutive
//    dx = 32 consecutive words: one wavefront.  A segment is 2R+1 = 65 (33) tasks long, not a multiple of 32, so about every other
//    warp-task straddles two segments whose rows start at the same bank (EXP_PITCH % 32 == 0): its sweep LDS.32 then take two
//    wavefronts.  ncu, per instruction (profiles/r2_k1_lds_bank_conflicts.txt): every sweep LDS averages 1.475 wavefronts, together
//    17.8 M of the kernel's 18.4 M excess wavefronts per 4-frame launch; the remaining 0.6 M are the ATOMS.MIN on the best keys.
//    The shared-memory pipe still runs at only 0.46 wavefronts/clk/SM while the ALU pipe is 92 % busy, so this is not the limiter --
//    and the fix was measured to cost more than it saves: a pitch with K * pitch = 1 (mod 32) lines the two segments' banks up, but
//    such a pitch is odd, so the expansion can no longer store 16 bytes per lane; bit-identical, 0.889 -> 0.868 of the VABSDIFF4 peak
//    with word-wise expansion alone and 0.853 with the padded pitch (+-16: 0.836 -> 0.787; profiles/r2_k1_exppad_ab.txt).
//    The conflicts stay.
//  * Winner: key = (cost << 13) | scan_index, CREDUX.MIN over the warp, atomicMin in smem.
//    Lowest scan index wins ties by construction, exactly like the oracle's strict '<'.
#include <atomic>
#include "b2_common.cuh"

namespace {

// Strip width and residency, tuned on the B200 (1080p +-32, 32 frames):
//   NMB x CTAs/SM :  8x2 0.859   10x2 0.874   12x2 0.879   5x3 0.885   6x3 0.888   7x3 0.881   4x3 0.871   of the VABSDIFF4 peak.
// Three resident CTAs (80 registers, 67 KB of shared memory each) keep the ALU pipe fed while one of them waits for its
// TMA window / expands it; a wider strip only amortises the halo.
// +-16: strips of 10 MBs.  Swept on the B200 with 192/256/320/384 threads (profiles/r2_k1_r16_strip_sweep.txt):
//   8 -> 0.821, 10 -> 0.838, 12 -> 0.817, 14 -> 0.829 of the VABSDIFF4 peak at 720p.
// 256 threads per CTA: a sweep of 192/256/320/384 threads found the ALU pipe itself to be the plateau (256 and 384 both 0.85 of the
// peak), not the rounding of 82 (+-32) / 41 (+-16) warp-tasks per full strip over the warps.
constexpr int K1_THREADS = 256;
constexpr int K1_MINCTAS = 3;
template <int R> struct K1Cfg;
// NMB = macroblocks per CTA strip
template <> struct K1Cfg<32> { static constexpr int K = 13, NG = 5, NMB = 6; };      // 65 = 5 x 13
template <> struct K1Cfg<16> { static constexpr int K = 11, NG = 3, NMB = 10; };     // 33 = 3 x 11

template <int R> struct K1Smem {
    static constexpr int NMB = K1Cfg<R>::NMB;
    static constexpr int ND = 2 * R + 1;
    static constexpr int WIN_W = NMB * 16 + 2 * R;      // bytes per raw window row
    static constexpr int WIN_H = 16 + 2 * R;
    static constexpr int RAW_BYTES = WIN_W * WIN_H;
    static constexpr int EXP_PITCH = WIN_W;             // words per expanded row
    static constexpr int EXP_BYTES = EXP_PITCH * WIN_H * 4;
    static constexpr int CUR_BYTES = NMB * 16 * 16;
    // layout (all 128-B aligned)
    static constexpr int OFF_RAW = 0;
    static constexpr int OFF_CUR = (RAW_BYTES + 16 + 127) & ~127;
    static constexpr int OFF_EXP = OFF_CUR + CUR_BYTES;
    static constexpr int OFF_COSTX = OFF_EXP + EXP_BYTES;
    static constexpr int OFF_COSTY = OFF_COSTX + NMB * ND * 4;
    static constexpr int OFF_BEST = OFF_COSTY + NMB * ND * 4;
    static constexpr int OFF_BAR = (OFF_BEST + NMB * 9 * 4 + 7) & ~7;    // 9 best keys per MB in the partition variant
    static constexpr int TOTAL = OFF_BAR + 8 + 128;     // +128: manual alignment slack
};

// PART (row N1, partitions = 2): the same sweep also yields the SAD of every 8x8 quadrant, hence the best vector of each of
// the nine shape parts (16x16 | 16x8 top,bottom | 8x16 left,right | four 8x8).  The number of VABSDIFF4 is unchanged; a lane
// sweeps the top half of the current MB, packs the two 8x8 SADs of its K candidates into K registers, sweeps the bottom
// half, and then forms 9 sums / keys per candidate (9 running minima, 9 CREDUX.MIN + 9 shared atomicMin per warp task).
template <int R, bool PART>
__global__ void __launch_bounds__(K1_THREADS, PART ? 2 : K1_MINCTAS)      // the partition variant needs ~90 registers: two CTAs
k1_me_fullpel_kernel(const __grid_constant__ CUtensorMap tm_cur,
                     const __grid_constant__ CUtensorMap tm_ref,
                     int mbw, int mbh, const b2_mv_t *__restrict__ pmv, int lambda,
                     b2_mv_t *__restrict__ mv_out, uint32_t *__restrict__ cost_out,
                     b2_mv_t *__restrict__ mv9_out, uint32_t *__restrict__ cost9_out)
{
    using S = K1Smem<R>;
    constexpr int NWARPS = K1_THREADS / 32;
    constexpr int K = K1Cfg<R>::K, NG = K1Cfg<R>::NG, ND = S::ND, NMB = K1Cfg<R>::NMB;
    static_assert(K * NG == ND, "dy groups must tile the search range");

    extern __shared__ uint8_t smem_raw_[];
    uint8_t *smem = smem_raw_ + ((128u - (smem_u32(smem_raw_) & 127u)) & 127u);   // keeps the shared address space
    uint8_t *s_raw = smem + S::OFF_RAW;
    uint8_t *s_cur = smem + S::OFF_CUR;
    uint32_t *s_exp = (uint32_t *)(smem + S::OFF_EXP);
    uint32_t *s_costx = (uint32_t *)(smem + S::OFF_COSTX);
    uint32_t *s_costy = (uint32_t *)(smem + S::OFF_COSTY);
    uint32_t *s_best = (uint32_t *)(smem + S::OFF_BEST);
    uint64_t *s_bar = (uint64_t *)(smem + S::OFF_BAR);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int mb0 = blockIdx.x * NMB, mby = blockIdx.y, frame = blockIdx.z;
    const int nmb = min(NMB, mbw - mb0);

    if (tid == 0) {
        mbar_init(s_bar, 1);
        fence_mbar_init();
    }
    __syncthreads();
    if (tid == 0) {
        mbar_expect_tx(s_bar, S::RAW_BYTES + S::CUR_BYTES);
        tma_load_3d(s_raw, &tm_ref, B2_PAD + mb0 * 16 - R, B2_PAD + mby * 16 - R, frame, s_bar);
        tma_load_3d(s_cur, &tm_cur, B2_PAD + mb0 * 16, B2_PAD + mby * 16, frame, s_bar);
    }

    // while the TMA is in flight: motion-vector cost tables and best-key init
    const size_t mb_base = ((size_t)frame * mbh + mby) * mbw + mb0;
    for (int i = tid; i < NMB * ND; i += K1_THREADS) {
        int m = i / ND, d = i - m * ND;
        int px = 0, py = 0;
        if (pmv != nullptr && m < nmb) { b2_mv_t p = pmv[mb_base + m]; px = p.x; py = p.y; }
        // pre-shifted so that key = (SAD << 13) + kx + ky = ((SAD + costx + costy) << 13) | scan index
        s_costx[i] = ((uint32_t)(lambda * b2_mvbits(4 * (d - R) - px)) << 13) + (uint32_t)d;
        s_costy[i] = ((uint32_t)(lambda * b2_mvbits(4 * (d - R) - py)) << 13) + (uint32_t)(d * ND);
    }
    if (tid < NMB * (PART ? 9 : 1)) s_best[tid] = 0xffffffffu;

    mbar_wait(s_bar, 0);

    // expand: word x of a row = pixels x..x+3 (little endian), all 4 byte alignments
    {
        constexpr int WPR = S::WIN_W / 4;             // aligned words per raw row
        const uint32_t *raw32 = (const uint32_t *)s_raw;
        for (int i = tid; i < WPR * S::WIN_H; i += K1_THREADS) {
            int r = i / WPR, j = i - r * WPR;
            uint32_t lo = raw32[i], hi = raw32[i + 1];    // last word of the buffer: 16 B slack
            uint4 o;
            o.x = lo;
            o.y = __funnelshift_r(lo, hi, 8);
            o.z = __funnelshift_r(lo, hi, 16);
            o.w = __funnelshift_r(lo, hi, 24);
            *(uint4 *)(s_exp + r * S::EXP_PITCH + 4 * j) = o;
        }
    }
    __syncthreads();

    const int total = nmb * NG * ND;                  // lane-tasks: (mb, dy-group, dx)
    for (int t0 = warp * 32; t0 < total; t0 += NWARPS * 32) {
        const int t = t0 + lane;
        const bool active = t < total;
        const int tt = active ? t : t0;               // idle lanes shadow lane 0's task
        const int m = tt / (NG * ND);
        const int rem = tt - m * (NG * ND);
        const int g = rem / ND;
        const int dxi = rem - g * ND;

        if constexpr (PART) {
            uint32_t top[K];                               // SAD(top-left 8x8) | SAD(top-right 8x8) << 16
            uint32_t best[9];
#pragma unroll
            for (int p = 0; p < 9; p++) best[p] = 0xffffffffu;
            const uint32_t kx = s_costx[m * ND + dxi];
            const uint32_t *ky = s_costy + m * ND + g * K;
#pragma unroll
            for (int half = 0; half < 2; half++) {
                uint32_t cur[32];                          // 8 rows of the current macroblock
                {
                    const uint4 *c4 = (const uint4 *)(s_cur + m * 16) + half * 8 * (NMB * 16 / 16);
#pragma unroll
                    for (int y = 0; y < 8; y++) {
                        uint4 v = c4[y * (NMB * 16 / 16)];
                        cur[y * 4 + 0] = v.x; cur[y * 4 + 1] = v.y; cur[y * 4 + 2] = v.z; cur[y * 4 + 3] = v.w;
                    }
                }
                uint32_t accl[K], accr[K];
#pragma unroll
                for (int k = 0; k < K; k++) accl[k] = accr[k] = 0;
                const uint32_t *wp = s_exp + (g * K + half * 8) * S::EXP_PITCH + m * 16 + dxi;
#pragma unroll
                for (int r = 0; r < K + 7; r++) {
                    const uint32_t w0 = wp[r * S::EXP_PITCH + 0];
                    const uint32_t w1 = wp[r * S::EXP_PITCH + 4];
                    const uint32_t w2 = wp[r * S::EXP_PITCH + 8];
                    const uint32_t w3 = wp[r * S::EXP_PITCH + 12];
#pragma unroll
                    for (int k = 0; k < K; k++) {
                        const int y = r - k;
                        if (y >= 0 && y < 8) {
                            accl[k] = vsad4_acc(w0, cur[y * 4 + 0], accl[k]);
                            accl[k] = vsad4_acc(w1, cur[y * 4 + 1], accl[k]);
                            accr[k] = vsad4_acc(w2, cur[y * 4 + 2], accr[k]);
                            accr[k] = vsad4_acc(w3, cur[y * 4 + 3], accr[k]);
                        }
                    }
                }
                if (half == 0) {
#pragma unroll
                    for (int k = 0; k < K; k++) top[k] = accl[k] | (accr[k] << 16);
                } else if (active) {
                    uint32_t pend[9];                          // keys of the previous candidate: merged two at a time (VIMNMX3)
#pragma unroll
                    for (int k = 0; k < K; k++) {
                        const uint32_t tl = top[k] & 0xffffu, tr = top[k] >> 16, bl = accl[k], br = accr[k];
                        const uint32_t kc = kx + ky[k];
                        const uint32_t st = tl + tr, sb = bl + br;
                        const uint32_t c[9] = {(st + sb) * 8192u + kc, st * 8192u + kc, sb * 8192u + kc, (tl + bl) * 8192u + kc,
                                               (tr + br) * 8192u + kc, tl * 8192u + kc,  tr * 8192u + kc, bl * 8192u + kc, br * 8192u + kc};
#pragma unroll
                        for (int p = 0; p < 9; p++) {
                            if (k & 1) best[p] = __vimin3_u32(best[p], pend[p], c[p]);
                            else if (k == K - 1) best[p] = min(best[p], c[p]);
                            else pend[p] = c[p];
                        }
                    }
                }
            }
            const int m0 = __shfl_sync(0xffffffffu, m, 0);
            if (__all_sync(0xffffffffu, m == m0)) {
#pragma unroll
                for (int p = 0; p < 9; p++) {
                    const uint32_t wmin = __reduce_min_sync(0xffffffffu, best[p]);
                    if (lane == 0) atomicMin(&s_best[m0 * 9 + p], wmin);
                }
            } else if (active) {
#pragma unroll
                for (int p = 0; p < 9; p++) atomicMin(&s_best[m * 9 + p], best[p]);
            }
        } else {
        // current macroblock -> 64 registers
        uint32_t cur[64];
        {
            const uint4 *c4 = (const uint4 *)(s_cur + m * 16);
#pragma unroll
            for (int y = 0; y < 16; y++) {
                uint4 v = c4[y * (NMB * 16 / 16)];
                cur[y * 4 + 0] = v.x; cur[y * 4 + 1] = v.y; cur[y * 4 + 2] = v.z; cur[y * 4 + 3] = v.w;
            }
        }
        uint32_t acc[K];
#pragma unroll
        for (int k = 0; k < K; k++) acc[k] = 0;

        const uint32_t *wp = s_exp + (g * K) * S::EXP_PITCH + m * 16 + dxi;
#pragma unroll
        for (int r = 0; r < K + 15; r++) {
            const uint32_t w0 = wp[r * S::EXP_PITCH + 0];
            const uint32_t w1 = wp[r * S::EXP_PITCH + 4];
            const uint32_t w2 = wp[r * S::EXP_PITCH + 8];
            const uint32_t w3 = wp[r * S::EXP_PITCH + 12];
#pragma unroll
            for (int k = 0; k < K; k++) {
                const int y = r - k;                  // current row that meets reference row r at dy = g*K+k
                if (y >= 0 && y < 16) {
                    acc[k] = vsad4_acc(w0, cur[y * 4 + 0], acc[k]);
                    acc[k] = vsad4_acc(w1, cur[y * 4 + 1], acc[k]);
                    acc[k] = vsad4_acc(w2, cur[y * 4 + 2], acc[k]);
                    acc[k] = vsad4_acc(w3, cur[y * 4 + 3], acc[k]);
                }
            }
        }

        uint32_t key = 0xffffffffu;
        if (active) {
            const uint32_t kx = s_costx[m * ND + dxi];
            const uint32_t *ky = s_costy + m * ND + g * K;
            // three-input minimum (VIMNMX3): half as many ALU-pipe instructions beside the VABSDIFF4 stream
#pragma unroll
            for (int k = 0; k + 1 < K; k += 2) key = __vimin3_u32(key, acc[k] * 8192u + (kx + ky[k]), acc[k + 1] * 8192u + (kx + ky[k + 1]));
            if (K & 1) key = min(key, acc[K - 1] * 8192u + (kx + ky[K - 1]));
        }
        const int m0 = __shfl_sync(0xffffffffu, m, 0);
        if (__all_sync(0xffffffffu, m == m0)) {
            const uint32_t wmin = __reduce_min_sync(0xffffffffu, key);
            if (lane == 0) atomicMin(&s_best[m0], wmin);
        } else if (active) {
            atomicMin(&s_best[m], key);
        }
        }
    }
    __syncthreads();

    if (tid < nmb * (PART ? 9 : 1)) {
        const uint32_t key = s_best[tid];
        const int idx = (int)(key & 8191u);
        const int dyi = idx / ND, dxi = idx - dyi * ND;
        b2_mv_t mv;
        mv.x = (int16_t)(dxi - R);
        mv.y = (int16_t)(dyi - R);
        if constexpr (PART) {
            const int mm = tid / 9, p = tid - mm * 9;
            mv9_out[(mb_base + mm) * 9 + p] = mv;
            cost9_out[(mb_base + mm) * 9 + p] = key >> 13;
            if (p == 0) { mv_out[mb_base + mm] = mv; cost_out[mb_base + mm] = key >> 13; }
        } else {
            mv_out[mb_base + tid] = mv;
            cost_out[mb_base + tid] = key >> 13;
        }
    }
}

// ---- lossless pruning: successive elimination in front of the same sweep (engine option me_prune) ---------------------------
// |sum(cur MB) - sum(ref block)| <= SAD(cur MB, ref block) (triangle inequality), so a candidate whose
//     |C - S(dx,dy)| + mvcost(dx,dy)  >  U,     U = exact cost of any candidate already evaluated,
// cannot be the minimum and cannot tie with it either; dropping it leaves argmin AND tie-break of the exhaustive scan untouched
// (x264's own "esa" search is built on the same inequality).  The unit that is kept or dropped is the sweep's lane-task
// (mb, dy-group of KS rows, dx): it is dropped when NONE of its KS candidates can pass, i.e. when
//     dist(C, [min_k S, max_k S]) + mvcost_x(dx) + min_k mvcost_y  >  U
// -- the interval form of the bound; K1a below delivers min | max of the 16x16 block sums over KS consecutive rows for every
// position of the padded reference plane, so the test is ONE shared-memory word per lane-task.  Per strip:
//   1. TMA window + current tile, cost tables, expansion: as k1_me_fullpel_kernel;
//   2. the raw window is dead after the expansion: the NG rows of (min | max) words the strip needs arrive by TMA into the same
//      shared memory (NG one-row boxes on a second mbarrier);
//   3. meanwhile one warp per macroblock evaluates two candidates exactly -- the zero vector and the rounded predictor (the
//      co-located vector of the previous frame) -- which gives U and the first best key;
//   4. bound test per lane-task (a warp walks 32 consecutive dx of one macroblock: ~20 instructions per lane-task); a survivor
//      goes into the queue of ITS shared-memory bank, q = (16 * mb + dx) mod 32 (one shared atomicAdd, no two lanes of a warp hit
//      the same counter);
//   5. the register-tiled sweep of k1_me_fullpel_kernel runs over the queues: lane q of warp-task i takes entry i of queue q.  The
//      expanded rows are a multiple of 32 words long, so the 32 lanes of every sweep load hit 32 different banks whatever rows and
//      macroblocks they work on (a plain survivor list gave 1.9 wavefronts per load: the band of survivors of neighbouring dy groups
//      overlaps in x; ncu: profiles/r2_k1_pruned_ncu.txt).  Queues that overflow (more than QCAP survivors: predictors that point
//      nowhere) make the strip fall back to sweeping every lane-task in natural order.
// What is skipped is reported, never folded into the roofline figure: `swept` counts the candidates that ran (b2_engine_k1_stats).
// KS (rows per lane-task): 5 (+-32) / 3 (+-16) instead of the exhaustive kernel's 13 / 11.  Fewer rows = finer pruning but fewer
// VABSDIFF4 per shared-memory load (13 -> 5 rows: 7.4 -> 4.0 per LDS.32, still ALU-bound when the loads are conflict-free); measured
// faster at 1080p +-32: 0.871 -> 0.803 ms on the synthetic pan, 0.908 -> 0.886 ms on natural-like content (profiles/r2_k1_pruned_forms.txt).
template <int R> constexpr int K1_PRUNE_KS = R == 32 ? 5 : 3;
constexpr int K1_PRUNE_MINCTAS = 3;
// partial-distortion exit inside the sweep: reference rows after which it is tested, K + FIRST, K + FIRST + STEP, ... <= K + LAST
// (every candidate has then seen at least FIRST + 1 rows); swept on the B200: profiles/r2_k1_pde_schedule.txt
constexpr int K1_PDE_FIRST = 5, K1_PDE_LAST = 9, K1_PDE_STEP = 4;

constexpr int k1_cmax(int a, int b) { return a > b ? a : b; }
template <int R, int KS> struct K1SeaSmem {
    using S = K1Smem<R>;                                          // the exhaustive kernel's strips (and tensor maps)
    static constexpr int NMB = S::NMB;
    static constexpr int ND = S::ND, NG = ND / KS;
    static_assert(NG * KS == ND, "dy groups must tile the search range");
    static_assert(S::EXP_PITCH % 32 == 0, "bank queues need expanded rows of a multiple of 32 words");
    static_assert(NMB <= 16 && NG <= 16 && ND <= 128, "queue entries are m | g << 4 | dx << 8");
    static constexpr int NX = (NMB - 1) * 16 + ND;               // candidate columns of a strip
    static constexpr int MP = (NX + 31) & ~31;                   // words per row of (min | max) sums: every row is its own TMA box, 128-B aligned
    static constexpr int M_BYTES = MP * NG * 4;
    static constexpr int NTASK = NMB * NG * ND;
    // entries per bank queue: all lane-tasks of a bank when that is small, else 128 (60-80 % of them: a strip whose predictors point
    // nowhere overflows and takes the natural-order path)
    static constexpr int QCAP = NTASK / 32 + 8 < 128 ? ((NTASK / 32 + 8 + 7) & ~7) : 128;
    static constexpr int Q_BYTES = 32 * QCAP * 2;
    // region 0: raw window while it is expanded, then the (min | max) rows followed by the 32 bank queues
    static constexpr int OFF_Q = (M_BYTES + 127) & ~127;
    static constexpr int R0_BYTES = k1_cmax(S::RAW_BYTES + 16, OFF_Q + Q_BYTES);
    static constexpr int OFF_R0 = 0;
    static constexpr int OFF_CUR = (R0_BYTES + 127) & ~127;
    static constexpr int OFF_EXP = OFF_CUR + S::CUR_BYTES;
    static constexpr int OFF_COSTX = OFF_EXP + S::EXP_BYTES;
    static constexpr int OFF_COSTY = OFF_COSTX + NMB * ND * 4;
    static constexpr int OFF_BEST = OFF_COSTY + NMB * ND * 4;
    static constexpr int OFF_CSUM = OFF_BEST + NMB * 4;
    static constexpr int OFF_PMV = OFF_CSUM + NMB * 4;           // NMB x {x, y}
    static constexpr int OFF_TG = OFF_PMV + NMB * 8;             // NMB x NG: U - smallest vertical vector cost of the group
    static constexpr int OFF_CNT = OFF_TG + NMB * NG * 4;        // 32 queue lengths + overflow flag
    static constexpr int OFF_BAR = (OFF_CNT + 33 * 4 + 7) & ~7;
    static constexpr int TOTAL = OFF_BAR + 16 + 128;             // +128: manual alignment slack
};
static_assert(K1_PRUNE_MINCTAS * (K1SeaSmem<32, K1_PRUNE_KS<32>>::TOTAL + 1024) <= 228 * 1024, "pruned K1 (+-32, 5 rows): the CTAs per SM asked for do not fit");

template <int R, int KS>
__global__ void __launch_bounds__(K1_THREADS, K1_PRUNE_MINCTAS)
k1_me_fullpel_sea_kernel(const __grid_constant__ CUtensorMap tm_cur, const __grid_constant__ CUtensorMap tm_ref,
                         const __grid_constant__ CUtensorMap tm_mm, int mbw, int mbh, const b2_mv_t *__restrict__ pmv, int lambda,
                         b2_mv_t *__restrict__ mv_out, uint32_t *__restrict__ cost_out, unsigned long long *__restrict__ swept)
{
    using Q = K1SeaSmem<R, KS>;
    using S = typename Q::S;
    constexpr int NWARPS = K1_THREADS / 32;
    constexpr int K = KS, NG = Q::NG, ND = S::ND, NMB = Q::NMB, QCAP = Q::QCAP;

    extern __shared__ uint8_t smem_raw_[];
    uint8_t *smem = smem_raw_ + ((128u - (smem_u32(smem_raw_) & 127u)) & 127u);
    uint8_t *s_raw = smem + Q::OFF_R0;
    const uint32_t *s_mm = (const uint32_t *)(smem + Q::OFF_R0);
    uint16_t *s_queue = (uint16_t *)(smem + Q::OFF_R0 + Q::OFF_Q);
    uint8_t *s_cur = smem + Q::OFF_CUR;
    uint32_t *s_exp = (uint32_t *)(smem + Q::OFF_EXP);
    uint32_t *s_costx = (uint32_t *)(smem + Q::OFF_COSTX);
    uint32_t *s_costy = (uint32_t *)(smem + Q::OFF_COSTY);
    uint32_t *s_best = (uint32_t *)(smem + Q::OFF_BEST);
    int *s_csum = (int *)(smem + Q::OFF_CSUM);
    int *s_pmv = (int *)(smem + Q::OFF_PMV);
    int *s_tg = (int *)(smem + Q::OFF_TG);
    int *s_cnt = (int *)(smem + Q::OFF_CNT);          // [32] queue lengths, [32] overflow flag
    uint64_t *s_bar = (uint64_t *)(smem + Q::OFF_BAR);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int mb0 = blockIdx.x * NMB, mby = blockIdx.y, frame = blockIdx.z;
    const int nmb = min(NMB, mbw - mb0);
    const size_t mb_base = ((size_t)frame * mbh + mby) * mbw + mb0;

    if (tid == 0) {
        mbar_init(&s_bar[0], 1);
        mbar_init(&s_bar[1], 1);
        fence_mbar_init();
    }
    if (tid < 33) s_cnt[tid] = 0;
    if (tid >= 64 && tid < 64 + NMB) {     // predictors: one global load per macroblock
        const int m = tid - 64;
        int px = 0, py = 0;
        if (pmv != nullptr && m < nmb) { const b2_mv_t p = pmv[mb_base + m]; px = p.x; py = p.y; }
        s_pmv[2 * m] = px; s_pmv[2 * m + 1] = py;
    }
    __syncthreads();
    if (tid == 0) {
        mbar_expect_tx(&s_bar[0], S::RAW_BYTES + S::CUR_BYTES);
        tma_load_3d(s_raw, &tm_ref, B2_PAD + mb0 * 16 - R, B2_PAD + mby * 16 - R, frame, &s_bar[0]);
        tma_load_3d(s_cur, &tm_cur, B2_PAD + mb0 * 16, B2_PAD + mby * 16, frame, &s_bar[0]);
    }

    for (int i = tid; i < NMB * ND; i += K1_THREADS) {
        const int m = i / ND, d = i - m * ND;
        s_costx[i] = ((uint32_t)(lambda * b2_mvbits(4 * (d - R) - s_pmv[2 * m])) << 13) + (uint32_t)d;
        s_costy[i] = ((uint32_t)(lambda * b2_mvbits(4 * (d - R) - s_pmv[2 * m + 1])) << 13) + (uint32_t)(d * ND);
    }

    mbar_wait(&s_bar[0], 0);
    {
        constexpr int WPR = S::WIN_W / 4;
        const uint32_t *raw32 = (const uint32_t *)s_raw;
        for (int i = tid; i < WPR * S::WIN_H; i += K1_THREADS) {
            int r = i / WPR, j = i - r * WPR;
            uint32_t lo = raw32[i], hi = raw32[i + 1];
            uint4 o;
            o.x = lo;
            o.y = __funnelshift_r(lo, hi, 8);
            o.z = __funnelshift_r(lo, hi, 16);
            o.w = __funnelshift_r(lo, hi, 24);
            *(uint4 *)(s_exp + r * S::EXP_PITCH + 4 * j) = o;
        }
    }
    fence_proxy_async();                  // this thread's generic reads of the raw window precede the TMA writes into the same bytes
    __syncthreads();                      // expansion and cost tables complete; the raw window is dead from here on
    if (tid == 0) {
        mbar_expect_tx(&s_bar[1], Q::M_BYTES);
        for (int g = 0; g < NG; g++)
            tma_load_3d(s_raw + g * Q::MP * 4, &tm_mm, B2_PAD + mb0 * 16 - R, B2_PAD + mby * 16 - R + g * K, frame, &s_bar[1]);
    }

    // thresholds while those rows are in flight: exact keys of the zero vector and of the rounded predictor; then U - min_k mvcost_y
    // per dy group
    for (int m = warp; m < nmb; m += NWARPS) {
        const int px = s_pmv[2 * m], py = s_pmv[2 * m + 1];
        const int cdx = min(max((px + 2) >> 2, -R), R) + R, cdy = min(max((py + 2) >> 2, -R), R) + R;
        uint32_t sa = 0, sb = 0, cs = 0;
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const int w = lane + 32 * h, y = w >> 2, c = w & 3;
            const uint32_t cw = ((const uint32_t *)s_cur)[y * (NMB * 4) + m * 4 + c];
            sa = vsad4_acc(s_exp[(R + y) * S::EXP_PITCH + m * 16 + R + 4 * c], cw, sa);
            sb = vsad4_acc(s_exp[(cdy + y) * S::EXP_PITCH + m * 16 + cdx + 4 * c], cw, sb);
            cs = __dp4a(cw, 0x01010101u, cs);
        }
        sa = __reduce_add_sync(0xffffffffu, sa);
        sb = __reduce_add_sync(0xffffffffu, sb);
        cs = __reduce_add_sync(0xffffffffu, cs);
        const uint32_t ka = sa * 8192u + s_costx[m * ND + R] + s_costy[m * ND + R];
        const uint32_t kb = sb * 8192u + s_costx[m * ND + cdx] + s_costy[m * ND + cdy];
        const uint32_t kk = min(ka, kb);
        if (lane == 0) {
            s_best[m] = kk;
            s_csum[m] = (int)cs;
        }
        for (int g = lane; g < NG; g += 32) {
            uint32_t mn = 0xffffffffu;
#pragma unroll
            for (int k = 0; k < K; k++) mn = min(mn, s_costy[m * ND + g * K + k] >> 13);
            s_tg[m * NG + g] = (int)(kk >> 13) - (int)mn;
        }
    }
    __syncthreads();
    mbar_wait(&s_bar[1], 0);

    // bound test.  A warp takes a UNIT = (macroblock, block of 32 columns, parity of the dy group): a lane keeps its column, so the
    // column's vector cost, the macroblock's sum and the queue number are loaded once and the groups are walked with immediate
    // offsets (about 10 instructions per lane-task; per-lane-task decoding cost 50).  The search range is 32 * FULL + 1 columns wide:
    // the left-over column of all NG groups of a macroblock makes one more round (lane = group).  Survivors go to their bank's
    // queue; entry i of all 32 queues is one row of 32 u16.
    {
        constexpr int FULL = (ND - 1) / 32;
        static_assert(FULL * 32 + 1 == ND && NG <= 32 && (FULL == 1 || FULL == 2), "unit layout of the bound test");
        auto append = [&](int q, uint32_t entry) {
            const int slot = atomicAdd(&s_cnt[q], 1);
            if (slot < QCAP) s_queue[slot * 32 + q] = (uint16_t)entry;
            else s_cnt[32] = 1;
        };
        const int units = nmb * FULL * 2;
        for (int u = warp; u < units; u += NWARPS) {
            const int m = u / (FULL * 2), rem = u - m * (FULL * 2), par = rem & 1;
            const int dxi = (rem >> 1) * 32 + lane;
            const int c = s_csum[m];
            const int cx = (int)(s_costx[m * ND + dxi] >> 13);
            const uint32_t *mmp = s_mm + par * Q::MP + m * 16 + dxi;
            const int *tgp = s_tg + m * NG + par;
            const int q = (m * 16 + dxi) & 31;
            const uint32_t ent = (uint32_t)(m | par << 4 | dxi << 8);
#pragma unroll
            for (int g2 = 0; g2 < (NG + 1) / 2; g2++) {
                if (2 * g2 + par < NG) {
                    const int t = tgp[2 * g2] - cx;
                    const uint32_t mm = mmp[2 * g2 * Q::MP];
                    const int d = max((int)(mm & 0xffffu) - c, c - (int)(mm >> 16));  // distance of C to [min, max]; negative inside
                    if (t >= 0 && d <= t) append(q, ent + (uint32_t)(2 * g2 << 4));
                }
            }
        }
        for (int m = warp; m < nmb; m += NWARPS) {
            if (lane < NG) {
                const int g = lane, dxi = ND - 1;
                const int t = s_tg[m * NG + g] - (int)(s_costx[m * ND + dxi] >> 13);
                const uint32_t mm = s_mm[g * Q::MP + m * 16 + dxi];
                const int c = s_csum[m];
                const int d = max((int)(mm & 0xffffu) - c, c - (int)(mm >> 16));
                if (t >= 0 && d <= t) append((m * 16 + dxi) & 31, (uint32_t)(m | g << 4 | dxi << 8));
            }
        }
    }
    __syncthreads();

    // one lane-task of the sweep: K candidates (dy = g*K .. g*K+K-1 at dx) of macroblock m; returns the smallest key.
    // Partial-distortion exit: a SAD only grows row by row, so once the PARTIAL key of every candidate of every lane of the warp
    // exceeds the macroblock's best key so far, none of them can become the minimum (keys are unique per candidate) and the warp
    // drops the rest of the task; checked after reference rows K + 5 and K + 9 (each candidate has then seen at least 6 / 10 rows).
    auto lane_task = [&](int m, int g, int dxi, bool active) -> uint32_t {
        uint32_t cur[64];
        {
            const uint4 *c4 = (const uint4 *)(s_cur + m * 16);
#pragma unroll
            for (int y = 0; y < 16; y++) {
                uint4 v = c4[y * (NMB * 16 / 16)];
                cur[y * 4 + 0] = v.x; cur[y * 4 + 1] = v.y; cur[y * 4 + 2] = v.z; cur[y * 4 + 3] = v.w;
            }
        }
        uint32_t acc[K], kc[K];
        {
            const uint32_t kx = s_costx[m * ND + dxi];
            const uint32_t *ky = s_costy + m * ND + g * K;
#pragma unroll
            for (int k = 0; k < K; k++) { acc[k] = 0; kc[k] = kx + ky[k]; }
        }
        const uint32_t *wp = s_exp + (g * K) * S::EXP_PITCH + m * 16 + dxi;
        bool dropped = false;
#pragma unroll
        for (int r = 0; r < K + 15; r++) {
            const uint32_t w0 = wp[r * S::EXP_PITCH + 0];
            const uint32_t w1 = wp[r * S::EXP_PITCH + 4];
            const uint32_t w2 = wp[r * S::EXP_PITCH + 8];
            const uint32_t w3 = wp[r * S::EXP_PITCH + 12];
#pragma unroll
            for (int k = 0; k < K; k++) {
                const int y = r - k;
                if (y >= 0 && y < 16) {
                    acc[k] = vsad4_acc(w0, cur[y * 4 + 0], acc[k]);
                    acc[k] = vsad4_acc(w1, cur[y * 4 + 1], acc[k]);
                    acc[k] = vsad4_acc(w2, cur[y * 4 + 2], acc[k]);
                    acc[k] = vsad4_acc(w3, cur[y * 4 + 3], acc[k]);
                }
            }
            if (r >= K + K1_PDE_FIRST && r <= K + K1_PDE_LAST && ((r - (K + K1_PDE_FIRST)) % K1_PDE_STEP) == 0) {
                bool hopeless = true;
                if (active) {
                    const uint32_t bk = ((volatile uint32_t *)s_best)[m];
#pragma unroll
                    for (int k = 0; k < K; k++) hopeless = hopeless && acc[k] * 8192u + kc[k] > bk;
                }
                if (__all_sync(0xffffffffu, hopeless)) { dropped = true; break; }
            }
        }
        uint32_t key = 0xffffffffu;
        if (active && !dropped) {
#pragma unroll
            for (int k = 0; k + 1 < K; k += 2) key = __vimin3_u32(key, acc[k] * 8192u + kc[k], acc[k + 1] * 8192u + kc[k + 1]);
            if (K & 1) key = min(key, acc[K - 1] * 8192u + kc[K - 1]);
        }
        return key;
    };

    long long executed;
    if (s_cnt[32] == 0) {
        const int mine = s_cnt[lane];
        const int rounds = __reduce_max_sync(0xffffffffu, mine);
        for (int i = warp; i < rounds; i += NWARPS) {
            const bool active = i < mine;
            // idle lanes sweep a harmless task of their own bank: (mb 0, group 0, dx = lane)
            const int tt = active ? (int)s_queue[i * 32 + lane] : lane << 8;
            const int m = tt & 15, g = (tt >> 4) & 15, dxi = tt >> 8;
            const uint32_t key = lane_task(m, g, dxi, active);
            if (active) atomicMin(&s_best[m], key);
        }
        int sum = mine;
#pragma unroll
        for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
        executed = (long long)sum * K;
    } else {
        // a queue overflowed: every lane-task, in the exhaustive kernel's order
        const int total = nmb * NG * ND;
        for (int t0 = warp * 32; t0 < total; t0 += NWARPS * 32) {
            const int t = t0 + lane;
            const bool active = t < total;
            const int tt = active ? t : t0;
            const int m = tt / (NG * ND);
            const int rem = tt - m * (NG * ND);
            const int g = rem / ND;
            const int dxi = rem - g * ND;
            const uint32_t key = lane_task(m, g, dxi, active);
            const int m0 = __shfl_sync(0xffffffffu, m, 0);
            if (__all_sync(0xffffffffu, m == m0)) {
                const uint32_t wmin = __reduce_min_sync(0xffffffffu, key);
                if (lane == 0) atomicMin(&s_best[m0], wmin);
            } else if (active) {
                atomicMin(&s_best[m], key);
            }
        }
        executed = (long long)total * K;
    }
    __syncthreads();

    if (tid < nmb) {
        const uint32_t key = s_best[tid];
        const int idx = (int)(key & 8191u);
        const int dyi = idx / ND, dxi = idx - dyi * ND;
        b2_mv_t mv;
        mv.x = (int16_t)(dxi - R);
        mv.y = (int16_t)(dyi - R);
        mv_out[mb_base + tid] = mv;
        cost_out[mb_base + tid] = key >> 13;
    }
    if (tid == 0 && swept != nullptr) atomicAdd(swept, (unsigned long long)executed);
}

// K1a: for every position (Y, X) of a padded luma plane, min | max << 16 over the KS rows Y..Y+KS-1 of the 16x16 block sums
// S[Y][X] = sum of plane[Y..Y+15][X..X+15] (at most 65,280: u16), as one u32 -- what the pruned search tests a lane-task with.
// Same [n][rows][pitch] geometry as the plane; positions whose blocks leave the allocation hold 0 | 0xffff (never prune).
// HBM-bound by design (1 B read + 4 B written per pixel).  One CTA per 128 x 48 tile; every pass works on PAIRS of adjacent
// columns packed as u16x2 (VIADD.16x2 / VIMNMX.U16x2): vertical 16-sums by a sliding column walk (three row segments so that
// 216 threads walk), the horizontal 16-sum as two levels of 4, then the row-window minimum / maximum.
constexpr int K1A_TW = 128, K1A_TH = 48;
template <int KS>
__global__ void __launch_bounds__(256) k1a_block_sums_kernel(const uint8_t *__restrict__ planes, int pitch, int rows, size_t plane_stride,
                                                             uint32_t *__restrict__ mm_out)
{
    constexpr int SR = K1A_TH + KS - 1;                   // rows of block sums a tile needs
    constexpr int IR = SR + 15;                           // input rows
    constexpr int WPR = (K1A_TW + 16) / 4;                // input words per row
    constexpr int PPR = (K1A_TW + 16) / 2;                // column pairs per row
    // the input tile is dead once the vertical sums exist: the sums of 4 columns reuse its memory (30 instead of 40 KB per CTA: seven
    // CTAs per SM instead of five -- the kernel is a chain of short phases and lives on occupancy)
    constexpr int A_WORDS = IR * WPR > SR * PPR ? IR * WPR : SR * PPR;
    __shared__ uint32_t s_a[A_WORDS];
    __shared__ uint32_t s_v[SR][PPR];                     // vertical 16-sums (pairs); later the block sums themselves ([SR][K1A_TW / 2] used)
    uint32_t (*s_in)[WPR] = (uint32_t (*)[WPR])s_a;
    uint32_t (*s_q)[PPR] = (uint32_t (*)[PPR])s_a;        // sums of 4 columns: pair p = (q[2p], q[2p+1])
    const int tid = threadIdx.x;
    const int x0 = blockIdx.x * K1A_TW, y0 = blockIdx.y * K1A_TH;
    const uint8_t *plane = planes + (size_t)blockIdx.z * plane_stride;
    uint32_t *out = mm_out + (size_t)blockIdx.z * plane_stride;         // same element stride: the plane of words mirrors the luma plane
    for (int i = tid; i < IR * WPR; i += 256) {
        const int r = i / WPR, w = i - r * WPR;
        const int yy = min(y0 + r, rows - 1), xx = x0 + 4 * w;
        s_in[r][w] = xx + 3 < pitch ? *(const uint32_t *)(plane + (size_t)yy * pitch + xx) : 0u;
    }
    __syncthreads();
    {
        constexpr int NSEG = 3, SEG = (SR + NSEG - 1) / NSEG;
        const int seg = tid / PPR, cp = tid - seg * PPR;
        if (seg < NSEG) {
            const uint16_t *col = (const uint16_t *)&s_in[0][0] + cp;   // two adjacent bytes of every row
            constexpr int P = WPR * 2;                                   // row pitch in u16
            const int r0 = seg * SEG, r1 = min(SR, r0 + SEG);
            uint32_t acc = 0;
#pragma unroll
            for (int j = 0; j < 16; j++) acc += __byte_perm((uint32_t)col[(r0 + j) * P], 0u, 0x4140);
            s_v[r0][cp] = acc;
            for (int r = r0 + 1; r < r1; r++) {
                acc += __byte_perm((uint32_t)col[(r + 15) * P], 0u, 0x4140) - __byte_perm((uint32_t)col[(r - 1) * P], 0u, 0x4140);
                s_v[r][cp] = acc;                                        // both halves stay below 4,081: no carry between them
            }
        }
    }
    __syncthreads();
    for (int i = tid; i < SR * (PPR - 2); i += 256) {                    // q[x] = v[x] + v[x+1] + v[x+2] + v[x+3] for the pair (2p, 2p+1)
        const int y = i / (PPR - 2), p = i - y * (PPR - 2);
        const uint32_t w0 = s_v[y][p], w1 = s_v[y][p + 1], w2 = s_v[y][p + 2];
        s_q[y][p] = __vadd2(__vadd2(w0, __funnelshift_r(w0, w1, 16)), __vadd2(w1, __funnelshift_r(w1, w2, 16)));
    }
    __syncthreads();
    for (int i = tid; i < SR * (K1A_TW / 2); i += 256) {                 // block sums into s_v (its vertical sums are dead)
        const int y = i / (K1A_TW / 2), p = i - y * (K1A_TW / 2);
        s_v[y][p] = __vadd2(__vadd2(s_q[y][p], s_q[y][p + 2]), __vadd2(s_q[y][p + 4], s_q[y][p + 6]));
    }
    __syncthreads();
    for (int i = tid; i < K1A_TH * (K1A_TW / 2); i += 256) {
        const int y = i / (K1A_TW / 2), p = i - y * (K1A_TW / 2);
        const int Y = y0 + y, X = x0 + 2 * p;
        if (Y < rows && X < pitch) {
            uint32_t lo = s_v[y][p], hi = lo;
#pragma unroll
            for (int j = 1; j < KS; j++) {
                const uint32_t v = s_v[y + j][p];
                lo = __vminu2(lo, v); hi = __vmaxu2(hi, v);
            }
            const bool rows_ok = Y + KS - 1 + 16 <= rows;
            uint2 o;
            o.x = rows_ok && X + 16 <= pitch ? (lo & 0xffffu) | (hi << 16) : 0xffff0000u;
            o.y = rows_ok && X + 17 <= pitch ? (lo >> 16) | (hi & 0xffff0000u) : 0xffff0000u;
            *(uint2 *)(out + (size_t)Y * pitch + X) = o;
        }
    }
}

template <int R, bool PART>
int launch_k1p(const CUtensorMap &tm_cur, const CUtensorMap &tm_ref, int mbw, int mbh, int nframes, const b2_mv_t *pmv, int lambda,
               b2_mv_t *mv_out, uint32_t *cost_out, b2_mv_t *mv9_out, uint32_t *cost9_out, cudaStream_t st)
{
    // function attributes are per device: one process may drive several GPUs, each from its own host thread
    static std::atomic<bool> attr_set[64];
    int dev = 0;
    B2_CUDA_OK(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64 || !attr_set[dev].load(std::memory_order_acquire)) {
        B2_CUDA_OK(cudaFuncSetAttribute(k1_me_fullpel_kernel<R, PART>, cudaFuncAttributeMaxDynamicSharedMemorySize, K1Smem<R>::TOTAL));
        if (dev >= 0 && dev < 64) attr_set[dev].store(true, std::memory_order_release);
    }
    constexpr int NMB = K1Cfg<R>::NMB;
    dim3 grid((mbw + NMB - 1) / NMB, mbh, nframes);
    k1_me_fullpel_kernel<R, PART><<<grid, K1_THREADS, K1Smem<R>::TOTAL, st>>>(tm_cur, tm_ref, mbw, mbh, pmv, lambda, mv_out, cost_out,
                                                                              mv9_out, cost9_out);
    B2_CUDA_OK(cudaGetLastError());
    return 0;
}
template <int R>
int launch_k1(const CUtensorMap &tm_cur, const CUtensorMap &tm_ref, int mbw, int mbh, int nframes, const b2_mv_t *pmv, int lambda,
              b2_mv_t *mv_out, uint32_t *cost_out, b2_mv_t *mv9_out, uint32_t *cost9_out, cudaStream_t st)
{
    if (mv9_out) return launch_k1p<R, true>(tm_cur, tm_ref, mbw, mbh, nframes, pmv, lambda, mv_out, cost_out, mv9_out, cost9_out, st);
    return launch_k1p<R, false>(tm_cur, tm_ref, mbw, mbh, nframes, pmv, lambda, mv_out, cost_out, nullptr, nullptr, st);
}

template <int R>
int launch_k1_sea(const CUtensorMap &tm_cur, const CUtensorMap &tm_ref, const CUtensorMap &tm_mm, int mbw, int mbh, int nframes,
                  const b2_mv_t *pmv, int lambda, b2_mv_t *mv_out, uint32_t *cost_out, unsigned long long *swept, cudaStream_t st)
{
    constexpr int KS = K1_PRUNE_KS<R>;
    static std::atomic<bool> attr_set[64];
    int dev = 0;
    B2_CUDA_OK(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64 || !attr_set[dev].load(std::memory_order_acquire)) {
        B2_CUDA_OK(cudaFuncSetAttribute(k1_me_fullpel_sea_kernel<R, KS>, cudaFuncAttributeMaxDynamicSharedMemorySize, K1SeaSmem<R, KS>::TOTAL));
        if (dev >= 0 && dev < 64) attr_set[dev].store(true, std::memory_order_release);
    }
    constexpr int NMB = K1Cfg<R>::NMB;
    dim3 grid((mbw + NMB - 1) / NMB, mbh, nframes);
    k1_me_fullpel_sea_kernel<R, KS><<<grid, K1_THREADS, K1SeaSmem<R, KS>::TOTAL, st>>>(tm_cur, tm_ref, tm_mm, mbw, mbh, pmv, lambda, mv_out,
                                                                                       cost_out, swept);
    B2_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // namespace

extern "C" int b2_k1_strip_mbs(int R) { return R == 16 ? K1Cfg<16>::NMB : K1Cfg<32>::NMB; }

// window/current-tile box sizes needed to build the tensor maps
extern "C" int b2_k1_window_box(int R, int *bw, int *bh)
{
    if (R != 16 && R != 32) return -1;
    *bw = b2_k1_strip_mbs(R) * 16 + 2 * R;
    *bh = 16 + 2 * R;
    return 0;
}

// d_* are device pointers; the tensor maps describe [nframes][rows][pitch] padded luma planes
// with boxes {128+2R, 16+2R, 1} (ref) and {128, 16, 1} (cur).
int b2_launch_me_fullpel(int R, const CUtensorMap *tm_cur, const CUtensorMap *tm_ref, int mbw, int mbh,
                         int nframes, const b2_mv_t *d_pmv, int lambda, b2_mv_t *d_mv, uint32_t *d_cost,
                         b2_mv_t *d_mv9, uint32_t *d_cost9, cudaStream_t st)
{
    switch (R) {
    case 32: return launch_k1<32>(*tm_cur, *tm_ref, mbw, mbh, nframes, d_pmv, lambda, d_mv, d_cost, d_mv9, d_cost9, st);
    case 16: return launch_k1<16>(*tm_cur, *tm_ref, mbw, mbh, nframes, d_pmv, lambda, d_mv, d_cost, d_mv9, d_cost9, st);
    default:
        fprintf(stderr, "b2enc: merange %d not supported (16 or 32)\n", R);
        return -1;
    }
}

// ---- pruned search (me_prune): K1a (min | max of the block sums per lane-task), then K1 with successive elimination -----------
// rows per lane-task the pruned search uses for +-R (K1a has to be run with the same number)
extern "C" int b2_k1_prune_rows(int R)
{
    if (R == 32) return K1_PRUNE_KS<32>;
    if (R == 16) return K1_PRUNE_KS<16>;
    return -1;
}
// words per row of the (min | max) box a strip fetches (the box is {this, 1, 1}; a strip issues one per dy group)
extern "C" int b2_k1_mm_box(int R)
{
    if (R == 32) return K1SeaSmem<32, K1_PRUNE_KS<32>>::MP;
    if (R == 16) return K1SeaSmem<16, K1_PRUNE_KS<16>>::MP;
    return -1;
}

int b2_launch_block_sums(int ks, const uint8_t *d_planes, int pitch, int rows, int nplanes, uint32_t *d_mm, cudaStream_t st)
{
    dim3 grid((pitch + K1A_TW - 1) / K1A_TW, (rows + K1A_TH - 1) / K1A_TH, nplanes);
    const size_t stride = (size_t)pitch * rows;
    switch (ks) {
    case 5: k1a_block_sums_kernel<5><<<grid, 256, 0, st>>>(d_planes, pitch, rows, stride, d_mm); break;
    case 3: k1a_block_sums_kernel<3><<<grid, 256, 0, st>>>(d_planes, pitch, rows, stride, d_mm); break;
    case 1: k1a_block_sums_kernel<1><<<grid, 256, 0, st>>>(d_planes, pitch, rows, stride, d_mm); break;      // the plain block sums (tests)
    default: fprintf(stderr, "b2enc: block sums over %d rows not built\n", ks); return -1;
    }
    B2_CUDA_OK(cudaGetLastError());
    return 0;
}

// candidate vectors of an exhaustive launch: what `swept` is compared with
extern "C" long long b2_k1_candidates(int R, int mbw, int mbh, int nframes)
{
    return (long long)(2 * R + 1) * (2 * R + 1) * mbw * mbh * nframes;
}

int b2_launch_me_fullpel_pruned(int R, const CUtensorMap *tm_cur, const CUtensorMap *tm_ref, const CUtensorMap *tm_mm, int mbw, int mbh,
                                int nframes, const b2_mv_t *d_pmv, int lambda, b2_mv_t *d_mv, uint32_t *d_cost,
                                unsigned long long *d_swept, cudaStream_t st)
{
    switch (R) {
    case 32: return launch_k1_sea<32>(*tm_cur, *tm_ref, *tm_mm, mbw, mbh, nframes, d_pmv, lambda, d_mv, d_cost, d_swept, st);
    case 16: return launch_k1_sea<16>(*tm_cur, *tm_ref, *tm_mm, mbw, mbh, nframes, d_pmv, lambda, d_mv, d_cost, d_swept, st);
    default:
        fprintf(stderr, "b2enc: merange %d not supported (16 or 32)\n", R);
        return -1;
    }
}
