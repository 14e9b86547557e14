// k7_intra_recon.cu -- K7: reconstruction of intra macroblocks on RECONSTRUCTED neighbours.
//
// Replaces x264's intra macroblock encode (behind x264_encoder_encode, av_encode.c:970); bit-exact
// against oracle/b2o_encode.c:b2o_recon_intra_mb and, through the decoder drift test, identical to
// libavcodec's H.264 decoder.
//
// Intra prediction reads reconstructed left / top / top-left / top-right neighbours, so macroblocks on
// one anti-diagonal d = mbx + 2*mby are independent and diagonals are a serial chain (inter MBs of the
// frame were already reconstructed by K5).  Prediction never reads across a slice boundary, and slices are
// whole macroblock rows (b2_slice_row, b2enc_types.h), so every slice is a chain of its own: the unit of work
// is one (frame, slice), walking d = mbx + 2*(mby - row0) over its own rows.  The chain is pure latency, so
// the kernel is built to make one link short:
//   * one THREAD-BLOCK CLUSTER per unit (up to 8 CTAs x 16 warps), hardware cluster barrier
//     (barrier.cluster release/acquire) between diagonals -> every MB of a diagonal has its own warps;
//   * luma and chroma of a macroblock are separate warp tasks (they depend on different planes);
//   * I4x4 luma: the MB's neighbourhood lives in a per-warp shared-memory tile; the sixteen blocks run as
//     a 10-step wavefront (s = bx + 2*by), two blocks per step on the two half-warps, ONE LANE PER PIXEL:
//     prediction per pixel, 4x4 DCT / IDCT as shuffle butterflies inside the 16-lane group;
//   * I16x16 luma and chroma: one lane per 4x4 block, DC Hadamards by shuffle.
// Bound: latency of the dependency chain; algorithmic bytes are those of the intra MBs only.
#include "b2_mbcode.cuh"

namespace {

using namespace b2;

constexpr int K7_WARPS_I = 16, K7_WARPS_P = 16;
constexpr int TP = 48;                      // tile pitch; pixel (x,y) of the MB sits at tile[(y+1)*TP + x + 16]

struct K7Warp {
    __align__(16) uint8_t tile[17 * TP];    // rows y=-1..15, cols x=-1..23 (top-right: 4 extra for I4x4, 8 for I8x8)
    __align__(16) uint8_t src[16 * 16];
    // I8x8 (row N1): edge tables of the current 8x8 block, its prediction and the residual / coefficient tile
    I8Edge edge;
    uint8_t raw[32];
    uint8_t p8[64];
    int d8[64];
};

__device__ __forceinline__ void cluster_barrier()
{
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ unsigned cluster_ctarank()
{
    unsigned r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ unsigned cluster_nctarank()
{
    unsigned r;
    asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
    return r;
}

// publish this task's nnz bits: a fire-and-forget reduction (RED.OR, nothing returned), so the warp does not sit out an L2 round
// trip at the end of every link of the dependency chain; cbp is derived from the finished masks by k7_cbp_kernel afterwards
__device__ __forceinline__ void publish_mask(b2_mbinfo_t *mi, uint32_t bits, bool)
{
    if (bits) atomicOr(&mi->nnz_mask, bits);
}

// ---- per-pixel intra 4x4 prediction straight from the shared-memory tile ---------------------------------
// t0 -> tile sample (x = bx, y = by-1); lf -> tile sample (x = bx-1, y = by).  Unavailable neighbours are
// never read by a legal mode except DC (handled through `avail`) and the top-right replication.
__device__ __forceinline__ int pred4x4_px(int mode, const uint8_t *t0, const uint8_t *lf, int avail, int x, int y)
{
#define TT(i) ((int)t0[((i) >= 4 && !(avail & 8)) ? 3 : (i)])      /* TT(-1) = top-left */
#define LL(i) ((i) < 0 ? (int)t0[-1] : (int)lf[(i) * TP])
#define F3(a, b, c) (((a) + 2 * (b) + (c) + 2) >> 2)
#define F2(a, b) (((a) + (b) + 1) >> 1)
    switch (mode) {
    case B2_I4_V: return TT(x);
    case B2_I4_H: return LL(y);
    case B2_I4_DC: {
        const bool hasT = avail & 2, hasL = avail & 1;
        int s = 0;
        if (hasT) s += (int)t0[0] + t0[1] + t0[2] + t0[3];
        if (hasL) s += (int)lf[0] + lf[TP] + lf[2 * TP] + lf[3 * TP];
        return (hasT && hasL) ? (s + 4) >> 3 : (hasT || hasL) ? (s + 2) >> 2 : 128;
    }
    case B2_I4_DDL: return (x == 3 && y == 3) ? (TT(6) + 3 * TT(7) + 2) >> 2 : F3(TT(x + y), TT(x + y + 1), TT(x + y + 2));
    case B2_I4_DDR:
        if (x > y) return F3(TT(x - y - 2), TT(x - y - 1), TT(x - y));
        if (x < y) return F3(LL(y - x - 2), LL(y - x - 1), LL(y - x));
        return F3(TT(0), TT(-1), LL(0));
    case B2_I4_VR: {
        const int z = 2 * x - y, k = x - (y >> 1);
        if (z >= 0 && !(z & 1)) return F2(TT(k - 1), TT(k));
        if (z >= 0) return F3(TT(k - 2), TT(k - 1), TT(k));
        if (z == -1) return F3(LL(0), TT(-1), TT(0));
        return F3(LL(y - 1), LL(y - 2), LL(y - 3));
    }
    case B2_I4_HD: {
        const int z = 2 * y - x, k = y - (x >> 1);
        if (z >= 0 && !(z & 1)) return F2(LL(k - 1), LL(k));
        if (z >= 0) return F3(LL(k - 2), LL(k - 1), LL(k));
        if (z == -1) return F3(LL(0), TT(-1), TT(0));
        return F3(TT(x - 1), TT(x - 2), TT(x - 3));
    }
    case B2_I4_VL: {
        const int k = x + (y >> 1);
        return (y & 1) ? F3(TT(k), TT(k + 1), TT(k + 2)) : F2(TT(k), TT(k + 1));
    }
    default: {                                // HU
        const int z = x + 2 * y, k = y + (x >> 1);
        if (z > 5) return LL(3);
        if (z == 5) return (LL(2) + 3 * LL(3) + 2) >> 2;
        return (z & 1) ? F3(LL(k), LL(k + 1), LL(k + 2)) : F2(LL(k), LL(k + 1));
    }
    }
#undef TT
#undef LL
#undef F3
#undef F2
}

// forward 4x4 core transform of one value per lane (lane p = y*4+x inside a 16-lane group)
__device__ __forceinline__ int dct4x4_px(int d, int x, int y)
{
    const int r = y << 2;
    const int a0 = __shfl_sync(0xffffffffu, d, r + 0, 16), a1 = __shfl_sync(0xffffffffu, d, r + 1, 16);
    const int a2 = __shfl_sync(0xffffffffu, d, r + 2, 16), a3 = __shfl_sync(0xffffffffu, d, r + 3, 16);
    const int t = x == 0 ? a0 + a1 + a2 + a3 : x == 1 ? 2 * a0 + a1 - a2 - 2 * a3 : x == 2 ? a0 - a1 - a2 + a3 : a0 - 2 * a1 + 2 * a2 - a3;
    const int b0 = __shfl_sync(0xffffffffu, t, 0 + x, 16), b1 = __shfl_sync(0xffffffffu, t, 4 + x, 16);
    const int b2v = __shfl_sync(0xffffffffu, t, 8 + x, 16), b3 = __shfl_sync(0xffffffffu, t, 12 + x, 16);
    return y == 0 ? b0 + b1 + b2v + b3 : y == 1 ? 2 * b0 + b1 - b2v - 2 * b3 : y == 2 ? b0 - b1 - b2v + b3 : b0 - 2 * b1 + 2 * b2v - b3;
}
// normative inverse: rows, columns, (x+32)>>6
__device__ __forceinline__ int idct4x4_px(int w, int x, int y)
{
    const int r = y << 2;
    const int c0 = __shfl_sync(0xffffffffu, w, r + 0, 16), c1 = __shfl_sync(0xffffffffu, w, r + 1, 16);
    const int c2 = __shfl_sync(0xffffffffu, w, r + 2, 16), c3 = __shfl_sync(0xffffffffu, w, r + 3, 16);
    int e0 = c0 + c2, e1 = c0 - c2, e2 = (c1 >> 1) - c3, e3 = c1 + (c3 >> 1);
    const int t = x == 0 ? e0 + e3 : x == 1 ? e1 + e2 : x == 2 ? e1 - e2 : e0 - e3;
    const int f0 = __shfl_sync(0xffffffffu, t, 0 + x, 16), f1 = __shfl_sync(0xffffffffu, t, 4 + x, 16);
    const int f2 = __shfl_sync(0xffffffffu, t, 8 + x, 16), f3 = __shfl_sync(0xffffffffu, t, 12 + x, 16);
    e0 = f0 + f2; e1 = f0 - f2; e2 = (f1 >> 1) - f3; e3 = f1 + (f3 >> 1);
    const int v = y == 0 ? e0 + e3 : y == 1 ? e1 + e2 : y == 2 ? e1 - e2 : e0 - e3;
    return (v + 32) >> 6;
}

// blocks of wavefront step s = bx + 2*by for the two half-warps (-1: none)
__device__ __constant__ int8_t c_i4_wave[10][2] = {{0, -1}, {1, -1}, {4, 2}, {5, 3}, {6, 8}, {7, 9}, {12, 10}, {13, 11}, {14, -1}, {15, -1}};
__device__ __constant__ uint8_t c_izz[16] = {0, 1, 5, 6, 2, 4, 7, 12, 3, 8, 11, 13, 9, 10, 14, 15};   // raster -> scan position

// z-order index of the block at (x,y) in units of 4 px
__device__ __forceinline__ int zidx(int x, int y) { return (x & 1) | ((y & 1) << 1) | ((x >> 1) << 2) | ((y >> 1) << 3); }

// ---- luma task ------------------------------------------------------------------------------------------
__device__ void k7_luma_task(int lane, K7Warp &ws, const FramePlanes &fp, int frame, int mbx, int mby, int mbw, int row0, int qp,
                             b2_mbinfo_t *mi, b2_mbcoef_t *cf)
{
    const int mba = mb_avail(mbx, mby, mbw, row0);
    const bool hasT = mba & 2, hasL = mba & 1;
    const int mb_type = mi->mb_type;
    const size_t offy = (size_t)(B2_PAD + mby * 16) * fp.pitch + B2_PAD + mbx * 16;
    const uint8_t *sy = fp.cur[0] + frame * fp.stride_y + offy;
    uint8_t *ry = fp.rec[0] + frame * fp.stride_y + offy;
    const QParams q = make_qparams(qp, true);
    uint32_t bits = 0;

    if (mb_type == B2_MB_I16x16) {
        const int mode = mi->i16_mode;
        const int l16 = lane & 15;
        const int topv = hasT ? ry[-(ptrdiff_t)fp.pitch + l16] : 0;
        const int leftv = hasL ? ry[(size_t)l16 * fp.pitch - 1] : 0;
        const int tlv = (mba & 4) ? ry[-(ptrdiff_t)fp.pitch - 1] : 0;
        const int bx = blk_x(l16) * 4, by = blk_y(l16) * 4;
        int t4[4], l4[4];
#pragma unroll
        for (int i = 0; i < 4; i++) { t4[i] = __shfl_sync(0xffffffffu, topv, bx + i); l4[i] = __shfl_sync(0xffffffffu, leftv, by + i); }
        int sumT = lane < 16 ? topv : 0, sumL = lane < 16 ? leftv : 0;
        int hterm = 0, vterm = 0;
        {
            const int i = l16 & 7;
            const int ta = __shfl_sync(0xffffffffu, topv, 8 + i), tb = __shfl_sync(0xffffffffu, topv, (6 - i) & 15);
            const int la = __shfl_sync(0xffffffffu, leftv, 8 + i), lb = __shfl_sync(0xffffffffu, leftv, (6 - i) & 15);
            if (lane < 8) { hterm = (i + 1) * (ta - (i == 7 ? tlv : tb)); vterm = (i + 1) * (la - (i == 7 ? tlv : lb)); }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            sumT += __shfl_xor_sync(0xffffffffu, sumT, o); sumL += __shfl_xor_sync(0xffffffffu, sumL, o);
            hterm += __shfl_xor_sync(0xffffffffu, hterm, o); vterm += __shfl_xor_sync(0xffffffffu, vterm, o);
        }
        const int t15 = __shfl_sync(0xffffffffu, topv, 15), l15 = __shfl_sync(0xffffffffu, leftv, 15);
        const int pa = 16 * (l15 + t15), pb = (5 * hterm + 32) >> 6, pc = (5 * vterm + 32) >> 6;
        const int dc = (hasT && hasL) ? (sumT + sumL + 16) >> 5 : (hasT || hasL) ? (sumT + sumL + 8) >> 4 : 128;
        int src[16], pred[16], w[16], z[16];
#pragma unroll
        for (int i = 0; i < 16; i++) src[i] = pred[i] = 0;
        if (lane < 16) {
            load_src4x4(sy + (size_t)by * fp.pitch + bx, fp.pitch, src);
#pragma unroll
            for (int y = 0; y < 4; y++)
#pragma unroll
                for (int x = 0; x < 4; x++)
                    pred[y * 4 + x] = mode == B2_I16_V ? t4[x] : mode == B2_I16_H ? l4[y] : mode == B2_I16_DC ? dc
                                      : b2_clip255((pa + pb * (bx + x - 7) + pc * (by + y - 7) + 16) >> 5);
        }
#pragma unroll
        for (int i = 0; i < 16; i++) w[i] = src[i] - pred[i];
        dct4x4(w);
        // 4x4 Hadamard of the 16 DCs: lane r (< 16) produces output raster position r = v*4+u
        const int v = (l16 >> 2), u = l16 & 3;
        int acc = 0;
#pragma unroll
        for (int s = 0; s < 16; s++) {
            const int dcs = __shfl_sync(0xffffffffu, w[0], zidx(s & 3, s >> 2));
            acc += h4_sign(v, s >> 2) * h4_sign(u, s & 3) * dcs;
        }
        const int zdc = quant_dc((acc + 1) >> 1, q);
        int acc2 = 0;
#pragma unroll
        for (int s = 0; s < 16; s++) {
            const int zs = __shfl_sync(0xffffffffu, zdc, s);
            acc2 += h4_sign(v, s >> 2) * h4_sign(u, s & 3) * zs;
        }
        const int dq_r = q.s >= 6 ? (acc2 * q.ls[0]) * (1 << (q.s - 6)) : (acc2 * q.ls[0] + (1 << (5 - q.s))) >> (6 - q.s);
        const int my_dc = __shfl_sync(0xffffffffu, dq_r, blk_y(l16) * 4 + blk_x(l16));
        const bool luma_dc = __ballot_sync(0xffffffffu, lane < 16 && zdc != 0) != 0;
        int nnz = 0;
        if (lane < 16) {
            cf->blk[24][c_izz[l16]] = (int16_t)zdc;
            nnz = quant4x4(w, z, q, true);
            store_levels_zigzag(cf->blk[l16], z);
            dequant4x4(z, w, q, true);
            w[0] = my_dc;
            idct4x4(w);
            store_rec4x4(ry + (size_t)by * fp.pitch + bx, fp.pitch, pred, w);
        }
        bits = __ballot_sync(0xffffffffu, lane < 16 && nnz != 0) & 0xffffu;
        if (luma_dc) bits |= 1u << 24;
    } else if (mb_type == B2_MB_I8x8) {
        // ---- I8x8 (row N1): the four 8x8 blocks are a serial chain (each predicts from the previous ones); per block the
        // warp filters the edge (8.3.2.2.1), predicts two samples per lane, and runs the 8x8 transform with one lane per
        // column / row through the shared-memory tile d8 ----
        if (lane < 25) {                                      // top row x = -1..23
            const int x = lane - 1;
            const bool ok = x < 0 ? (mba & 4) != 0 : x < 16 ? hasT : (mba & 8) != 0;
            ws.tile[x + 16] = ok ? ry[-(ptrdiff_t)fp.pitch + x] : 0;
        }
        if (lane < 16) {
            ws.tile[(lane + 1) * TP + 15] = hasL ? ry[(size_t)lane * fp.pitch - 1] : 0;
            *(uint4 *)&ws.src[lane * 16] = *(const uint4 *)(sy + (size_t)lane * fp.pitch);
        }
        const int modes = mi->i8_modes;
        const int qbits8 = 16 + qp / 6, f8 = ((1 << qbits8) * 21) >> 6, sh = qp / 6, rem = qp % 6;
        __syncwarp();
        uint32_t mask = 0;
#pragma unroll 1
        for (int q8 = 0; q8 < 4; q8++) {
            const int qx = (q8 & 1) * 8, qy = (q8 >> 1) * 8, qa = blk8_avail(q8, mba), mode = (modes >> (4 * q8)) & 15;
            const uint8_t *t0 = &ws.tile[qy * TP + qx + 16];              // sample (x = qx, y = qy-1)
            if (lane < 25) {                                               // raw edge, substituted where unavailable
                int v = 128;
                if (lane < 8) { if (qa & 1) v = t0[(8 - lane) * TP - 1]; }                       // p[-1, 7-lane]
                else if (lane == 8) { if (qa & 4) v = t0[-1]; }
                else if (qa & 2) v = t0[(lane - 9 < 8 || (qa & 8)) ? lane - 9 : 7];
                ws.raw[lane] = (uint8_t)v;
            }
            __syncwarp();
            if (lane < 25) ws.edge.E[lane] = (uint8_t)i8_filter_edge(ws.raw, lane, qa);
            __syncwarp();
            if (lane < 24) {
                const uint8_t *E = ws.edge.E;
                ws.edge.F2[lane] = (uint8_t)((E[lane] + E[lane + 1] + 1) >> 1);
                ws.edge.F3[lane] = lane < 23 ? (uint8_t)((E[lane] + 2 * E[lane + 1] + E[lane + 2] + 2) >> 2) : (uint8_t)((E[23] + 3 * E[24] + 2) >> 2);
            } else if (lane == 24) {
                const uint8_t *E = ws.edge.E;
                int st = 0, sl = 0;
#pragma unroll
                for (int i = 0; i < 8; i++) { st += E[9 + i]; sl += E[i]; }
                const bool hT = qa & 2, hL = qa & 1;
                ws.edge.dc = (uint8_t)((hT && hL) ? (st + sl + 8) >> 4 : hT ? (st + 4) >> 3 : hL ? (sl + 4) >> 3 : 128);
                ws.edge.hu13 = (uint8_t)((E[1] + 3 * E[0] + 2) >> 2);
            }
            __syncwarp();
#pragma unroll
            for (int j = 0; j < 2; j++) {
                const int p = lane + 32 * j, X = p & 7, Y = p >> 3;
                const int pr = pred8x8_px(mode, ws.edge, X, Y);
                ws.p8[p] = (uint8_t)pr;
                ws.d8[p] = (int)ws.src[(qy + Y) * 16 + qx + X] - pr;
            }
            __syncwarp();
            if (lane < 8) {                                                // forward: columns, then rows + quantiser
                int a[8], o[8];
#pragma unroll
                for (int y = 0; y < 8; y++) a[y] = ws.d8[y * 8 + lane];
                fdct8_1d(a, o);
#pragma unroll
                for (int y = 0; y < 8; y++) ws.d8[y * 8 + lane] = o[y];
            }
            __syncwarp();
            int z[8];
            if (lane < 8) {
                int a[8], o[8];
#pragma unroll
                for (int x = 0; x < 8; x++) a[x] = ws.d8[lane * 8 + x];
                fdct8_1d(a, o);
#pragma unroll
                for (int x = 0; x < 8; x++) {
                    const uint32_t mf = c_quant8_mf[rem][c_cls8[(lane & 3) * 4 + (x & 3)]];
                    const int v = (int)(((uint32_t)abs(o[x]) * mf + (uint32_t)f8) >> qbits8);
                    z[x] = o[x] < 0 ? -v : v;
                }
            }
            __syncwarp();
            if (lane < 8) {
#pragma unroll
                for (int x = 0; x < 8; x++) ws.d8[lane * 8 + x] = z[x];
            }
            __syncwarp();
            uint32_t mask4 = 0;
#pragma unroll
            for (int j = 0; j < 2; j++) {                                  // levels in 8x8 zig-zag order -> blk[4q..4q+3]
                const int sp = lane + 32 * j;
                const int v = ws.d8[c_zigzag8[sp]];
                ((int16_t *)cf->blk[4 * q8])[sp] = (int16_t)v;
                const uint32_t nzb = __ballot_sync(0xffffffffu, v != 0);
#pragma unroll
                for (int k = 0; k < 4; k++)
                    if (nzb & (0x11111111u << k)) mask4 |= 1u << k;       // interleaved quarter k = scan positions == k mod 4
            }
            __syncwarp();
            if (mask4) {                                                   // normative scaling + inverse: rows, then columns
                if (lane < 8) {
                    int a[8], o[8];
#pragma unroll
                    for (int x = 0; x < 8; x++) {
                        const int ls = 16 * c_dequant8_v[rem][c_cls8[(lane & 3) * 4 + (x & 3)]];
                        a[x] = sh >= 6 ? (z[x] * ls) * (1 << (sh - 6)) : (z[x] * ls + (1 << (5 - sh))) >> (6 - sh);
                    }
                    idct8_1d(a, o);
#pragma unroll
                    for (int x = 0; x < 8; x++) ws.d8[lane * 8 + x] = o[x];
                }
                __syncwarp();
                if (lane < 8) {
                    int a[8], o[8];
#pragma unroll
                    for (int y = 0; y < 8; y++) a[y] = ws.d8[y * 8 + lane];
                    idct8_1d(a, o);
#pragma unroll
                    for (int y = 0; y < 8; y++) ws.d8[y * 8 + lane] = (o[y] + 32) >> 6;
                }
                __syncwarp();
            }
#pragma unroll
            for (int j = 0; j < 2; j++) {
                const int p = lane + 32 * j, X = p & 7, Y = p >> 3;
                const int v = (int)ws.p8[p] + (mask4 ? ws.d8[p] : 0);
                ws.tile[(qy + Y + 1) * TP + qx + X + 16] = (uint8_t)b2_clip255(v);
            }
            __syncwarp();
            mask |= mask4 << (4 * q8);
        }
        bits = mask & 0xffffu;
        if (lane < 16) {
            *(uint4 *)(ry + (size_t)lane * fp.pitch) = *(const uint4 *)&ws.tile[(lane + 1) * TP + 16];
            mi->i4_mode[lane] = (uint8_t)((modes >> (4 * (lane >> 2))) & 15);
        }
        if (lane == 0) mi->transform8x8 = 1;
        if (lane == 24) {
            uint4 z4 = make_uint4(0, 0, 0, 0);
            ((uint4 *)cf->blk[24])[0] = z4; ((uint4 *)cf->blk[24])[1] = z4;
        }
    } else {
        // ---- I4x4: shared-memory tile, 10-step wavefront, two blocks per step, one lane per pixel ----
        if (lane < 21) {                                      // top row x = -1..19
            const int x = lane - 1;
            const bool ok = x < 0 ? (mba & 4) != 0 : x < 16 ? hasT : (mba & 8) != 0;
            ws.tile[x + 16] = ok ? ry[-(ptrdiff_t)fp.pitch + x] : 0;
        }
        if (lane < 16) {
            ws.tile[(lane + 1) * TP + 15] = hasL ? ry[(size_t)lane * fp.pitch - 1] : 0;
            *(uint4 *)&ws.src[lane * 16] = *(const uint4 *)(sy + (size_t)lane * fp.pitch);
        }
        // lane b (< 16) holds mode | avail << 8 of block b; each step fetches its block's word by shuffle
        const int blkinfo = lane < 16 ? ((int)mi->i4_mode[lane] | (blk_avail(lane, mba) << 8)) : 0;
        __syncwarp();
        const int half = lane >> 4, p = lane & 15, x = p & 3, y = p >> 2;
        const int cls = pos_class(p);
        const uint32_t mf = (uint32_t)q.mf[cls];
        const int lsm = q.lsm[cls];
        const int izz = c_izz[p];
        uint32_t mymask = 0;
#pragma unroll 1
        for (int s = 0; s < 10; s++) {
            const int blk = c_i4_wave[s][half];
            const bool act = blk >= 0;
            const int b = act ? blk : 0;
            const int bx = blk_x(b) * 4, by = blk_y(b) * 4;
            const int bi = __shfl_sync(0xffffffffu, blkinfo, b);
            const uint8_t *t0 = &ws.tile[by * TP + bx + 16];              // (x = bx, y = by-1)
            const int pred = pred4x4_px(bi & 255, t0, t0 + TP - 1, bi >> 8, x, y);
            const int d = (int)ws.src[(by + y) * 16 + bx + x] - pred;
            const int w = dct4x4_px(d, x, y);
            const int zq = (int)(((uint32_t)abs(w) * mf + (uint32_t)q.f) >> q.qbits);
            const int z = w < 0 ? -zq : zq;
            const uint32_t nz = __ballot_sync(0xffffffffu, act && z != 0);
            const int wq = (z * lsm + q.rnd) >> q.sh;
            const int res = idct4x4_px(wq, x, y);
            if (act) {
                cf->blk[b][izz] = (int16_t)z;
                ws.tile[(by + y + 1) * TP + bx + x + 16] = (uint8_t)b2_clip255(pred + res);
                if ((nz >> (half * 16)) & 0xffffu) mymask |= 1u << b;
            }
            __syncwarp();
        }
        bits = (__shfl_sync(0xffffffffu, mymask, 0) | __shfl_sync(0xffffffffu, mymask, 16)) & 0xffffu;
        if (lane < 16) *(uint4 *)(ry + (size_t)lane * fp.pitch) = *(const uint4 *)&ws.tile[(lane + 1) * TP + 16];
        if (lane == 24) {
            uint4 z4 = make_uint4(0, 0, 0, 0);
            ((uint4 *)cf->blk[24])[0] = z4; ((uint4 *)cf->blk[24])[1] = z4;
        }
    }
    if (lane == 0) publish_mask(mi, bits, true);
}

// ---- chroma task: lanes 0..7 own (plane, 4x4 block) ---------------------------------------------------------
__device__ void k7_chroma_task(int lane, const FramePlanes &fp, int frame, int mbx, int mby, int mbw, int row0, int qp,
                               b2_mbinfo_t *mi, b2_mbcoef_t *cf)
{
    const int mba = mb_avail(mbx, mby, mbw, row0);
    const bool hasT = mba & 2, hasL = mba & 1;
    const bool act = lane < 8;
    const int pl = (lane >> 2) & 1, k = lane & 3, cbx = (k & 1) * 4, cby = (k >> 1) * 4;
    const int qpc = chroma_qp(qp);
    const QParams q = make_qparams(qpc, true);
    const size_t offc = (size_t)(B2_PADC + mby * 8) * fp.pitchc + B2_PADC + mbx * 8;
    uint8_t *rc = fp.rec[1 + pl] + frame * fp.stride_c + offc;
    int src[16], pred[16];
#pragma unroll
    for (int i = 0; i < 16; i++) src[i] = pred[i] = 0;
    if (act) {
        const int mode = mi->chroma_mode;
        load_src4x4(fp.cur[1 + pl] + frame * fp.stride_c + offc + (size_t)cby * fp.pitchc + cbx, fp.pitchc, src);
        int top[8], left[8], tl = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) { top[i] = hasT ? rc[-(ptrdiff_t)fp.pitchc + i] : 0; left[i] = hasL ? rc[(size_t)i * fp.pitchc - 1] : 0; }
        if (mba & 4) tl = rc[-(ptrdiff_t)fp.pitchc - 1];
        if (mode == B2_IC_DC) {
            const int t0 = top[0] + top[1] + top[2] + top[3], t1 = top[4] + top[5] + top[6] + top[7];
            const int l0 = left[0] + left[1] + left[2] + left[3], l1 = left[4] + left[5] + left[6] + left[7];
            int dcv;
            if (k == 0) dcv = (hasT && hasL) ? (t0 + l0 + 4) >> 3 : hasT ? (t0 + 2) >> 2 : hasL ? (l0 + 2) >> 2 : 128;
            else if (k == 1) dcv = hasT ? (t1 + 2) >> 2 : hasL ? (l0 + 2) >> 2 : 128;
            else if (k == 2) dcv = hasL ? (l1 + 2) >> 2 : hasT ? (t0 + 2) >> 2 : 128;
            else dcv = (hasT && hasL) ? (t1 + l1 + 4) >> 3 : hasT ? (t1 + 2) >> 2 : hasL ? (l1 + 2) >> 2 : 128;
#pragma unroll
            for (int i = 0; i < 16; i++) pred[i] = dcv;
        } else if (mode == B2_IC_H) {
#pragma unroll
            for (int i = 0; i < 16; i++) pred[i] = left[cby + (i >> 2)];
        } else if (mode == B2_IC_V) {
#pragma unroll
            for (int i = 0; i < 16; i++) pred[i] = top[cbx + (i & 3)];
        } else {
            int Hc = 0, Vc = 0;
#pragma unroll
            for (int i = 0; i < 4; i++) {
                Hc += (i + 1) * (top[4 + i] - (i == 3 ? tl : top[2 - i]));
                Vc += (i + 1) * (left[4 + i] - (i == 3 ? tl : left[2 - i]));
            }
            const int pa = 16 * (left[7] + top[7]), pb = (34 * Hc + 32) >> 6, pc = (34 * Vc + 32) >> 6;
#pragma unroll
            for (int i = 0; i < 16; i++)
                pred[i] = b2_clip255((pa + pb * (cbx + (i & 3) - 3) + pc * (cby + (i >> 2) - 3) + 16) >> 5);
        }
    }
    const int cfl = code_chroma4x4(lane, act, src, pred, q, qpc, cf, rc + (size_t)cby * fp.pitchc + cbx, fp.pitchc);
    const uint32_t ac = __ballot_sync(0xffffffffu, act && (cfl & 1)) & 0xffu;
    const uint32_t dc = __ballot_sync(0xffffffffu, act && (cfl & 2)) & 0xffu;
    uint32_t bits = ac << 16;
    if (dc & 0x0fu) bits |= 1u << 25;
    if (dc & 0xf0u) bits |= 1u << 26;
    if (lane == 25) ((uint4 *)cf->blk[25])[1] = make_uint4(0, 0, 0, 0);
    if (lane == 0) publish_mask(mi, bits, false);
}

// WARPS = warps per CTA.  Measured: shrinking the P-frame CTA to 4 warps (so that it fits beside two K1 CTAs in the register
// file) LOSES 16 % of the stage throughput -- P frames after a scene change hold thousands of intra MBs and the chain of a
// stream group then waits on K7 -- so both variants use 16
template <int WARPS>
__global__ void __launch_bounds__(WARPS * 32)
k7_intra_wavefront_kernel(FramePlanes fp, int mbw, int mbh, int nslices, int qp, b2_mbinfo_t *__restrict__ info,
                          b2_mbcoef_t *__restrict__ coef)
{
    constexpr int K7_WARPS = WARPS;
    extern __shared__ int s_diag_cnt[];                 // [ndiag] diagonal holds intra MBs | [ndiag] list of those diagonals
    __shared__ K7Warp s_warp[K7_WARPS];
    const int frame = blockIdx.y / nslices, slice = blockIdx.y - frame * nslices;   // the unit: rows [row0, row0 + srows)
    const int row0 = b2_slice_row(slice, nslices, mbh), srows = b2_slice_row(slice + 1, nslices, mbh) - row0;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int ncta = (int)cluster_nctarank(), crank = (int)cluster_ctarank();
    const int gwarp = crank * K7_WARPS + warp, nwarps = ncta * K7_WARPS;
    const int ndiag = mbw + 2 * (srows - 1);
    b2_mbinfo_t *finfo = info + (size_t)frame * mbw * mbh;
    b2_mbcoef_t *fcoef = coef + (size_t)frame * mbw * mbh;
    // Anti-diagonals that hold intra macroblocks, as an ascending list (identical in every CTA of the cluster).  P frames hold
    // few: testing every diagonal in the main loop was 255 dependent shared-memory reads, most of a sparse frame's K7 time.
    int *s_diag_list = s_diag_cnt + ndiag;
    __shared__ int s_nlist;
    for (int i = threadIdx.x; i < ndiag; i += blockDim.x) s_diag_cnt[i] = 0;
    __syncthreads();
    const int mb0 = row0 * mbw, nmb = srows * mbw;                           // the unit's macroblocks, from mb0
    for (int i0 = threadIdx.x; i0 < nmb; i0 += 4 * blockDim.x) {            // four independent loads in flight per thread
        uint8_t ty[4];
#pragma unroll
        for (int j = 0; j < 4; j++) { const int i = i0 + j * blockDim.x; ty[j] = i < nmb ? finfo[mb0 + i].mb_type : (uint8_t)B2_MB_P16x16; }
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int i = i0 + j * blockDim.x;
            if (ty[j] != B2_MB_P16x16) s_diag_cnt[(i % mbw) + 2 * (i / mbw)] = 1;                 // same value from every writer
        }
    }
    __syncthreads();
    if (warp == 0) {
        int n = 0;
        for (int d0 = 0; d0 < ndiag; d0 += 32) {
            const int d = d0 + lane;
            const bool used = d < ndiag && s_diag_cnt[d] != 0;
            const unsigned m = __ballot_sync(0xffffffffu, used);
            if (used) s_diag_list[n + __popc(m & ((1u << lane) - 1u))] = d;
            n += __popc(m);
        }
        if (lane == 0) s_nlist = n;
    }
    __syncthreads();
    const int nlist = s_nlist;
    for (int k = 0; k < nlist; k++) {
        const int d = s_diag_list[k];
        const int y_lo = max(0, (d - mbw + 2) >> 1), y_hi = min(srows - 1, d >> 1);     // rows relative to row0
        const int ntask = 2 * (y_hi - y_lo + 1);        // (MB, luma|chroma)
        for (int t = gwarp; t < ntask; t += nwarps) {
            const int y = y_lo + (t >> 1), mbx = d - 2 * y, mby = row0 + y;
            const int i = mby * mbw + mbx;
            if (finfo[i].mb_type != B2_MB_P16x16) {
                if (t & 1) k7_chroma_task(lane, fp, frame, mbx, mby, mbw, row0, qp, &finfo[i], &fcoef[i]);
                else k7_luma_task(lane, s_warp[warp], fp, frame, mbx, mby, mbw, row0, qp, &finfo[i], &fcoef[i]);
            }
        }
        if (ncta > 1) cluster_barrier();
        else __syncthreads();
    }
}

// coded_block_pattern of the intra macroblocks from their finished masks (luma and chroma tasks OR their bits in independently)
__global__ void __launch_bounds__(256)
k7_cbp_kernel(b2_mbinfo_t *__restrict__ info, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int t = info[i].mb_type;
    if (t != B2_MB_P16x16) info[i].cbp = (uint8_t)cbp_from_mask(t, info[i].nnz_mask);
}

}  // namespace

void b2_intra_recon_shape(int mbw, int mbh, int slices, int all_intra, int *ncta, int *rounds, int *dyn_smem)
{
    const int ns = b2_slice_count(slices, mbh);
    int rows = 0;                                                        // the tallest slice sizes every unit
    for (int k = 0; k < ns; k++) rows = max(rows, b2_slice_row(k + 1, ns, mbh) - b2_slice_row(k, ns, mbh));
    const int ndiag = mbw + 2 * (rows - 1);
    const int maxdiag = rows < (mbw + 1) / 2 ? rows : (mbw + 1) / 2;    // macroblocks on the longest anti-diagonal
    // I frames: every MB of a diagonal gets its own luma + chroma warp (cluster of up to 8 CTAs per slice).  P frames hold few,
    // scattered intra MBs: one CTA per (frame, slice) keeps the footprint small so that other streams' kernels keep the rest.
    const int warps = all_intra ? K7_WARPS_I : K7_WARPS_P;
    int n = 1;
    if (all_intra)
        while (n < 8 && n * warps < 2 * maxdiag) n *= 2;
    *ncta = n;
    *rounds = (2 * maxdiag + n * warps - 1) / (n * warps);           // (MB, luma | chroma) tasks of the longest diagonal per warp
    *dyn_smem = 2 * ndiag * (int)sizeof(int);                        // per diagonal: holds intra MBs | list entry
}

int b2_launch_intra_recon(const uint8_t *const cur[3], uint8_t *const rec[3], int pitch, int pitchc, size_t stride_y,
                          size_t stride_c, int mbw, int mbh, int slices, int nframes, int qp, int all_intra, b2_mbinfo_t *d_info,
                          b2_mbcoef_t *d_coef, cudaStream_t st)
{
    const int ns = b2_slice_count(slices, mbh);
    FramePlanes fp;
    for (int i = 0; i < 3; i++) { fp.cur[i] = cur[i]; fp.ref[i] = nullptr; fp.rec[i] = rec[i]; }
    fp.pitch = pitch; fp.pitchc = pitchc; fp.stride_y = stride_y; fp.stride_c = stride_c;
    int ncta, rounds, dyn_smem;
    b2_intra_recon_shape(mbw, mbh, ns, all_intra, &ncta, &rounds, &dyn_smem);
    // The diagonal tables grow with mbw + 2*mbh (of the tallest slice) and sit beside the per-warp tiles; the kernel does not opt in to more than the
    // default dynamic shared memory (48 KB in all with the static part: ndiag <= 3134).  Every size within H.264 level 6.2
    // stays below that (ndiag <= 2240, at 2112x16880); a taller picture is refused here rather than failing at launch.
    // (a property of the kernel binary, the same for both instantiations' 16 warps: read once per process)
    static_assert(K7_WARPS_I == K7_WARPS_P, "one shared-memory limit for both schedules");
    static const int max_dyn = [] {
        cudaFuncAttributes fa;
        return cudaFuncGetAttributes(&fa, k7_intra_wavefront_kernel<K7_WARPS_I>) == cudaSuccess ? fa.maxDynamicSharedSizeBytes : -1;
    }();
    if (dyn_smem > max_dyn) {
        fprintf(stderr, "b2enc: K7 needs %d bytes of dynamic shared memory for %d x %d macroblocks in %d slices (%d diagonals), at most %d\n",
                dyn_smem, mbw, mbh, ns, dyn_smem / (2 * (int)sizeof(int)), max_dyn);
        return -1;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(ncta, nframes * ns, 1);
    cfg.blockDim = dim3((all_intra ? K7_WARPS_I : K7_WARPS_P) * 32, 1, 1);
    cfg.dynamicSmemBytes = dyn_smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = ncta; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    if (all_intra) B2_CUDA_OK(cudaLaunchKernelEx(&cfg, k7_intra_wavefront_kernel<K7_WARPS_I>, fp, mbw, mbh, ns, qp, d_info, d_coef));
    else B2_CUDA_OK(cudaLaunchKernelEx(&cfg, k7_intra_wavefront_kernel<K7_WARPS_P>, fp, mbw, mbh, ns, qp, d_info, d_coef));
    const int n = mbw * mbh * nframes;
    k7_cbp_kernel<<<(n + 255) / 256, 256, 0, st>>>(d_info, n);
    B2_CUDA_OK(cudaGetLastError());
    return 0;
}
