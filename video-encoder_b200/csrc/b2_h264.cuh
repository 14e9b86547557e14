// b2_h264.cuh -- per-thread device building blocks of the H.264 arithmetic used by K2/K3/K5/K7.
// One thread owns one 4x4 block in registers; warps cooperate through shuffles.
// Normative pieces follow ITU-T H.264 (8.3 intra prediction, 8.4.2.2 interpolation, 8.5 transform
// and scaling); encoder-side pieces (forward DCT, dead-zone quantiser, SATD) follow the frozen
// definitions in oracle/ (SURVEY.md Appendix A).  In the reference all of it is inside
// x264_encoder_encode (av_encode.c:970).
#pragma once
#include "b2_common.cuh"

namespace b2 {

__device__ __constant__ uint16_t c_quant_mf[6][3] = {{13107, 8066, 5243}, {11916, 7490, 4660}, {10082, 6554, 4194},
                                                     {9362, 5825, 3647},  {8192, 5243, 3355},  {7282, 4559, 2893}};
__device__ __constant__ uint8_t c_dequant_v[6][3] = {{10, 13, 16}, {11, 14, 18}, {13, 16, 20},
                                                     {14, 18, 23}, {16, 20, 25}, {18, 23, 29}};
__device__ __constant__ uint8_t c_zigzag[16] = {0, 1, 4, 8, 5, 2, 3, 6, 9, 12, 13, 10, 7, 11, 14, 15};
__device__ __constant__ uint8_t c_chroma_qp[22] = {29, 30, 31, 32, 32, 33, 34, 34, 35, 35, 36,
                                                   36, 37, 37, 37, 38, 38, 38, 39, 39, 39, 39};

// 4x4 block index (z order) <-> position in units of 4 pixels
__device__ __forceinline__ int blk_x(int b) { return (b & 1) | ((b >> 1) & 2); }
__device__ __forceinline__ int blk_y(int b) { return ((b >> 1) & 1) | ((b >> 2) & 2); }
__device__ __forceinline__ int chroma_qp(int qp) { return qp < 30 ? qp : c_chroma_qp[qp - 30]; }

struct QParams {
    int qbits, f, mf[3];        // quantiser
    int ls[3], s;               // dequantiser: LevelScale = 16*V, s = qp/6
    int lsm[3], rnd, sh;        // 4x4 scaling as one multiply-add-shift: w = (z * lsm + rnd) >> sh  (8.5.12.1 for both branches of qP/6 >= 4)
};
__device__ __forceinline__ QParams make_qparams(int qp, bool intra)
{
    QParams q;
    q.qbits = 15 + qp / 6;
    q.f = ((1 << q.qbits) * (intra ? 21 : 11)) >> 6;
    q.s = qp / 6;
#pragma unroll
    for (int i = 0; i < 3; i++) { q.mf[i] = c_quant_mf[qp % 6][i]; q.ls[i] = 16 * c_dequant_v[qp % 6][i]; }
    q.sh = q.s >= 4 ? 0 : 4 - q.s;
    q.rnd = q.s >= 4 ? 0 : 1 << (3 - q.s);
#pragma unroll
    for (int i = 0; i < 3; i++) q.lsm[i] = q.s >= 4 ? q.ls[i] << (q.s - 4) : q.ls[i];
    return q;
}
// position class of raster index i: 0 = (even,even), 2 = (odd,odd), 1 otherwise
__device__ __forceinline__ constexpr int pos_class(int i)
{
    return (((i & 1) && ((i >> 2) & 1)) ? 2 : (((i | (i >> 2)) & 1) ? 1 : 0));
}

// ---- transforms on a register-resident 4x4 (raster order) ------------------------------------------
__device__ __forceinline__ void dct4x4(int d[16])
{
#pragma unroll
    for (int y = 0; y < 4; y++) {
        int s03 = d[y * 4 + 0] + d[y * 4 + 3], d03 = d[y * 4 + 0] - d[y * 4 + 3];
        int s12 = d[y * 4 + 1] + d[y * 4 + 2], d12 = d[y * 4 + 1] - d[y * 4 + 2];
        d[y * 4 + 0] = s03 + s12; d[y * 4 + 1] = 2 * d03 + d12; d[y * 4 + 2] = s03 - s12; d[y * 4 + 3] = d03 - 2 * d12;
    }
#pragma unroll
    for (int x = 0; x < 4; x++) {
        int s03 = d[x] + d[12 + x], d03 = d[x] - d[12 + x];
        int s12 = d[4 + x] + d[8 + x], d12 = d[4 + x] - d[8 + x];
        d[x] = s03 + s12; d[4 + x] = 2 * d03 + d12; d[8 + x] = s03 - s12; d[12 + x] = d03 - 2 * d12;
    }
}

// normative inverse (8.5.12.2): rows, then columns, then (x+32)>>6.  In place: w -> residual.
__device__ __forceinline__ void idct4x4(int w[16])
{
#pragma unroll
    for (int y = 0; y < 4; y++) {
        int e0 = w[y * 4 + 0] + w[y * 4 + 2], e1 = w[y * 4 + 0] - w[y * 4 + 2];
        int e2 = (w[y * 4 + 1] >> 1) - w[y * 4 + 3], e3 = w[y * 4 + 1] + (w[y * 4 + 3] >> 1);
        w[y * 4 + 0] = e0 + e3; w[y * 4 + 1] = e1 + e2; w[y * 4 + 2] = e1 - e2; w[y * 4 + 3] = e0 - e3;
    }
#pragma unroll
    for (int x = 0; x < 4; x++) {
        int e0 = w[x] + w[8 + x], e1 = w[x] - w[8 + x];
        int e2 = (w[4 + x] >> 1) - w[12 + x], e3 = w[4 + x] + (w[12 + x] >> 1);
        w[x] = (e0 + e3 + 32) >> 6; w[4 + x] = (e1 + e2 + 32) >> 6;
        w[8 + x] = (e1 - e2 + 32) >> 6; w[12 + x] = (e0 - e3 + 32) >> 6;
    }
}

// dead-zone quantiser; z raster; returns number of non-zero levels
__device__ __forceinline__ int quant4x4(const int w[16], int z[16], const QParams &q, bool skip_dc)
{
    int nnz = 0;
#pragma unroll
    for (int i = 0; i < 16; i++) {
        if (i == 0 && skip_dc) { z[0] = 0; continue; }
        int a = abs(w[i]);
        // |w| <= 9180 and mf <= 13107: the product plus the dead-zone offset stays below 2^31
        int v = (int)(((uint32_t)a * (uint32_t)q.mf[pos_class(i)] + (uint32_t)q.f) >> q.qbits);
        z[i] = w[i] < 0 ? -v : v;
        nnz += v != 0;
    }
    return nnz;
}
__device__ __forceinline__ int quant_dc(int x, const QParams &q)
{
    int a = abs(x);
    // |x| <= 16*4080/2 (luma DC Hadamard) -> a*mf <= 4.3e8 < 2^31
    int v = (int)(((uint32_t)a * (uint32_t)q.mf[0] + 2u * (uint32_t)q.f) >> (q.qbits + 1));
    return x < 0 ? -v : v;
}
// normative scaling (8.5.12.1), flat matrices; w[0] untouched when skip_dc
__device__ __forceinline__ void dequant4x4(const int z[16], int w[16], const QParams &q, bool skip_dc)
{
#pragma unroll
    for (int i = 0; i < 16; i++) {
        if (i == 0 && skip_dc) continue;
        w[i] = (z[i] * q.lsm[pos_class(i)] + q.rnd) >> q.sh;
    }
}

// ---- SATD in the transform domain for the "flat" intra predictors ------------------------------------------------------------
// H (src - pred) H^T = H src H^T - H pred H^T, and a predictor that is constant along columns (vertical), along rows
// (horizontal) or everywhere (DC) has a transform with one non-zero row, column or coefficient.  With the source block's
// transform T kept per lane, those modes cost a 4-point Hadamard of the edge and four |.| instead of a prediction, a
// difference block and a full 4x4 Hadamard -- exact by linearity, 9 of K3's 17 SATDs per lane.
// Common output order of the 4-point Hadamard: rows (1,1,1,1) (1,1,-1,-1) (1,-1,-1,1) (1,-1,1,-1).
__device__ __forceinline__ void had4(int v0, int v1, int v2, int v3, int &o0, int &o1, int &o2, int &o3)
{
    const int a = v0 + v1, b = v0 - v1, c = v2 + v3, d = v2 - v3;
    o0 = a + c; o1 = a - c; o2 = b - d; o3 = b + d;
}
__device__ __forceinline__ int dp4a_u8s8(uint32_t u8x4, uint32_t s8x4, int acc)
{
    int d;
    asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(u8x4), "r"(s8x4), "r"(acc));
    return d;
}
struct SrcHad {
    int T[16];        // T[j * 4 + k]: vertical frequency j, horizontal frequency k
    int A, R0, C0;    // sum |T|, sum_k |T[0][k]|, sum_j |T[j][0]|
};
// rows: the four source rows as little-endian u8x4 words (byte x = column x)
__device__ __forceinline__ void src_hadamard(const uint32_t rows[4], SrcHad &h)
{
    int c[16];
#pragma unroll
    for (int y = 0; y < 4; y++) {                    // horizontal pass on the dot-product unit
        c[4 * y + 0] = dp4a_u8s8(rows[y], 0x01010101u, 0); c[4 * y + 1] = dp4a_u8s8(rows[y], 0xffff0101u, 0);
        c[4 * y + 2] = dp4a_u8s8(rows[y], 0x01ffff01u, 0); c[4 * y + 3] = dp4a_u8s8(rows[y], 0xff01ff01u, 0);
    }
#pragma unroll
    for (int k = 0; k < 4; k++) had4(c[k], c[4 + k], c[8 + k], c[12 + k], h.T[k], h.T[4 + k], h.T[8 + k], h.T[12 + k]);
    int a = 0;
#pragma unroll
    for (int i = 0; i < 16; i++) a += abs(h.T[i]);
    h.A = a;
    h.R0 = abs(h.T[0]) + abs(h.T[1]) + abs(h.T[2]) + abs(h.T[3]);
    h.C0 = abs(h.T[0]) + abs(h.T[4]) + abs(h.T[8]) + abs(h.T[12]);
}
// pred[y][x] = t[x]
__device__ __forceinline__ uint32_t satd_pred_v(const SrcHad &h, int t0, int t1, int t2, int t3)
{
    int k0, k1, k2, k3;
    had4(t0, t1, t2, t3, k0, k1, k2, k3);
    return (uint32_t)(h.A - h.R0 + abs(h.T[0] - 4 * k0) + abs(h.T[1] - 4 * k1) + abs(h.T[2] - 4 * k2) + abs(h.T[3] - 4 * k3)) >> 1;
}
// pred[y][x] = l[y]
__device__ __forceinline__ uint32_t satd_pred_h(const SrcHad &h, int l0, int l1, int l2, int l3)
{
    int j0, j1, j2, j3;
    had4(l0, l1, l2, l3, j0, j1, j2, j3);
    return (uint32_t)(h.A - h.C0 + abs(h.T[0] - 4 * j0) + abs(h.T[4] - 4 * j1) + abs(h.T[8] - 4 * j2) + abs(h.T[12] - 4 * j3)) >> 1;
}
// pred[y][x] = dc
__device__ __forceinline__ uint32_t satd_pred_dc(const SrcHad &h, int dc)
{
    return (uint32_t)(h.A - abs(h.T[0]) + abs(h.T[0] - 16 * dc)) >> 1;
}

// SATD of a 4x4 difference block: (sum |H d H^T|) >> 1.  The last butterfly stage is folded into the absolute values with
// |a + b| + |a - b| = 2 max(|a|, |b|): the sum is even and the final shift disappears.
__device__ __forceinline__ uint32_t satd4x4(const int d[16])
{
    int t[16];
#pragma unroll
    for (int y = 0; y < 4; y++) {
        int s01 = d[y * 4 + 0] + d[y * 4 + 1], d01 = d[y * 4 + 0] - d[y * 4 + 1];
        int s23 = d[y * 4 + 2] + d[y * 4 + 3], d23 = d[y * 4 + 2] - d[y * 4 + 3];
        t[y * 4 + 0] = s01 + s23; t[y * 4 + 1] = s01 - s23; t[y * 4 + 2] = d01 - d23; t[y * 4 + 3] = d01 + d23;
    }
    uint32_t s = 0;
#pragma unroll
    for (int x = 0; x < 4; x++) {
        int s01 = t[x] + t[4 + x], d01 = t[x] - t[4 + x];
        int s23 = t[8 + x] + t[12 + x], d23 = t[8 + x] - t[12 + x];
        s += max(abs(s01), abs(s23)) + max(abs(d01), abs(d23));
    }
    return s;
}

// ---- 8x8 transform path (High profile, SURVEY.md 8f row N1) -----------------------------------------------
// normAdjust8x8 position classes [y&3][x&3] (8.5.9), quantiser / scaling constants per class
__device__ __constant__ uint8_t c_cls8[16] = {0, 3, 4, 3, 3, 1, 5, 1, 4, 5, 2, 5, 3, 1, 5, 1};
__device__ __constant__ uint16_t c_quant8_mf[6][6] = {
    {13107, 11428, 20972, 12222, 16777, 15481}, {11916, 10826, 19174, 11058, 14980, 14290},
    {10082, 8943, 15978, 9675, 12710, 11985},   {9362, 8228, 14913, 8931, 11984, 11259},
    {8192, 7346, 13159, 7740, 10486, 9777},     {7282, 6428, 11570, 6830, 9118, 8640}};
__device__ __constant__ uint8_t c_dequant8_v[6][6] = {{20, 18, 32, 19, 25, 24}, {22, 19, 35, 21, 28, 26}, {26, 23, 42, 24, 33, 31},
                                                      {28, 25, 45, 26, 35, 33}, {32, 28, 51, 30, 40, 38}, {36, 32, 58, 34, 46, 43}};
// 8x8 frame zig-zag (Figure 8-8): scan position -> raster index y*8+x
__device__ __constant__ uint8_t c_zigzag8[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                                 41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                                 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

// forward 8-point butterflies (encoder side; x264's dct8 form, frozen in oracle/b2o_transform8.c)
__device__ __forceinline__ void fdct8_1d(const int s[8], int d[8])
{
    const int s07 = s[0] + s[7], s16 = s[1] + s[6], s25 = s[2] + s[5], s34 = s[3] + s[4];
    const int a0 = s07 + s34, a1 = s16 + s25, a2 = s07 - s34, a3 = s16 - s25;
    const int d07 = s[0] - s[7], d16 = s[1] - s[6], d25 = s[2] - s[5], d34 = s[3] - s[4];
    const int a4 = d16 + d25 + (d07 + (d07 >> 1));
    const int a5 = d07 - d34 - (d25 + (d25 >> 1));
    const int a6 = d07 + d34 - (d16 + (d16 >> 1));
    const int a7 = d16 - d25 + (d34 + (d34 >> 1));
    d[0] = a0 + a1; d[1] = a4 + (a7 >> 2); d[2] = a2 + (a3 >> 1); d[3] = a5 + (a6 >> 2);
    d[4] = a0 - a1; d[5] = a6 - (a5 >> 2); d[6] = (a2 >> 1) - a3; d[7] = (a4 >> 2) - a7;
}
// normative inverse 8-point butterflies (8.5.13)
__device__ __forceinline__ void idct8_1d(const int d[8], int o[8])
{
    const int a0 = d[0] + d[4], a2 = d[0] - d[4], a4 = (d[2] >> 1) - d[6], a6 = d[2] + (d[6] >> 1);
    const int b0 = a0 + a6, b2 = a2 + a4, b4 = a2 - a4, b6 = a0 - a6;
    const int a1 = -d[3] + d[5] - d[7] - (d[7] >> 1);
    const int a3 = d[1] + d[7] - d[3] - (d[3] >> 1);
    const int a5 = -d[1] + d[7] + d[5] + (d[5] >> 1);
    const int a7 = d[3] + d[5] + d[1] + (d[1] >> 1);
    const int b1 = a1 + (a7 >> 2), b3 = a3 + (a5 >> 2), b5 = (a3 >> 2) - a5, b7 = a7 - (a1 >> 2);
    o[0] = b0 + b7; o[1] = b2 + b5; o[2] = b4 + b3; o[3] = b6 + b1;
    o[4] = b6 - b1; o[5] = b4 - b3; o[6] = b2 - b5; o[7] = b0 - b7;
}
// 2-D 4x4 Hadamard of a difference block, unnormalised (the SATD is (sum |t|) >> 1)
__device__ __forceinline__ void hadamard4x4(const int d[16], int t[16])
{
#pragma unroll
    for (int y = 0; y < 4; y++) {
        int s01 = d[y * 4 + 0] + d[y * 4 + 1], d01 = d[y * 4 + 0] - d[y * 4 + 1];
        int s23 = d[y * 4 + 2] + d[y * 4 + 3], d23 = d[y * 4 + 2] - d[y * 4 + 3];
        t[y * 4 + 0] = s01 + s23; t[y * 4 + 1] = s01 - s23; t[y * 4 + 2] = d01 - d23; t[y * 4 + 3] = d01 + d23;
    }
#pragma unroll
    for (int x = 0; x < 4; x++) {
        int s01 = t[x] + t[4 + x], d01 = t[x] - t[4 + x];
        int s23 = t[8 + x] + t[12 + x], d23 = t[8 + x] - t[12 + x];
        t[x] = s01 + s23; t[4 + x] = s01 - s23; t[8 + x] = d01 - d23; t[12 + x] = d01 + d23;
    }
}

// sign (+1/-1) of entry [v][u] of H4 = rows ++++ / ++-- / +--+ / +-+-
__device__ __forceinline__ int h4_sign(int v, int u)
{
    // bit u of row mask v is 1 where the entry is negative
    const unsigned masks = 0x0u | (0xCu << 4) | (0x6u << 8) | (0xAu << 12);
    return ((masks >> (4 * v + u)) & 1u) ? -1 : 1;
}

// store 16 raster levels of one block in zig-zag order as int16 (two 16-byte stores)
__device__ __forceinline__ void store_levels_zigzag(int16_t *dst, const int z[16])
{
    uint32_t p[8];
#pragma unroll
    for (int i = 0; i < 8; i++) {
        // c_zigzag is compile-time here
        constexpr int zz[16] = {0, 1, 4, 8, 5, 2, 3, 6, 9, 12, 13, 10, 7, 11, 14, 15};
        p[i] = ((uint32_t)(uint16_t)(int16_t)z[zz[2 * i]]) | ((uint32_t)(uint16_t)(int16_t)z[zz[2 * i + 1]] << 16);
    }
    uint4 *d4 = (uint4 *)dst;
    d4[0] = make_uint4(p[0], p[1], p[2], p[3]);
    d4[1] = make_uint4(p[4], p[5], p[6], p[7]);
}

// ---- intra 4x4 prediction (8.3.1.2); T[-1..7], L[-1..3] passed as pointers offset by one ---------
// avail bits: 1 left, 2 top, 4 top-left, 8 top-right (same as the oracle's B2O_AV_*)
__device__ __forceinline__ bool i4_mode_ok(int mode, int avail)
{
    switch (mode) {
    case B2_I4_V: case B2_I4_DDL: case B2_I4_VL: return (avail & 2) != 0;
    case B2_I4_H: case B2_I4_HU: return (avail & 1) != 0;
    case B2_I4_DC: return true;
    default: return (avail & 7) == 7;
    }
}

// E layout: E[0]=M (top-left), E[1..8]=T0..T7, E[9..12]=L0..L3, all already substituted
// (128 for unavailable, T3 replicated when top-right is missing)
__device__ __forceinline__ void pred4x4(int mode, const int E[13], int avail, int pred[16])
{
    const int *T = E + 1, *L = E + 9;
    const int M = E[0];
#define B2F3(a, b, c) (((a) + 2 * (b) + (c) + 2) >> 2)
#define B2F2(a, b) (((a) + (b) + 1) >> 1)
    switch (mode) {
    case B2_I4_V:
#pragma unroll
        for (int i = 0; i < 16; i++) pred[i] = T[i & 3];
        break;
    case B2_I4_H:
#pragma unroll
        for (int i = 0; i < 16; i++) pred[i] = L[i >> 2];
        break;
    case B2_I4_DC: {
        const bool hasT = avail & 2, hasL = avail & 1;
        int s = 0;
        if (hasT) s += T[0] + T[1] + T[2] + T[3];
        if (hasL) s += L[0] + L[1] + L[2] + L[3];
        const int dc = (hasT && hasL) ? (s + 4) >> 3 : (hasT || hasL) ? (s + 2) >> 2 : 128;
#pragma unroll
        for (int i = 0; i < 16; i++) pred[i] = dc;
        break;
    }
    case B2_I4_DDL: {
        int d[7];
#pragma unroll
        for (int k = 0; k < 6; k++) d[k] = B2F3(T[k], T[k + 1], T[k + 2]);
        d[6] = (T[6] + 3 * T[7] + 2) >> 2;
#pragma unroll
        for (int y = 0; y < 4; y++)
#pragma unroll
            for (int x = 0; x < 4; x++) pred[y * 4 + x] = d[x + y];
        break;
    }
    case B2_I4_DDR: {
        // diagonal index k = x - y + 3 in 0..6 over the edge sequence L3 L2 L1 L0 M T0 T1 T2 T3
        const int e[9] = {L[3], L[2], L[1], L[0], M, T[0], T[1], T[2], T[3]};
        int d[7];
#pragma unroll
        for (int k = 0; k < 7; k++) d[k] = B2F3(e[k], e[k + 1], e[k + 2]);
#pragma unroll
        for (int y = 0; y < 4; y++)
#pragma unroll
            for (int x = 0; x < 4; x++) pred[y * 4 + x] = d[x - y + 3];
        break;
    }
    case B2_I4_VR: {
        const int e[9] = {L[3], L[2], L[1], L[0], M, T[0], T[1], T[2], T[3]};
#pragma unroll
        for (int y = 0; y < 4; y++)
#pragma unroll
            for (int x = 0; x < 4; x++) {
                const int z = 2 * x - y;
                int v;
                if (z >= 0 && !(z & 1)) v = B2F2(e[4 + x - (y >> 1)], e[5 + x - (y >> 1)]);
                else if (z >= 0) v = B2F3(e[3 + x - (y >> 1)], e[4 + x - (y >> 1)], e[5 + x - (y >> 1)]);
                else if (z == -1) v = B2F3(L[0], M, T[0]);
                else v = B2F3(e[4 - y], e[5 - y], e[6 - y]);      // L[y-1], L[y-2], L[y-3]
                pred[y * 4 + x] = v;
            }
        break;
    }
    case B2_I4_HD: {
        const int e[9] = {L[3], L[2], L[1], L[0], M, T[0], T[1], T[2], T[3]};
#pragma unroll
        for (int y = 0; y < 4; y++)
#pragma unroll
            for (int x = 0; x < 4; x++) {
                const int z = 2 * y - x;
                int v;
                if (z >= 0 && !(z & 1)) v = B2F2(e[4 - (y - (x >> 1))], e[3 - (y - (x >> 1))]);   // L[y'-1], L[y']
                else if (z >= 0) v = B2F3(e[5 - (y - (x >> 1))], e[4 - (y - (x >> 1))], e[3 - (y - (x >> 1))]);
                else if (z == -1) v = B2F3(L[0], M, T[0]);
                else v = B2F3(e[4 + x], e[3 + x], e[2 + x]);      // T[x-1], T[x-2], T[x-3]
                pred[y * 4 + x] = v;
            }
        break;
    }
    case B2_I4_VL:
#pragma unroll
        for (int y = 0; y < 4; y++)
#pragma unroll
            for (int x = 0; x < 4; x++) {
                const int k = x + (y >> 1);
                pred[y * 4 + x] = (y & 1) ? B2F3(T[k], T[k + 1], T[k + 2]) : B2F2(T[k], T[k + 1]);
            }
        break;
    default:   // HU
#pragma unroll
        for (int y = 0; y < 4; y++)
#pragma unroll
            for (int x = 0; x < 4; x++) {
                const int z = x + 2 * y, k = y + (x >> 1);
                int v;
                if (z > 5) v = L[3];
                else if (z == 5) v = (L[2] + 3 * L[3] + 2) >> 2;
                else if (z & 1) v = B2F3(L[k], L[k + 1], L[k + 2]);
                else v = B2F2(L[k], L[k + 1]);
                pred[y * 4 + x] = v;
            }
        break;
    }
#undef B2F3
#undef B2F2
}

// ---- intra 8x8 prediction (8.3.2.2) from edge tables -------------------------------------------------------
// Edge sequence of one 8x8 block after the reference-sample filter 8.3.2.2.1, bottom-left to top-right:
//   E[7-y] = p'[-1,y] (y = 0..7), E[8] = p'[-1,-1], E[9+x] = p'[x,-1] (x = 0..15)
// and its two smoothings  F2[i] = (E[i] + E[i+1] + 1) >> 1 (i = 0..23),  F3[i] = (E[i] + 2 E[i+1] + E[i+2] + 2) >> 2
// (i = 0..22), F3[23] = (E[23] + 3 E[24] + 2) >> 2.  Every directional predictor is one lookup:
struct I8Edge {
    uint8_t E[25], F2[24], F3[24];
    uint8_t hu13;                      // (E[1] + 3 E[0] + 2) >> 2, the z = 13 sample of Horizontal-Up
    uint8_t dc;                        // DC value for this block's availability
    uint8_t pad[5];
};                                     // 80 bytes

// filtered edge sample i (0..24) from the raw edge R (same indexing, unavailable samples already substituted:
// 128, top-right replicated); avail bits as for 4x4 blocks
__device__ __forceinline__ int i8_filter_edge(const uint8_t *R, int i, int avail)
{
    const bool hasL = avail & 1, hasT = avail & 2, hasTL = avail & 4;
    if (i < 8) {                                           // left column, y = 7 - i
        if (!hasL) return 128;
        if (i == 0) return (R[1] + 3 * R[0] + 2) >> 2;     // y = 7: (p[-1,6] + 3 p[-1,7] + 2) >> 2
        if (i == 7 && !hasTL) return (3 * R[7] + R[6] + 2) >> 2;
        return (R[i - 1] + 2 * R[i] + R[i + 1] + 2) >> 2;
    }
    if (i == 8) {
        if (!hasTL) return 128;
        if (!hasT) return (3 * R[8] + R[7] + 2) >> 2;
        if (!hasL) return (3 * R[8] + R[9] + 2) >> 2;
        return (R[7] + 2 * R[8] + R[9] + 2) >> 2;
    }
    if (!hasT) return 128;
    if (i == 24) return (R[23] + 3 * R[24] + 2) >> 2;
    if (i == 9 && !hasTL) return (3 * R[9] + R[10] + 2) >> 2;
    return (R[i - 1] + 2 * R[i] + R[i + 1] + 2) >> 2;
}

// one predicted sample (X,Y in 0..7) of mode `mode`
__device__ __forceinline__ int pred8x8_px(int mode, const I8Edge &t, int X, int Y)
{
    switch (mode) {
    case B2_I4_V: return t.E[9 + X];
    case B2_I4_H: return t.E[7 - Y];
    case B2_I4_DC: return t.dc;
    case B2_I4_DDL: return t.F3[9 + X + Y];
    case B2_I4_DDR: return t.F3[7 + X - Y];
    case B2_I4_VR: {
        const int z = 2 * X - Y, k = X - (Y >> 1);
        if (z < -1) return t.F3[8 - Y + 2 * X];
        return (z & 1) ? t.F3[7 + k] : t.F2[8 + k];
    }
    case B2_I4_HD: {
        const int z = 2 * Y - X, k = Y - (X >> 1);
        if (z < -1) return t.F3[6 + X - 2 * Y];
        return (z & 1) ? t.F3[7 - k] : t.F2[7 - k];
    }
    case B2_I4_VL: {
        const int k = X + (Y >> 1);
        return (Y & 1) ? t.F3[9 + k] : t.F2[9 + k];
    }
    default: {                                             // HU
        const int z = X + 2 * Y, k = Y + (X >> 1);
        if (z > 13) return t.E[0];
        if (z == 13) return t.hu13;
        return (z & 1) ? t.F3[5 - k] : t.F2[6 - k];
    }
    }
}

// availability of 8x8 block q (raster 2x2) given the MB's availability
__device__ __forceinline__ int blk8_avail(int q, int mba)
{
    const int qx = q & 1, qy = q >> 1;
    int a = 0;
    if (qx || (mba & 1)) a |= 1;
    if (qy || (mba & 2)) a |= 2;
    if ((qx && qy) || (qx && !qy && (mba & 2)) || (!qx && qy && (mba & 1)) || (!qx && !qy && (mba & 4))) a |= 4;
    if (q == 0 ? (mba & 2) != 0 : q == 1 ? (mba & 8) != 0 : q == 2) a |= 8;
    return a;
}

// MB-level neighbour availability; row0 = first row of the macroblock's slice (b2_slice_row0, b2enc_types.h): the neighbours
// above are in another slice, so unavailable, when mby == row0
__device__ __forceinline__ int mb_avail(int mbx, int mby, int mbw, int row0)
{
    int a = 0;
    if (mbx > 0) a |= 1;
    if (mby > row0) a |= 2;
    if (mbx > 0 && mby > row0) a |= 4;
    if (mby > row0 && mbx < mbw - 1) a |= 8;
    return a;
}
// availability of 4x4 block b (z order) given the MB's availability
__device__ __forceinline__ int blk_avail(int b, int mba)
{
    const int bx = blk_x(b), by = blk_y(b);
    int a = 0;
    if (bx > 0 || (mba & 1)) a |= 1;
    if (by > 0 || (mba & 2)) a |= 2;
    if ((bx > 0 && by > 0) || (bx > 0 && by == 0 && (mba & 2)) || (bx == 0 && by > 0 && (mba & 1)) ||
        (bx == 0 && by == 0 && (mba & 4)))
        a |= 4;
    if (by == 0) {
        if (bx < 3 ? (mba & 2) : (mba & 8)) a |= 8;
    } else if (bx < 3 && b != 3 && b != 11 && b != 7 && b != 13 && b != 15) {
        a |= 8;
    }
    return a;
}

// gather the 13 edge samples of a 4x4 block from a plane (p -> block's top-left pixel)
__device__ __forceinline__ void load_edge4x4(const uint8_t *p, int pitch, int avail, int E[13])
{
    const uint8_t *top = p - pitch;
    E[0] = (avail & 4) ? top[-1] : 128;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        E[1 + i] = (avail & 2) ? top[i] : 128;
        E[9 + i] = (avail & 1) ? p[i * pitch - 1] : 128;
    }
#pragma unroll
    for (int i = 4; i < 8; i++) E[1 + i] = (avail & 8) ? top[i] : E[4];
}

// ---- luma quarter-pel sample (8.4.2.2.1) straight from a plane ------------------------------------
__device__ __forceinline__ int tap6(int a, int b, int c, int d, int e, int f) { return a - 5 * b + 20 * c + 20 * d - 5 * e + f; }
__device__ __forceinline__ int hb1(const uint8_t *q) { return tap6(q[-2], q[-1], q[0], q[1], q[2], q[3]); }
__device__ __forceinline__ int vh1(const uint8_t *q, int p)
{
    return tap6(q[-2 * p], q[-p], q[0], q[p], q[2 * p], q[3 * p]);
}
__device__ __forceinline__ int half_b(const uint8_t *q) { return b2_clip255((hb1(q) + 16) >> 5); }
__device__ __forceinline__ int half_h(const uint8_t *q, int p) { return b2_clip255((vh1(q, p) + 16) >> 5); }
__device__ __forceinline__ int half_j(const uint8_t *q, int p)
{
    int j1 = tap6(hb1(q - 2 * p), hb1(q - p), hb1(q), hb1(q + p), hb1(q + 2 * p), hb1(q + 3 * p));
    return b2_clip255((j1 + 512) >> 10);
}
// q -> integer sample G; (fx,fy) quarter-pel fraction
__device__ __forceinline__ int qpel_sample(const uint8_t *q, int p, int fx, int fy)
{
#define B2AVG(a, b) (((a) + (b) + 1) >> 1)
    switch (fy * 4 + fx) {
    case 0: return q[0];
    case 1: return B2AVG(q[0], half_b(q));
    case 2: return half_b(q);
    case 3: return B2AVG(q[1], half_b(q));
    case 4: return B2AVG(q[0], half_h(q, p));
    case 5: return B2AVG(half_b(q), half_h(q, p));
    case 6: return B2AVG(half_b(q), half_j(q, p));
    case 7: return B2AVG(half_b(q), half_h(q + 1, p));
    case 8: return half_h(q, p);
    case 9: return B2AVG(half_h(q, p), half_j(q, p));
    case 10: return half_j(q, p);
    case 11: return B2AVG(half_j(q, p), half_h(q + 1, p));
    case 12: return B2AVG(q[p], half_h(q, p));
    case 13: return B2AVG(half_h(q, p), half_b(q + p));
    case 14: return B2AVG(half_j(q, p), half_b(q + p));
    default: return B2AVG(half_h(q + 1, p), half_b(q + p));
    }
#undef B2AVG
}

}  // namespace b2
