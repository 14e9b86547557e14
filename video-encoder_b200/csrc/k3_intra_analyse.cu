// k3_intra_analyse.cu -- K3: intra mode analysis on SOURCE pixels (I16x16: 4 modes, I4x4: 9 modes per
// block, chroma 8x8: 4 modes), SATD + lambda*bits costs.
//
// Replaces x264's intra analysis (behind x264_encoder_encode, av_encode.c:970); bit-exact against
// oracle/b2o_intra.c:b2o_intra_analyse.  Because predictions are built from source neighbours, every
// macroblock and every 4x4 block is independent (SURVEY.md 7.2 item 2-ii): 16 threads per MB, one per
// 4x4 block, 16-lane shuffle reductions for the MB-level sums.
// Bound: integer ALU / L1; algorithmic bytes = 1.5*W*H source read + 32 B/MB written.
#include "b2_h264.cuh"

namespace {

constexpr int K3_THREADS = 128;                 // 8 macroblocks per CTA

__device__ __forceinline__ int sum16(int v)      // sum over the 16-lane group
{
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o, 16);
    return v;
}

template <bool I8>
__global__ void __launch_bounds__(K3_THREADS)
k3_intra_analyse_kernel(const uint8_t *__restrict__ cur_y, const uint8_t *__restrict__ cur_u,
                        const uint8_t *__restrict__ cur_v, int pitch, int pitchc, size_t stride_y, size_t stride_c,
                        int mbw, int mbh, int nslices, int nmb_total, int lambda, b2_mbinfo_t *__restrict__ info,
                        uint32_t *__restrict__ cost_i16, uint32_t *__restrict__ cost_i4, uint32_t *__restrict__ cost_i8)
{
    const int gt = blockIdx.x * K3_THREADS + threadIdx.x;
    int mbi = gt >> 4;                            // global MB index over all frames
    const int b = gt & 15;                        // 4x4 block (z order) owned by this lane
    const bool valid = mbi < nmb_total;
    if (!valid) mbi = nmb_total - 1;              // keep the lane in the shuffles
    const int per_frame = mbw * mbh;
    const int frame = mbi / per_frame, r = mbi - frame * per_frame;
    const int mby = r / mbw, mbx = r - mby * mbw;
    const int mba = b2::mb_avail(mbx, mby, mbw, nslices > 1 ? b2_slice_row0(mby, nslices, mbh) : 0);
    const int bx = b2::blk_x(b) * 4, by = b2::blk_y(b) * 4;

    const uint8_t *sy = cur_y + frame * stride_y + (size_t)(B2_PAD + mby * 16) * pitch + B2_PAD + mbx * 16;
    const uint8_t *sb = sy + (size_t)by * pitch + bx;

    int src[16];
    uint32_t srow[4];
#pragma unroll
    for (int y = 0; y < 4; y++) {
        const uint32_t w = *(const uint32_t *)(sb + (size_t)y * pitch);
        srow[y] = w;
#pragma unroll
        for (int x = 0; x < 4; x++) src[y * 4 + x] = (w >> (8 * x)) & 255;
    }
    // the block's own Hadamard transform: vertical / horizontal / DC predictors are priced against it (b2_h264.cuh)
    b2::SrcHad sh;
    b2::src_hadamard(srow, sh);

    // ---- I4x4: 9 modes on this lane's block --------------------------------------------------------
    uint32_t best4 = 0xffffffffu; int mode4 = B2_I4_DC;
    {
        const int ba = b2::blk_avail(b, mba);
        int E[13];
        b2::load_edge4x4(sb, pitch, ba, E);
#pragma unroll
        for (int m = 0; m < 9; m++) {
            if (!b2::i4_mode_ok(m, ba)) continue;
            uint32_t sat;
            if (m == B2_I4_V) sat = b2::satd_pred_v(sh, E[1], E[2], E[3], E[4]);
            else if (m == B2_I4_H) sat = b2::satd_pred_h(sh, E[9], E[10], E[11], E[12]);
            else if (m == B2_I4_DC) {
                const bool hT = ba & 2, hL = ba & 1;
                const int sum = (hT ? E[1] + E[2] + E[3] + E[4] : 0) + (hL ? E[9] + E[10] + E[11] + E[12] : 0);
                sat = b2::satd_pred_dc(sh, (hT && hL) ? (sum + 4) >> 3 : (hT || hL) ? (sum + 2) >> 2 : 128);
            } else {
                int pred[16], d[16];
                b2::pred4x4(m, E, ba, pred);
#pragma unroll
                for (int i = 0; i < 16; i++) d[i] = src[i] - pred[i];
                sat = b2::satd4x4(d);
            }
            uint32_t c = sat + (uint32_t)(lambda * (m == B2_I4_DC ? 1 : 4));
            if (c < best4) { best4 = c; mode4 = m; }
        }
    }
    const uint32_t sum4 = (uint32_t)sum16((int)best4) + (uint32_t)(lambda * 24);

    // ---- I8x8 (row N1, only with the 8x8 transform): the four lanes of a quad (z-order blocks 4q..4q+3) share the 8x8
    // block's filtered edge tables in shared memory; every mode is evaluated (no divergence around the shuffles) and
    // illegal ones are masked when the minimum is taken.  Cost = SA8D (8x8 Hadamard = butterflies over the quad's four
    // 4x4 Hadamards) + lambda * bits, as in oracle/b2o_intra.c.
    uint32_t sum8 = 0; int modes8 = 0;
    if (I8) {
        __shared__ b2::I8Edge s_edge[K3_THREADS / 4];
        __shared__ uint8_t s_raw[K3_THREADS / 4][32];
        const int quad = threadIdx.x >> 2, k = b & 3, q = b >> 2;
        const int qx = (q & 1) * 8, qy = (q >> 1) * 8, sx = (k & 1) * 4, sy4 = (k >> 1) * 4;
        const int qa = b2::blk8_avail(q, mba);
        b2::I8Edge &et = s_edge[quad];
        uint8_t *R = s_raw[quad];
        const uint8_t *qp0 = sy + (size_t)qy * pitch + qx;             // top-left pixel of the 8x8 block
        {   // raw edge: lane k loads T[4k..4k+3], L[2k], L[2k+1]; lane 0 the corner
            uint32_t tw = 0x80808080u;
            if (qa & 2) {
                if (k < 2 || (qa & 8)) tw = *(const uint32_t *)(qp0 - (ptrdiff_t)pitch + 4 * k);
                else tw = 0x01010101u * qp0[-(ptrdiff_t)pitch + 7];   // top-right missing: replicate p[7,-1]
            }
#pragma unroll
            for (int i = 0; i < 4; i++) R[9 + 4 * k + i] = (uint8_t)(tw >> (8 * i));
            R[7 - 2 * k] = (qa & 1) ? qp0[(size_t)(2 * k) * pitch - 1] : 128;
            R[6 - 2 * k] = (qa & 1) ? qp0[(size_t)(2 * k + 1) * pitch - 1] : 128;
            if (k == 0) R[8] = (qa & 4) ? qp0[-(ptrdiff_t)pitch - 1] : 128;
        }
        __syncwarp();
        for (int i = k; i < 25; i += 4) et.E[i] = (uint8_t)b2::i8_filter_edge(R, i, qa);
        __syncwarp();
        for (int i = k; i < 24; i += 4) {
            et.F2[i] = (uint8_t)((et.E[i] + et.E[i + 1] + 1) >> 1);
            et.F3[i] = i < 23 ? (uint8_t)((et.E[i] + 2 * et.E[i + 1] + et.E[i + 2] + 2) >> 2) : (uint8_t)((et.E[23] + 3 * et.E[24] + 2) >> 2);
        }
        if (k == 0) {
            int st = 0, sl = 0;
#pragma unroll
            for (int i = 0; i < 8; i++) { st += et.E[9 + i]; sl += et.E[i]; }
            const bool hT = qa & 2, hL = qa & 1;
            et.dc = (uint8_t)((hT && hL) ? (st + sl + 8) >> 4 : hT ? (st + 4) >> 3 : hL ? (sl + 4) >> 3 : 128);
            et.hu13 = (uint8_t)((et.E[1] + 3 * et.E[0] + 2) >> 2);
        }
        __syncwarp();
        uint32_t best8 = 0xffffffffu; int mode8 = B2_I4_DC;
#pragma unroll
        for (int m = 0; m < 9; m++) {                    // unrolled: the predictor switch and the parity tests fold per mode
            int d[16], t[16];
#pragma unroll
            for (int i = 0; i < 16; i++) d[i] = src[i] - b2::pred8x8_px(m, et, sx + (i & 3), sy4 + (i >> 2));
            b2::hadamard4x4(d, t);
            uint32_t s8 = 0;
#pragma unroll
            for (int i = 0; i < 16; i++) {
                int o = __shfl_xor_sync(0xffffffffu, t[i], 1);
                int u = (k & 1) ? o - t[i] : t[i] + o;
                o = __shfl_xor_sync(0xffffffffu, u, 2);
                u = (k & 2) ? o - u : u + o;
                s8 += abs(u);
            }
            s8 += __shfl_xor_sync(0xffffffffu, s8, 1);
            s8 += __shfl_xor_sync(0xffffffffu, s8, 2);
            const uint32_t c = ((s8 + 2) >> 2) + (uint32_t)(lambda * (m == B2_I4_DC ? 1 : 4));
            if (b2::i4_mode_ok(m, qa) && c < best8) { best8 = c; mode8 = m; }
        }
        sum8 = (uint32_t)sum16(k == 0 ? (int)best8 : 0) + (uint32_t)(lambda * 8);
        // modes of the four quads -> 16-bit word on every lane of the group
        const int gb = (threadIdx.x & 31) & 16;
        modes8 = __shfl_sync(0xffffffffu, mode8, gb + 0) | (__shfl_sync(0xffffffffu, mode8, gb + 4) << 4) |
                 (__shfl_sync(0xffffffffu, mode8, gb + 8) << 8) | (__shfl_sync(0xffffffffu, mode8, gb + 12) << 12);
    }

    // ---- I16x16: lane i holds top[i] and left[i] ----------------------------------------------------
    const int lane16 = b;                        // 0..15 inside the group (group = 16 consecutive lanes)
    const int grp_base = (threadIdx.x & 31) & 16;
    const bool hasT = mba & 2, hasL = mba & 1;
    const int topv = hasT ? sy[-(ptrdiff_t)pitch + lane16] : 0;
    const int leftv = hasL ? sy[(size_t)lane16 * pitch - 1] : 0;
    const int tlv = (mba & 4) ? sy[-(ptrdiff_t)pitch - 1] : 0;
    uint32_t best16 = 0xffffffffu; int mode16 = B2_I16_DC;
    {
        // per-lane copies of the 4 top / 4 left samples this block needs
        int t4[4], l4[4];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            t4[i] = __shfl_sync(0xffffffffu, topv, grp_base + bx + i);
            l4[i] = __shfl_sync(0xffffffffu, leftv, grp_base + by + i);
        }
        const int sumT = sum16(topv), sumL = sum16(leftv);
        // plane parameters: H = sum_{i<8} (i+1)(top[8+i]-top[6-i]) with top[-1] = top-left
        int hterm = 0, vterm = 0;
        {
            const int i = lane16 & 7;
            const int ta = __shfl_sync(0xffffffffu, topv, grp_base + 8 + i);
            const int tb = __shfl_sync(0xffffffffu, topv, grp_base + ((6 - i) & 15));
            const int la = __shfl_sync(0xffffffffu, leftv, grp_base + 8 + i);
            const int lb = __shfl_sync(0xffffffffu, leftv, grp_base + ((6 - i) & 15));
            if (lane16 < 8) {
                hterm = (i + 1) * (ta - (i == 7 ? tlv : tb));
                vterm = (i + 1) * (la - (i == 7 ? tlv : lb));
            }
        }
        const int Hs = sum16(hterm), Vs = sum16(vterm);
        const int t15 = __shfl_sync(0xffffffffu, topv, grp_base + 15), l15 = __shfl_sync(0xffffffffu, leftv, grp_base + 15);
        const int pa = 16 * (l15 + t15), pb = (5 * Hs + 32) >> 6, pc = (5 * Vs + 32) >> 6;
        const int dc = (hasT && hasL) ? (sumT + sumL + 16) >> 5 : (hasT || hasL) ? (sumT + sumL + 8) >> 4 : 128;
        const int ue_bits[4] = {1, 3, 3, 5};
#pragma unroll
        for (int m = 0; m < 4; m++) {
            const bool ok = m == B2_I16_V ? hasT : m == B2_I16_H ? hasL : m == B2_I16_DC ? true : (mba & 7) == 7;
            uint32_t sat;
            if (m == B2_I16_V) sat = b2::satd_pred_v(sh, t4[0], t4[1], t4[2], t4[3]);
            else if (m == B2_I16_H) sat = b2::satd_pred_h(sh, l4[0], l4[1], l4[2], l4[3]);
            else if (m == B2_I16_DC) sat = b2::satd_pred_dc(sh, dc);
            else {
                int d[16];
#pragma unroll
                for (int y = 0; y < 4; y++)
#pragma unroll
                    for (int x = 0; x < 4; x++)
                        d[y * 4 + x] = src[y * 4 + x] - b2_clip255((pa + pb * (bx + x - 7) + pc * (by + y - 7) + 16) >> 5);
                sat = b2::satd4x4(d);
            }
            const uint32_t c = (uint32_t)sum16((int)sat) + (uint32_t)(lambda * ue_bits[m]);
            if (ok && c < best16) { best16 = c; mode16 = m; }
        }
    }

    // ---- chroma 8x8: lanes 0..7 own (plane, 4x4 block) ------------------------------------------------
    uint32_t bestc = 0xffffffffu; int modec = B2_IC_DC;
    {
        const int pl = (b >> 2) & 1, k = b & 3, cbx = (k & 1) * 4, cby = (k >> 1) * 4;
        const uint8_t *cp = (pl ? cur_v : cur_u) + frame * stride_c + (size_t)(B2_PADC + mby * 8) * pitchc + B2_PADC + mbx * 8;
        int top[8], left[8], tl = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) { top[i] = hasT ? cp[-(ptrdiff_t)pitchc + i] : 0; left[i] = hasL ? cp[(size_t)i * pitchc - 1] : 0; }
        if (mba & 4) tl = cp[-(ptrdiff_t)pitchc - 1];
        int csrc[16];
        uint32_t crow[4];
#pragma unroll
        for (int y = 0; y < 4; y++) {
            const uint32_t w = *(const uint32_t *)(cp + (size_t)(cby + y) * pitchc + cbx);
            crow[y] = w;
#pragma unroll
            for (int x = 0; x < 4; x++) csrc[y * 4 + x] = (w >> (8 * x)) & 255;
        }
        b2::SrcHad ch;
        b2::src_hadamard(crow, ch);
        const int t0 = top[0] + top[1] + top[2] + top[3], t1 = top[4] + top[5] + top[6] + top[7];
        const int l0 = left[0] + left[1] + left[2] + left[3], l1 = left[4] + left[5] + left[6] + left[7];
        int dcv;
        if (k == 0) dcv = (hasT && hasL) ? (t0 + l0 + 4) >> 3 : hasT ? (t0 + 2) >> 2 : hasL ? (l0 + 2) >> 2 : 128;
        else if (k == 1) dcv = hasT ? (t1 + 2) >> 2 : hasL ? (l0 + 2) >> 2 : 128;
        else if (k == 2) dcv = hasL ? (l1 + 2) >> 2 : hasT ? (t0 + 2) >> 2 : 128;
        else dcv = (hasT && hasL) ? (t1 + l1 + 4) >> 3 : hasT ? (t1 + 2) >> 2 : hasL ? (l1 + 2) >> 2 : 128;
        int Hc = 0, Vc = 0;
#pragma unroll
        for (int i = 0; i < 4; i++) {
            Hc += (i + 1) * (top[4 + i] - (i == 3 ? tl : top[2 - i]));
            Vc += (i + 1) * (left[4 + i] - (i == 3 ? tl : left[2 - i]));
        }
        const int pa = 16 * (left[7] + top[7]), pb = (34 * Hc + 32) >> 6, pc = (34 * Vc + 32) >> 6;
        const int ue_bits[4] = {1, 3, 3, 5};
#pragma unroll
        for (int m = 0; m < 4; m++) {
            const bool ok = m == B2_IC_DC ? true : m == B2_IC_H ? hasL : m == B2_IC_V ? hasT : (mba & 7) == 7;
            uint32_t sat;
            if (m == B2_IC_DC) sat = b2::satd_pred_dc(ch, dcv);
            else if (m == B2_IC_H) sat = b2::satd_pred_h(ch, left[cby], left[cby + 1], left[cby + 2], left[cby + 3]);
            else if (m == B2_IC_V) sat = b2::satd_pred_v(ch, top[cbx], top[cbx + 1], top[cbx + 2], top[cbx + 3]);
            else {
                int d[16];
#pragma unroll
                for (int y = 0; y < 4; y++)
#pragma unroll
                    for (int x = 0; x < 4; x++)
                        d[y * 4 + x] = csrc[y * 4 + x] - b2_clip255((pa + pb * (cbx + x - 3) + pc * (cby + y - 3) + 16) >> 5);
                sat = b2::satd4x4(d);
            }
            const int part = b < 8 ? (int)sat : 0;
            const uint32_t c = (uint32_t)sum16(part) + (uint32_t)(lambda * ue_bits[m]);
            if (ok && c < bestc) { bestc = c; modec = m; }
        }
    }

    if (valid) {
        info[mbi].i4_mode[b] = (uint8_t)mode4;
        if (b == 0) {
            info[mbi].i16_mode = (uint8_t)mode16;
            info[mbi].chroma_mode = (uint8_t)modec;
            cost_i16[mbi] = best16;
            cost_i4[mbi] = sum4;
            if (I8) { cost_i8[mbi] = sum8; info[mbi].i8_modes = (uint16_t)modes8; }
        }
    }
}

}  // namespace

int b2_launch_intra_analyse(const uint8_t *d_y, const uint8_t *d_u, const uint8_t *d_v, int pitch, int pitchc,
                            size_t stride_y, size_t stride_c, int mbw, int mbh, int slices, int nframes, int lambda,
                            b2_mbinfo_t *d_info, uint32_t *d_c16, uint32_t *d_c4, uint32_t *d_c8, cudaStream_t st)
{
    const int nmb = mbw * mbh * nframes, ns = b2_slice_count(slices, mbh);
    const int blocks = (nmb * 16 + K3_THREADS - 1) / K3_THREADS;
    if (d_c8)
        k3_intra_analyse_kernel<true><<<blocks, K3_THREADS, 0, st>>>(d_y, d_u, d_v, pitch, pitchc, stride_y, stride_c, mbw, mbh, ns, nmb,
                                                                     lambda, d_info, d_c16, d_c4, d_c8);
    else
        k3_intra_analyse_kernel<false><<<blocks, K3_THREADS, 0, st>>>(d_y, d_u, d_v, pitch, pitchc, stride_y, stride_c, mbw, mbh, ns, nmb,
                                                                      lambda, d_info, d_c16, d_c4, nullptr);
    B2_CUDA_OK(cudaGetLastError());
    return 0;
}
