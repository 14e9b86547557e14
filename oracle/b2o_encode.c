/* b2o_encode.c -- ORACLE (test infrastructure only; see b2o.h).
 * Frame-level encode stage = everything x264_encoder_encode (av_encode.c:970) does per frame
 * up to, but excluding, entropy coding: motion search, intra analysis, mode decision,
 * transform/quant and decoder-identical reconstruction.  The CUDA engine's per-MB output
 * (b2_mbinfo_t, b2_mbcoef_t) and its reconstructed planes must equal this bit for bit. */
#include <stdlib.h>
#include <string.h>
#include "b2o.h"

static void copy_block(uint8_t *dst, int dp, const uint8_t *src, int sp, int w, int h)
{
    for (int y = 0; y < h; y++) memcpy(dst + (size_t)y * dp, src + (size_t)y * sp, w);
}

static void finish_cbp(b2_mbinfo_t *mi, uint32_t mask)
{
    int cbp = 0;
    if (mi->mb_type == B2_MB_I16x16) {
        if (mask & 0xffffu) cbp = 15;
    } else {
        for (int q = 0; q < 4; q++)
            if (mask & (0xfu << (4 * q))) cbp |= 1 << q;
    }
    if (mask & 0x00ff0000u) cbp |= 2 << 4;
    else if (mask & 0x06000000u) cbp |= 1 << 4;
    mi->cbp = (uint8_t)cbp;
    mi->nnz_mask = mask;
}

static uint32_t code_chroma(const b2o_params_t *prm, const b2o_frame_t *cur, b2o_frame_t *recon, int mbx, int mby,
                            int intra, b2_mbcoef_t *coef)
{
    int qpc = b2o_chroma_qp(prm->qp);
    size_t off = (size_t)(mby * 8) * cur->pitchc + mbx * 8;
    uint32_t m = b2o_code_chroma8x8(cur->u + off, cur->pitchc, recon->u + off, recon->pitchc, qpc, intra, 0, coef);
    m |= b2o_code_chroma8x8(cur->v + off, cur->pitchc, recon->v + off, recon->pitchc, qpc, intra, 1, coef);
    return m;
}

void b2o_recon_inter_mb(const b2o_params_t *prm, const b2o_frame_t *cur, const b2o_frame_t *ref,
                        b2o_frame_t *recon, int mbx, int mby, b2_mbinfo_t *mi, b2_mbcoef_t *coef)
{
    uint8_t *ry = recon->y + (size_t)(mby * 16) * recon->pitch + mbx * 16;
    const uint8_t *sy = cur->y + (size_t)(mby * 16) * cur->pitch + mbx * 16;
    size_t offc = (size_t)(mby * 8) * recon->pitchc + mbx * 8;
    memset(coef, 0, sizeof(*coef));
    for (int q = 0; q < 4; q++) {             /* inter prediction per 8x8 quadrant (all four vectors are equal for 16x16) */
        const b2_mv_t mv = b2o_quad_mv(mi, q);
        const int qx = (q & 1) * 8, qy = (q >> 1) * 8;
        b2o_mc_luma(ref->y, ref->pitch, mbx * 16 + qx, mby * 16 + qy, mv.x, mv.y, 8, 8, ry + qy * recon->pitch + qx, recon->pitch);
        b2o_mc_chroma(ref->u, ref->pitchc, mbx * 8 + qx / 2, mby * 8 + qy / 2, mv.x, mv.y, 4, 4,
                      recon->u + offc + (qy / 2) * recon->pitchc + qx / 2, recon->pitchc);
        b2o_mc_chroma(ref->v, ref->pitchc, mbx * 8 + qx / 2, mby * 8 + qy / 2, mv.x, mv.y, 4, 4,
                      recon->v + offc + (qy / 2) * recon->pitchc + qx / 2, recon->pitchc);
    }
    uint32_t mask = 0;
    /* transform size (row N1): like x264's non-RD analysis, the 8x8 transform is used when the 8x8-Hadamard cost of
     * the prediction error is below its 4x4-Hadamard cost; ry holds the motion-compensated prediction here */
    int t8 = prm->transform8x8 && b2o_sa8d16x16(sy, cur->pitch, ry, recon->pitch) < b2o_satd16x16(sy, cur->pitch, ry, recon->pitch);
    if (t8) {
        for (int q = 0; q < 4; q++) {
            int o = (q >> 1) * 8 * cur->pitch + (q & 1) * 8, orc = (q >> 1) * 8 * recon->pitch + (q & 1) * 8;
            mask |= (uint32_t)b2o_code_luma8x8(sy + o, cur->pitch, ry + orc, recon->pitch, prm->qp, 0, coef->blk[4 * q]) << (4 * q);
        }
        if (!(mask & 0xffffu)) t8 = 0;       /* transform_size_8x8_flag is only sent with coded luma: inferred 0 otherwise */
    } else {
        for (int b = 0; b < 16; b++) {
            int o = b2o_blk_y[b] * 4 * cur->pitch + b2o_blk_x[b] * 4;
            int orc = b2o_blk_y[b] * 4 * recon->pitch + b2o_blk_x[b] * 4;
            if (b2o_code_luma4x4(sy + o, cur->pitch, ry + orc, recon->pitch, prm->qp, 0, coef->blk[b])) mask |= 1u << b;
        }
    }
    mi->transform8x8 = (uint8_t)t8;
    mask |= code_chroma(prm, cur, recon, mbx, mby, 0, coef);
    finish_cbp(mi, mask);
}

void b2o_recon_intra_mb(const b2o_params_t *prm, const b2o_frame_t *cur, b2o_frame_t *recon,
                        int mbx, int mby, b2_mbinfo_t *mi, b2_mbcoef_t *coef)
{
    uint8_t *ry = recon->y + (size_t)(mby * 16) * recon->pitch + mbx * 16;
    const uint8_t *sy = cur->y + (size_t)(mby * 16) * cur->pitch + mbx * 16;
    int mba = b2o_mb_avail(mbx, mby, cur->mbw);
    uint32_t mask = 0;
    memset(coef, 0, sizeof(*coef));
    if (mi->mb_type == B2_MB_I16x16) {
        uint8_t pred[256];
        b2o_pred16x16(mi->i16_mode, ry, recon->pitch, mba, pred);
        copy_block(ry, recon->pitch, pred, 16, 16, 16);
        mask |= b2o_code_luma16x16(sy, cur->pitch, ry, recon->pitch, prm->qp, coef);
    } else if (mi->mb_type == B2_MB_I8x8) {
        for (int q = 0; q < 4; q++) {
            uint8_t pred[64];
            int mode = (mi->i8_modes >> (4 * q)) & 15;
            int o = (q >> 1) * 8 * cur->pitch + (q & 1) * 8;
            uint8_t *rb = ry + (q >> 1) * 8 * recon->pitch + (q & 1) * 8;
            b2o_pred8x8l(mode, rb, recon->pitch, b2o_blk8_avail(q, mba), pred);
            copy_block(rb, recon->pitch, pred, 8, 8, 8);
            mask |= (uint32_t)b2o_code_luma8x8(sy + o, cur->pitch, rb, recon->pitch, prm->qp, 1, coef->blk[4 * q]) << (4 * q);
            for (int k = 0; k < 4; k++) mi->i4_mode[4 * q + k] = (uint8_t)mode;
        }
        mi->transform8x8 = 1;
    } else {
        for (int b = 0; b < 16; b++) {
            uint8_t pred[16];
            int o = b2o_blk_y[b] * 4 * cur->pitch + b2o_blk_x[b] * 4;
            uint8_t *rb = ry + b2o_blk_y[b] * 4 * recon->pitch + b2o_blk_x[b] * 4;
            b2o_pred4x4(mi->i4_mode[b], rb, recon->pitch, b2o_blk_avail(b, mba), pred);
            copy_block(rb, recon->pitch, pred, 4, 4, 4);
            if (b2o_code_luma4x4(sy + o, cur->pitch, rb, recon->pitch, prm->qp, 1, coef->blk[b])) mask |= 1u << b;
        }
    }
    uint8_t pu[64], pv[64];
    size_t offc = (size_t)(mby * 8) * recon->pitchc + mbx * 8;
    b2o_pred8x8c(mi->chroma_mode, recon->u + offc, recon->pitchc, mba, pu);
    b2o_pred8x8c(mi->chroma_mode, recon->v + offc, recon->pitchc, mba, pv);
    copy_block(recon->u + offc, recon->pitchc, pu, 8, 8, 8);
    copy_block(recon->v + offc, recon->pitchc, pv, 8, 8, 8);
    mask |= code_chroma(prm, cur, recon, mbx, mby, 1, coef);
    finish_cbp(mi, mask);
}

void b2o_recon_intra_frame(int qp, const b2o_frame_t *cur, b2o_frame_t *recon, b2_mbinfo_t *info, b2_mbcoef_t *coef)
{
    b2o_params_t prm;
    memset(&prm, 0, sizeof(prm));
    prm.qp = qp;
    for (int mby = 0; mby < cur->mbh; mby++)
        for (int mbx = 0; mbx < cur->mbw; mbx++) {
            int i = mby * cur->mbw + mbx;
            if (info[i].mb_type != B2_MB_P16x16) b2o_recon_intra_mb(&prm, cur, recon, mbx, mby, &info[i], &coef[i]);
        }
}

void b2o_encode_frame(const b2o_params_t *prm, int frame_type,
                      const b2o_frame_t *cur, const b2o_frame_t *ref, b2o_frame_t *recon,
                      const b2_mv_t *prev_mv, b2_mbinfo_t *info, b2_mbcoef_t *coef)
{
    int n = cur->mbw * cur->mbh;
    int lambda = b2o_lambda(prm->qp);
    uint32_t *c16 = (uint32_t *)malloc(sizeof(uint32_t) * n), *c4 = (uint32_t *)malloc(sizeof(uint32_t) * n);
    uint32_t *cinter = (uint32_t *)malloc(sizeof(uint32_t) * n);
    uint32_t *c8 = prm->transform8x8 ? (uint32_t *)malloc(sizeof(uint32_t) * n) : NULL;
    b2_mv_t *mvf = (b2_mv_t *)malloc(sizeof(b2_mv_t) * n), *mvq = (b2_mv_t *)malloc(sizeof(b2_mv_t) * n);
    const int parts = prm->partitions && prm->subpel && frame_type == B2_FRAME_P;
    b2_mv_t (*mv4)[4] = parts ? (b2_mv_t (*)[4])malloc(sizeof(b2_mv_t) * 4 * n) : NULL;
    uint8_t *part = parts ? (uint8_t *)malloc(n) : NULL;
    memset(info, 0, sizeof(b2_mbinfo_t) * n);

    int do_intra = frame_type == B2_FRAME_I || prm->intra_in_p;
    if (do_intra) b2o_intra_analyse(cur, lambda, info, c16, c4, c8);
    if (frame_type == B2_FRAME_P) {
        if (parts && prm->partitions == 2) {
            uint32_t *cfull = (uint32_t *)malloc(sizeof(uint32_t) * n);
            b2o_me_parts_wide(cur, ref, prm->merange, prev_mv, lambda, 1, mvf, cfull, part, mv4, cinter);
            for (int i = 0; i < n; i++) mvq[i] = mv4[i][0];
            free(cfull);
        } else if (b2o_me_fullpel(cur, ref, prm->merange, prev_mv, lambda, mvf, cinter), parts) {
            b2o_me_subpel_part(cur, ref, mvf, prev_mv, lambda, part, mv4, cinter);
            for (int i = 0; i < n; i++) mvq[i] = mv4[i][0];
        } else if (prm->subpel) {
            b2o_me_subpel(cur, ref, mvf, prev_mv, lambda, mvq, cinter);
        } else {
            for (int i = 0; i < n; i++) {       /* SATD-domain cost at the full-pel winner */
                int mbx = i % cur->mbw, mby = i / cur->mbw;
                b2_mv_t p = {0, 0};
                if (prev_mv) p = prev_mv[i];
                mvq[i].x = (int16_t)(mvf[i].x * 4); mvq[i].y = (int16_t)(mvf[i].y * 4);
                const uint8_t *r = ref->y + (ptrdiff_t)(mby * 16 + mvf[i].y) * ref->pitch + mbx * 16 + mvf[i].x;
                cinter[i] = b2o_satd16x16(cur->y + (size_t)(mby * 16) * cur->pitch + mbx * 16, cur->pitch, r, ref->pitch)
                          + (uint32_t)lambda * (uint32_t)(b2o_mvbits(mvq[i].x - p.x) + b2o_mvbits(mvq[i].y - p.y));
            }
        }
    }
    /* decision */
    for (int i = 0; i < n; i++) {
        uint32_t ci = 0xffffffffu; int it = B2_MB_I16x16;
        if (do_intra) {
            ci = c16[i];
            if (c4[i] < ci) { ci = c4[i]; it = B2_MB_I4x4; }
            if (c8 && c8[i] < ci) { ci = c8[i]; it = B2_MB_I8x8; }
        }
        if (frame_type == B2_FRAME_P && !(do_intra && ci < cinter[i])) {
            info[i].mb_type = B2_MB_P16x16; info[i].mvx = mvq[i].x; info[i].mvy = mvq[i].y; info[i].cost = cinter[i];
            if (parts && part[i] != B2_PART_16x16) {
                info[i].part = part[i];
                for (int q = 1; q < 4; q++) info[i].mv8[q - 1] = mv4[i][q];
            }
        } else {
            info[i].mb_type = (uint8_t)it; info[i].mvx = info[i].mvy = 0; info[i].cost = ci;
        }
    }
    /* reconstruction, raster order (intra MBs read reconstructed left/top neighbours) */
    for (int mby = 0; mby < cur->mbh; mby++)
        for (int mbx = 0; mbx < cur->mbw; mbx++) {
            int i = mby * cur->mbw + mbx;
            if (info[i].mb_type == B2_MB_P16x16) b2o_recon_inter_mb(prm, cur, ref, recon, mbx, mby, &info[i], &coef[i]);
            else b2o_recon_intra_mb(prm, cur, recon, mbx, mby, &info[i], &coef[i]);
        }
    if (prm->deblock) b2o_deblock_frame(recon, info, prm->qp, prm->deblock_alpha, prm->deblock_beta);
    b2o_frame_extend(recon);
    free(c16); free(c4); free(cinter); free(mvf); free(mvq); free(c8); free(mv4); free(part);
}
