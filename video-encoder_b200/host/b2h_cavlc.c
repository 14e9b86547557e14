/*
 * b2h_cavlc.c -- H.264 Baseline (CAVLC) slice writer, SPS/PPS and NAL packing: the serial host
 * stage that follows the CUDA encode stage.  Stands where the entropy-coding tail of
 * x264_encoder_encode (av_encode.c:970) stands in the reference.  ITU-T H.264 7.3 / 9.1 / 9.2;
 * tables 9-4 (coded_block_pattern), 9-5 (coeff_token), 9-7/9-8/9-9 (total_zeros), 9-10
 * (run_before).  One slice per picture, one reference frame, POC type 2; the in-loop filter is signalled per
 * slice from b2h_seq_t (disable_deblocking_filter_idc, slice_alpha_c0_offset_div2, slice_beta_offset_div2; SURVEY.md 8f row N2).
 */
#include <stdlib.h>
#include <string.h>

#include "b2h_priv.h"

/* ---- parameter sets --------------------------------------------------------------------------*/
static int level_idc_for(int mbw, int mbh, int fps_num, int fps_den)
{
    /* smallest level whose MaxFS / MaxMBPS cover the stream (Table A-1) */
    /* level 1b (idc 11 + constraint_set3) and the levels that differ from their predecessor only in bit rate (2 vs 1.3, 4.1 vs 4)
     * are not listed: with constant QP there is no bit-rate bound to tell them apart, the smaller idc covers the stream */
    static const struct { int idc, fs; long mbps; } lv[] = {
        {10, 99, 1485}, {11, 396, 3000}, {12, 396, 6000}, {13, 396, 11880}, {21, 792, 19800}, {22, 1620, 20250},
        {30, 1620, 40500}, {31, 3600, 108000}, {32, 5120, 216000}, {40, 8192, 245760}, {42, 8704, 522240},
        {50, 22080, 589824}, {51, 36864, 983040}, {52, 36864, 2073600}};
    long fs = (long)mbw * mbh;
    double rate = fps_den > 0 ? (double)fps_num / fps_den : 30.0;
    for (unsigned i = 0; i < sizeof(lv) / sizeof(lv[0]); i++)
        if (fs <= lv[i].fs && fs * rate <= (double)lv[i].mbps) return lv[i].idc;
    return 52;
}

size_t b2h_write_sps(const b2h_seq_t *s, uint8_t *out, size_t cap)
{
    uint8_t rb[128];
    bs_t b;
    int mbw = (s->width + 15) >> 4, mbh = (s->height + 15) >> 4;
    bs_init(&b, rb, sizeof(rb));
    /* profile_idc / constraint flags: Constrained Baseline (CAVLC, 4x4), Main (CABAC) or High (8x8 transform);
     * the reference reads these three bytes back from the SPS NAL (av_encode.c:703-705) */
    const int profile = s->transform8x8 ? 100 : (s->cabac ? 77 : 66);
    bs_put(&b, 8, (uint32_t)profile);
    bs_put(&b, 8, profile == 66 ? 0xC0 : (profile == 77 ? 0x40 : 0x00));
    bs_put(&b, 8, (uint32_t)level_idc_for(mbw, mbh, s->fps_num, s->fps_den));
    bs_ue(&b, 0);                              /* seq_parameter_set_id                           */
    if (profile == 100) {
        bs_ue(&b, 1);                          /* chroma_format_idc 4:2:0                        */
        bs_ue(&b, 0); bs_ue(&b, 0);            /* bit_depth_luma_minus8, bit_depth_chroma_minus8 */
        bs_put(&b, 1, 0);                      /* qpprime_y_zero_transform_bypass_flag           */
        bs_put(&b, 1, 0);                      /* seq_scaling_matrix_present_flag                */
    }
    bs_ue(&b, 4);                              /* log2_max_frame_num_minus4 -> 8 bits            */
    bs_ue(&b, 2);                              /* pic_order_cnt_type 2: output order = decode order */
    bs_ue(&b, 1);                              /* max_num_ref_frames                             */
    bs_put(&b, 1, 0);                          /* gaps_in_frame_num_value_allowed_flag           */
    bs_ue(&b, (uint32_t)(mbw - 1));
    bs_ue(&b, (uint32_t)(mbh - 1));
    bs_put(&b, 1, 1);                          /* frame_mbs_only_flag                            */
    bs_put(&b, 1, 1);                          /* direct_8x8_inference_flag                      */
    int cr = (mbw * 16 - s->width) / 2, cbm = (mbh * 16 - s->height) / 2;
    if (cr || cbm) {
        bs_put(&b, 1, 1);
        bs_ue(&b, 0); bs_ue(&b, (uint32_t)cr); bs_ue(&b, 0); bs_ue(&b, (uint32_t)cbm);
    } else {
        bs_put(&b, 1, 0);
    }
    bs_put(&b, 1, 1);                          /* vui_parameters_present_flag                    */
    {
        int sar = s->sar_w > 0 && s->sar_h > 0;
        bs_put(&b, 1, (uint32_t)sar);          /* aspect_ratio_info_present_flag                 */
        if (sar) { bs_put(&b, 8, 255); bs_put(&b, 16, (uint32_t)s->sar_w); bs_put(&b, 16, (uint32_t)s->sar_h); }
        bs_put(&b, 1, 0);                      /* overscan_info_present_flag                     */
        bs_put(&b, 1, 0);                      /* video_signal_type_present_flag                 */
        bs_put(&b, 1, 0);                      /* chroma_loc_info_present_flag                   */
        int timing = s->fps_num > 0 && s->fps_den > 0;
        bs_put(&b, 1, (uint32_t)timing);
        if (timing) {
            bs_put(&b, 32, (uint32_t)s->fps_den);
            bs_put(&b, 32, (uint32_t)s->fps_num * 2u);
            bs_put(&b, 1, 1);                  /* fixed_frame_rate_flag                          */
        }
        bs_put(&b, 1, 0);                      /* nal_hrd_parameters_present_flag                */
        bs_put(&b, 1, 0);                      /* vcl_hrd_parameters_present_flag                */
        bs_put(&b, 1, 0);                      /* pic_struct_present_flag                        */
        bs_put(&b, 1, 1);                      /* bitstream_restriction_flag                     */
        bs_put(&b, 1, 1);                      /* motion_vectors_over_pic_boundaries_flag        */
        bs_ue(&b, 0); bs_ue(&b, 0);            /* max_bytes_per_pic_denom, max_bits_per_mb_denom */
        bs_ue(&b, 9); bs_ue(&b, 9);            /* log2_max_mv_length_horizontal / vertical       */
        bs_ue(&b, 0);                          /* max_num_reorder_frames                         */
        bs_ue(&b, 1);                          /* max_dec_frame_buffering                        */
    }
    bs_trailing(&b);
    return b.overflow ? 0 : nal_pack(3, B2H_NAL_SPS, rb, b.pos, out, cap);
}

size_t b2h_write_pps(const b2h_seq_t *s, uint8_t *out, size_t cap)
{
    uint8_t rb[32];
    bs_t b;
    bs_init(&b, rb, sizeof(rb));
    bs_ue(&b, 0); bs_ue(&b, 0);                /* pps id, sps id                                  */
    bs_put(&b, 1, s->cabac ? 1 : 0);           /* entropy_coding_mode_flag                        */
    bs_put(&b, 1, 0);                          /* bottom_field_pic_order_in_frame_present_flag    */
    bs_ue(&b, 0);                              /* num_slice_groups_minus1                         */
    bs_ue(&b, 0); bs_ue(&b, 0);                /* num_ref_idx_l0/l1_default_active_minus1         */
    bs_put(&b, 1, 0); bs_put(&b, 2, 0);        /* weighted_pred_flag, weighted_bipred_idc         */
    bs_se(&b, s->qp - 26);                     /* pic_init_qp_minus26                             */
    bs_se(&b, 0);                              /* pic_init_qs_minus26                             */
    bs_se(&b, 0);                              /* chroma_qp_index_offset                          */
    bs_put(&b, 1, 1);                          /* deblocking_filter_control_present_flag          */
    bs_put(&b, 1, 0);                          /* constrained_intra_pred_flag                     */
    bs_put(&b, 1, 0);                          /* redundant_pic_cnt_present_flag                  */
    if (s->transform8x8) {
        bs_put(&b, 1, 1);                      /* transform_8x8_mode_flag                         */
        bs_put(&b, 1, 0);                      /* pic_scaling_matrix_present_flag                 */
        bs_se(&b, 0);                          /* second_chroma_qp_index_offset                   */
    }
    bs_trailing(&b);
    return b.overflow ? 0 : nal_pack(3, B2H_NAL_PPS, rb, b.pos, out, cap);
}

/* ---- CAVLC tables ------------------------------------------------------------------------------*/
/* index [table][4*total_coeff + trailing_ones]; table 0: 0<=nC<2, 1: 2<=nC<4, 2: 4<=nC<8, 3: 8<=nC */
static const uint8_t coeff_token_len[4][4 * 17] = {
    {1, 0, 0, 0, 6, 2, 0, 0, 8, 6, 3, 0, 9, 8, 7, 5, 10, 9, 8, 6, 11, 10, 9, 7, 13, 11, 10, 8, 13, 13, 11, 9,
     13, 13, 13, 10, 14, 14, 13, 11, 14, 14, 14, 13, 15, 15, 14, 14, 15, 15, 15, 14, 16, 15, 15, 15, 16, 16, 16, 15,
     16, 16, 16, 16, 16, 16, 16, 16},
    {2, 0, 0, 0, 6, 2, 0, 0, 6, 5, 3, 0, 7, 6, 6, 4, 8, 6, 6, 4, 8, 7, 7, 5, 9, 8, 8, 6, 11, 9, 9, 6,
     11, 11, 11, 7, 12, 11, 11, 9, 12, 12, 12, 11, 12, 12, 12, 11, 13, 13, 13, 12, 13, 13, 13, 13, 13, 14, 13, 13,
     14, 14, 14, 13, 14, 14, 14, 14},
    {4, 0, 0, 0, 6, 4, 0, 0, 6, 5, 4, 0, 6, 5, 5, 4, 7, 5, 5, 4, 7, 5, 5, 4, 7, 6, 6, 4, 7, 6, 6, 4,
     8, 7, 7, 5, 8, 8, 7, 6, 9, 8, 8, 7, 9, 9, 8, 8, 9, 9, 9, 8, 10, 9, 9, 9, 10, 10, 10, 10,
     10, 10, 10, 10, 10, 10, 10, 10},
    {6, 0, 0, 0, 6, 6, 0, 0, 6, 6, 6, 0, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6,
     6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6, 6,
     6, 6, 6, 6, 6, 6, 6, 6}};
static const uint8_t coeff_token_bits[4][4 * 17] = {
    {1, 0, 0, 0, 5, 1, 0, 0, 7, 4, 1, 0, 7, 6, 5, 3, 7, 6, 5, 3, 7, 6, 5, 4, 15, 6, 5, 4, 11, 14, 5, 4,
     8, 10, 13, 4, 15, 14, 9, 4, 11, 10, 13, 12, 15, 14, 9, 12, 11, 10, 13, 8, 15, 1, 9, 12, 11, 14, 13, 8,
     7, 10, 9, 12, 4, 6, 5, 8},
    {3, 0, 0, 0, 11, 2, 0, 0, 7, 7, 3, 0, 7, 10, 9, 5, 7, 6, 5, 4, 4, 6, 5, 6, 7, 6, 5, 8, 15, 6, 5, 4,
     11, 14, 13, 4, 15, 10, 9, 4, 11, 14, 13, 12, 8, 10, 9, 8, 15, 14, 13, 12, 11, 10, 9, 12, 7, 11, 6, 8,
     9, 8, 10, 1, 7, 6, 5, 4},
    {15, 0, 0, 0, 15, 14, 0, 0, 11, 15, 13, 0, 8, 12, 14, 12, 15, 10, 11, 11, 11, 8, 9, 10, 9, 14, 13, 9, 8, 10, 9, 8,
     15, 14, 13, 13, 11, 14, 10, 12, 15, 10, 13, 12, 11, 14, 9, 12, 8, 10, 13, 8, 13, 7, 9, 12, 9, 12, 11, 10,
     5, 8, 7, 6, 1, 4, 3, 2},
    {3, 0, 0, 0, 0, 1, 0, 0, 4, 5, 6, 0, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22, 23, 24, 25, 26, 27,
     28, 29, 30, 31, 32, 33, 34, 35, 36, 37, 38, 39, 40, 41, 42, 43, 44, 45, 46, 47, 48, 49, 50, 51, 52, 53, 54, 55,
     56, 57, 58, 59, 60, 61, 62, 63}};
static const uint8_t chroma_dc_coeff_token_len[4 * 5] = {2, 0, 0, 0, 6, 1, 0, 0, 6, 6, 3, 0, 6, 7, 7, 6, 6, 8, 8, 7};
static const uint8_t chroma_dc_coeff_token_bits[4 * 5] = {1, 0, 0, 0, 7, 1, 0, 0, 4, 6, 1, 0, 3, 3, 2, 5, 2, 3, 2, 0};

/* [total_coeff-1][total_zeros] */
static const uint8_t total_zeros_len[15][16] = {
    {1, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 9},
    {3, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 6, 6, 6, 6},
    {4, 3, 3, 3, 4, 4, 3, 3, 4, 5, 5, 6, 5, 6},
    {5, 3, 4, 4, 3, 3, 3, 4, 3, 4, 5, 5, 5},
    {4, 4, 4, 3, 3, 3, 3, 3, 4, 5, 4, 5},
    {6, 5, 3, 3, 3, 3, 3, 3, 4, 3, 6},
    {6, 5, 3, 3, 3, 2, 3, 4, 3, 6},
    {6, 4, 5, 3, 2, 2, 3, 3, 6},
    {6, 6, 4, 2, 2, 3, 2, 5},
    {5, 5, 3, 2, 2, 2, 4},
    {4, 4, 3, 3, 1, 3},
    {4, 4, 2, 1, 3},
    {3, 3, 1, 2},
    {2, 2, 1},
    {1, 1}};
static const uint8_t total_zeros_bits[15][16] = {
    {1, 3, 2, 3, 2, 3, 2, 3, 2, 3, 2, 3, 2, 3, 2, 1},
    {7, 6, 5, 4, 3, 5, 4, 3, 2, 3, 2, 3, 2, 1, 0},
    {5, 7, 6, 5, 4, 3, 4, 3, 2, 3, 2, 1, 1, 0},
    {3, 7, 5, 4, 6, 5, 4, 3, 3, 2, 2, 1, 0},
    {5, 4, 3, 7, 6, 5, 4, 3, 2, 1, 1, 0},
    {1, 1, 7, 6, 5, 4, 3, 2, 1, 1, 0},
    {1, 1, 5, 4, 3, 3, 2, 1, 1, 0},
    {1, 1, 1, 3, 3, 2, 2, 1, 0},
    {1, 0, 1, 3, 2, 1, 1, 1},
    {1, 0, 1, 3, 2, 1, 1},
    {0, 1, 1, 2, 1, 3},
    {0, 1, 1, 1, 1},
    {0, 1, 1, 1},
    {0, 1, 1},
    {0, 1}};
static const uint8_t chroma_dc_total_zeros_len[3][4] = {{1, 2, 3, 3}, {1, 2, 2, 0}, {1, 1, 0, 0}};
static const uint8_t chroma_dc_total_zeros_bits[3][4] = {{1, 1, 1, 0}, {1, 1, 0, 0}, {1, 0, 0, 0}};
/* [min(zeros_left,7)-1][run_before] */
static const uint8_t run_len[7][16] = {
    {1, 1}, {1, 2, 2}, {2, 2, 2, 2}, {2, 2, 2, 3, 3}, {2, 2, 3, 3, 3, 3}, {2, 3, 3, 3, 3, 3, 3},
    {3, 3, 3, 3, 3, 3, 3, 4, 5, 6, 7, 8, 9, 10, 11}};
static const uint8_t run_bits[7][16] = {
    {1, 0}, {1, 1, 0}, {3, 2, 1, 0}, {3, 2, 1, 1, 0}, {3, 2, 3, 2, 1, 0}, {3, 0, 1, 3, 2, 5, 4},
    {7, 6, 5, 4, 3, 2, 1, 1, 1, 1, 1, 1, 1, 1, 1}};

/* Table 9-4: codeNum -> coded_block_pattern (chroma_format_idc 1), intra4x4 / inter */
static const uint8_t cbp_from_code_intra[48] = {47, 31, 15, 0, 23, 27, 29, 30, 7, 11, 13, 14, 39, 43, 45, 46,
                                                16, 3, 5, 10, 12, 19, 21, 26, 28, 35, 37, 42, 44, 1, 2, 4,
                                                8, 17, 18, 20, 24, 6, 9, 22, 25, 32, 33, 34, 36, 40, 38, 41};
static const uint8_t cbp_from_code_inter[48] = {0, 16, 1, 2, 4, 8, 32, 3, 5, 10, 12, 15, 47, 7, 11, 13,
                                                14, 6, 9, 31, 35, 37, 42, 44, 33, 34, 36, 40, 39, 43, 45, 46,
                                                17, 18, 20, 24, 19, 21, 26, 28, 23, 27, 29, 30, 22, 25, 38, 41};

const uint8_t b2h_blk_x[16] = {0, 1, 0, 1, 2, 3, 2, 3, 0, 1, 0, 1, 2, 3, 2, 3};
const uint8_t b2h_blk_y[16] = {0, 0, 1, 1, 0, 0, 1, 1, 2, 2, 3, 3, 2, 2, 3, 3};
#define blk_x b2h_blk_x
#define blk_y b2h_blk_y

/* exported for the table self-test (tests/test_cavlc_tables.py) */
const uint8_t *b2h_table(int which, int *rows, int *cols)
{
    switch (which) {
    case 0: *rows = 4; *cols = 68; return &coeff_token_len[0][0];
    case 1: *rows = 4; *cols = 68; return &coeff_token_bits[0][0];
    case 2: *rows = 1; *cols = 20; return chroma_dc_coeff_token_len;
    case 3: *rows = 1; *cols = 20; return chroma_dc_coeff_token_bits;
    case 4: *rows = 15; *cols = 16; return &total_zeros_len[0][0];
    case 5: *rows = 15; *cols = 16; return &total_zeros_bits[0][0];
    case 6: *rows = 3; *cols = 4; return &chroma_dc_total_zeros_len[0][0];
    case 7: *rows = 3; *cols = 4; return &chroma_dc_total_zeros_bits[0][0];
    case 8: *rows = 7; *cols = 16; return &run_len[0][0];
    case 9: *rows = 7; *cols = 16; return &run_bits[0][0];
    case 10: *rows = 1; *cols = 48; return cbp_from_code_intra;
    case 11: *rows = 1; *cols = 48; return cbp_from_code_inter;
    default: *rows = *cols = 0; return NULL;
    }
}

b2h_entropy_t *b2h_entropy_create(int mbw, int mbh)
{
    b2h_entropy_t *e = (b2h_entropy_t *)calloc(1, sizeof(*e));
    if (!e) return NULL;
    e->mbw = mbw; e->mbh = mbh;
    size_t n = (size_t)mbw * mbh;
    e->nnz_y = (uint8_t *)malloc(n * 16);
    e->nnz_c[0] = (uint8_t *)malloc(n * 4);
    e->nnz_c[1] = (uint8_t *)malloc(n * 4);
    e->i4 = (int8_t *)malloc(n * 16);
    e->ref4 = (int8_t *)malloc(n * 16);
    e->mv4 = (b2_mv_t *)malloc(n * 16 * sizeof(b2_mv_t));
    e->mbf = (uint8_t *)calloc(n, 1); e->cbp = (uint8_t *)calloc(n, 1); e->cmode = (uint8_t *)calloc(n, 1);
    e->mvd[0] = (uint8_t *)calloc(n, 16); e->mvd[1] = (uint8_t *)calloc(n, 16);
    e->rbsp_cap = n * 2048 + 4096;
    e->rbsp = (uint8_t *)malloc(e->rbsp_cap);
    if (!e->nnz_y || !e->nnz_c[0] || !e->nnz_c[1] || !e->i4 || !e->ref4 || !e->mv4 || !e->rbsp || !e->mbf || !e->cbp || !e->cmode ||
        !e->mvd[0] || !e->mvd[1]) {
        b2h_entropy_destroy(e);
        return NULL;
    }
    for (int i = 0; i < 48; i++) {
        e->cbp_code_intra[cbp_from_code_intra[i]] = (uint8_t)i;
        e->cbp_code_inter[cbp_from_code_inter[i]] = (uint8_t)i;
    }
    return e;
}

void b2h_entropy_destroy(b2h_entropy_t *e)
{
    if (!e) return;
    free(e->nnz_y); free(e->nnz_c[0]); free(e->nnz_c[1]); free(e->i4); free(e->ref4); free(e->mv4); free(e->rbsp);
    free(e->mbf); free(e->cbp); free(e->cmode); free(e->mvd[0]); free(e->mvd[1]);
    free(e);
}

/* ---- residual_block_cavlc (7.3.5.3.2 / 9.2) ----------------------------------------------------*/
/* l[0..maxn) in scan order; nC < 0 selects the chroma DC tables.  Returns total_coeff. */
static int write_residual(bs_t *b, const int16_t *l, int maxn, int nC)
{
    int level[16], run[16];
    int total = 0, t1 = 0, last = -1, zeros = 0;
    /* walk from the highest frequency down: level[0] is the last non-zero coefficient */
    for (int i = maxn - 1; i >= 0; i--) {
        if (l[i]) {
            if (last < 0) last = i;
            level[total] = l[i];
            run[total] = 0;
            total++;
        } else if (total) {
            run[total - 1]++;      /* zeros preceding (in scan order) the previously found coeff */
        }
    }
    if (total) zeros = last + 1 - total;
    for (int i = 0; i < total && i < 3; i++) {
        if (level[i] == 1 || level[i] == -1) t1++;
        else break;
    }
    if (nC < 0) {
        bs_put(b, chroma_dc_coeff_token_len[4 * total + t1], chroma_dc_coeff_token_bits[4 * total + t1]);
    } else {
        int tab = nC < 2 ? 0 : nC < 4 ? 1 : nC < 8 ? 2 : 3;
        bs_put(b, coeff_token_len[tab][4 * total + t1], coeff_token_bits[tab][4 * total + t1]);
    }
    if (!total) return 0;
    for (int i = 0; i < t1; i++) bs_put(b, 1, level[i] < 0);
    int suffix_len = (total > 10 && t1 < 3) ? 1 : 0;
    for (int i = t1; i < total; i++) {
        int lv = level[i];
        int code = lv > 0 ? 2 * lv - 2 : -2 * lv - 1;
        if (i == t1 && t1 < 3) code -= 2;
        if (suffix_len == 0) {
            if (code < 14) {
                bs_put(b, code + 1, 1);
            } else if (code < 30) {
                bs_put(b, 15, 1); bs_put(b, 4, (uint32_t)(code - 14));
            } else {
                bs_put(b, 16, 1); bs_put(b, 12, (uint32_t)(code - 30));
            }
        } else {
            if (code < (15 << suffix_len)) {
                bs_put(b, (code >> suffix_len) + 1, 1);
                bs_put(b, suffix_len, (uint32_t)code & ((1u << suffix_len) - 1));
            } else {
                bs_put(b, 16, 1); bs_put(b, 12, (uint32_t)(code - (15 << suffix_len)));
            }
        }
        if (suffix_len == 0) suffix_len = 1;
        if (abs(lv) > (3 << (suffix_len - 1)) && suffix_len < 6) suffix_len++;
    }
    if (total < maxn) {
        if (nC < 0) bs_put(b, chroma_dc_total_zeros_len[total - 1][zeros], chroma_dc_total_zeros_bits[total - 1][zeros]);
        else bs_put(b, total_zeros_len[total - 1][zeros], total_zeros_bits[total - 1][zeros]);
    }
    int zleft = zeros;
    for (int i = 0; i < total - 1 && zleft > 0; i++) {
        int zi = (zleft > 7 ? 7 : zleft) - 1;
        bs_put(b, run_len[zi][run[i]], run_bits[zi][run[i]]);
        zleft -= run[i];
    }
    return total;
}

/* ---- neighbour helpers ---------------------------------------------------------------------------*/
/* y0: first block row of the slice (blocks above it are in another slice) */
static inline int pred_nc(const uint8_t *map, int stride, int x, int y, int y0)
{
    int hasA = x > 0, hasB = y > y0;
    int nA = hasA ? map[y * stride + x - 1] : 0, nB = hasB ? map[(y - 1) * stride + x] : 0;
    if (hasA && hasB) return (nA + nB + 1) >> 1;
    return hasA ? nA : (hasB ? nB : 0);
}

void b2h_slice_header(bs_t *b, const b2h_seq_t *s, int is_p, int frame_num, int idr_pic_id, int first_mb)
{
    bs_ue(b, (uint32_t)first_mb);                  /* first_mb_in_slice                   */
    bs_ue(b, is_p ? 5 : 7);                        /* slice_type: all slices P / all I    */
    bs_ue(b, 0);                                   /* pic_parameter_set_id                */
    bs_put(b, 8, (uint32_t)frame_num & 255u);      /* frame_num, log2_max_frame_num = 8   */
    if (!is_p) bs_ue(b, (uint32_t)idr_pic_id & 0xffffu);
    if (is_p) {
        bs_put(b, 1, 0);                           /* num_ref_idx_active_override_flag    */
        bs_put(b, 1, 0);                           /* ref_pic_list_modification_flag_l0   */
        bs_put(b, 1, 0);                           /* adaptive_ref_pic_marking_mode_flag  */
    } else {
        bs_put(b, 1, 0);                           /* no_output_of_prior_pics_flag        */
        bs_put(b, 1, 0);                           /* long_term_reference_flag            */
    }
    if (s->cabac && is_p) bs_ue(b, 0);             /* cabac_init_idc                      */
    bs_se(b, 0);                                   /* slice_qp_delta                      */
    if (s->deblock) {
        bs_ue(b, 0);                               /* disable_deblocking_filter_idc = 0   */
        bs_se(b, s->deblock_alpha);                /* slice_alpha_c0_offset_div2          */
        bs_se(b, s->deblock_beta);                 /* slice_beta_offset_div2              */
    } else {
        bs_ue(b, 1);                               /* disable_deblocking_filter_idc = 1   */
    }
}

void b2h_info_pack(const b2_mbinfo_t *info, b2_mbinfo_packed_t *packed, int n)
{
    for (int i = 0; i < n; i++) packed[i] = b2_mbinfo_pack(&info[i]);
}
void b2h_info_unpack(const b2_mbinfo_packed_t *packed, b2_mbinfo_t *info, int n)
{
    for (int i = 0; i < n; i++) b2_mbinfo_unpack(&packed[i], &info[i]);
}

/* ---- slice ---------------------------------------------------------------------------------------*/
const int16_t b2h_zero_levels[64] = {0};

static size_t write_slice(b2h_entropy_t *e, const b2h_seq_t *s, int frame_type, int frame_num, int idr_pic_id, int first_row,
                          int nrows, const b2_mbinfo_t *info, b2h_levels_t *lv, uint8_t *out, size_t cap);

size_t b2h_write_slice_rows(b2h_entropy_t *e, const b2h_seq_t *s, int frame_type, int frame_num, int idr_pic_id, int first_row,
                            int nrows, const b2_mbinfo_t *info, const b2_mbcoef_t *coef, uint8_t *out, size_t cap)
{
    b2h_levels_t lv = {coef, NULL, 0, 0};
    return write_slice(e, s, frame_type, frame_num, idr_pic_id, first_row, nrows, info, &lv, out, cap);
}

size_t b2h_write_slice_rows_packed(b2h_entropy_t *e, const b2h_seq_t *s, int frame_type, int frame_num, int idr_pic_id, int first_row,
                                   int nrows, const b2_mbinfo_t *info, const uint8_t *packed, size_t packed_bytes, uint8_t *out,
                                   size_t cap)
{
    /* the stream holds the whole picture: the slice's first macroblock follows the present blocks of the ones in front of it */
    size_t pos = 0;
    for (int i = 0; first_row > 0 && i < first_row * e->mbw; i++) pos += 32u * (size_t)__builtin_popcount(b2_coef_present(&info[i]));
    b2h_levels_t lv = {NULL, packed, pos, packed_bytes};
    return write_slice(e, s, frame_type, frame_num, idr_pic_id, first_row, nrows, info, &lv, out, cap);
}

size_t b2h_write_slice(b2h_entropy_t *e, const b2h_seq_t *s, int frame_type, int frame_num, int idr_pic_id,
                       const b2_mbinfo_t *info, const b2_mbcoef_t *coef, uint8_t *out, size_t cap)
{
    return b2h_write_slice_rows(e, s, frame_type, frame_num, idr_pic_id, 0, e->mbh, info, coef, out, cap);
}

size_t b2h_write_slice_packed(b2h_entropy_t *e, const b2h_seq_t *s, int frame_type, int frame_num, int idr_pic_id,
                              const b2_mbinfo_t *info, const uint8_t *packed, size_t packed_bytes, uint8_t *out, size_t cap)
{
    return b2h_write_slice_rows_packed(e, s, frame_type, frame_num, idr_pic_id, 0, e->mbh, info, packed, packed_bytes, out, cap);
}

static size_t write_slice(b2h_entropy_t *e, const b2h_seq_t *s, int frame_type, int frame_num, int idr_pic_id, int first_row,
                          int nrows, const b2_mbinfo_t *info, b2h_levels_t *lv, uint8_t *out, size_t cap)
{
    bs_t bs, *b = &bs;
    const int mbw = e->mbw, is_p = frame_type == B2_FRAME_P;
    const int ys = 4 * mbw, cs = 2 * mbw;
    if (first_row < 0 || nrows < 1 || first_row + nrows > e->mbh) return 0;
    e->row0 = first_row;
    const int y4top = 4 * first_row, y2top = 2 * first_row;
    if (s->cabac) return b2h_write_slice_cabac(e, s, frame_type, frame_num, idr_pic_id, nrows, info, lv, out, cap);
    bs_init(b, e->rbsp, e->rbsp_cap);
    b2h_slice_header(b, s, is_p, frame_num, idr_pic_id, first_row * mbw);

    /* slice_data() */
    int skip_run = 0;
    for (int mby = first_row; mby < first_row + nrows; mby++)
        for (int mbx = 0; mbx < mbw; mbx++) {
            const int mi = mby * mbw + mbx;
            const b2_mbinfo_t *m = &info[mi];
            const int16_t *cblk[B2_COEF_BLOCKS];
            b2h_levels_mb(lv, m, mi, cblk);
            const int cbp_l = m->cbp & 15, cbp_c = m->cbp >> 4;
            /* reset this MB's neighbour state; filled in below as blocks are coded */
            for (int r = 0; r < 4; r++) { memset(e->nnz_y + (mby * 4 + r) * ys + mbx * 4, 0, 4); memset(e->i4 + (mby * 4 + r) * ys + mbx * 4, 2, 4); }
            for (int p = 0; p < 2; p++)
                for (int r = 0; r < 2; r++) memset(e->nnz_c[p] + (mby * 2 + r) * cs + mbx * 2, 0, 2);

            if (m->mb_type == B2_MB_P16x16) {
                if (m->part == B2_PART_16x16 && m->cbp == 0) {
                    const b2_mv_t skipmv = b2h_skip_mv(e, mbx, mby);
                    if (m->mvx == skipmv.x && m->mvy == skipmv.y) {                          /* P_Skip */
                        b2h_fill_mv(e, mbx * 4, mby * 4, 4, 4, skipmv, 0);
                        skip_run++;
                        continue;
                    }
                }
                bs_ue(b, (uint32_t)skip_run); skip_run = 0;
                bs_ue(b, m->part);                             /* mb_type P_L0_16x16 / P_L0_L0_16x8 / P_L0_L0_8x16 / P_8x8 */
                if (m->part == B2_PART_8x8)
                    for (int k = 0; k < 4; k++) bs_ue(b, 0);   /* sub_mb_type P_L0_8x8 */
                {
                    int px, py, pw, ph, dir;
                    const int np = b2h_part_geom(m->part, 0, &px, &py, &pw, &ph, &dir);
                    for (int a = 0; a < np; a++) {             /* mvd_l0 per partition; ref_idx is not sent with one reference */
                        b2h_part_geom(m->part, a, &px, &py, &pw, &ph, &dir);
                        const b2_mv_t mv = b2h_mb_mv(m, px, py);
                        const b2_mv_t mvp = b2h_mv_pred(e, mbx * 4 + px, mby * 4 + py, pw, dir);
                        bs_se(b, mv.x - mvp.x);
                        bs_se(b, mv.y - mvp.y);
                        b2h_fill_mv(e, mbx * 4 + px, mby * 4 + py, pw, ph, mv, 0);
                    }
                }
                bs_ue(b, e->cbp_code_inter[m->cbp]);
                if (cbp_l && s->transform8x8) bs_put(b, 1, m->transform8x8 != 0);     /* transform_size_8x8_flag */
            } else {
                { b2_mv_t z = {0, 0}; b2h_fill_mv(e, mbx * 4, mby * 4, 4, 4, z, -1); }   /* inter MBs fill their blocks partition by partition */
                if (is_p) { bs_ue(b, (uint32_t)skip_run); skip_run = 0; }
                if (m->mb_type != B2_MB_I16x16) {
                    const int i8 = m->mb_type == B2_MB_I8x8;
                    bs_ue(b, is_p ? 5 : 0);                    /* I_NxN */
                    if (s->transform8x8) bs_put(b, 1, (uint32_t)i8);                  /* transform_size_8x8_flag */
                    for (int k = 0; k < 16; k += i8 ? 4 : 1) {
                        int x = mbx * 4 + blk_x[k], y = mby * 4 + blk_y[k];
                        int pred = 2;
                        if (x > 0 && y > y4top) {
                            int a = e->i4[y * ys + x - 1], bb = e->i4[(y - 1) * ys + x];
                            pred = a < bb ? a : bb;
                        }
                        int mode = m->i4_mode[k];
                        if (mode == pred) bs_put(b, 1, 1);
                        else bs_put(b, 4, (uint32_t)(mode < pred ? mode : mode - 1));   /* flag 0 + rem (3 bits) */
                        e->i4[y * ys + x] = (int8_t)mode;
                        if (i8) e->i4[y * ys + x + 1] = e->i4[(y + 1) * ys + x] = e->i4[(y + 1) * ys + x + 1] = (int8_t)mode;
                    }
                    bs_ue(b, m->chroma_mode);
                    bs_ue(b, e->cbp_code_intra[m->cbp]);
                } else {
                    bs_ue(b, (uint32_t)((is_p ? 5 : 0) + 1 + m->i16_mode + 4 * cbp_c + (cbp_l ? 12 : 0)));
                    bs_ue(b, m->chroma_mode);
                }
            }
            if (m->cbp || m->mb_type == B2_MB_I16x16) bs_se(b, 0);       /* mb_qp_delta */

            /* residual() */
            if (m->mb_type == B2_MB_I16x16) {
                write_residual(b, cblk[24], 16, pred_nc(e->nnz_y, ys, mbx * 4, mby * 4, y4top));
                if (cbp_l)
                    for (int k = 0; k < 16; k++) {
                        int x = mbx * 4 + blk_x[k], y = mby * 4 + blk_y[k];
                        e->nnz_y[y * ys + x] = (uint8_t)write_residual(b, cblk[k] + 1, 15, pred_nc(e->nnz_y, ys, x, y, y4top));
                    }
            } else if (m->transform8x8 && s->transform8x8) {
                /* 8x8 transform with CAVLC (7.3.5.3.2): the 64 levels are split into four interleaved 4x4 blocks */
                for (int k = 0; k < 16; k++) {
                    if (!(cbp_l & (1 << (k >> 2)))) continue;
                    int x = mbx * 4 + blk_x[k], y = mby * 4 + blk_y[k];
                    int16_t l4[16];
                    const int16_t *l8 = cblk[k & ~3];
                    for (int i = 0; i < 16; i++) l4[i] = l8[4 * i + (k & 3)];
                    e->nnz_y[y * ys + x] = (uint8_t)write_residual(b, l4, 16, pred_nc(e->nnz_y, ys, x, y, y4top));
                }
            } else {
                for (int k = 0; k < 16; k++) {
                    if (!(cbp_l & (1 << (k >> 2)))) continue;
                    int x = mbx * 4 + blk_x[k], y = mby * 4 + blk_y[k];
                    e->nnz_y[y * ys + x] = (uint8_t)write_residual(b, cblk[k], 16, pred_nc(e->nnz_y, ys, x, y, y4top));
                }
            }
            if (cbp_c) {
                write_residual(b, cblk[25], 4, -1);
                write_residual(b, cblk[25] + 4, 4, -1);
                if (cbp_c == 2)
                    for (int p = 0; p < 2; p++)
                        for (int k = 0; k < 4; k++) {
                            int x = mbx * 2 + (k & 1), y = mby * 2 + (k >> 1);
                            e->nnz_c[p][y * cs + x] =
                                (uint8_t)write_residual(b, cblk[16 + 4 * p + k] + 1, 15, pred_nc(e->nnz_c[p], cs, x, y, y2top));
                        }
            }
        }
    if (is_p && skip_run) bs_ue(b, (uint32_t)skip_run);
    bs_trailing(b);
    if (b->overflow) return 0;
    return nal_pack(is_p ? 2 : 3, is_p ? B2H_NAL_SLICE : B2H_NAL_IDR, e->rbsp, b->pos, out, cap);
}
