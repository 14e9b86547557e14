/*
 * b2h_entropy.h -- host-side serial stage: H.264 slice writer (CAVLC, b2h_cavlc.c, or CABAC,
 * b2h_cabac.c) + SPS/PPS + NAL packing.  In the reference this stage is the tail of x264_encoder_encode (av_encode.c:970)
 * and is left on the host by BASELINE.json's north_star ("entropy coding and muxing left on
 * the serial stage").  libx264 is not available in this image, so a minimal writer is part of
 * the product; its output is pinned by decoding it with libavcodec's H.264 decoder.
 */
#ifndef B2H_ENTROPY_H
#define B2H_ENTROPY_H
#include <stddef.h>
#include <stdint.h>
#include "b2enc_types.h"
#ifdef __cplusplus
extern "C" {
#endif

enum { B2H_NAL_SLICE = 1, B2H_NAL_IDR = 5, B2H_NAL_SEI = 6, B2H_NAL_SPS = 7, B2H_NAL_PPS = 8 };

typedef struct {
    int width, height;          /* display size; coded size is rounded up to 16 */
    int fps_num, fps_den;
    int sar_w, sar_h;
    int qp;                     /* pic_init_qp (all slices use slice_qp_delta = 0) */
    int deblock;                /* 1: disable_deblocking_filter_idc = 0 (filter on), 0: idc = 1            */
    int cabac;                  /* 1: entropy_coding_mode_flag = 1 (CABAC, Main profile), 0: CAVLC (Constrained Baseline) */
    int transform8x8;           /* 1: transform_8x8_mode_flag = 1 (High profile)                            */
    int deblock_alpha, deblock_beta;   /* slice_alpha_c0_offset_div2 / slice_beta_offset_div2 (-6..6)          */
} b2h_seq_t;

typedef struct b2h_entropy b2h_entropy_t;   /* per-encoder scratch (neighbour maps) */

b2h_entropy_t *b2h_entropy_create(int mbw, int mbh);
void b2h_entropy_destroy(b2h_entropy_t *e);

/* Each writer emits ONE complete NAL unit (header byte + RBSP with emulation prevention, no
 * start code / length prefix) into out[0..cap) and returns its size, or 0 on overflow. */
size_t b2h_write_sps(const b2h_seq_t *s, uint8_t *out, size_t cap);
size_t b2h_write_pps(const b2h_seq_t *s, uint8_t *out, size_t cap);
/* the whole picture as one slice; info / coef [mbh * mbw] */
size_t b2h_write_slice(b2h_entropy_t *e, const b2h_seq_t *s, int frame_type /* B2_FRAME_* */, int frame_num,
                       int idr_pic_id, const b2_mbinfo_t *info, const b2_mbcoef_t *coef,
                       uint8_t *out, size_t cap);
/* same, reading the levels from the engine's packed stream (b2_engine_packed, layout in b2enc_types.h) */
size_t b2h_write_slice_packed(b2h_entropy_t *e, const b2h_seq_t *s, int frame_type, int frame_num, int idr_pic_id,
                              const b2_mbinfo_t *info, const uint8_t *packed, size_t packed_bytes, uint8_t *out, size_t cap);
/* the slice of macroblock rows [first_row, first_row + nrows) of a picture cut into row-aligned slices (b2_slice_row,
 * b2enc_types.h); info / coef / packed hold the whole picture.  A writer reads nothing above first_row, so writers with their
 * own scratch (b2h_entropy_create) may write the slices of one picture at the same time. */
size_t b2h_write_slice_rows(b2h_entropy_t *e, const b2h_seq_t *s, int frame_type, int frame_num, int idr_pic_id, int first_row,
                            int nrows, const b2_mbinfo_t *info, const b2_mbcoef_t *coef, uint8_t *out, size_t cap);
size_t b2h_write_slice_rows_packed(b2h_entropy_t *e, const b2h_seq_t *s, int frame_type, int frame_num, int idr_pic_id,
                                   int first_row, int nrows, const b2_mbinfo_t *info, const uint8_t *packed, size_t packed_bytes,
                                   uint8_t *out, size_t cap);

/* the 24-byte decision records that cross PCIe (b2_mbinfo_packed_t, include/b2enc_types.h) <-> b2_mbinfo_t, n macroblocks */
void b2h_info_pack(const b2_mbinfo_t *info, b2_mbinfo_packed_t *packed, int n);
void b2h_info_unpack(const b2_mbinfo_packed_t *packed, b2_mbinfo_t *info, int n);

#ifdef __cplusplus
}
#endif
#endif
