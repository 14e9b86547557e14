/*
 * b2enc.h -- the DROP-IN BOUNDARY: C-ABI of libb2enc.so mirroring, call for call, the third-party
 * API subset that the reference's hot path uses (SURVEY.md 8b).  x264.h / swscale.h are not available
 * in this image, so mirror types are declared here with the field names the reference touches; a
 * maintainer switches av_encode.c over with the #define block shown in INTEGRATION.md.
 *
 *   reference call (av_encode.c)                         replacement
 *   ---------------------------------------------------  ---------------------------------------------
 *   sws_getContext(...)                      :427-430     b2_sws_getContext
 *   sws_scale(...)                           :545-547     b2_sws_scale
 *   sws_freeContext(...)                     :441         b2_sws_freeContext
 *   x264_param_default_preset(&p,preset,tune):384         b2_param_default_preset
 *   x264_param_apply_profile(&p,profile)     :403         b2_param_apply_profile
 *   x264_encoder_open(&p)                    :408         b2_encoder_open
 *   x264_picture_alloc(&pic,CSP_I420,w,h)    :415         b2_picture_alloc      (pinned host memory)
 *   x264_picture_clean(&pic)                 :442         b2_picture_clean
 *   x264_encoder_encode(h,&nal,&n,in,out)    :970,:1078   b2_encoder_encode
 *   x264_encoder_delayed_frames(h)           :1076        b2_encoder_delayed_frames
 *   x264_encoder_close(h)                    :443         b2_encoder_close
 *   MP4AddH264VideoTrack(.., profile, compat, level, 3) + MP4AddH264Sequence/PictureParameterSet
 *                                            :638-640,:703-727  b2_avcc_write   (the avcC record itself)
 *
 * Error convention = the reference's: int 0 / non-zero (or <0), NULL handles, message on stderr
 * (av_encode.c:385,404,409,416,433,973).  No CPU fallback exists: without a CUDA device
 * b2_encoder_open / b2_sws_getContext return NULL.
 */
#ifndef B2ENC_H
#define B2ENC_H
#include <stdint.h>
#include "b2enc_types.h"
#ifdef __cplusplus
extern "C" {
#endif

/* ---- libswscale subset ------------------------------------------------------------------------------*/
#define B2_SWS_FAST_BILINEAR 1
#define B2_SWS_HOST_OUTPUT 0x10000000    /* extension flag for b2_sws_getContext: always write the destination planes (see b2_sws_scale) */
typedef struct b2_sws_context b2_sws_context_t;
/* same-size conversion only (the reference never scales: av_encode.c:427-430); srcFormat = B2_FMT_*,
 * dstFormat must be B2_FMT_YUV420P.  NULL on error. */
b2_sws_context_t *b2_sws_getContext(int srcW, int srcH, int srcFormat, int dstW, int dstH, int dstFormat, int flags,
                                    void *srcFilter, void *dstFilter, const double *param);
/* whole frame per call (srcSliceY = 0, srcSliceH = srcH, as at av_encode.c:545-547); src has been read when it returns
 * (the reference frees it right away, :550).  The conversion itself runs on the GPU (kernel K0).
 * When dst are the planes of a b2_picture_alloc picture -- the reference's only use: x264.pic_in, :415, :545-547 -- the
 * conversion is DEFERRED into the b2_encoder_encode call that picture is handed to next (:970): the source is staged in
 * page-locked memory belonging to the picture, uploaded once, and K0 writes straight into the encoder's device planes.
 * The picture's host planes are NOT written in that form (the reference never reads them); pass B2_SWS_HOST_OUTPUT to
 * b2_sws_getContext, or any other destination memory, to get sws_scale's host-out behaviour (host -> GPU -> host round
 * trip).  Returns the height of the output slice, < 0 on error. */
int b2_sws_scale(b2_sws_context_t *c, const uint8_t *const src[], const int srcStride[], int srcSliceY, int srcSliceH,
                 uint8_t *const dst[], const int dstStride[]);
void b2_sws_freeContext(b2_sws_context_t *c);

/* ---- libx264 subset ---------------------------------------------------------------------------------*/
#define B2_CSP_I420 1
#define B2_TYPE_AUTO 0
#define B2_TYPE_IDR 1
#define B2_TYPE_P 3
#define B2_RC_CQP 0
#define B2_RC_CRF 1
enum { B2_NAL_SLICE = 1, B2_NAL_SLICE_IDR = 5, B2_NAL_SEI = 6, B2_NAL_SPS = 7, B2_NAL_PPS = 8, B2_NAL_FILLER = 12 };

typedef struct {
    /* fields the reference writes (av_encode.c:389-401) */
    int i_width, i_height;
    int b_annexb;                       /* 0: 4-byte big-endian length prefix per NAL (what the MP4 muxer needs) */
    int i_fps_num, i_fps_den;
    struct { int i_sar_width, i_sar_height; } vui;
    struct { int i_rc_method; float f_rf_constant; int i_qp_constant; } rc;
    /* extensions (not in the reference; defaults chosen by b2_param_default_preset) */
    int i_keyint_max;                   /* closed-GOP length                                    */
    int i_gop_slots;                    /* closed GOPs in flight per GPU, each on its own CUDA stream (default 32; 1 = zero delay) */
    int i_merange;                      /* 16 or 32                                             */
    int b_subpel;                       /* half + quarter-pel refinement                        */
    int b_intra_in_p;
    int i_device;                       /* CUDA device ordinal                                  */
    int i_csp_in;                       /* B2_FMT_* of the pictures handed to b2_encoder_encode */
    int b_deblocking_filter;            /* in-loop deblocking filter (x264 field of the same name; default 1) */
    int b_cabac;                        /* CABAC entropy coding (x264 field of the same name; default 1, cleared by
                                           profile "baseline" exactly like x264_param_apply_profile)             */
    int b_transform_8x8;                /* adaptive 8x8 transform (x264: analyse.b_transform_8x8; High profile;
                                           cleared by profiles "baseline" and "main")                            */
    int b_partitions;                   /* inter partitions 16x8 / 8x16 / 8x8 (x264: analyse.inter & X264_ANALYSE_PSUB16x16).
                                           1: refined per 8x8 quadrant within +-3/4 pel of the 16x16 vector; 2: every part gets
                                           its own exhaustive full-pel search (K1 partition variant); default 0              */
    int i_deblocking_filter_alphac0;    /* loop-filter offsets, x264 fields of the same names ([-6,6]; tune film sets -1:-1, */
    int i_deblocking_filter_beta;       /* as x264 does): slice_alpha_c0_offset_div2 / slice_beta_offset_div2               */
    int i_devices;                      /* GPUs one stream is spread over by closed GOP: GOP k is encoded on device
                                           i_device + k % i_devices; the output is byte-identical for every value.
                                           0 (default) = environment variable B2ENC_DEVICES, else 1                          */
    int b_me_prune;                     /* lossless pruning of the exhaustive full-pel search (successive elimination, the idea
                                           behind x264's me=esa): the stream is byte-identical with 0 and 1, only the time differs.
                                           Default 1; the environment variable B2ENC_ME_PRUNE=0/1 overrides it.  Takes effect for
                                           i_merange 32 (presets slow and up); at +-16 the exhaustive kernel is the faster one      */
    int i_slice_count;                  /* slices per picture (x264 field of the same name): row-aligned, slice k covers macroblock
                                           rows [(k mbh + n/2) / n, ((k+1) mbh + n/2) / n), n clamped to the picture's mbh rows.
                                           0 (default) = environment variable B2ENC_SLICES, else 1.  With i_gop_slots = 1 the
                                           slices of a picture are entropy-coded on several cores at once                          */
} b2_param_t;

typedef struct {
    int i_csp;
    int i_plane;
    int i_stride[4];
    uint8_t *plane[4];
} b2_image_t;

typedef struct {
    int i_type;                         /* in: B2_TYPE_AUTO (av_encode.c:543); out: slice type  */
    int64_t i_pts;                      /* in: av_encode.c:544; out: pts of the returned frame  */
    int64_t i_dts;                      /* out (av_encode.c:775)                                */
    int b_keyframe;                     /* out (av_encode.c:783)                                */
    b2_image_t img;
    void *opaque;
} b2_picture_t;

typedef struct {
    int i_ref_idc;
    int i_type;                         /* B2_NAL_* (av_encode.c:683-729)                       */
    int i_payload;                      /* bytes incl. the 4-byte length prefix / start code    */
    uint8_t *p_payload;                 /* all NALs of one frame are contiguous from nal[0].p_payload (av_encode.c:802) */
} b2_nal_t;

typedef struct b2_encoder b2_t;

int b2_param_default_preset(b2_param_t *p, const char *preset, const char *tune);
int b2_param_apply_profile(b2_param_t *p, const char *profile);
b2_t *b2_encoder_open(b2_param_t *p);
int b2_picture_alloc(b2_picture_t *pic, int i_csp, int i_width, int i_height);
void b2_picture_clean(b2_picture_t *pic);
/* returns the payload size of the returned frame (> 0), 0 when no frame is output yet, < 0 on error.
 * pic_in == NULL flushes (av_encode.c:1078).  NAL memory is owned by the encoder and valid until the
 * next call (the reference deep-copies it: av_encode.c:789-812). */
int b2_encoder_encode(b2_t *h, b2_nal_t **pp_nal, int *pi_nal, b2_picture_t *pic_in, b2_picture_t *pic_out);
int b2_encoder_delayed_frames(b2_t *h);
void b2_encoder_close(b2_t *h);

/* ---- MP4 side of the hand-off (SURVEY.md 8f row N3) -----------------------------------------------------*/
/* Writes the AVCDecoderConfigurationRecord (payload of the `avcC` box) for one SPS and one PPS NAL unit (without the
 * 4-byte length prefix: nal.p_payload + 4, nal.i_payload - 4 -- what the reference passes to
 * MP4AddH264SequenceParameterSet / MP4AddH264PictureParameterSet, av_encode.c:722, :727).  Replaces the libmp4v2 calls
 * av_encode.c:638-640 and :703-727.  Returns the record size, < 0 on error (bad NALs or cap too small). */
int b2_avcc_write(const uint8_t *sps, int sps_size, const uint8_t *pps, int pps_size, uint8_t *out, int cap);

#ifdef __cplusplus
}
#endif
#endif
