/*
 * b2enc_engine.h -- C-ABI of the B200 encode-stage engine (libb2enc.so): the pixel-parallel part of
 * what the reference does per frame between av_encode.c:545 (sws_scale into pic_in) and the entropy
 * coder inside x264_encoder_encode (av_encode.c:970):
 *     convert -> full-pel SAD search -> sub-pel SATD refine -> intra analysis -> decision ->
 *     DCT/quant/dequant/IDCT/reconstruction -> border extension.
 * One engine = one GPU.  It encodes `slots` independent units (closed GOPs of one stream, or live
 * streams) in lock-step: every call advances all slots by one frame, so each kernel launch covers
 * slots x macroblocks.  Frames inside a closed GOP are a serial chain (P needs the previous
 * reconstruction); different GOPs / streams share nothing (SURVEY.md 8e), hence no collective.
 * Plain pointers and sizes only.  All int functions return 0 on success, <0 on error (stderr message).
 */
#ifndef B2ENC_ENGINE_H
#define B2ENC_ENGINE_H
#include <stddef.h>
#include "b2enc_types.h"
#ifdef __cplusplus
extern "C" {
#endif

typedef struct b2_engine b2_engine_t;

typedef struct {
    int device;        /* CUDA device ordinal                                             */
    int width, height; /* picture size (any; coded size is rounded up to 16)              */
    int slots;         /* units encoded in lock-step (closed GOPs or streams)             */
    int in_fmt;        /* B2_FMT_* layout of the raw input pictures                       */
    int in_ring;       /* raw input pictures kept resident per slot (>= 1)                */
    int merange;       /* 16 or 32: exhaustive search +-merange                           */
    int qp;            /* constant QP, 10..51                                             */
    int subpel;        /* 1: half + quarter-pel SATD refinement                           */
    int intra_in_p;    /* 1: intra/inter decision in P frames                             */
    int profile;       /* 1: record per-kernel CUDA-event timings (b2_engine_kernel_ms)   */
    int streams;       /* stream groups the slots are split into (0 = automatic); groups   */
                       /* run on separate CUDA streams so that their kernels overlap       */
    int deblock;       /* 1: in-loop deblocking filter (K8) on every reconstructed frame    */
    int transform8x8;  /* 1: adaptive 8x8 transform for inter macroblocks (SA8D < SATD), row N1 */
    int partitions;    /* inter partitions 16x8 / 8x16 / 8x8 (need subpel), row N1: 1 = refined per quadrant     */
                       /* within +-3/4 pel of the 16x16 vector, 2 = own exhaustive full-pel search per part      */
    int pack_levels;   /* 1: levels leave the GPU packed (only blocks with a non-zero level, K9):   */
                       /* b2_engine_packed* replace b2_engine_coef*, which then return NULL         */
    int deblock_alpha, deblock_beta;   /* loop-filter offsets (slice_alpha_c0_offset_div2 / slice_beta_offset_div2, -6..6) */
    int me_prune;      /* 1: lossless pruning of the exhaustive full-pel search (successive elimination: candidates whose      */
                       /* block-sum lower bound exceeds an exactly evaluated cost are skipped).  Vectors, costs and tie-break  */
                       /* are those of the exhaustive scan; the time is content dependent.  Used for merange 32 without the    */
                       /* wide partition search (partitions == 2); elsewhere the exhaustive kernel is the faster one and runs. */
    int slices;        /* row-aligned slices per picture (x264 i_slice_count; split: b2_slice_row, b2enc_types.h); 0 or 1: one. */
                       /* Intra analysis (K3) and reconstruction (K7) see no neighbour in another slice; K7 runs every   */
                       /* (frame, slice) as its own wavefront.  The loop filter (K8) crosses slice boundaries.             */
} b2_engine_cfg_t;

b2_engine_t *b2_engine_create(const b2_engine_cfg_t *cfg);      /* NULL on error */
void b2_engine_destroy(b2_engine_t *e);

/* tight byte size of one raw input picture in cfg.in_fmt */
size_t b2_engine_input_bytes(const b2_engine_t *e);
/* pinned host staging for (slot, ring position); fill it directly or through b2_engine_put_frame */
uint8_t *b2_engine_host_input(b2_engine_t *e, int slot, int ring);
/* copy a strided picture (plane pointers + strides as sws_scale takes them, av_encode.c:545) into
 * the pinned staging of (slot, ring); the source may be freed on return (cf. av_encode.c:550) */
int b2_engine_put_frame(b2_engine_t *e, int slot, int ring, const uint8_t *const src[4], const int stride[4]);
/* the same hand-over without the host copy: when the picture lives in page-locked memory (b2_picture_alloc, the mirror of
 * x264_picture_alloc av_encode.c:415) its planes are DMA'd straight into the device ring and the call returns once the
 * source has been read; the following b2_engine_h2d skips that entry.  Returns 0, 1 = source not page-locked (fall back to
 * b2_engine_put_frame), -1 = error.  May be called from another host thread than h2d/encode/d2h for a different ring position. */
int b2_engine_put_frame_direct(b2_engine_t *e, int slot, int ring, const uint8_t *const src[4], const int stride[4]);
/* GOP-streaming hand-over (used by b2_encoder_encode): one picture from ANY host memory into (slot, ring); returns as soon as
 * the source has been read (page-locked sources: DMA + wait; pageable ones: copy into a page-locked bounce buffer whose upload
 * completes behind the caller's back).  No b2_engine_h2d follows -- the next encode of the slot's group waits for the upload.
 * May run on another host thread than encode_group / d2h_group for ring entries that are not being encoded. */
int b2_engine_put_picture(b2_engine_t *e, int slot, int ring, const uint8_t *const src[4], const int stride[4]);
/* the same without waiting for the DMA of a page-locked source: returns a ticket (> 0) that b2_engine_put_wait blocks on before
 * the source may be overwritten; 0: the source has already been read; < 0: error */
long b2_engine_put_picture_async(b2_engine_t *e, int slot, int ring, const uint8_t *const src[4], const int stride[4]);
int b2_engine_put_wait(b2_engine_t *e, long ticket);
/* change cfg.in_fmt of an idle engine (the ring is re-allocated when the picture size differs) */
int b2_engine_set_input_format(b2_engine_t *e, int fmt);
/* async pinned-host -> device copy of ring position `ring` for slots [slot0, slot0+nslots) */
int b2_engine_h2d(b2_engine_t *e, int slot0, int nslots, int ring);
/* async: encode ring position `ring` of slots [0,nslots) as one frame each (B2_FRAME_I / B2_FRAME_P) */
int b2_engine_encode(b2_engine_t *e, int frame_type, int nslots, int ring);
/* stream groups: contiguous slot ranges with their own compute stream.  Groups may be advanced
 * independently (e.g. with staggered GOP phases so that only one group is in an I frame at a time). */
int b2_engine_groups(const b2_engine_t *e);
int b2_engine_group_range(const b2_engine_t *e, int group, int *slot0, int *nslots);
int b2_engine_encode_group(b2_engine_t *e, int group, int frame_type, int ring);
int b2_engine_d2h_group(b2_engine_t *e, int group);
/* group-level hand-off: result set (0/1) the group's last b2_engine_d2h_group copies into; whether that copy has landed
 * (1 yes, 0 not yet, <0 error) / wait for it (the thread sleeps); host views of a result set.  A set stays valid until the
 * group's next but one b2_engine_d2h_group. */
int b2_engine_group_result_set(const b2_engine_t *e, int group);
int b2_engine_group_done(b2_engine_t *e, int group, int set);
int b2_engine_group_wait(b2_engine_t *e, int group, int set);
const b2_mbinfo_t *b2_engine_info_set(b2_engine_t *e, int set, int slot);
/* cfg.pack_levels: the decisions cross PCIe as 24-byte records (b2_mbinfo_packed_t: everything the serial stage reads; not `cost`,
 * `i8_modes` or the intra analysis modes of macroblocks that ended up inter).  Every b2_engine_info* view expands them on first use;
 * this returns the records themselves. */
const b2_mbinfo_packed_t *b2_engine_info_packed_set(b2_engine_t *e, int set, int slot);
const uint8_t *b2_engine_packed_set(b2_engine_t *e, int set, int slot, size_t *bytes);
/* async device -> pinned-host copy of the last encode's per-MB results for slots [0,nslots) */
int b2_engine_d2h(b2_engine_t *e, int nslots);
int b2_engine_sync(b2_engine_t *e);
/* host views of the results fetched by the last b2_engine_d2h (valid until the next but one d2h) */
const b2_mbinfo_t *b2_engine_info(b2_engine_t *e, int slot);
const b2_mbcoef_t *b2_engine_coef(b2_engine_t *e, int slot);
size_t b2_engine_result_bytes(const b2_engine_t *e);           /* fixed D2H bytes per slot per frame (pack_levels: + the packed stream) */
/* cfg.pack_levels: the slot's level stream (layout: b2enc_types.h, b2_coef_present) and its size in bytes */
const uint8_t *b2_engine_packed(b2_engine_t *e, int slot, size_t *bytes);
const uint8_t *b2_engine_packed_ticket(b2_engine_t *e, int ticket, int slot, size_t *bytes);
long long b2_engine_packed_bytes_total(b2_engine_t *e);        /* packed bytes produced since creation (synchronises) */
/* pipelined consumption: the ticket of the last b2_engine_d2h stays valid until the next but one b2_engine_d2h, so
 * the host can entropy-code step t while the GPU already runs step t+1 */
int b2_engine_ticket(const b2_engine_t *e);
int b2_engine_wait_ticket(b2_engine_t *e, int ticket);         /* waits for that copy only, not for later GPU work */
const b2_mbinfo_t *b2_engine_info_ticket(b2_engine_t *e, int ticket, int slot);
const b2_mbcoef_t *b2_engine_coef_ticket(b2_engine_t *e, int ticket, int slot);

/* parity / debugging (synchronous): coded-size planes, tight layout */
int b2_engine_get_recon(b2_engine_t *e, int slot, uint8_t *y, uint8_t *u, uint8_t *v);
int b2_engine_get_cur(b2_engine_t *e, int slot, uint8_t *y, uint8_t *u, uint8_t *v);
enum { B2_STAGE_MV_FULL = 0, B2_STAGE_COST_FULL, B2_STAGE_MV_QPEL, B2_STAGE_COST_INTER, B2_STAGE_COST_I16, B2_STAGE_COST_I4 };
int b2_engine_get_stage(b2_engine_t *e, int slot, int what, void *out);   /* 4 bytes per MB */
void b2_engine_geometry(const b2_engine_t *e, int *mbw, int *mbh, int *w16, int *h16);

/* timing on the engine's compute stream (CUDA events) */
int b2_engine_timer_start(b2_engine_t *e);
int b2_engine_timer_stop(b2_engine_t *e, float *ms);            /* synchronises */
/* cfg.profile: accumulated device ms and launch count per kernel since the last reset.
 * which: 0 K0 convert, 1 K6 border(cur), 2 K1 full-pel, 3 K2 sub-pel, 4 K3 intra, 5 K5 decide+inter,
 *        6 K7 intra recon, 7 K6 border(recon), 8 K8 deblock, 9 K9 pack levels */
enum { B2_NKERNELS = 10 };
int b2_engine_kernel_ms(b2_engine_t *e, int which, double *ms_total, long *launches);
void b2_engine_profile_reset(b2_engine_t *e);
long b2_engine_launch_count(const b2_engine_t *e);              /* kernels launched since creation */
/* cfg.me_prune: candidate vectors the pruned search evaluated since creation and what the exhaustive search evaluates for the
 * same steps (executed vs algorithmic work, SURVEY.md 8d).  Synchronises the device.  -1 when pruning is off. */
int b2_engine_k1_stats(b2_engine_t *e, unsigned long long *swept, unsigned long long *all);

#ifdef __cplusplus
}
#endif
#endif
