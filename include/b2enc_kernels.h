/*
 * b2enc_kernels.h -- kernel-level C-ABI entry points of libb2enc.so (host buffers in, host
 * buffers out, plain pointers and sizes).  They exist so that every CUDA kernel can be checked
 * bit-exactly against "the reference's linked C functions" (BASELINE.json north_star): in the
 * reference those are libx264's / libswscale's internal pixel, dct and quant functions reached
 * through av_encode.c:545 (sws_scale) and av_encode.c:970 (x264_encoder_encode).
 * All functions return 0 on success, a negative value on error (message on stderr), mirroring
 * the reference's int/NULL error convention (av_encode.c:385,409,416,433,973).
 */
#ifndef B2ENC_KERNELS_H
#define B2ENC_KERNELS_H
#include <stddef.h>
#include "b2enc_types.h"
#ifdef __cplusplus
extern "C" {
#endif

/* number of CUDA devices visible; <= 0 when the CUDA path cannot run (no fallback exists) */
int b2_device_count(void);

/* PCI bus id ("0000:1b:00.0") of a CUDA device, so that a host process can pin itself to the GPU's NUMA node before
 * allocating the pinned staging buffers */
int b2_device_pci_bus_id(int device, char *out, int len);

/* free / total memory of a CUDA device in bytes */
int b2_device_mem_info(int device, size_t *free_bytes, size_t *total_bytes);

/* K1: exhaustive full-pel SAD search (replaces the full-pel ME inside x264_encoder_encode,
 * av_encode.c:970).  cur_y/ref_y: [nframes][h][w] unpadded luma, w and h multiples of 16.
 * pmv: [nframes][mbh*mbw] quarter-pel predictors or NULL.  Outputs per MB, raster order.
 * If kernel_ms != NULL the kernel is re-run `iters` times and the mean device time of one
 * launch (CUDA events) is stored there. */
int b2k_me_fullpel(const uint8_t *cur_y, const uint8_t *ref_y, int w, int h, int nframes, int merange,
                   const b2_mv_t *pmv, int lambda, b2_mv_t *mv_out, uint32_t *cost_out,
                   int iters, float *kernel_ms);

/* K1 with lossless pruning (successive elimination: K1a block sums of the reference, then the same sweep over the lane-tasks
 * -- KS consecutive dy at one dx -- whose lower bound dist(sum(cur), [min, max of the block sums]) + mvcost does not exceed an
 * exactly evaluated cost).  Results are identical to b2k_me_fullpel's by construction; swept / all = candidate vectors that were
 * evaluated / that the exhaustive kernel evaluates.  kernel_ms: K1 alone; sums_ms: K1a alone. */
int b2k_me_fullpel_pruned(const uint8_t *cur_y, const uint8_t *ref_y, int w, int h, int nframes, int merange,
                          const b2_mv_t *pmv, int lambda, b2_mv_t *mv_out, uint32_t *cost_out, int iters, float *kernel_ms,
                          float *sums_ms, unsigned long long *swept_candidates, unsigned long long *all_candidates);
/* K1a alone on the padded (B2_PAD, replicated border) planes; out [nframes][rows][pitch] u32 (may be NULL to query the geometry):
 * position (Y,X) = min | max << 16 over rows Y..Y+ks-1 of S[.][X], S[Y][X] = sum of padded[Y..Y+15][X..X+15]; 0 | 0xffff where a
 * block leaves the allocation.  ks in {1, 3, 5} */
int b2k_block_sums(const uint8_t *y, int w, int h, int nframes, int ks, uint32_t *out, int *pitch_out, int *rows_out);
/* K8 (in-loop deblocking, H.264 8.7) alone on planes in the engine's padded layout: pitch = w + 2*B2_PAD,
 * pitchc = (w/2 + 2*B2_PADC + 15) & ~15, rows h + 2*B2_PAD / h/2 + 2*B2_PADC, nframes frames one after the other per plane;
 * w and h multiples of 16; info [nframes][mbh*mbw]; qp 0..51, offsets (slice_alpha_c0_offset_div2 / slice_beta_offset_div2)
 * -6..6.  All frames go through one launch and the planes are filtered in place; y == NULL only reports the shape.
 * Out (each may be NULL): wavefront 0 (row pipeline) / 1 (anti-diagonal wavefront), ncta = CTAs per frame actually launched,
 * rounds = rows / macroblocks of a diagonal per warp. */
int b2k_deblock(uint8_t *y, uint8_t *u, uint8_t *v, int w, int h, int nframes, int qp, int alpha_off, int beta_off,
                const b2_mbinfo_t *info, int *wavefront, int *ncta, int *rounds);
/* K7 (intra reconstruction on reconstructed neighbours, 8.3 / 8.5) and its cbp pass alone, in one launch, on planes in the
 * padded layout of b2k_deblock: cur_* the source, rec_* the reconstruction (inter macroblocks already reconstructed; read as
 * neighbours, never written); nframes frames one after the other; info / coef [nframes][mbh*mbw]; qp 10..51.
 * all_intra 1: the I-frame schedule (a cluster of up to 8 CTAs per frame), 0: the P-frame schedule (one CTA per frame).
 * Preconditions, as the engine leaves them after K5: intra records are zero apart from mb_type, i16_mode, chroma_mode, i4_mode,
 * i8_modes and cost -- in particular nnz_mask == 0, because K7 ORs its masks in -- and every mode is legal for the
 * neighbours available to its block (K7 does not check).  coef need not be cleared: K7 writes all 26 x 16 levels of an intra
 * macroblock.  Writes cbp, nnz_mask, and for I8x8 i4_mode and transform8x8, of intra records; leaves inter macroblocks alone.
 * rec_*, info and coef are updated in place (padding included); rec_y == NULL only reports the shape.  Refuses a picture whose
 * diagonal tables exceed the kernel's dynamic shared memory (mbw + 2*(mbh-1) > 3134 on a B200).
 * Out (each may be NULL): ncta = CTAs per frame, rounds = tasks of the longest diagonal per warp, dyn_smem = bytes per CTA. */
int b2k_intra_recon(const uint8_t *cur_y, const uint8_t *cur_u, const uint8_t *cur_v, uint8_t *rec_y, uint8_t *rec_u, uint8_t *rec_v,
                    int w, int h, int nframes, int qp, int all_intra, b2_mbinfo_t *info, b2_mbcoef_t *coef, int *ncta, int *rounds,
                    int *dyn_smem);
/* rows per lane-task of the pruned search for +-merange: 5 (+-32) or 3 (+-16) */
int b2_k1_prune_rows(int merange);

/* K1, partition variant (row N1, partitions = 2): best full-pel vector and cost of each of the nine shape parts per MB
 * (16x16 | 16x8 top,bottom | 8x16 left,right | four 8x8), outputs [nframes][mbs][9] */
int b2k_me_fullpel_parts(const uint8_t *cur_y, const uint8_t *ref_y, int w, int h, int nframes, int merange,
                         const b2_mv_t *pmv, int lambda, b2_mv_t *mv9_out, uint32_t *cost9_out, int iters, float *kernel_ms);

/* sustained VABSDIFF4 lane-instructions/s of the chip (roofline denominator of K1) */
double b2_bench_vabsdiff4_peak(int device, int outer, int reps, double *ms_best);

#ifdef __cplusplus
}
#endif
#endif
