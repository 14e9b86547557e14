// b2_internal.h -- internal launcher prototypes (device pointers + stream); not part of the C-ABI.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/b2enc_types.h"

// padded layout of the device planes of a coded size w16 x h16: luma pitch / rows, chroma pitch (a multiple of 16) / rows
inline void b2_padded_layout(int w16, int h16, int *pitch, int *rows, int *pitchc, int *rowsc)
{
    *pitch = w16 + 2 * B2_PAD; *rows = h16 + 2 * B2_PAD;
    *pitchc = (w16 / 2 + 2 * B2_PADC + 15) & ~15; *rowsc = h16 / 2 + 2 * B2_PADC;
}

int b2_make_plane_tmap(CUtensorMap *tm, const void *base, int pitch, int rows, int nplanes, int bw, int bh);
int b2_launch_extend_border(uint8_t *d_planes, int pitch, int rows, int nplanes, int pad, int iw, int ih,
                            cudaStream_t st);
// all three planes of `nframes` frames in one launch (luma pad B2_PAD, chroma pad B2_PADC, interior = coded size)
int b2_launch_extend_border_yuv(uint8_t *d_y, uint8_t *d_u, uint8_t *d_v, int pitch, int rows, int pitchc, int rowsc,
                                size_t stride_y, size_t stride_c, int w16, int h16, int nframes, cudaStream_t st);
extern "C" int b2_k1_window_box(int R, int *bw, int *bh);
extern "C" int b2_k1_strip_mbs(int R);                    // macroblocks per K1 strip: the current-tile box is {16 * this, 16, 1}
int b2_launch_me_fullpel(int R, const CUtensorMap *tm_cur, const CUtensorMap *tm_ref, int mbw, int mbh,
                         int nframes, const b2_mv_t *d_pmv, int lambda, b2_mv_t *d_mv, uint32_t *d_cost,
                         b2_mv_t *d_mv9 /* NULL, or [nmb][9] best vector of every shape part */, uint32_t *d_cost9, cudaStream_t st);

// pruned search (successive elimination, lossless): K1a = min | max over `ks` rows of the 16x16 block sums of the reference planes
// (one u32 per position), then K1 over the surviving lane-tasks only
int b2_make_plane_tmap32(CUtensorMap *tm, const void *base, int pitch, int rows, int nplanes, int bw);   // u32 planes, box {bw, 1, 1}
extern "C" int b2_k1_prune_rows(int R);
extern "C" int b2_k1_mm_box(int R);
extern "C" long long b2_k1_candidates(int R, int mbw, int mbh, int nframes);
int b2_launch_block_sums(int ks, const uint8_t *d_planes, int pitch, int rows, int nplanes, uint32_t *d_mm /* [nplanes][rows][pitch] */,
                         cudaStream_t st);
int b2_launch_me_fullpel_pruned(int R, const CUtensorMap *tm_cur, const CUtensorMap *tm_ref, const CUtensorMap *tm_mm, int mbw, int mbh,
                                int nframes, const b2_mv_t *d_pmv, int lambda, b2_mv_t *d_mv, uint32_t *d_cost,
                                unsigned long long *d_swept /* NULL, or += candidates evaluated */, cudaStream_t st);

int b2_launch_convert(int fmt, const uint8_t *d_in, size_t in_stride, uint8_t *d_y, uint8_t *d_u, uint8_t *d_v, int pitch,
                      int pitchc, size_t stride_y, size_t stride_c, int w, int h, int nframes, cudaStream_t st);
int b2_launch_me_subpel(const uint8_t *d_cur, const uint8_t *d_ref, int pitch, size_t plane_stride, int mbw, int mbh,
                        int nframes, const b2_mv_t *d_mv_full, const b2_mv_t *d_pmv, int lambda, int subpel,
                        b2_mv_t *d_mv_out, uint32_t *d_cost_out, uint8_t *d_pred_out, uint8_t *d_part_out /* NULL: 16x16 only */,
                        b2_mv_t *d_mv8_out /* [nmb][3] */, const b2_mv_t *d_mv9 /* NULL, or K1<PART>'s vectors: wide partition search */,
                        const uint32_t *d_cost9, cudaStream_t st);
int b2_launch_intra_analyse(const uint8_t *d_y, const uint8_t *d_u, const uint8_t *d_v, int pitch, int pitchc,
                            size_t stride_y, size_t stride_c, int mbw, int mbh, int nframes, int lambda,
                            b2_mbinfo_t *d_info, uint32_t *d_c16, uint32_t *d_c4, uint32_t *d_c8 /* NULL: no I8x8 analysis */,
                            cudaStream_t st);
int b2_launch_decide_inter(const uint8_t *const cur[3], const uint8_t *const ref[3], uint8_t *const rec[3], int pitch,
                           int pitchc, size_t stride_y, size_t stride_c, int mbw, int mbh, int nframes, int is_p,
                           int do_intra, int qp, const b2_mv_t *d_mvq, const uint32_t *d_cost_inter, const uint32_t *d_c16,
                           const uint32_t *d_c4, const uint32_t *d_c8, b2_mbinfo_t *d_info, b2_mbcoef_t *d_coef, b2_mv_t *d_prev_mv,
                           const uint8_t *d_pred_y, int transform8x8, const uint8_t *d_part, const b2_mv_t *d_mv8, cudaStream_t st);
// K7's launch shape for frames of mbw x mbh macroblocks: ncta = CTAs per frame (one cluster; 1 unless all_intra), rounds =
// (macroblock, luma | chroma) tasks of the longest anti-diagonal per warp, dyn_smem = dynamic shared memory of one CTA
void b2_intra_recon_shape(int mbw, int mbh, int all_intra, int *ncta, int *rounds, int *dyn_smem);
// refuses (-1, before any launch) a picture whose diagonal tables exceed the kernel's dynamic shared memory (ndiag > 3134)
int b2_launch_intra_recon(const uint8_t *const cur[3], uint8_t *const rec[3], int pitch, int pitchc, size_t stride_y,
                          size_t stride_c, int mbw, int mbh, int nframes, int qp, int all_intra, b2_mbinfo_t *d_info,
                          b2_mbcoef_t *d_coef, cudaStream_t st);
int b2_lambda_for_qp(int qp);
// K8's launch shape for `nframes` frames of mbw x mbh macroblocks: wavefront 0 = row pipeline, 1 = anti-diagonal wavefront;
// ncta = CTAs per frame (one cluster); rounds = rows (row pipeline) / macroblocks of one diagonal (wavefront) per warp.  Above
// 8 CTAs of rows it allows the non-portable cluster size on the current device; where that is refused it reports 8 CTAs.
void b2_deblock_shape(int mbw, int mbh, int nframes, int *wavefront, int *ncta, int *rounds);
int b2_launch_deblock(uint8_t *const rec[3], int pitch, int pitchc, size_t stride_y, size_t stride_c, int mbw, int mbh,
                      int nframes, int qp, int alpha_off, int beta_off, const b2_mbinfo_t *d_info,
                      int *d_flags /* [nframes][8] cross-CTA progress flags (scratch) */, cudaStream_t st);
// K9: pack the non-zero level blocks of every frame (k9a, compute stream) and copy exactly the used bytes to pinned host memory (k9b)
int b2_pack_chunks(int nmb);               // chunks per frame: d_chunk_cnt holds nframes x this many counters (scratch)
int b2_launch_pack_levels(const b2_mbinfo_t *d_info, const b2_mbcoef_t *d_coef, uint8_t *d_packed, size_t packed_stride,
                          uint32_t *d_nblocks, unsigned long long *d_cum_bytes, uint32_t *d_chunk_cnt,
                          b2_mbinfo_packed_t *d_pinfo /* [nframes][nmb] 24-byte decision records for the copy-out */, int nmb, int nframes,
                          cudaStream_t st);
int b2_launch_pack_copy_out(const uint8_t *d_packed, size_t packed_stride, const uint32_t *d_nblocks, uint8_t *h_packed,
                            uint32_t *h_nblocks, int nframes, cudaStream_t st);
