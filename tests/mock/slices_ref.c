/*
 * slices_ref.c -- TEST INFRASTRUCTURE: the oracle (oracle/) with several row-aligned slices per picture.
 *
 * A slice is whole macroblock rows (b2_slice_row, include/b2enc_types.h) and intra prediction never reads across a slice
 * boundary, so the intra analysis and reconstruction of a slice are those of the unsliced oracle run on a picture that starts at
 * the slice's first row: a view of the same planes whose row 0 is that row.  Nothing else in the encode stage is slice-aware --
 * the motion search, sub-pel refinement and inter reconstruction read the reference wherever the vector points, and a view reads
 * exactly the samples the whole picture reads -- so an encoded frame is the slices encoded one by one (each into a scratch
 * frame, because a view's border extension would overwrite its neighbours), followed by the loop filter over the whole picture,
 * which runs across slice boundaries (disable_deblocking_filter_idc 0).
 *
 * With B2S_MOCK it also wraps the mock engine (tests/mock/mock_engine.c, compiled with b2o_encode_frame -> b2s_mock_encode_frame
 * and b2_engine_create -> b2s_mock_engine_create) so that the host pipeline sees cfg.slices honoured.
 */
#include <stdlib.h>
#include <string.h>
#include "b2o.h"

/* rows [r0, r0 + n) of f as a picture of their own */
static b2o_frame_t rows_view(const b2o_frame_t *f, int r0, int n)
{
    b2o_frame_t v = *f;
    v.h = v.h16 = 16 * n;
    v.mbh = n;
    v.y = f->y + (size_t)(16 * r0) * f->pitch;
    v.u = f->u + (size_t)(8 * r0) * f->pitchc;
    v.v = f->v + (size_t)(8 * r0) * f->pitchc;
    v.buf[0] = v.buf[1] = v.buf[2] = NULL;
    return v;
}

int b2s_slice_rows(int slices, int mbh, int *first)
{
    const int n = b2_slice_count(slices, mbh);
    for (int k = 0; k <= n; k++) first[k] = b2_slice_row(k, n, mbh);
    return n;
}

void b2s_intra_analyse(const b2o_frame_t *cur, int slices, int lambda, b2_mbinfo_t *info, uint32_t *c16, uint32_t *c4, uint32_t *c8)
{
    const int ns = b2_slice_count(slices, cur->mbh);
    for (int k = 0; k < ns; k++) {
        const int r0 = b2_slice_row(k, ns, cur->mbh), n = b2_slice_row(k + 1, ns, cur->mbh) - r0;
        const size_t o = (size_t)r0 * cur->mbw;
        const b2o_frame_t v = rows_view(cur, r0, n);
        b2o_intra_analyse(&v, lambda, info + o, c16 + o, c4 + o, c8 ? c8 + o : NULL);
    }
}

void b2s_recon_intra_frame(int qp, int slices, const b2o_frame_t *cur, b2o_frame_t *recon, b2_mbinfo_t *info, b2_mbcoef_t *coef)
{
    const int ns = b2_slice_count(slices, cur->mbh);
    for (int k = 0; k < ns; k++) {
        const int r0 = b2_slice_row(k, ns, cur->mbh), n = b2_slice_row(k + 1, ns, cur->mbh) - r0;
        const size_t o = (size_t)r0 * cur->mbw;
        const b2o_frame_t vc = rows_view(cur, r0, n);
        b2o_frame_t vr = rows_view(recon, r0, n);
        b2o_recon_intra_frame(qp, &vc, &vr, info + o, coef + o);
    }
}

static void copy_rows(uint8_t *dst, const uint8_t *src, int pitch, int w, int rows)
{
    for (int y = 0; y < rows; y++) memcpy(dst + (size_t)y * pitch, src + (size_t)y * pitch, (size_t)w);
}

int b2s_encode_frame(const b2o_params_t *prm, int slices, int frame_type, const b2o_frame_t *cur, const b2o_frame_t *ref,
                     b2o_frame_t *recon, const b2_mv_t *prev_mv, b2_mbinfo_t *info, b2_mbcoef_t *coef)
{
    const int ns = b2_slice_count(slices, cur->mbh);
    b2o_frame_t scratch;
    if (b2o_frame_alloc(&scratch, cur->w16, cur->h16)) return -1;
    b2o_params_t p = *prm;
    p.deblock = 0;                                           /* the filter runs once over the whole picture, below */
    for (int k = 0; k < ns; k++) {
        const int r0 = b2_slice_row(k, ns, cur->mbh), n = b2_slice_row(k + 1, ns, cur->mbh) - r0;
        const size_t o = (size_t)r0 * cur->mbw;
        const b2o_frame_t vc = rows_view(cur, r0, n);
        b2o_frame_t vref, vs = rows_view(&scratch, r0, n);
        if (ref) vref = rows_view(ref, r0, n);
        b2o_encode_frame(&p, frame_type, &vc, ref ? &vref : NULL, &vs, prev_mv ? prev_mv + o : NULL, info + o, coef + o);
        copy_rows(recon->y + (size_t)(16 * r0) * recon->pitch, vs.y, recon->pitch, cur->w16, 16 * n);
        copy_rows(recon->u + (size_t)(8 * r0) * recon->pitchc, vs.u, recon->pitchc, cur->w16 / 2, 8 * n);
        copy_rows(recon->v + (size_t)(8 * r0) * recon->pitchc, vs.v, recon->pitchc, cur->w16 / 2, 8 * n);
    }
    b2o_frame_free(&scratch);
    if (prm->deblock) b2o_deblock_frame(recon, info, prm->qp, prm->deblock_alpha, prm->deblock_beta);
    b2o_frame_extend(recon);
    return 0;
}

#ifdef B2S_MOCK
#include "b2enc_engine.h"
/* The mock engine builds its b2o_params_t without a slice count; the count of the engine being created is kept here.  The host
 * pipeline opens every engine of an encoder with the same cfg, and the tests run one encoder at a time. */
static int mock_slices = 1;
b2_engine_t *b2s_mock_engine_create(const b2_engine_cfg_t *cfg);
b2_engine_t *b2_engine_create(const b2_engine_cfg_t *cfg)
{
    if (cfg) __atomic_store_n(&mock_slices, cfg->slices, __ATOMIC_RELAXED);
    return b2s_mock_engine_create(cfg);
}
void b2s_mock_encode_frame(const b2o_params_t *prm, int frame_type, const b2o_frame_t *cur, const b2o_frame_t *ref, b2o_frame_t *recon,
                           const b2_mv_t *prev_mv, b2_mbinfo_t *info, b2_mbcoef_t *coef)
{
    b2s_encode_frame(prm, __atomic_load_n(&mock_slices, __ATOMIC_RELAXED), frame_type, cur, ref, recon, prev_mv, info, coef);
}
#endif
