// b2_kernel_api.cu -- kernel-level C-ABI (include/b2enc_kernels.h): host buffers in/out.
#include "b2_common.cuh"
#include "b2_internal.h"
#include "../../include/b2enc_kernels.h"

extern "C" int b2_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

// free / total device memory in bytes (b2_encoder_open sizes its GOP slots with it)
extern "C" int b2_device_mem_info(int device, size_t *free_bytes, size_t *total_bytes)
{
    int prev = 0;
    cudaGetDevice(&prev);
    if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); return -1; }
    size_t f = 0, t = 0;
    const cudaError_t r = cudaMemGetInfo(&f, &t);
    cudaSetDevice(prev);
    if (r != cudaSuccess) { cudaGetLastError(); return -1; }
    if (free_bytes) *free_bytes = f;
    if (total_bytes) *total_bytes = t;
    return 0;
}

namespace {
struct DevBuf {
    void *p = nullptr;
    ~DevBuf() { if (p) cudaFree(p); }
    int alloc(size_t n) { return cudaMalloc(&p, n) == cudaSuccess ? 0 : -1; }
};

// upload [n][h][w] unpadded planes into a padded stack and replicate the border
int upload_padded(DevBuf &buf, const uint8_t *host, int w, int h, int n, int pad, int *pitch, int *rows)
{
    *pitch = w + 2 * pad; *rows = h + 2 * pad;
    if (buf.alloc((size_t)*pitch * *rows * n)) { fprintf(stderr, "b2enc: cudaMalloc failed\n"); return -1; }
    for (int i = 0; i < n; i++) {
        uint8_t *dst = (uint8_t *)buf.p + (size_t)i * *pitch * *rows + (size_t)pad * *pitch + pad;
        B2_CUDA_OK(cudaMemcpy2D(dst, *pitch, host + (size_t)i * w * h, w, w, h, cudaMemcpyHostToDevice));
    }
    return b2_launch_extend_border((uint8_t *)buf.p, *pitch, *rows, n, pad, w, h, 0);
}
}  // namespace

struct PruneOut { unsigned long long *swept, *all; float *sums_ms; };      // non-NULL: run the pruned search (K1a + K1 over survivors)
static int me_fullpel_impl(const uint8_t *cur_y, const uint8_t *ref_y, int w, int h, int nframes, int merange, const b2_mv_t *pmv,
                           int lambda, b2_mv_t *mv_out, uint32_t *cost_out, b2_mv_t *mv9_out, uint32_t *cost9_out, int iters,
                           float *kernel_ms, const PruneOut *prune = nullptr);

extern "C" int b2k_me_fullpel_pruned(const uint8_t *cur_y, const uint8_t *ref_y, int w, int h, int nframes, int merange,
                                     const b2_mv_t *pmv, int lambda, b2_mv_t *mv_out, uint32_t *cost_out, int iters, float *kernel_ms,
                                     float *sums_ms, unsigned long long *swept_candidates, unsigned long long *all_candidates)
{
    unsigned long long sw = 0, al = 0;
    float sm = 0;
    const PruneOut po = {&sw, &al, &sm};
    const int r = me_fullpel_impl(cur_y, ref_y, w, h, nframes, merange, pmv, lambda, mv_out, cost_out, nullptr, nullptr, iters, kernel_ms, &po);
    if (swept_candidates) *swept_candidates = sw;
    if (all_candidates) *all_candidates = al;
    if (sums_ms) *sums_ms = sm;
    return r;
}

// K1a alone: (min | max << 16) over `ks` rows of the 16x16 block sums of `nframes` w x h planes after padding by B2_PAD with
// replicated borders; out: [nframes][rows][pitch] u32.  ks = 1 gives the plain block sums in both halves.
extern "C" int b2k_block_sums(const uint8_t *y, int w, int h, int nframes, int ks, uint32_t *out, int *pitch_out, int *rows_out)
{
    DevBuf d_ref, d_mm;
    int pitch, rows;
    if (upload_padded(d_ref, y, w, h, nframes, B2_PAD, &pitch, &rows)) return -1;
    if (pitch_out) *pitch_out = pitch;
    if (rows_out) *rows_out = rows;
    if (!out) return 0;
    const size_t n = (size_t)pitch * rows * nframes;
    if (d_mm.alloc(n * 4)) return -1;
    B2_CUDA_OK(cudaMemset(d_mm.p, 0, n * 4));
    if (b2_launch_block_sums(ks, (const uint8_t *)d_ref.p, pitch, rows, nframes, (uint32_t *)d_mm.p, 0)) return -1;
    B2_CUDA_OK(cudaMemcpy(out, d_mm.p, n * 4, cudaMemcpyDeviceToHost));
    return 0;
}

// K8 alone: the planes go to the device as they are (padding included), are filtered in one launch and come back whole, so
// that a caller can see any store outside the picture
extern "C" int b2k_deblock(uint8_t *y, uint8_t *u, uint8_t *v, int w, int h, int nframes, int qp, int alpha_off, int beta_off,
                           const b2_mbinfo_t *info, int *wavefront, int *ncta, int *rounds)
{
    if ((w & 15) || (h & 15) || w <= 0 || h <= 0 || nframes <= 0 || qp < 0 || qp > 51 || alpha_off < -6 || alpha_off > 6 ||
        beta_off < -6 || beta_off > 6) {
        fprintf(stderr, "b2enc: b2k_deblock needs w,h multiples of 16, qp 0..51, offsets -6..6\n");
        return -1;
    }
    const int mbw = w / 16, mbh = h / 16;
    int wf, nc, rd;
    b2_deblock_shape(mbw, mbh, nframes, &wf, &nc, &rd);
    if (wavefront) *wavefront = wf;
    if (ncta) *ncta = nc;
    if (rounds) *rounds = rd;
    if (!y) return 0;
    if (!u || !v || !info) return -1;
    int pitch, rows, pitchc, rowsc;
    b2_padded_layout(w, h, &pitch, &rows, &pitchc, &rowsc);
    const size_t ny = (size_t)pitch * rows * nframes, nc_bytes = (size_t)pitchc * rowsc * nframes;
    const size_t ni = (size_t)mbw * mbh * nframes * sizeof(b2_mbinfo_t);
    DevBuf d_y, d_u, d_v, d_info;
    if (d_y.alloc(ny) || d_u.alloc(nc_bytes) || d_v.alloc(nc_bytes) || d_info.alloc(ni)) { fprintf(stderr, "b2enc: cudaMalloc failed\n"); return -1; }
    B2_CUDA_OK(cudaMemcpy(d_y.p, y, ny, cudaMemcpyHostToDevice));
    B2_CUDA_OK(cudaMemcpy(d_u.p, u, nc_bytes, cudaMemcpyHostToDevice));
    B2_CUDA_OK(cudaMemcpy(d_v.p, v, nc_bytes, cudaMemcpyHostToDevice));
    B2_CUDA_OK(cudaMemcpy(d_info.p, info, ni, cudaMemcpyHostToDevice));
    uint8_t *const rec[3] = {(uint8_t *)d_y.p, (uint8_t *)d_u.p, (uint8_t *)d_v.p};
    if (b2_launch_deblock(rec, pitch, pitchc, (size_t)pitch * rows, (size_t)pitchc * rowsc, mbw, mbh, nframes, qp, alpha_off, beta_off,
                          (const b2_mbinfo_t *)d_info.p, nullptr, 0))
        return -1;
    B2_CUDA_OK(cudaDeviceSynchronize());
    B2_CUDA_OK(cudaMemcpy(y, d_y.p, ny, cudaMemcpyDeviceToHost));
    B2_CUDA_OK(cudaMemcpy(u, d_u.p, nc_bytes, cudaMemcpyDeviceToHost));
    B2_CUDA_OK(cudaMemcpy(v, d_v.p, nc_bytes, cudaMemcpyDeviceToHost));
    return 0;
}

// K7 (+ its cbp pass) alone: as b2k_deblock, the planes, records and levels go to the device as they are and come back whole, so
// that a caller can see any store outside an intra macroblock
extern "C" int b2k_intra_recon(const uint8_t *cur_y, const uint8_t *cur_u, const uint8_t *cur_v, uint8_t *rec_y, uint8_t *rec_u,
                               uint8_t *rec_v, int w, int h, int nframes, int slices, int qp, int all_intra, b2_mbinfo_t *info,
                               b2_mbcoef_t *coef, int *ncta, int *rounds, int *dyn_smem)
{
    if ((w & 15) || (h & 15) || w <= 0 || h <= 0 || nframes <= 0 || qp < 10 || qp > 51) {
        fprintf(stderr, "b2enc: b2k_intra_recon needs w,h multiples of 16, qp 10..51\n");
        return -1;
    }
    const int mbw = w / 16, mbh = h / 16;
    int nc, rd, ds;
    b2_intra_recon_shape(mbw, mbh, slices, all_intra, &nc, &rd, &ds);
    if (ncta) *ncta = nc;
    if (rounds) *rounds = rd;
    if (dyn_smem) *dyn_smem = ds;
    if (!rec_y) return 0;
    if (!cur_y || !cur_u || !cur_v || !rec_u || !rec_v || !info || !coef) return -1;
    int pitch, rows, pitchc, rowsc;
    b2_padded_layout(w, h, &pitch, &rows, &pitchc, &rowsc);
    const size_t sy = (size_t)pitch * rows, sc = (size_t)pitchc * rowsc, ny = sy * nframes, nc_bytes = sc * nframes;
    const size_t nmb = (size_t)mbw * mbh * nframes, ni = nmb * sizeof(b2_mbinfo_t), ncf = nmb * sizeof(b2_mbcoef_t);
    DevBuf d_cy, d_cu, d_cv, d_ry, d_ru, d_rv, d_info, d_coef;
    if (d_cy.alloc(ny) || d_cu.alloc(nc_bytes) || d_cv.alloc(nc_bytes) || d_ry.alloc(ny) || d_ru.alloc(nc_bytes) || d_rv.alloc(nc_bytes) ||
        d_info.alloc(ni) || d_coef.alloc(ncf)) {
        fprintf(stderr, "b2enc: cudaMalloc failed\n");
        return -1;
    }
    B2_CUDA_OK(cudaMemcpy(d_cy.p, cur_y, ny, cudaMemcpyHostToDevice));
    B2_CUDA_OK(cudaMemcpy(d_cu.p, cur_u, nc_bytes, cudaMemcpyHostToDevice));
    B2_CUDA_OK(cudaMemcpy(d_cv.p, cur_v, nc_bytes, cudaMemcpyHostToDevice));
    B2_CUDA_OK(cudaMemcpy(d_ry.p, rec_y, ny, cudaMemcpyHostToDevice));
    B2_CUDA_OK(cudaMemcpy(d_ru.p, rec_u, nc_bytes, cudaMemcpyHostToDevice));
    B2_CUDA_OK(cudaMemcpy(d_rv.p, rec_v, nc_bytes, cudaMemcpyHostToDevice));
    B2_CUDA_OK(cudaMemcpy(d_info.p, info, ni, cudaMemcpyHostToDevice));
    B2_CUDA_OK(cudaMemcpy(d_coef.p, coef, ncf, cudaMemcpyHostToDevice));
    const uint8_t *const cur[3] = {(const uint8_t *)d_cy.p, (const uint8_t *)d_cu.p, (const uint8_t *)d_cv.p};
    uint8_t *const rec[3] = {(uint8_t *)d_ry.p, (uint8_t *)d_ru.p, (uint8_t *)d_rv.p};
    if (b2_launch_intra_recon(cur, rec, pitch, pitchc, sy, sc, mbw, mbh, slices, nframes, qp, all_intra, (b2_mbinfo_t *)d_info.p,
                              (b2_mbcoef_t *)d_coef.p, 0))
        return -1;
    B2_CUDA_OK(cudaDeviceSynchronize());
    B2_CUDA_OK(cudaMemcpy(rec_y, d_ry.p, ny, cudaMemcpyDeviceToHost));
    B2_CUDA_OK(cudaMemcpy(rec_u, d_ru.p, nc_bytes, cudaMemcpyDeviceToHost));
    B2_CUDA_OK(cudaMemcpy(rec_v, d_rv.p, nc_bytes, cudaMemcpyDeviceToHost));
    B2_CUDA_OK(cudaMemcpy(info, d_info.p, ni, cudaMemcpyDeviceToHost));
    B2_CUDA_OK(cudaMemcpy(coef, d_coef.p, ncf, cudaMemcpyDeviceToHost));
    return 0;
}

extern "C" int b2k_me_fullpel(const uint8_t *cur_y, const uint8_t *ref_y, int w, int h, int nframes, int merange,
                              const b2_mv_t *pmv, int lambda, b2_mv_t *mv_out, uint32_t *cost_out,
                              int iters, float *kernel_ms)
{
    return me_fullpel_impl(cur_y, ref_y, w, h, nframes, merange, pmv, lambda, mv_out, cost_out, nullptr, nullptr, iters, kernel_ms);
}

extern "C" int b2k_me_fullpel_parts(const uint8_t *cur_y, const uint8_t *ref_y, int w, int h, int nframes, int merange,
                                    const b2_mv_t *pmv, int lambda, b2_mv_t *mv9_out, uint32_t *cost9_out, int iters, float *kernel_ms)
{
    if (!mv9_out || !cost9_out) return -1;
    return me_fullpel_impl(cur_y, ref_y, w, h, nframes, merange, pmv, lambda, nullptr, nullptr, mv9_out, cost9_out, iters, kernel_ms);
}

static int me_fullpel_impl(const uint8_t *cur_y, const uint8_t *ref_y, int w, int h, int nframes, int merange, const b2_mv_t *pmv,
                           int lambda, b2_mv_t *mv_out, uint32_t *cost_out, b2_mv_t *mv9_out, uint32_t *cost9_out, int iters,
                           float *kernel_ms, const PruneOut *prune)
{
    if ((w & 15) || (h & 15) || w <= 0 || h <= 0 || nframes <= 0) {
        fprintf(stderr, "b2enc: b2k_me_fullpel needs w,h multiples of 16\n");
        return -1;
    }
    int bw, bh;
    if (b2_k1_window_box(merange, &bw, &bh)) { fprintf(stderr, "b2enc: merange %d not supported\n", merange); return -1; }
    const int mbw = w / 16, mbh = h / 16;
    const size_t nmb = (size_t)mbw * mbh * nframes;
    DevBuf d_cur, d_ref, d_pmv, d_mv, d_cost, d_mv9, d_cost9;
    int pitch, rows;
    if (upload_padded(d_cur, cur_y, w, h, nframes, B2_PAD, &pitch, &rows)) return -1;
    if (upload_padded(d_ref, ref_y, w, h, nframes, B2_PAD, &pitch, &rows)) return -1;
    if (d_mv.alloc(nmb * sizeof(b2_mv_t)) || d_cost.alloc(nmb * 4)) return -1;
    if (mv9_out && (d_mv9.alloc(nmb * 9 * sizeof(b2_mv_t)) || d_cost9.alloc(nmb * 9 * 4))) return -1;
    if (pmv) {
        if (d_pmv.alloc(nmb * sizeof(b2_mv_t))) return -1;
        B2_CUDA_OK(cudaMemcpy(d_pmv.p, pmv, nmb * sizeof(b2_mv_t), cudaMemcpyHostToDevice));
    }
    CUtensorMap tm_cur, tm_ref, tm_sum;
    if (b2_make_plane_tmap(&tm_cur, d_cur.p, pitch, rows, nframes, 16 * b2_k1_strip_mbs(merange), 16)) return -1;
    if (b2_make_plane_tmap(&tm_ref, d_ref.p, pitch, rows, nframes, bw, bh)) return -1;
    DevBuf d_sum, d_swept;
    if (prune) {
        if (mv9_out) return -1;
        const int mbox = b2_k1_mm_box(merange);
        if (mbox < 0) return -1;
        if (d_sum.alloc((size_t)pitch * rows * nframes * 4) || d_swept.alloc(8)) return -1;
        B2_CUDA_OK(cudaMemset(d_sum.p, 0, (size_t)pitch * rows * nframes * 4));
        B2_CUDA_OK(cudaMemset(d_swept.p, 0, 8));
        if (b2_make_plane_tmap32(&tm_sum, d_sum.p, pitch, rows, nframes, mbox)) return -1;
    }
    const int ks = prune ? b2_k1_prune_rows(merange) : 0;
    auto launch = [&](bool with_sums, unsigned long long *swept) -> int {
        if (!prune)
            return b2_launch_me_fullpel(merange, &tm_cur, &tm_ref, mbw, mbh, nframes, (const b2_mv_t *)d_pmv.p, lambda,
                                        (b2_mv_t *)d_mv.p, (uint32_t *)d_cost.p, (b2_mv_t *)d_mv9.p, (uint32_t *)d_cost9.p, 0);
        if (with_sums && b2_launch_block_sums(ks, (const uint8_t *)d_ref.p, pitch, rows, nframes, (uint32_t *)d_sum.p, 0)) return -1;
        return b2_launch_me_fullpel_pruned(merange, &tm_cur, &tm_ref, &tm_sum, mbw, mbh, nframes, (const b2_mv_t *)d_pmv.p, lambda,
                                           (b2_mv_t *)d_mv.p, (uint32_t *)d_cost.p, swept, 0);
    };
    if (launch(true, (unsigned long long *)d_swept.p)) return -1;
    B2_CUDA_OK(cudaDeviceSynchronize());
    if (prune) {
        B2_CUDA_OK(cudaMemcpy(prune->swept, d_swept.p, 8, cudaMemcpyDeviceToHost));
        *prune->all = (unsigned long long)b2_k1_candidates(merange, mbw, mbh, nframes);
    }
    if (kernel_ms) {
        cudaEvent_t e0, e1;
        cudaEventCreate(&e0); cudaEventCreate(&e1);
        if (iters < 1) iters = 1;
        if (prune) {                                           // K1a on its own: it runs once per reference frame
            cudaEventRecord(e0, 0);
            for (int i = 0; i < iters; i++) b2_launch_block_sums(ks, (const uint8_t *)d_ref.p, pitch, rows, nframes, (uint32_t *)d_sum.p, 0);
            cudaEventRecord(e1, 0);
            B2_CUDA_OK(cudaEventSynchronize(e1));
            float ms = 0;
            cudaEventElapsedTime(&ms, e0, e1);
            *prune->sums_ms = ms / iters;
        }
        cudaEventRecord(e0, 0);
        for (int i = 0; i < iters; i++) launch(false, nullptr);
        cudaEventRecord(e1, 0);
        B2_CUDA_OK(cudaEventSynchronize(e1));
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        *kernel_ms = ms / iters;
        cudaEventDestroy(e0); cudaEventDestroy(e1);
    }
    if (mv_out) B2_CUDA_OK(cudaMemcpy(mv_out, d_mv.p, nmb * sizeof(b2_mv_t), cudaMemcpyDeviceToHost));
    if (cost_out) B2_CUDA_OK(cudaMemcpy(cost_out, d_cost.p, nmb * 4, cudaMemcpyDeviceToHost));
    if (mv9_out) {
        B2_CUDA_OK(cudaMemcpy(mv9_out, d_mv9.p, nmb * 9 * sizeof(b2_mv_t), cudaMemcpyDeviceToHost));
        B2_CUDA_OK(cudaMemcpy(cost9_out, d_cost9.p, nmb * 9 * 4, cudaMemcpyDeviceToHost));
    }
    return 0;
}

// PCI bus id ("0000:1b:00.0") of a CUDA device: lets the host pin itself to the GPU's NUMA node before it allocates
// the pinned staging buffers (bench.py / b2enc.bind_to_gpu_numa)
extern "C" int b2_device_pci_bus_id(int device, char *out, int len)
{
    if (!out || len < 13) return -1;
    if (cudaDeviceGetPCIBusId(out, len, device) != cudaSuccess) { cudaGetLastError(); return -1; }
    return 0;
}
