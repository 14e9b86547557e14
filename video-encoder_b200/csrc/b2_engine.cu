// b2_engine.cu -- the encode-stage engine behind include/b2enc_engine.h: device memory layout,
// streams/events (pinned host -> device ring -> kernels -> pinned host results, double buffered) and
// the per-frame kernel schedule.  This is the "frame queue" row (a0) of SURVEY.md 8a: the
// reference's strictly synchronous one-AVFrame/one-pic_in loop (av_encode.c:968-975) becomes
// copy-in stream || compute stream || copy-out stream over `slots` lock-stepped GOPs/streams.
//
// HBM layout per engine (S = slots):
//   raw input ring      [S][ring][in_bytes]              tight pictures as uploaded
//   cur Y/U/V           [S][rows][pitch] / [S][rowsc][pitchc]   64/32-px replicated border
//   recon Y/U/V  x2     same shape; ping-pong reference / reconstruction
//   per-MB scratch      mv_full, cost_full, mv_qpel, cost_inter, cost_i16, cost_i4, prev_mv  [S][nmb]
//   results x2          b2_mbinfo_t [S][nmb] (48 B) + b2_mbcoef_t [S][nmb] (832 B), ping-pong
//   packed levels x2    [S][nmb*832] worst case, only the used prefix is copied out (cfg.pack_levels, K9)
#include <stdlib.h>
#include <string.h>
#include <vector>
#include <mutex>
#include <atomic>
#include <memory>
#include "b2_common.cuh"
#include "b2_internal.h"
#include "../../include/b2enc_engine.h"

int b2_lambda_for_qp(int qp)
{
    static const uint8_t tab[52] = {1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 4, 4, 4,
                                    5, 6, 6, 7, 8, 9, 10, 11, 13, 14, 16, 18, 20, 23, 25, 29, 32, 36, 40, 45, 51, 57,
                                    64, 72, 81, 91};
    return tab[qp < 0 ? 0 : (qp > 51 ? 51 : qp)];
}

struct ProfRec { int k; cudaEvent_t e0, e1; };

// Test hook (default off): B2ENC_TEST_FAULT=no_h2d_wait makes an encode NOT wait for the upload of its ring entry,
// =no_d2h_wait makes it NOT wait for the copy-out of the result set it is about to overwrite.  tests/test_bench_path.py must
// fail with either (scripts/gpu_fault_injection.sh): that is the proof that those tests see the inter-stream ordering.
static int test_fault()
{
    static const int f = [] {
        const char *e = getenv("B2ENC_TEST_FAULT");
        return !e ? 0 : !strcmp(e, "no_h2d_wait") ? 1 : !strcmp(e, "no_d2h_wait") ? 2 : 0;
    }();
    return f;
}

// A stream group: a contiguous range of slots advanced together on its own compute stream.  Groups
// share nothing, so their kernels overlap on the GPU: while one group sits in the latency-bound intra
// wavefront (K7) the others keep the SMs busy with the ALU-bound search (K1).
struct Group {
    int slot0 = 0, n = 0;
    cudaStream_t st = nullptr;
    CUtensorMap tm_cur, tm_ref[2];
    CUtensorMap tm_sum;                    // cfg.me_prune: (min | max) block-sum words
    int ref_idx = 0;                       // d_rec[ref_idx] holds this group's latest reconstruction
    int res_set = 0, host_set = 0;
    int last_n = 0;                        // slots covered by the most recent encode
    cudaEvent_t ev_enc[2] = {}, ev_d2h[2] = {}, ev_join = nullptr;
    bool d2h_used[2] = {false, false};
    std::vector<cudaEvent_t> ev_k0;
    std::vector<char> h2d_pending;
};

struct b2_engine {
    b2_engine_cfg_t cfg;
    int w16, h16, mbw, mbh, nmb;
    int pitch, rows, pitchc, rowsc;
    size_t stride_y, stride_c, in_bytes, in_stride;
    int lambda;
    uint8_t *d_in = nullptr, *h_in = nullptr;
    std::mutex h_in_mu;
    uint8_t *d_cur[3] = {}, *d_rec[2][3] = {};
    b2_mv_t *d_mvf = nullptr, *d_mvq = nullptr, *d_prev_mv = nullptr;
    uint32_t *d_cost_full = nullptr, *d_cost_inter = nullptr, *d_c16 = nullptr, *d_c4 = nullptr, *d_c8 = nullptr;
    uint8_t *d_pred = nullptr;             // [S][nmb][256] motion-compensated luma prediction (K2 -> K5)
    uint8_t *d_part = nullptr;             // cfg.partitions: [S][nmb] partition shape chosen by K2
    b2_mv_t *d_mv8 = nullptr;              //                 [S][nmb][3] vectors of quadrants 1..3
    b2_mv_t *d_mv9 = nullptr;              // cfg.partitions == 2: [S][nmb][9] best full-pel vector of every shape part (K1<PART>)
    uint32_t *d_cost9 = nullptr;           //                      and its cost
    b2_mbinfo_t *d_info[2] = {}, *h_info[2] = {};
    // cfg.pack_levels: the decisions cross PCIe as 24-byte records (K9a writes them); h_info is then filled on the host, per slot,
    // the first time a view of it is asked for (info_stale: the slot's records are newer than its h_info)
    b2_mbinfo_packed_t *d_pinfo[2] = {}, *h_pinfo[2] = {};
    std::vector<uint8_t> info_stale[2];
    b2_mbcoef_t *d_coef[2] = {}, *h_coef[2] = {};
    // cfg.pack_levels: packed level streams [S][pack_stride] per result set (device + pinned host), blocks used per slot
    uint8_t *d_pack[2] = {}, *h_pack[2] = {};
    uint32_t *d_pack_n[2] = {}, *h_pack_n[2] = {};
    unsigned long long *d_pack_cum = nullptr;
    uint32_t *d_pack_chunk = nullptr;              // K9a scratch: present blocks per chunk of macroblocks, [S][chunks]
    uint32_t *d_sum = nullptr;             // cfg.me_prune: [S][rows][pitch] min | max of the reference planes' block sums (K1a), refilled per P step
    unsigned long long *d_k1_swept = nullptr;      // cfg.me_prune: candidates the pruned K1 launches evaluated, accumulated on the device
    long long k1_all = 0;                          //               ... and what the exhaustive kernel would have run
    int *d_k8_flags = nullptr;                     // K8 row pipeline: cross-CTA progress flags [S][8]
    size_t pack_stride = 0;
    std::vector<Group> groups;
    // result tickets: which result set each group copied out in one of the last two b2_engine_d2h calls
    struct Ticket { std::vector<int> set; } ticket[2];
    int cur_ticket = 0;
    cudaStream_t st = nullptr, st_in = nullptr, st_out = nullptr;     // st: timer / join stream
    // b2_engine_put_frame_direct: DMA straight from the caller's pinned picture into the device ring (own stream; may run on
    // another host thread than h2d/encode/d2h as long as the two work on different ring positions)
    cudaStream_t st_put = nullptr;
    std::vector<uint8_t> in_direct;                                   // [slot * in_ring + ring]: entry is already on the device
    std::vector<cudaEvent_t> ev_h2d;
    // b2_engine_put_picture (GOP-streaming hosts): per slot, the event behind its latest upload and a flag that the group's
    // next encode still has to wait for it (set by the caller's thread, consumed by the thread that issues the encodes);
    // pageable sources go through two page-locked bounce buffers
    std::vector<cudaEvent_t> ev_put;
    std::unique_ptr<std::atomic<uint8_t>[]> put_pending;
    cudaEvent_t ev_putq[8] = {};                    // b2_engine_put_picture_async: ticket t -> ev_putq[t % 8]
    long put_seq = 0;
    uint8_t *h_bounce[2] = {nullptr, nullptr};
    cudaEvent_t ev_bounce[2] = {nullptr, nullptr};
    int bounce_next = 0;
    cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr;
    long launches = 0;
    double k_ms[B2_NKERNELS] = {};
    long k_n[B2_NKERNELS] = {};
    std::vector<ProfRec> prof_pending;
    std::vector<cudaEvent_t> ev_pool;
};

#define ENG_OK(expr)                                                                                 \
    do {                                                                                             \
        cudaError_t _e = (expr);                                                                     \
        if (_e != cudaSuccess) {                                                                     \
            fprintf(stderr, "b2enc: CUDA error %s at %s:%d: %s\n", cudaGetErrorName(_e), __FILE__,   \
                    __LINE__, cudaGetErrorString(_e));                                               \
            return -1;                                                                               \
        }                                                                                            \
    } while (0)

static size_t input_bytes(int fmt, int w, int h)
{
    int rb[3], rows[3];
    const int np = b2_fmt_layout(fmt, w, h, rb, rows);
    size_t n = 0;
    for (int p = 0; p < np; p++) n += (size_t)rb[p] * rows[p];
    return np && b2_fmt_size_ok(fmt, w, h) ? n : 0;
}

static int engine_alloc(b2_engine *e)
{
    const b2_engine_cfg_t &c = e->cfg;
    const size_t S = c.slots;
    ENG_OK(cudaMalloc(&e->d_in, e->in_stride * c.in_ring * S));
    // the pinned staging ring (in_stride * in_ring * S bytes: gigabytes for a drop-in batch) is allocated on first use
    // (b2_engine_host_input): callers that hand over page-locked pictures through b2_engine_put_frame_direct never need it
    for (int p = 0; p < 3; p++) {
        const size_t sz = (p ? e->stride_c : e->stride_y) * S;
        ENG_OK(cudaMalloc(&e->d_cur[p], sz));
        ENG_OK(cudaMalloc(&e->d_rec[0][p], sz));
        ENG_OK(cudaMalloc(&e->d_rec[1][p], sz));
        ENG_OK(cudaMemset(e->d_cur[p], 0, sz));
        ENG_OK(cudaMemset(e->d_rec[0][p], 0, sz));
        ENG_OK(cudaMemset(e->d_rec[1][p], 0, sz));
    }
    const size_t n = (size_t)e->nmb * S;
    ENG_OK(cudaMalloc(&e->d_mvf, n * 4)); ENG_OK(cudaMalloc(&e->d_mvq, n * 4)); ENG_OK(cudaMalloc(&e->d_prev_mv, n * 4));
    ENG_OK(cudaMalloc(&e->d_cost_full, n * 4)); ENG_OK(cudaMalloc(&e->d_cost_inter, n * 4));
    ENG_OK(cudaMalloc(&e->d_c16, n * 4)); ENG_OK(cudaMalloc(&e->d_c4, n * 4));
    ENG_OK(cudaMalloc(&e->d_pred, n * 256));
    ENG_OK(cudaMemset(e->d_prev_mv, 0, n * 4)); ENG_OK(cudaMemset(e->d_mvf, 0, n * 4)); ENG_OK(cudaMemset(e->d_mvq, 0, n * 4));
    ENG_OK(cudaMemset(e->d_cost_full, 0, n * 4)); ENG_OK(cudaMemset(e->d_cost_inter, 0, n * 4));
    ENG_OK(cudaMemset(e->d_c16, 0, n * 4)); ENG_OK(cudaMemset(e->d_c4, 0, n * 4));
    if (c.transform8x8) { ENG_OK(cudaMalloc(&e->d_c8, n * 4)); ENG_OK(cudaMemset(e->d_c8, 0, n * 4)); }
    if (c.partitions && c.subpel) {
        ENG_OK(cudaMalloc(&e->d_part, n)); ENG_OK(cudaMemset(e->d_part, 0, n));
        ENG_OK(cudaMalloc(&e->d_mv8, n * 3 * sizeof(b2_mv_t))); ENG_OK(cudaMemset(e->d_mv8, 0, n * 3 * sizeof(b2_mv_t)));
        if (c.partitions == 2) {
            ENG_OK(cudaMalloc(&e->d_mv9, n * 9 * sizeof(b2_mv_t))); ENG_OK(cudaMalloc(&e->d_cost9, n * 9 * 4));
            ENG_OK(cudaMemset(e->d_mv9, 0, n * 9 * sizeof(b2_mv_t))); ENG_OK(cudaMemset(e->d_cost9, 0, n * 9 * 4));
        }
    }
    for (int s = 0; s < 2; s++) {
        ENG_OK(cudaMalloc(&e->d_info[s], n * sizeof(b2_mbinfo_t)));
        ENG_OK(cudaMalloc(&e->d_coef[s], n * sizeof(b2_mbcoef_t)));
        if (c.pack_levels) {
            e->h_info[s] = (b2_mbinfo_t *)malloc(n * sizeof(b2_mbinfo_t));       // filled from the packed records on demand: plain memory
            if (!e->h_info[s]) return -1;
            memset(e->h_info[s], 0, n * sizeof(b2_mbinfo_t));
            ENG_OK(cudaMalloc(&e->d_pinfo[s], n * sizeof(b2_mbinfo_packed_t)));
            ENG_OK(cudaHostAlloc(&e->h_pinfo[s], n * sizeof(b2_mbinfo_packed_t), cudaHostAllocDefault));
            e->info_stale[s].assign(S, 0);
        } else {
            ENG_OK(cudaHostAlloc(&e->h_info[s], n * sizeof(b2_mbinfo_t), cudaHostAllocDefault));
        }
        if (c.pack_levels) {
            e->pack_stride = (size_t)e->nmb * sizeof(b2_mbcoef_t);
            ENG_OK(cudaMalloc(&e->d_pack[s], e->pack_stride * S));
            ENG_OK(cudaHostAlloc(&e->h_pack[s], e->pack_stride * S, cudaHostAllocDefault));     // UVA: the device writes it directly
            ENG_OK(cudaMalloc(&e->d_pack_n[s], S * sizeof(uint32_t)));
            ENG_OK(cudaHostAlloc(&e->h_pack_n[s], S * sizeof(uint32_t), cudaHostAllocDefault));
            memset(e->h_pack_n[s], 0, S * sizeof(uint32_t));
        } else {
            ENG_OK(cudaHostAlloc(&e->h_coef[s], n * sizeof(b2_mbcoef_t), cudaHostAllocDefault));
        }
    }
    // lossless pruning of the full-pel search: +-32 only -- at +-16 the 33 x 33 candidates leave too little to prune against the
    // per-strip costs of the bound test (measured slower than the exhaustive kernel: profiles/r2_pruned_legs.txt); the wide
    // partition search keeps the exhaustive kernel too (nine minima per macroblock)
    if (c.me_prune && c.partitions != 2 && c.merange == 32) {
        ENG_OK(cudaMalloc(&e->d_sum, e->stride_y * S * sizeof(uint32_t)));
        ENG_OK(cudaMemset(e->d_sum, 0, e->stride_y * S * sizeof(uint32_t)));
        ENG_OK(cudaMalloc(&e->d_k1_swept, sizeof(unsigned long long)));
        ENG_OK(cudaMemset(e->d_k1_swept, 0, sizeof(unsigned long long)));
    }
    ENG_OK(cudaMalloc(&e->d_k8_flags, S * 8 * sizeof(int)));
    ENG_OK(cudaMemset(e->d_k8_flags, 0, S * 8 * sizeof(int)));
    if (c.pack_levels) {
        ENG_OK(cudaMalloc(&e->d_pack_cum, sizeof(unsigned long long)));
        ENG_OK(cudaMemset(e->d_pack_cum, 0, sizeof(unsigned long long)));
        ENG_OK(cudaMalloc(&e->d_pack_chunk, S * b2_pack_chunks(e->nmb) * sizeof(uint32_t)));
    }
    ENG_OK(cudaStreamCreateWithFlags(&e->st, cudaStreamNonBlocking));
    ENG_OK(cudaStreamCreateWithFlags(&e->st_in, cudaStreamNonBlocking));
    ENG_OK(cudaStreamCreateWithFlags(&e->st_put, cudaStreamNonBlocking));
    e->in_direct.assign((size_t)c.in_ring * S, 0);
    e->ev_put.resize(S);
    e->put_pending.reset(new std::atomic<uint8_t>[S]);
    for (size_t s = 0; s < S; s++) {
        ENG_OK(cudaEventCreateWithFlags(&e->ev_put[s], cudaEventDisableTiming));
        e->put_pending[s].store(0);
    }
    for (int k = 0; k < 2; k++) ENG_OK(cudaEventCreateWithFlags(&e->ev_bounce[k], cudaEventDisableTiming));
    for (int k = 0; k < 8; k++) ENG_OK(cudaEventCreateWithFlags(&e->ev_putq[k], cudaEventDisableTiming));
    {   // the copy-out stream runs K9b (a small kernel that writes the packed levels into pinned memory) while the compute
        // streams keep every SM busy with K1: at the highest priority its CTAs are placed as soon as any resident CTA retires.
        // (Measured at 64 GOPs per GPU: no difference in e2e, 5,110-5,166 frames/s either way -- kept because a late K9b
        // would hold a result set and stall the step after next.)
        int prio_lo = 0, prio_hi = 0;
        ENG_OK(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
        ENG_OK(cudaStreamCreateWithPriority(&e->st_out, cudaStreamNonBlocking, prio_hi));
    }
    e->ev_h2d.resize(c.in_ring);
    for (int r = 0; r < c.in_ring; r++) ENG_OK(cudaEventCreateWithFlags(&e->ev_h2d[r], cudaEventDisableTiming));
    ENG_OK(cudaEventCreate(&e->ev_t0)); ENG_OK(cudaEventCreate(&e->ev_t1));
    int bw, bh;
    if (b2_k1_window_box(c.merange, &bw, &bh)) { fprintf(stderr, "b2enc: merange must be 16 or 32\n"); return -1; }
    // stream groups: contiguous, near-equal slot ranges
    int G = c.streams > 0 ? c.streams : (c.slots >= 8 ? 4 : (c.slots >= 2 ? 2 : 1));
    if (G > c.slots) G = c.slots;
    e->groups.resize(G);
    int s0 = 0;
    for (int g = 0; g < G; g++) {
        Group &gr = e->groups[g];
        gr.slot0 = s0; gr.n = c.slots / G + (g < c.slots % G ? 1 : 0);
        s0 += gr.n;
        ENG_OK(cudaStreamCreateWithFlags(&gr.st, cudaStreamNonBlocking));
        for (int s = 0; s < 2; s++) {
            ENG_OK(cudaEventCreateWithFlags(&gr.ev_enc[s], cudaEventDisableTiming));
            // a host thread waiting for a result set sleeps instead of spinning: the cores belong to the entropy stage
            ENG_OK(cudaEventCreateWithFlags(&gr.ev_d2h[s], cudaEventDisableTiming | cudaEventBlockingSync));
        }
        ENG_OK(cudaEventCreateWithFlags(&gr.ev_join, cudaEventDisableTiming));
        gr.ev_k0.resize(c.in_ring); gr.h2d_pending.assign(c.in_ring, 0);
        for (int r = 0; r < c.in_ring; r++) ENG_OK(cudaEventCreateWithFlags(&gr.ev_k0[r], cudaEventDisableTiming));
        if (b2_make_plane_tmap(&gr.tm_cur, e->d_cur[0] + gr.slot0 * e->stride_y, e->pitch, e->rows, gr.n, 16 * b2_k1_strip_mbs(c.merange), 16)) return -1;
        if (b2_make_plane_tmap(&gr.tm_ref[0], e->d_rec[0][0] + gr.slot0 * e->stride_y, e->pitch, e->rows, gr.n, bw, bh)) return -1;
        if (b2_make_plane_tmap(&gr.tm_ref[1], e->d_rec[1][0] + gr.slot0 * e->stride_y, e->pitch, e->rows, gr.n, bw, bh)) return -1;
        if (e->d_sum && b2_make_plane_tmap32(&gr.tm_sum, e->d_sum + gr.slot0 * e->stride_y, e->pitch, e->rows, gr.n, b2_k1_mm_box(c.merange)))
            return -1;
    }
    return 0;
}

extern "C" b2_engine_t *b2_engine_create(const b2_engine_cfg_t *cfg)
{
    if (!cfg || cfg->width < 16 || cfg->height < 16 || cfg->slots < 1 || cfg->in_ring < 1) {
        fprintf(stderr, "b2enc: bad engine configuration\n");
        return nullptr;
    }
    if (cfg->qp < 10 || cfg->qp > 51) { fprintf(stderr, "b2enc: qp must be in 10..51\n"); return nullptr; }
    if (cfg->merange != 16 && cfg->merange != 32) { fprintf(stderr, "b2enc: merange must be 16 or 32\n"); return nullptr; }
    // every stream group wants its own hardware queue (the default of 8 connections makes groups share queues, and a group
    // that waits on an event then holds up the kernels of the group queued behind it); read when the context is created
    setenv("CUDA_DEVICE_MAX_CONNECTIONS", "32", 0);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
        cudaGetLastError();
        fprintf(stderr, "b2enc: no CUDA device; the encode stage has no CPU fallback\n");
        return nullptr;
    }
    if (cudaSetDevice(cfg->device) != cudaSuccess) { fprintf(stderr, "b2enc: cannot select device %d\n", cfg->device); return nullptr; }
    b2_engine *e = new b2_engine();
    e->cfg = *cfg;
    e->w16 = (cfg->width + 15) & ~15; e->h16 = (cfg->height + 15) & ~15;
    e->mbw = e->w16 / 16; e->mbh = e->h16 / 16; e->nmb = e->mbw * e->mbh;
    b2_padded_layout(e->w16, e->h16, &e->pitch, &e->rows, &e->pitchc, &e->rowsc);
    e->stride_y = (size_t)e->pitch * e->rows; e->stride_c = (size_t)e->pitchc * e->rowsc;
    e->in_bytes = input_bytes(cfg->in_fmt, cfg->width, cfg->height);
    if (!e->in_bytes) { fprintf(stderr, "b2enc: unsupported input format %d\n", cfg->in_fmt); delete e; return nullptr; }
    e->in_stride = (e->in_bytes + 255) & ~(size_t)255;
    e->lambda = b2_lambda_for_qp(cfg->qp);
    if (engine_alloc(e)) { b2_engine_destroy(e); return nullptr; }
    return e;
}

extern "C" void b2_engine_destroy(b2_engine_t *e)
{
    if (!e) return;
    cudaSetDevice(e->cfg.device);
    cudaDeviceSynchronize();
    cudaFree(e->d_in); cudaFreeHost(e->h_in);
    for (int p = 0; p < 3; p++) { cudaFree(e->d_cur[p]); cudaFree(e->d_rec[0][p]); cudaFree(e->d_rec[1][p]); }
    cudaFree(e->d_mvf); cudaFree(e->d_mvq); cudaFree(e->d_prev_mv); cudaFree(e->d_cost_full); cudaFree(e->d_cost_inter);
    cudaFree(e->d_c16); cudaFree(e->d_c4); cudaFree(e->d_c8); cudaFree(e->d_pred); cudaFree(e->d_part); cudaFree(e->d_mv8); cudaFree(e->d_mv9); cudaFree(e->d_cost9);
    for (int s = 0; s < 2; s++) {
        cudaFree(e->d_info[s]); cudaFree(e->d_coef[s]); cudaFreeHost(e->h_coef[s]);
        if (e->cfg.pack_levels) free(e->h_info[s]); else cudaFreeHost(e->h_info[s]);
        cudaFree(e->d_pinfo[s]); cudaFreeHost(e->h_pinfo[s]);
        cudaFree(e->d_pack[s]); cudaFreeHost(e->h_pack[s]); cudaFree(e->d_pack_n[s]); cudaFreeHost(e->h_pack_n[s]);
    }
    cudaFree(e->d_pack_cum); cudaFree(e->d_pack_chunk); cudaFree(e->d_k8_flags); cudaFree(e->d_sum); cudaFree(e->d_k1_swept);
    for (auto &gr : e->groups) {
        for (int s = 0; s < 2; s++) { if (gr.ev_enc[s]) cudaEventDestroy(gr.ev_enc[s]); if (gr.ev_d2h[s]) cudaEventDestroy(gr.ev_d2h[s]); }
        if (gr.ev_join) cudaEventDestroy(gr.ev_join);
        for (auto ev : gr.ev_k0) cudaEventDestroy(ev);
        if (gr.st) cudaStreamDestroy(gr.st);
    }
    for (auto ev : e->ev_h2d) cudaEventDestroy(ev);
    for (auto ev : e->ev_put) cudaEventDestroy(ev);
    for (int k = 0; k < 2; k++) { if (e->ev_bounce[k]) cudaEventDestroy(e->ev_bounce[k]); cudaFreeHost(e->h_bounce[k]); }
    for (int k = 0; k < 8; k++) if (e->ev_putq[k]) cudaEventDestroy(e->ev_putq[k]);
    for (auto ev : e->ev_pool) cudaEventDestroy(ev);
    for (auto &r : e->prof_pending) { cudaEventDestroy(r.e0); cudaEventDestroy(r.e1); }
    if (e->ev_t0) cudaEventDestroy(e->ev_t0);
    if (e->ev_t1) cudaEventDestroy(e->ev_t1);
    if (e->st) cudaStreamDestroy(e->st);
    if (e->st_in) cudaStreamDestroy(e->st_in);
    if (e->st_put) cudaStreamDestroy(e->st_put);
    if (e->st_out) cudaStreamDestroy(e->st_out);
    delete e;
}

extern "C" size_t b2_engine_input_bytes(const b2_engine_t *e) { return e->in_bytes; }
extern "C" size_t b2_engine_result_bytes(const b2_engine_t *e)
{
    return e->cfg.pack_levels ? (size_t)e->nmb * sizeof(b2_mbinfo_packed_t)                      // + the packed level stream
                              : (size_t)e->nmb * (sizeof(b2_mbinfo_t) + sizeof(b2_mbcoef_t));
}
extern "C" void b2_engine_geometry(const b2_engine_t *e, int *mbw, int *mbh, int *w16, int *h16)
{
    if (mbw) *mbw = e->mbw;
    if (mbh) *mbh = e->mbh;
    if (w16) *w16 = e->w16;
    if (h16) *h16 = e->h16;
}
extern "C" int b2_engine_groups(const b2_engine_t *e) { return (int)e->groups.size(); }
extern "C" int b2_engine_group_range(const b2_engine_t *e, int group, int *slot0, int *nslots)
{
    if (group < 0 || group >= (int)e->groups.size()) return -1;
    if (slot0) *slot0 = e->groups[group].slot0;
    if (nslots) *nslots = e->groups[group].n;
    return 0;
}

static inline size_t in_off(const b2_engine *e, int slot, int ring) { return ((size_t)slot * e->cfg.in_ring + ring) * e->in_stride; }
static inline Group *group_of(b2_engine *e, int slot)
{
    for (auto &gr : e->groups)
        if (slot >= gr.slot0 && slot < gr.slot0 + gr.n) return &gr;
    return nullptr;
}

extern "C" uint8_t *b2_engine_host_input(b2_engine_t *e, int slot, int ring)
{
    if (slot < 0 || slot >= e->cfg.slots || ring < 0 || ring >= e->cfg.in_ring) return nullptr;
    if (!e->h_in) {
        std::lock_guard<std::mutex> lk(e->h_in_mu);
        if (!e->h_in) {
            cudaSetDevice(e->cfg.device);
            uint8_t *p = nullptr;
            if (cudaHostAlloc(&p, e->in_stride * e->cfg.in_ring * e->cfg.slots, cudaHostAllocDefault) != cudaSuccess) {
                fprintf(stderr, "b2enc: cannot allocate the pinned input ring\n");
                return nullptr;
            }
            e->h_in = p;
        }
    }
    return e->h_in + in_off(e, slot, ring);
}

extern "C" int b2_engine_put_frame(b2_engine_t *e, int slot, int ring, const uint8_t *const src[4], const int stride[4])
{
    uint8_t *dst = b2_engine_host_input(e, slot, ring);
    if (!dst) { fprintf(stderr, "b2enc: put_frame: bad slot/ring\n"); return -1; }
    int rb[3], rows[3];
    const int np = b2_fmt_layout(e->cfg.in_fmt, e->cfg.width, e->cfg.height, rb, rows);
    for (int p = 0; p < np; p++) {                      // tight planes, one after the other
        for (int y = 0; y < rows[p]; y++) memcpy(dst + (size_t)y * rb[p], src[p] + (size_t)y * stride[p], rb[p]);
        dst += (size_t)rb[p] * rows[p];
    }
    return 0;
}

// 0: copied; 1: the source is not page-locked host memory (use b2_engine_put_frame); -1: error
extern "C" int b2_engine_put_frame_direct(b2_engine_t *e, int slot, int ring, const uint8_t *const src[4], const int stride[4])
{
    if (slot < 0 || slot >= e->cfg.slots || ring < 0 || ring >= e->cfg.in_ring || !src || !src[0]) return -1;
    cudaSetDevice(e->cfg.device);
    int np0; { int rb0[3], rows0[3]; np0 = b2_fmt_layout(e->cfg.in_fmt, e->cfg.width, e->cfg.height, rb0, rows0); }
    for (int p = 0; p < np0; p++) {                     // every plane, every call: an address may have been freed and re-used
        cudaPointerAttributes a;
        const bool ok = src[p] && cudaPointerGetAttributes(&a, src[p]) == cudaSuccess && a.type == cudaMemoryTypeHost;
        cudaGetLastError();                             // an unregistered pointer is not an error here
        if (!ok) return 1;
    }
    Group *gr = group_of(e, slot);
    if (!gr) return -1;
    ENG_OK(cudaStreamWaitEvent(e->st_put, gr->ev_k0[ring], 0));     // the K0 that last read this ring entry
    int rb[3], rows[3];
    const int np = b2_fmt_layout(e->cfg.in_fmt, e->cfg.width, e->cfg.height, rb, rows);
    uint8_t *dst = e->d_in + in_off(e, slot, ring);
    for (int p = 0; p < np; p++) {
        ENG_OK(cudaMemcpy2DAsync(dst, rb[p], src[p], stride[p], rb[p], rows[p], cudaMemcpyHostToDevice, e->st_put));
        dst += (size_t)rb[p] * rows[p];
    }
    ENG_OK(cudaStreamSynchronize(e->st_put));            // the caller may refill the picture as soon as this returns
    e->in_direct[(size_t)slot * e->cfg.in_ring + ring] = 1;
    return 0;
}

// Hand one picture to (slot, ring) from any host memory; returns as soon as the source has been read.  Page-locked sources are
// DMA'd straight into the device ring (the call waits for the copy: the caller refills the picture, av_encode.c:415/:545);
// pageable ones are copied into one of two page-locked bounce buffers whose upload runs behind the caller's back.  No
// b2_engine_h2d follows: the next encode of the slot's group waits for the upload itself.  One caller thread at a time; it may
// be another thread than the one issuing encode_group / d2h_group as long as the slot's ring entry is not being encoded.
static long put_picture_impl(b2_engine_t *e, int slot, int ring, const uint8_t *const src[4], const int stride[4], bool wait)
{
    if (slot < 0 || slot >= e->cfg.slots || ring < 0 || ring >= e->cfg.in_ring || !src || !src[0]) return -1;
    cudaSetDevice(e->cfg.device);
    cudaPointerAttributes a;
    const bool pinned = cudaPointerGetAttributes(&a, src[0]) == cudaSuccess && a.type == cudaMemoryTypeHost;
    cudaGetLastError();                                 // an unregistered pointer is not an error here
    int rb[3], rows[3];
    const int np = b2_fmt_layout(e->cfg.in_fmt, e->cfg.width, e->cfg.height, rb, rows);
    uint8_t *dst = e->d_in + in_off(e, slot, ring);
    long ticket = 0;
    if (pinned) {
        bool tight = true;                              // planes back to back without row padding: one copy instead of 3 strided ones
        for (int p = 0; p < np; p++) tight &= stride[p] == rb[p] && (p == 0 || src[p] == src[p - 1] + (size_t)rb[p - 1] * rows[p - 1]);
        if (tight) ENG_OK(cudaMemcpyAsync(dst, src[0], e->in_bytes, cudaMemcpyHostToDevice, e->st_put));
        else
            for (int p = 0; p < np; p++) {
                ENG_OK(cudaMemcpy2DAsync(dst, rb[p], src[p], stride[p], rb[p], rows[p], cudaMemcpyHostToDevice, e->st_put));
                dst += (size_t)rb[p] * rows[p];
            }
        ENG_OK(cudaEventRecord(e->ev_put[slot], e->st_put));
        if (wait) ENG_OK(cudaStreamSynchronize(e->st_put));
        else {
            ticket = ++e->put_seq;
            ENG_OK(cudaEventRecord(e->ev_putq[ticket % 8], e->st_put));
        }
    } else {
        const int k = e->bounce_next;
        e->bounce_next ^= 1;
        if (!e->h_bounce[k]) ENG_OK(cudaHostAlloc(&e->h_bounce[k], e->in_stride, cudaHostAllocPortable));
        else ENG_OK(cudaEventSynchronize(e->ev_bounce[k]));         // its previous upload has left the buffer
        uint8_t *b = e->h_bounce[k];
        for (int p = 0; p < np; p++) {
            if (stride[p] == rb[p]) memcpy(b, src[p], (size_t)rb[p] * rows[p]);
            else for (int y = 0; y < rows[p]; y++) memcpy(b + (size_t)y * rb[p], src[p] + (size_t)y * stride[p], rb[p]);
            b += (size_t)rb[p] * rows[p];
        }
        ENG_OK(cudaMemcpyAsync(dst, e->h_bounce[k], e->in_bytes, cudaMemcpyHostToDevice, e->st_put));
        ENG_OK(cudaEventRecord(e->ev_bounce[k], e->st_put));
        ENG_OK(cudaEventRecord(e->ev_put[slot], e->st_put));
    }
    e->put_pending[slot].store(1, std::memory_order_release);
    return ticket;
}

extern "C" int b2_engine_put_picture(b2_engine_t *e, int slot, int ring, const uint8_t *const src[4], const int stride[4])
{
    return put_picture_impl(e, slot, ring, src, stride, true) < 0 ? -1 : 0;
}

// The same without waiting for the DMA of a page-locked source: returns a ticket > 0 that b2_engine_put_wait blocks on before the
// source may be overwritten (0: the source has already been read; < 0: error).  Used for the staging buffers of deferred
// b2_sws_scale conversions, which the library owns and double-buffers, so that the caller's thread never waits for PCIe.
extern "C" long b2_engine_put_picture_async(b2_engine_t *e, int slot, int ring, const uint8_t *const src[4], const int stride[4])
{
    return put_picture_impl(e, slot, ring, src, stride, false);
}
extern "C" int b2_engine_put_wait(b2_engine_t *e, long ticket)
{
    if (ticket <= 0) return 0;
    // the event of ticket t is re-recorded by ticket t + 8 on the same in-order stream: waiting for the newer record covers the older copy
    ENG_OK(cudaEventSynchronize(e->ev_putq[ticket % 8]));
    return 0;
}

// Change the raw input layout (B2_FMT_*) of an idle engine: the ring is re-allocated when the picture size differs.  Used by
// the drop-in encoder when sws_scale hands it pictures in the decoder's own format (the conversion then runs as K0).
extern "C" int b2_engine_set_input_format(b2_engine_t *e, int fmt)
{
    if (fmt == e->cfg.in_fmt) return 0;
    const size_t nb = input_bytes(fmt, e->cfg.width, e->cfg.height);
    if (!nb) { fprintf(stderr, "b2enc: unsupported input format %d for %dx%d\n", fmt, e->cfg.width, e->cfg.height); return -1; }
    cudaSetDevice(e->cfg.device);
    if (b2_engine_sync(e)) return -1;
    ENG_OK(cudaStreamSynchronize(e->st_put));
    const size_t ns = (nb + 255) & ~(size_t)255;
    if (ns != e->in_stride) {
        ENG_OK(cudaFree(e->d_in)); e->d_in = nullptr;
        cudaFreeHost(e->h_in); e->h_in = nullptr;
        for (int k = 0; k < 2; k++) { cudaFreeHost(e->h_bounce[k]); e->h_bounce[k] = nullptr; }
        ENG_OK(cudaMalloc(&e->d_in, ns * e->cfg.in_ring * e->cfg.slots));
    }
    e->cfg.in_fmt = fmt; e->in_bytes = nb; e->in_stride = ns;
    return 0;
}

extern "C" int b2_engine_h2d(b2_engine_t *e, int slot0, int nslots, int ring)
{
    if (slot0 < 0 || nslots < 1 || slot0 + nslots > e->cfg.slots || ring < 0 || ring >= e->cfg.in_ring) return -1;
    cudaSetDevice(e->cfg.device);
    // do not overwrite a ring entry that a previously issued K0 of an affected group still has to read
    for (auto &gr : e->groups)
        if (gr.slot0 < slot0 + nslots && slot0 < gr.slot0 + gr.n) ENG_OK(cudaStreamWaitEvent(e->st_in, gr.ev_k0[ring], 0));
    bool any_direct = false, all_direct = true;          // entries that b2_engine_put_frame_direct already placed on the device
    for (int s = slot0; s < slot0 + nslots; s++) {
        const bool d = e->in_direct[(size_t)s * e->cfg.in_ring + ring] != 0;
        any_direct |= d; all_direct &= d;
    }
    if (!all_direct && !e->h_in) { fprintf(stderr, "b2enc: h2d: no picture was handed over for this ring position\n"); return -1; }
    if (e->cfg.in_ring == 1 && !any_direct) {
        const size_t off = in_off(e, slot0, 0);
        ENG_OK(cudaMemcpyAsync(e->d_in + off, e->h_in + off, e->in_stride * nslots, cudaMemcpyHostToDevice, e->st_in));
    } else if (!any_direct) {
        // consecutive slots are in_ring pictures apart: one strided copy instead of one call per slot
        const size_t off = in_off(e, slot0, ring), pitch = e->in_stride * e->cfg.in_ring;
        ENG_OK(cudaMemcpy2DAsync(e->d_in + off, pitch, e->h_in + off, pitch, e->in_bytes, nslots, cudaMemcpyHostToDevice, e->st_in));
    } else {
        for (int s = slot0; s < slot0 + nslots; s++) {
            uint8_t &direct = e->in_direct[(size_t)s * e->cfg.in_ring + ring];
            if (direct) { direct = 0; continue; }
            const size_t off = in_off(e, s, ring);
            ENG_OK(cudaMemcpyAsync(e->d_in + off, e->h_in + off, e->in_bytes, cudaMemcpyHostToDevice, e->st_in));
        }
    }
    ENG_OK(cudaEventRecord(e->ev_h2d[ring], e->st_in));
    for (auto &gr : e->groups)
        if (gr.slot0 < slot0 + nslots && slot0 < gr.slot0 + gr.n) gr.h2d_pending[ring] = 1;
    return 0;
}

static cudaEvent_t pool_event(b2_engine *e)
{
    if (!e->ev_pool.empty()) { cudaEvent_t ev = e->ev_pool.back(); e->ev_pool.pop_back(); return ev; }
    cudaEvent_t ev;
    cudaEventCreate(&ev);
    return ev;
}
struct KScope {
    b2_engine *e; cudaStream_t st; int k; cudaEvent_t e0 = nullptr, e1 = nullptr;
    KScope(b2_engine *e_, cudaStream_t st_, int k_) : e(e_), st(st_), k(k_)
    {
        e->launches++;
        if (e->cfg.profile) { e0 = pool_event(e); e1 = pool_event(e); cudaEventRecord(e0, st); }
    }
    ~KScope() { if (e->cfg.profile) { cudaEventRecord(e1, st); e->prof_pending.push_back({k, e0, e1}); } }
};
static void prof_collect(b2_engine *e)
{
    for (auto &r : e->prof_pending) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, r.e0, r.e1) == cudaSuccess) { e->k_ms[r.k] += ms; e->k_n[r.k]++; }
        e->ev_pool.push_back(r.e0); e->ev_pool.push_back(r.e1);
    }
    e->prof_pending.clear();
}

// one frame for the first `ns` slots of group `gr`
static int encode_group(b2_engine *e, Group &gr, int frame_type, int ns, int ring)
{
    const b2_engine_cfg_t &c = e->cfg;
    const int is_p = frame_type == B2_FRAME_P;
    const int do_intra = !is_p || c.intra_in_p;
    const int set = gr.res_set ^ 1;
    cudaStream_t st = gr.st;
    if (gr.h2d_pending[ring]) { if (test_fault() != 1) ENG_OK(cudaStreamWaitEvent(st, e->ev_h2d[ring], 0)); gr.h2d_pending[ring] = 0; }
    for (int s = gr.slot0; s < gr.slot0 + ns; s++)          // pictures handed over by b2_engine_put_picture
        if (e->put_pending[s].exchange(0, std::memory_order_acquire)) ENG_OK(cudaStreamWaitEvent(st, e->ev_put[s], 0));
    if (gr.d2h_used[set] && test_fault() != 2) ENG_OK(cudaStreamWaitEvent(st, gr.ev_d2h[set], 0));        // result set still being copied out
    const size_t oy = gr.slot0 * e->stride_y, oc = gr.slot0 * e->stride_c, om = (size_t)gr.slot0 * e->nmb;
    uint8_t *curw[3] = {e->d_cur[0] + oy, e->d_cur[1] + oc, e->d_cur[2] + oc};
    const uint8_t *cur[3] = {curw[0], curw[1], curw[2]};
    const uint8_t *ref[3] = {e->d_rec[gr.ref_idx][0] + oy, e->d_rec[gr.ref_idx][1] + oc, e->d_rec[gr.ref_idx][2] + oc};
    uint8_t *rec[3] = {e->d_rec[gr.ref_idx ^ 1][0] + oy, e->d_rec[gr.ref_idx ^ 1][1] + oc, e->d_rec[gr.ref_idx ^ 1][2] + oc};
    b2_mbinfo_t *info = e->d_info[set] + om;
    b2_mbcoef_t *coef = e->d_coef[set] + om;
    const size_t n = (size_t)e->nmb * ns;

    {   // K0: raw picture -> padded planes (consecutive slots are `in_ring` pictures apart in the ring buffer)
        KScope k(e, st, 0);
        if (b2_launch_convert(c.in_fmt, e->d_in + in_off(e, gr.slot0, ring), e->in_stride * c.in_ring, curw[0], curw[1], curw[2],
                              e->pitch, e->pitchc, e->stride_y, e->stride_c, c.width, c.height, ns, st))
            return -1;
    }
    ENG_OK(cudaEventRecord(gr.ev_k0[ring], st));
    {
        KScope k(e, st, 1);
        if (b2_launch_extend_border_yuv(curw[0], curw[1], curw[2], e->pitch, e->rows, e->pitchc, e->rowsc, e->stride_y, e->stride_c,
                                        e->w16, e->h16, ns, st))
            return -1;
    }
    ENG_OK(cudaMemsetAsync(info, 0, n * sizeof(b2_mbinfo_t), st));
    if (is_p) {
        {
            KScope k(e, st, 2);
            if (e->d_sum) {
                // lossless pruning: block sums of this step's reference planes, then the search over the surviving candidates
                if (b2_launch_block_sums(b2_k1_prune_rows(c.merange), ref[0], e->pitch, e->rows, ns, e->d_sum + gr.slot0 * e->stride_y, st)) return -1;
                if (b2_launch_me_fullpel_pruned(c.merange, &gr.tm_cur, &gr.tm_ref[gr.ref_idx], &gr.tm_sum, e->mbw, e->mbh, ns, e->d_prev_mv + om,
                                                e->lambda, e->d_mvf + om, e->d_cost_full + om, e->d_k1_swept, st))
                    return -1;
                e->k1_all += b2_k1_candidates(c.merange, e->mbw, e->mbh, ns);
                e->launches++;                               // K1a
            } else if (b2_launch_me_fullpel(c.merange, &gr.tm_cur, &gr.tm_ref[gr.ref_idx], e->mbw, e->mbh, ns, e->d_prev_mv + om, e->lambda,
                                     e->d_mvf + om, e->d_cost_full + om, e->d_mv9 ? e->d_mv9 + om * 9 : nullptr,
                                     e->d_cost9 ? e->d_cost9 + om * 9 : nullptr, st))
                return -1;
        }
        {
            KScope k(e, st, 3);
            if (b2_launch_me_subpel(cur[0], ref[0], e->pitch, e->stride_y, e->mbw, e->mbh, ns, e->d_mvf + om, e->d_prev_mv + om,
                                    e->lambda, c.subpel, e->d_mvq + om, e->d_cost_inter + om, e->d_pred + om * 256,
                                    e->d_part ? e->d_part + om : nullptr, e->d_mv8 ? e->d_mv8 + om * 3 : nullptr,
                                    e->d_mv9 ? e->d_mv9 + om * 9 : nullptr, e->d_cost9 ? e->d_cost9 + om * 9 : nullptr, st))
                return -1;
        }
    }
    if (do_intra) {
        KScope k(e, st, 4);
        if (b2_launch_intra_analyse(cur[0], cur[1], cur[2], e->pitch, e->pitchc, e->stride_y, e->stride_c, e->mbw, e->mbh, c.slices, ns,
                                    e->lambda, info, e->d_c16 + om, e->d_c4 + om, e->d_c8 ? e->d_c8 + om : nullptr, st))
            return -1;
    }
    {
        KScope k(e, st, 5);
        if (b2_launch_decide_inter(cur, ref, rec, e->pitch, e->pitchc, e->stride_y, e->stride_c, e->mbw, e->mbh, ns, is_p, do_intra,
                                   c.qp, e->d_mvq + om, e->d_cost_inter + om, e->d_c16 + om, e->d_c4 + om, e->d_c8 ? e->d_c8 + om : nullptr, info, coef,
                                   e->d_prev_mv + om, e->d_pred + om * 256, c.transform8x8, e->d_part ? e->d_part + om : nullptr,
                                   e->d_mv8 ? e->d_mv8 + om * 3 : nullptr, st))
            return -1;
    }
    if (do_intra) {
        KScope k(e, st, 6);
        e->launches++;                                   // K7 + its cbp pass
        if (b2_launch_intra_recon(cur, rec, e->pitch, e->pitchc, e->stride_y, e->stride_c, e->mbw, e->mbh, c.slices, ns, c.qp, !is_p, info, coef, st))
            return -1;
    }
    if (c.deblock) {
        KScope k(e, st, 8);
        if (b2_launch_deblock(rec, e->pitch, e->pitchc, e->stride_y, e->stride_c, e->mbw, e->mbh, ns, c.qp, c.deblock_alpha, c.deblock_beta, info,
                              e->d_k8_flags + (size_t)gr.slot0 * 8, st)) return -1;
    }
    {
        KScope k(e, st, 7);
        if (b2_launch_extend_border_yuv(rec[0], rec[1], rec[2], e->pitch, e->rows, e->pitchc, e->rowsc, e->stride_y, e->stride_c,
                                        e->w16, e->h16, ns, st))
            return -1;
    }
    if (c.pack_levels) {
        KScope k(e, st, 9);
        e->launches++;                                   // K9a is two kernels (count, scatter)
        if (b2_launch_pack_levels(info, coef, e->d_pack[set] + gr.slot0 * e->pack_stride, e->pack_stride, e->d_pack_n[set] + gr.slot0,
                                  e->d_pack_cum, e->d_pack_chunk + (size_t)gr.slot0 * b2_pack_chunks(e->nmb), e->d_pinfo[set] + om, e->nmb, ns, st))
            return -1;
    }
    ENG_OK(cudaEventRecord(gr.ev_enc[set], st));
    gr.ref_idx ^= 1;
    gr.res_set = set;
    gr.last_n = ns;
    return 0;
}

extern "C" int b2_engine_encode_group(b2_engine_t *e, int group, int frame_type, int ring)
{
    if (group < 0 || group >= (int)e->groups.size() || ring < 0 || ring >= e->cfg.in_ring) return -1;
    cudaSetDevice(e->cfg.device);
    return encode_group(e, e->groups[group], frame_type, e->groups[group].n, ring);
}

extern "C" int b2_engine_encode(b2_engine_t *e, int frame_type, int nslots, int ring)
{
    if (nslots < 1 || nslots > e->cfg.slots || ring < 0 || ring >= e->cfg.in_ring) return -1;
    cudaSetDevice(e->cfg.device);
    for (auto &gr : e->groups) {
        const int ns = nslots - gr.slot0 < gr.n ? nslots - gr.slot0 : gr.n;
        if (ns <= 0) continue;
        if (encode_group(e, gr, frame_type, ns, ring)) return -1;
    }
    return 0;
}

static int d2h_group(b2_engine *e, Group &gr, int ns)
{
    const int set = gr.res_set;
    const size_t om = (size_t)gr.slot0 * e->nmb, n = (size_t)e->nmb * ns;
    ENG_OK(cudaStreamWaitEvent(e->st_out, gr.ev_enc[set], 0));
    if (e->cfg.pack_levels) {
        ENG_OK(cudaMemcpyAsync(e->h_pinfo[set] + om, e->d_pinfo[set] + om, n * sizeof(b2_mbinfo_packed_t), cudaMemcpyDeviceToHost, e->st_out));
        for (int s = gr.slot0; s < gr.slot0 + ns; s++) e->info_stale[set][s] = 1;
    } else {
        ENG_OK(cudaMemcpyAsync(e->h_info[set] + om, e->d_info[set] + om, n * sizeof(b2_mbinfo_t), cudaMemcpyDeviceToHost, e->st_out));
    }
    if (e->cfg.pack_levels) {
        if (b2_launch_pack_copy_out(e->d_pack[set] + gr.slot0 * e->pack_stride, e->pack_stride, e->d_pack_n[set] + gr.slot0,
                                    e->h_pack[set] + gr.slot0 * e->pack_stride, e->h_pack_n[set] + gr.slot0, ns, e->st_out))
            return -1;
        e->launches++;
    } else {
        ENG_OK(cudaMemcpyAsync(e->h_coef[set] + om, e->d_coef[set] + om, n * sizeof(b2_mbcoef_t), cudaMemcpyDeviceToHost, e->st_out));
    }
    ENG_OK(cudaEventRecord(gr.ev_d2h[set], e->st_out));
    gr.d2h_used[set] = true;
    gr.host_set = set;
    return 0;
}

extern "C" int b2_engine_d2h_group(b2_engine_t *e, int group)
{
    if (group < 0 || group >= (int)e->groups.size()) return -1;
    cudaSetDevice(e->cfg.device);
    Group &gr = e->groups[group];
    return d2h_group(e, gr, gr.last_n > 0 ? gr.last_n : gr.n);
}

// group-level hand-off (hosts that advance every group on its own, e.g. one closed GOP per group): the result set the
// group's last b2_engine_d2h_group copies into, whether / until that copy has landed, and views of a given set
extern "C" int b2_engine_group_result_set(const b2_engine_t *e, int group)
{
    return group < 0 || group >= (int)e->groups.size() ? -1 : e->groups[group].host_set;
}
extern "C" int b2_engine_group_done(b2_engine_t *e, int group, int set)
{
    if (group < 0 || group >= (int)e->groups.size() || set < 0 || set > 1) return -1;
    const cudaError_t r = cudaEventQuery(e->groups[group].ev_d2h[set]);
    if (r == cudaSuccess) return 1;
    if (r == cudaErrorNotReady) { cudaGetLastError(); return 0; }
    fprintf(stderr, "b2enc: CUDA error %s while waiting for a result set\n", cudaGetErrorName(r));
    return -1;
}
extern "C" int b2_engine_group_wait(b2_engine_t *e, int group, int set)
{
    if (group < 0 || group >= (int)e->groups.size() || set < 0 || set > 1) return -1;
    ENG_OK(cudaEventSynchronize(e->groups[group].ev_d2h[set]));
    return 0;
}
// host view of a slot's decisions in result set `set`; with cfg.pack_levels the 24-byte records that were copied out are
// expanded into it the first time it is asked for after a copy-out (the caller has waited for that copy: b2_engine_group_wait /
// b2_engine_wait_ticket / b2_engine_sync)
static const b2_mbinfo_t *info_view(b2_engine *e, int set, int slot)
{
    b2_mbinfo_t *dst = e->h_info[set] + (size_t)slot * e->nmb;
    if (e->cfg.pack_levels && e->info_stale[set][slot]) {
        const b2_mbinfo_packed_t *src = e->h_pinfo[set] + (size_t)slot * e->nmb;
        for (int i = 0; i < e->nmb; i++) b2_mbinfo_unpack(&src[i], &dst[i]);
        e->info_stale[set][slot] = 0;
    }
    return dst;
}
extern "C" const b2_mbinfo_t *b2_engine_info_set(b2_engine_t *e, int set, int slot)
{
    return set < 0 || set > 1 || slot < 0 || slot >= e->cfg.slots ? nullptr : info_view(e, set, slot);
}
// the 24-byte records themselves (cfg.pack_levels): for hosts that move them on without expanding them here
extern "C" const b2_mbinfo_packed_t *b2_engine_info_packed_set(b2_engine_t *e, int set, int slot)
{
    return set < 0 || set > 1 || slot < 0 || slot >= e->cfg.slots || !e->cfg.pack_levels ? nullptr : e->h_pinfo[set] + (size_t)slot * e->nmb;
}
extern "C" const uint8_t *b2_engine_packed_set(b2_engine_t *e, int set, int slot, size_t *bytes)
{
    if (set < 0 || set > 1 || slot < 0 || slot >= e->cfg.slots || !e->cfg.pack_levels) return nullptr;
    if (bytes) *bytes = (size_t)e->h_pack_n[set][slot] * 32;
    return e->h_pack[set] + (size_t)slot * e->pack_stride;
}

extern "C" int b2_engine_d2h(b2_engine_t *e, int nslots)
{
    if (nslots < 1 || nslots > e->cfg.slots) return -1;
    cudaSetDevice(e->cfg.device);
    e->cur_ticket ^= 1;
    auto &tk = e->ticket[e->cur_ticket];
    tk.set.assign(e->groups.size(), -1);
    for (size_t g = 0; g < e->groups.size(); g++) {
        Group &gr = e->groups[g];
        const int ns = nslots - gr.slot0 < gr.n ? nslots - gr.slot0 : gr.n;
        if (ns <= 0) continue;
        if (d2h_group(e, gr, ns)) return -1;
        tk.set[g] = gr.host_set;
    }
    return 0;
}

// ticket of the most recent b2_engine_d2h; stays valid until the next but one b2_engine_d2h
extern "C" int b2_engine_ticket(const b2_engine_t *e) { return e->cur_ticket; }
// block until the copies of that b2_engine_d2h have landed (later work may still be running on the GPU)
extern "C" int b2_engine_wait_ticket(b2_engine_t *e, int ticket)
{
    if (ticket < 0 || ticket > 1) return -1;
    cudaSetDevice(e->cfg.device);
    auto &tk = e->ticket[ticket];
    for (size_t g = 0; g < tk.set.size(); g++)
        if (tk.set[g] >= 0) ENG_OK(cudaEventSynchronize(e->groups[g].ev_d2h[tk.set[g]]));
    return 0;
}
extern "C" const b2_mbinfo_t *b2_engine_info_ticket(b2_engine_t *e, int ticket, int slot)
{
    if (ticket < 0 || ticket > 1) return nullptr;
    for (size_t g = 0; g < e->groups.size(); g++)
        if (slot >= e->groups[g].slot0 && slot < e->groups[g].slot0 + e->groups[g].n && g < e->ticket[ticket].set.size() &&
            e->ticket[ticket].set[g] >= 0)
            return info_view(e, e->ticket[ticket].set[g], slot);
    return nullptr;
}
extern "C" const b2_mbcoef_t *b2_engine_coef_ticket(b2_engine_t *e, int ticket, int slot)
{
    if (ticket < 0 || ticket > 1 || e->cfg.pack_levels) return nullptr;
    for (size_t g = 0; g < e->groups.size(); g++)
        if (slot >= e->groups[g].slot0 && slot < e->groups[g].slot0 + e->groups[g].n && g < e->ticket[ticket].set.size() &&
            e->ticket[ticket].set[g] >= 0)
            return e->h_coef[e->ticket[ticket].set[g]] + (size_t)slot * e->nmb;
    return nullptr;
}

extern "C" int b2_engine_sync(b2_engine_t *e)
{
    cudaSetDevice(e->cfg.device);
    ENG_OK(cudaStreamSynchronize(e->st_in));
    for (auto &gr : e->groups) ENG_OK(cudaStreamSynchronize(gr.st));
    ENG_OK(cudaStreamSynchronize(e->st));
    ENG_OK(cudaStreamSynchronize(e->st_out));
    prof_collect(e);
    return 0;
}

extern "C" const b2_mbinfo_t *b2_engine_info(b2_engine_t *e, int slot)
{
    Group *gr = group_of(e, slot);
    return gr ? info_view(e, gr->host_set, slot) : nullptr;
}
extern "C" const b2_mbcoef_t *b2_engine_coef(b2_engine_t *e, int slot)
{
    Group *gr = group_of(e, slot);
    return gr && !e->cfg.pack_levels ? e->h_coef[gr->host_set] + (size_t)slot * e->nmb : nullptr;
}
// packed levels (cfg.pack_levels): stream of the slot's last fetched frame and its size in bytes
extern "C" const uint8_t *b2_engine_packed(b2_engine_t *e, int slot, size_t *bytes)
{
    Group *gr = group_of(e, slot);
    if (!gr || !e->cfg.pack_levels) return nullptr;
    if (bytes) *bytes = (size_t)e->h_pack_n[gr->host_set][slot] * 32;
    return e->h_pack[gr->host_set] + (size_t)slot * e->pack_stride;
}
extern "C" const uint8_t *b2_engine_packed_ticket(b2_engine_t *e, int ticket, int slot, size_t *bytes)
{
    if (ticket < 0 || ticket > 1 || !e->cfg.pack_levels) return nullptr;
    for (size_t g = 0; g < e->groups.size(); g++)
        if (slot >= e->groups[g].slot0 && slot < e->groups[g].slot0 + e->groups[g].n && g < e->ticket[ticket].set.size() &&
            e->ticket[ticket].set[g] >= 0) {
            const int set = e->ticket[ticket].set[g];
            if (bytes) *bytes = (size_t)e->h_pack_n[set][slot] * 32;
            return e->h_pack[set] + (size_t)slot * e->pack_stride;
        }
    return nullptr;
}
// bytes of packed levels produced since the engine was created (synchronises)
extern "C" long long b2_engine_packed_bytes_total(b2_engine_t *e)
{
    if (!e->cfg.pack_levels || b2_engine_sync(e)) return -1;
    unsigned long long v = 0;
    if (cudaMemcpy(&v, e->d_pack_cum, sizeof(v), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
    return (long long)v;
}

static int get_planes(b2_engine *e, uint8_t *const src[3], int slot, uint8_t *y, uint8_t *u, uint8_t *v)
{
    cudaSetDevice(e->cfg.device);
    if (b2_engine_sync(e)) return -1;
    uint8_t *dst[3] = {y, u, v};
    for (int p = 0; p < 3; p++) {
        if (!dst[p]) continue;
        const int pitch = p ? e->pitchc : e->pitch, pad = p ? B2_PADC : B2_PAD, w = p ? e->w16 / 2 : e->w16, h = p ? e->h16 / 2 : e->h16;
        const uint8_t *s = src[p] + (size_t)slot * (p ? e->stride_c : e->stride_y) + (size_t)pad * pitch + pad;
        ENG_OK(cudaMemcpy2D(dst[p], w, s, pitch, w, h, cudaMemcpyDeviceToHost));
    }
    return 0;
}
extern "C" int b2_engine_get_recon(b2_engine_t *e, int slot, uint8_t *y, uint8_t *u, uint8_t *v)
{
    Group *gr = group_of(e, slot);
    if (!gr) return -1;
    return get_planes(e, e->d_rec[gr->ref_idx], slot, y, u, v);
}
extern "C" int b2_engine_get_cur(b2_engine_t *e, int slot, uint8_t *y, uint8_t *u, uint8_t *v)
{
    if (!group_of(e, slot)) return -1;
    return get_planes(e, e->d_cur, slot, y, u, v);
}
extern "C" int b2_engine_get_stage(b2_engine_t *e, int slot, int what, void *out)
{
    if (slot < 0 || slot >= e->cfg.slots) return -1;
    if (b2_engine_sync(e)) return -1;
    const void *src = nullptr;
    switch (what) {
    case B2_STAGE_MV_FULL: src = e->d_mvf; break;
    case B2_STAGE_COST_FULL: src = e->d_cost_full; break;
    case B2_STAGE_MV_QPEL: src = e->d_mvq; break;
    case B2_STAGE_COST_INTER: src = e->d_cost_inter; break;
    case B2_STAGE_COST_I16: src = e->d_c16; break;
    case B2_STAGE_COST_I4: src = e->d_c4; break;
    default: return -1;
    }
    ENG_OK(cudaMemcpy(out, (const uint8_t *)src + (size_t)slot * e->nmb * 4, (size_t)e->nmb * 4, cudaMemcpyDeviceToHost));
    return 0;
}

// The timer brackets ALL group streams: t0 is recorded after every group stream has reached this point
// and every group stream then waits for t0; t1 is recorded after every group stream has drained.
extern "C" int b2_engine_timer_start(b2_engine_t *e)
{
    cudaSetDevice(e->cfg.device);
    for (auto &gr : e->groups) { ENG_OK(cudaEventRecord(gr.ev_join, gr.st)); ENG_OK(cudaStreamWaitEvent(e->st, gr.ev_join, 0)); }
    ENG_OK(cudaEventRecord(e->ev_t0, e->st));
    for (auto &gr : e->groups) ENG_OK(cudaStreamWaitEvent(gr.st, e->ev_t0, 0));
    return 0;
}
extern "C" int b2_engine_timer_stop(b2_engine_t *e, float *ms)
{
    cudaSetDevice(e->cfg.device);
    for (auto &gr : e->groups) { ENG_OK(cudaEventRecord(gr.ev_join, gr.st)); ENG_OK(cudaStreamWaitEvent(e->st, gr.ev_join, 0)); }
    ENG_OK(cudaEventRecord(e->ev_t1, e->st));
    ENG_OK(cudaEventSynchronize(e->ev_t1));
    ENG_OK(cudaEventElapsedTime(ms, e->ev_t0, e->ev_t1));
    return 0;
}
extern "C" int b2_engine_kernel_ms(b2_engine_t *e, int which, double *ms_total, long *launches)
{
    if (which < 0 || which >= B2_NKERNELS) return -1;
    if (b2_engine_sync(e)) return -1;
    if (ms_total) *ms_total = e->k_ms[which];
    if (launches) *launches = e->k_n[which];
    return 0;
}
extern "C" void b2_engine_profile_reset(b2_engine_t *e)
{
    b2_engine_sync(e);
    for (int i = 0; i < B2_NKERNELS; i++) { e->k_ms[i] = 0; e->k_n[i] = 0; }
}
extern "C" long b2_engine_launch_count(const b2_engine_t *e) { return e->launches; }

// cfg.me_prune: candidate vectors the pruned K1 launches evaluated and what exhaustive launches of the same steps evaluate;
// synchronises the device (a reporting call, not for the hot path).  Returns -1 when pruning is off.
extern "C" int b2_engine_k1_stats(b2_engine_t *e, unsigned long long *swept, unsigned long long *all)
{
    if (!e || !e->d_k1_swept) return -1;
    cudaSetDevice(e->cfg.device);
    unsigned long long v = 0;
    if (cudaDeviceSynchronize() != cudaSuccess) return -1;
    if (cudaMemcpy(&v, e->d_k1_swept, sizeof(v), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
    if (swept) *swept = v;
    if (all) *all = (unsigned long long)e->k1_all;
    return 0;
}
