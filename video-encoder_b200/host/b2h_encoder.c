/*
 * b2h_encoder.c -- host side of the drop-in encoder boundary (include/b2enc.h): the x264 API subset
 * that av_encode.c calls (enc_x264_open :378-438, the encode loop :968-975, the drain loop :1076-1083),
 * implemented over the CUDA engine (include/b2enc_engine.h) and the host entropy stage (b2h_entropy.h: CABAC or CAVLC).
 *
 * Frame queue (row a0 of SURVEY.md 8a).  The caller still hands over one picture per call; the reference's strictly
 * synchronous loop becomes a GOP-streaming pipeline:
 *
 *   caller thread      picture -> device ring of the closed GOP being gathered (GOP k lives on GPU k % N, in a free slot of
 *                      that GPU's engine); returns a finished frame when the head of the display-order fifo is ready
 *   one thread per GPU advances every slot that has pictures: upload is already done, so a step is encode_group + d2h_group
 *                      of the slot's own CUDA stream, two steps in flight per slot; a slot starts as soon as its first picture
 *                      is there -- it does not wait for the GOP, let alone for a batch of GOPs -- and is free again when its
 *                      last result set has been fetched
 *   entropy workers    one frame per job (CABAC / CAVLC slice + parameter sets), from heap copies of the result sets, on all
 *                      host cores; finished frames land in the fifo slot of their frame number
 *
 * Closed GOPs share nothing, so which GPU or slot a GOP ran on, and how many were in flight, cannot change its bytes: the
 * N-GPU stream is byte-identical to the 1-GPU stream (SURVEY.md 8e, T5; tests/test_dropin.py, tests/test_multi_gpu.py).
 * The x264 contract main() relies on holds: 0 = no output yet, delayed_frames() = frames in - frames out, encode(NULL)
 * returns one frame per call until the encoder is empty (av_encode.c:971-974, :1076-1083).
 * i_gop_slots = 1 (tune zerolatency) encodes every picture synchronously in the caller's thread (zero delay).
 *
 * Slices (i_slice_count n > 1, b2_slice_row in b2enc_types.h): a picture is SPS/PPS (IDR) + n slice NALs.  With several GOP slots
 * an entropy job stays one frame and writes its slices one after the other (frames are already coded in parallel); in zero-delay
 * mode the slices of the one picture are written at the same time by a pool of min(n, cores - 1) threads started at open.
 */
#define _GNU_SOURCE                 /* syscall(SYS_gettid): per-thread nice value of the entropy workers */
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/resource.h>
#include <sys/syscall.h>
#include <time.h>
#include <unistd.h>
#include "b2enc.h"
#include "b2enc_engine.h"
#include "b2enc_kernels.h"
#include "b2h_entropy.h"
#include "b2h_picture.h"

typedef struct { int off, size, type, ref; } nalrec_t;
typedef struct {
    uint8_t *data;
    int size;
    int nal_count;
    nalrec_t *nal;              /* [slices + 2]; owned like data */
    int64_t pts;
    int key;
    int ready;
} outframe_t;

#define B2_MAX_WORKERS 64
#define B2_MAX_DEVICES 16
static double now_s(void) { struct timespec t; clock_gettime(CLOCK_MONOTONIC, &t); return (double)t.tv_sec + 1e-9 * (double)t.tv_nsec; }
static double thread_cpu_s(void) { struct timespec t; clock_gettime(CLOCK_THREAD_CPUTIME_ID, &t); return (double)t.tv_sec + 1e-9 * (double)t.tv_nsec; }

/* one frame to entropy-code; the per-MB decisions (as the 24-byte records that crossed PCIe; the worker expands them) and the
 * packed levels are heap copies of the engine's pinned result set, so the GPU may run ahead of the entropy workers (the engine
 * keeps only two result sets per slot) */
typedef struct { int64_t frame; int t; int64_t gop_index; uint8_t *res; size_t res_cap, packed_bytes; } job_t;
/* The copies are 1-4 MB each and come and go thousands of times per second: they are recycled through a small pool instead
 * of malloc/free, which at this size is an mmap + page faults + munmap (a TLB shoot-down across all the process's threads). */
#define B2_RES_POOL 96

enum { SLOT_FREE = 0, SLOT_OPEN = 1 /* pictures still arriving */, SLOT_CLOSED = 2 /* the GOP's last picture is in */ };
typedef struct {
    int state;
    int n;                      /* pictures handed over (caller thread writes, under mu)       */
    int issued, fetched;        /* steps issued to / fetched from the GPU (device thread only)  */
    int set[2];                 /* result set of step t in set[t & 1]                           */
    int64_t gop_index, frame0;  /* closed GOP number; frame number of its first picture         */
} slot_t;

typedef struct {
    struct b2_encoder *h;
    int device;
    b2_engine_t *eng;
    pthread_t thread;
    int started;
    pthread_cond_t cv;          /* pictures arrived / a GOP was closed on this GPU              */
    slot_t *slots;
} gpu_t;

struct b2_encoder {
    b2_param_t p;
    int qp, S, L, N, mbw, mbh, nmb;
    int fmt;                    /* raw layout of the pictures in the device rings (B2_FMT_*)    */
    gpu_t dev[B2_MAX_DEVICES];
    b2h_entropy_t *ent;
    b2h_seq_t seq;
    /* everything below is guarded by mu */
    pthread_mutex_t mu;
    pthread_cond_t cv_job, cv_space, cv_out;
    int nworkers;
    pthread_t workers[B2_MAX_WORKERS];
    b2h_entropy_t *went[B2_MAX_WORKERS];
    uint8_t *wscratch[B2_MAX_WORKERS];
    b2_mbinfo_t *winfo[B2_MAX_WORKERS];   /* the worker's expanded decision records */
    job_t *jobs;                /* ring */
    uint8_t *pool[B2_RES_POOL]; /* idle result-copy buffers */
    size_t pool_cap[B2_RES_POOL];
    int pool_n;
    int job_cap, job_head, job_count, job_limit;
    outframe_t *fifo;           /* frame f lives in fifo[f % fifo_cap]                          */
    int fifo_cap;
    int64_t frames_in, frames_out, cur_gop;
    int g_dev, g_slot;          /* slot of the GOP being gathered, -1: none                     */
    int error, stop;
    /* zero-delay mode */
    int gop_pos;
    int64_t gops_done;
    outframe_t zout;
    uint8_t *scratch;
    size_t scratch_cap;
    uint8_t *ret_buf;           /* payload of the frame returned by the last call */
    /* B2ENC_STATS=1: where the threads' time went, printed by b2_encoder_close (seconds; worker_busy under mu) */
    int stats;
    double st_open, st_caller_slot_wait, st_caller_put, st_worker_busy;
    double st_dev_cpu[B2_MAX_DEVICES], st_dev_copy[B2_MAX_DEVICES], st_dev_gpu_wait[B2_MAX_DEVICES], st_dev_idle[B2_MAX_DEVICES];
    long st_dev_rounds[B2_MAX_DEVICES];
    int ns;                     /* slices per picture                                              */
    b2_nal_t *nals;             /* [ns + 2] */
    /* zero-delay slice pool (i_gop_slots = 1, ns > 1), guarded by sp_mu: the caller posts one picture (sp_gen++), the threads take
     * slices k = sp_next++ and write slice k into sp_buf[k] (sp_len[k] bytes, 0 = overflow), the caller waits for sp_done == ns */
    int sp_n;
    pthread_t sp_thread[B2_MAX_WORKERS];
    b2h_entropy_t *sp_ent[B2_MAX_WORKERS];
    uint8_t **sp_buf;
    size_t *sp_cap, *sp_len;
    pthread_mutex_t sp_mu;
    pthread_cond_t sp_cv_go, sp_cv_done;
    long sp_gen;
    int sp_next, sp_done, sp_stop;
    const b2_mbinfo_t *sp_info;
    const uint8_t *sp_packed;
    size_t sp_packed_bytes;
    int sp_t;
    int64_t sp_gop_index;
};

/* ---- picture registry (b2h_picture.h) ------------------------------------------------------------------------------ */
static pthread_mutex_t pic_mu = PTHREAD_MUTEX_INITIALIZER;
static b2h_picrec_t *pic_list;

b2h_picrec_t *b2h_picture_find(const uint8_t *plane0)
{
    if (!plane0) return NULL;
    pthread_mutex_lock(&pic_mu);
    b2h_picrec_t *r = pic_list;
    while (r && r->base != plane0) r = r->next;
    pthread_mutex_unlock(&pic_mu);
    return r;
}

uint8_t *b2h_picture_stage(b2h_picrec_t *r, size_t bytes)
{
    const int k = r->cur ^ 1;
    if (r->busy_eng[k]) {                                 /* the upload of the picture before last */
        b2_engine_put_wait((b2_engine_t *)r->busy_eng[k], r->busy_ticket[k]);
        r->busy_eng[k] = NULL;
    }
    if (r->stage_bytes[k] < bytes) {
        b2_pinned_free(r->stage[k]);
        r->stage[k] = (uint8_t *)b2_pinned_alloc(bytes);
        r->stage_bytes[k] = r->stage[k] ? bytes : 0;
    }
    if (r->stage[k]) r->cur = k;
    return r->stage[k];
}

void b2h_picture_forget_engine(void *eng)
{
    pthread_mutex_lock(&pic_mu);
    for (b2h_picrec_t *r = pic_list; r; r = r->next)
        for (int k = 0; k < 2; k++)
            if (r->busy_eng[k] == eng) r->busy_eng[k] = NULL;
    pthread_mutex_unlock(&pic_mu);
}

int b2_picture_alloc(b2_picture_t *pic, int i_csp, int i_width, int i_height)
{
    if (!pic || i_csp != B2_CSP_I420 || i_width < 2 || i_height < 2) return -1;
    memset(pic, 0, sizeof(*pic));
    int cw = (i_width + 1) / 2, ch = (i_height + 1) / 2;
    size_t ny = (size_t)i_width * i_height, nc = (size_t)cw * ch;
    b2h_picrec_t *r = (b2h_picrec_t *)calloc(1, sizeof(*r));
    uint8_t *buf = r ? (uint8_t *)b2_pinned_alloc(ny + 2 * nc) : NULL;   /* pinned: H2D copies run at full PCIe rate */
    if (!buf) { free(r); return -1; }
    pic->img.i_csp = i_csp; pic->img.i_plane = 3;
    pic->img.plane[0] = buf; pic->img.plane[1] = buf + ny; pic->img.plane[2] = buf + ny + nc;
    pic->img.i_stride[0] = i_width; pic->img.i_stride[1] = cw; pic->img.i_stride[2] = cw;
    pic->opaque = buf;
    r->base = buf; r->bytes = ny + 2 * nc; r->width = i_width; r->height = i_height;
    pthread_mutex_lock(&pic_mu);
    r->next = pic_list; pic_list = r;
    pthread_mutex_unlock(&pic_mu);
    return 0;
}

void b2_picture_clean(b2_picture_t *pic)
{
    if (!pic) return;
    pthread_mutex_lock(&pic_mu);
    b2h_picrec_t **pp = &pic_list, *r = NULL;
    while (*pp && (*pp)->base != pic->opaque) pp = &(*pp)->next;
    if (*pp) { r = *pp; *pp = r->next; }
    pthread_mutex_unlock(&pic_mu);
    if (r) {
        for (int k = 0; k < 2; k++) {
            if (r->busy_eng[k]) b2_engine_put_wait((b2_engine_t *)r->busy_eng[k], r->busy_ticket[k]);
            b2_pinned_free(r->stage[k]);
        }
        free(r);
    }
    b2_pinned_free(pic->opaque);
    memset(pic, 0, sizeof(*pic));
}

/* ---- parameters ---------------------------------------------------------------------------------------------------- */
static const struct { const char *name; int merange, subpel, intra_in_p; } presets[] = {
    {"ultrafast", 16, 0, 0}, {"superfast", 16, 1, 1}, {"veryfast", 16, 1, 1}, {"faster", 16, 1, 1}, {"fast", 16, 1, 1},
    {"medium", 16, 1, 1},    {"slow", 32, 1, 1},      {"slower", 32, 1, 1},   {"veryslow", 32, 1, 1}, {"placebo", 32, 1, 1}};
static const char *tunes[] = {"film", "animation", "grain", "stillimage", "psnr", "ssim", "fastdecode", "zerolatency"};

int b2_param_default_preset(b2_param_t *p, const char *preset, const char *tune)
{
    if (!p) return -1;
    memset(p, 0, sizeof(*p));
    p->i_fps_num = 25; p->i_fps_den = 1;
    p->vui.i_sar_width = p->vui.i_sar_height = 0;
    p->rc.i_rc_method = B2_RC_CRF; p->rc.f_rf_constant = 23.0f; p->rc.i_qp_constant = 26;
    p->b_annexb = 1;
    /* 32 closed GOPs in flight per GPU: fewer leave the GPU waiting on the per-frame latency chain (K7 / K8); with the pruned search
     * 16 slots carry 3,058 and 32 slots 3,708 frames/s at 1080p (profiles/r2s3_slot_stream_probe_pruned.txt) */
    p->i_keyint_max = 32; p->i_gop_slots = 32; p->i_device = 0; p->i_devices = 0; p->b_me_prune = 1; p->i_csp_in = B2_FMT_YUV420P;
    p->b_deblocking_filter = 1;
    p->b_cabac = 1;                      /* x264 default at every preset but ultrafast */
    p->b_transform_8x8 = 0;
    int found = preset == NULL;
    p->i_merange = 16; p->b_subpel = 1; p->b_intra_in_p = 1;
    for (unsigned i = 0; preset && i < sizeof(presets) / sizeof(presets[0]); i++)
        if (!strcmp(preset, presets[i].name)) {
            p->i_merange = presets[i].merange; p->b_subpel = presets[i].subpel; p->b_intra_in_p = presets[i].intra_in_p;
            found = 1;
        }
    if (!found) { fprintf(stderr, "b2enc: invalid preset '%s'\n", preset); return -1; }
    if (preset && !strcmp(preset, "ultrafast")) { p->b_cabac = 0; p->b_deblocking_filter = 0; }     /* as x264's ultrafast */
    if (tune) {
        /* like x264: several tunes separated by ',', './' or ' ' */
        char buf[128];
        if (strlen(tune) >= sizeof(buf)) { fprintf(stderr, "b2enc: invalid tune '%s'\n", tune); return -1; }
        strcpy(buf, tune);
        char *save = NULL;
        for (char *tok = strtok_r(buf, ",./ ", &save); tok; tok = strtok_r(NULL, ",./ ", &save)) {
            int ok = 0;
            for (unsigned i = 0; i < sizeof(tunes) / sizeof(tunes[0]); i++) ok |= !strcmp(tok, tunes[i]);
            if (!ok) { fprintf(stderr, "b2enc: invalid tune '%s'\n", tok); return -1; }
            if (!strcmp(tok, "zerolatency")) p->i_gop_slots = 1;
            /* x264: film = deblock -1:-1, animation = 1:1, grain = -2:-2, stillimage = -3:-3 (the psy settings of those
             * tunes have no counterpart in a constant-QP, non-RD encoder) */
            if (!strcmp(tok, "film")) p->i_deblocking_filter_alphac0 = p->i_deblocking_filter_beta = -1;
            if (!strcmp(tok, "animation")) p->i_deblocking_filter_alphac0 = p->i_deblocking_filter_beta = 1;
            if (!strcmp(tok, "grain")) p->i_deblocking_filter_alphac0 = p->i_deblocking_filter_beta = -2;
            if (!strcmp(tok, "stillimage")) p->i_deblocking_filter_alphac0 = p->i_deblocking_filter_beta = -3;
        }
    }
    return 0;
}

int b2_param_apply_profile(b2_param_t *p, const char *profile)
{
    if (!p) return -1;
    if (!profile) return 0;
    /* like x264_param_apply_profile: a profile only removes tools.  baseline: CAVLC, 4x4 transform; main: no 8x8 transform */
    if (!strcmp(profile, "baseline")) { p->b_cabac = 0; p->b_transform_8x8 = 0; return 0; }
    if (!strcmp(profile, "main")) { p->b_transform_8x8 = 0; return 0; }
    if (!strcmp(profile, "high")) return 0;
    fprintf(stderr, "b2enc: invalid profile: %s\n", profile);
    return -1;
}

/* ---- open / close -------------------------------------------------------------------------------------------------- */
static void *worker_main(void *arg);
static void *dev_main(void *arg);
static void *slice_main(void *arg);

static int slice_count_wanted(const b2_param_t *p)
{
    int n = p->i_slice_count;
    if (n <= 0) {                                        /* an unmodified av_encode.c cannot set the field: environment */
        const char *e = getenv("B2ENC_SLICES");
        n = e ? atoi(e) : 1;
    }
    return n < 1 ? 1 : n;
}

static int device_count_wanted(const b2_param_t *p)
{
    int n = p->i_devices;
    if (n <= 0) {                                        /* an unmodified av_encode.c cannot set the field: environment */
        const char *e = getenv("B2ENC_DEVICES");
        n = e ? atoi(e) : 1;
    }
    return n < 1 ? 1 : n;
}

b2_t *b2_encoder_open(b2_param_t *p)
{
    if (!p || p->i_width < 16 || p->i_height < 16) { fprintf(stderr, "b2enc: bad picture size\n"); return NULL; }
    if ((long)((p->i_width + 15) / 16) * ((p->i_height + 15) / 16) > 36864) {          /* MaxFS of level 5.2, the largest there is */
        fprintf(stderr, "b2enc: %dx%d exceeds H.264 level 5.2 (36,864 macroblocks per frame)\n", p->i_width, p->i_height);
        return NULL;
    }
    b2_t *h = (b2_t *)calloc(1, sizeof(*h));
    if (!h) return NULL;
    h->p = *p;
    h->g_slot = -1;
    { const char *ev = getenv("B2ENC_STATS"); h->stats = ev && atoi(ev) > 0; h->st_open = now_s(); }
    int qp = p->rc.i_rc_method == B2_RC_CQP ? p->rc.i_qp_constant : (int)(p->rc.f_rf_constant + 0.5f);
    if (qp < 10 || qp > 51)
        fprintf(stderr, "b2enc: quality %d is outside the supported constant-QP range, using %d\n", qp, qp < 10 ? 10 : 51);
    h->qp = qp < 10 ? 10 : (qp > 51 ? 51 : qp);      /* CRF is mapped to a constant QP (north_star: fixed QP) */
    h->S = p->i_gop_slots > 0 ? p->i_gop_slots : 1;
    h->L = p->i_keyint_max > 0 ? p->i_keyint_max : 32;
    h->N = h->S == 1 ? 1 : device_count_wanted(p);
    h->fmt = p->i_csp_in;
    const int ndev = b2_device_count();
    if (ndev <= 0) { fprintf(stderr, "b2enc: no CUDA device; the encode stage has no CPU fallback\n"); free(h); return NULL; }
    if (h->N > B2_MAX_DEVICES) h->N = B2_MAX_DEVICES;
    if (p->i_device < 0 || p->i_device + h->N > ndev) {
        fprintf(stderr, "b2enc: devices %d..%d requested, %d visible\n", p->i_device, p->i_device + h->N - 1, ndev);
        free(h);
        return NULL;
    }
    pthread_mutex_init(&h->mu, NULL);
    pthread_cond_init(&h->cv_job, NULL); pthread_cond_init(&h->cv_space, NULL); pthread_cond_init(&h->cv_out, NULL);
    b2_engine_cfg_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.width = p->i_width; cfg.height = p->i_height;
    cfg.in_fmt = p->i_csp_in; cfg.merange = p->i_merange ? p->i_merange : 16; cfg.qp = h->qp;
    cfg.subpel = p->b_subpel; cfg.intra_in_p = p->b_intra_in_p; cfg.profile = 0; cfg.deblock = p->b_deblocking_filter;
    cfg.deblock_alpha = p->i_deblocking_filter_alphac0; cfg.deblock_beta = p->i_deblocking_filter_beta;
    cfg.transform8x8 = p->b_transform_8x8 != 0;
    cfg.partitions = p->b_partitions < 0 ? 0 : (p->b_partitions > 2 ? 2 : p->b_partitions);
    cfg.pack_levels = 1;                              /* only blocks with a non-zero level cross PCIe (K9) */
    {
        const char *ev = getenv("B2ENC_ME_PRUNE");
        cfg.me_prune = ev ? atoi(ev) != 0 : p->b_me_prune != 0;
    }
    /* every GOP slot holds its GOP's raw pictures on the device: shrink the slot count to what the GPU can hold */
    {
        const size_t w16 = ((size_t)p->i_width + 15) & ~(size_t)15, h16 = ((size_t)p->i_height + 15) & ~(size_t)15;
        const size_t per_slot = (size_t)h->L * w16 * h16 * 3 + 20 * (w16 + 128) * (h16 + 128);      /* ring (<= 3 B/px) + planes, block-sum words + results */
        size_t free_b = 0, total_b = 0;
        for (int d = 0; d < h->N && h->S > 1; d++) {
            if (b2_device_mem_info(p->i_device + d, &free_b, &total_b)) continue;
            int fit = (int)(free_b * 8 / 10 / per_slot);
            if (fit < 2) {
                fprintf(stderr, "b2enc: keyint %d x %dx%d needs %.1f GB per GOP slot, device %d has %.1f GB free\n", h->L,
                        p->i_width, p->i_height, per_slot / 1e9, p->i_device + d, free_b / 1e9);
                b2_encoder_close(h);
                return NULL;
            }
            if (fit < h->S) {
                fprintf(stderr, "b2enc: %d GOP slots of %d frames do not fit device %d, using %d\n", h->S, h->L, p->i_device + d, fit);
                h->S = fit;
            }
        }
    }
    cfg.slices = slice_count_wanted(p);
    cfg.slots = h->S; cfg.streams = h->S;             /* one stream group per slot: every GOP advances on its own */
    cfg.in_ring = h->S == 1 ? 1 : h->L;
    for (int d = 0; d < h->N; d++) {
        gpu_t *dv = &h->dev[d];
        dv->h = h; dv->device = p->i_device + d;
        cfg.device = dv->device;
        dv->eng = b2_engine_create(&cfg);
        dv->slots = (slot_t *)calloc((size_t)h->S, sizeof(slot_t));
        pthread_cond_init(&dv->cv, NULL);
        if (!dv->eng || !dv->slots) { b2_encoder_close(h); return NULL; }
    }
    int w16, h16;
    b2_engine_geometry(h->dev[0].eng, &h->mbw, &h->mbh, &w16, &h16);
    h->nmb = h->mbw * h->mbh;
    h->ent = b2h_entropy_create(h->mbw, h->mbh);
    h->seq.width = p->i_width; h->seq.height = p->i_height; h->seq.fps_num = p->i_fps_num; h->seq.fps_den = p->i_fps_den;
    h->seq.sar_w = p->vui.i_sar_width; h->seq.sar_h = p->vui.i_sar_height; h->seq.qp = h->qp;
    h->seq.deblock = p->b_deblocking_filter;
    h->seq.deblock_alpha = p->i_deblocking_filter_alphac0; h->seq.deblock_beta = p->i_deblocking_filter_beta;
    h->seq.cabac = p->b_cabac != 0; h->seq.transform8x8 = p->b_transform_8x8 != 0;
    h->ns = b2_slice_count(cfg.slices, h->mbh);
    h->scratch_cap = (size_t)h->nmb * 3072 + 65536 * (size_t)h->ns;
    h->scratch = (uint8_t *)malloc(h->scratch_cap);
    h->nals = (b2_nal_t *)calloc((size_t)h->ns + 2, sizeof(b2_nal_t));
    if (!h->ent || !h->scratch || !h->nals) { b2_encoder_close(h); return NULL; }
    pthread_mutex_init(&h->sp_mu, NULL);
    pthread_cond_init(&h->sp_cv_go, NULL); pthread_cond_init(&h->sp_cv_done, NULL);
    if (h->S == 1 && h->ns > 1) {
        long ncpu = sysconf(_SC_NPROCESSORS_ONLN);
        int nt = ncpu > 2 ? (int)ncpu - 1 : 1;
        if (nt > h->ns) nt = h->ns;
        if (nt > B2_MAX_WORKERS) nt = B2_MAX_WORKERS;
        h->sp_buf = (uint8_t **)calloc((size_t)h->ns, sizeof(uint8_t *));
        h->sp_cap = (size_t *)calloc((size_t)h->ns, sizeof(size_t)); h->sp_len = (size_t *)calloc((size_t)h->ns, sizeof(size_t));
        if (!h->sp_buf || !h->sp_cap || !h->sp_len) { b2_encoder_close(h); return NULL; }
        for (int k = 0; k < h->ns; k++) {
            const int rows = b2_slice_row(k + 1, h->ns, h->mbh) - b2_slice_row(k, h->ns, h->mbh);
            h->sp_cap[k] = (size_t)rows * h->mbw * 3072 + 65536;
            if (!(h->sp_buf[k] = (uint8_t *)malloc(h->sp_cap[k]))) { b2_encoder_close(h); return NULL; }
        }
        for (int i = 0; i < nt; i++)
            if (!(h->sp_ent[i] = b2h_entropy_create(h->mbw, h->mbh))) { b2_encoder_close(h); return NULL; }
        pthread_mutex_lock(&h->sp_mu);                   /* the threads look themselves up in sp_thread[] under the lock */
        for (int i = 0; i < nt; i++) {
            if (pthread_create(&h->sp_thread[i], NULL, slice_main, h)) break;
            h->sp_n++;
        }
        pthread_mutex_unlock(&h->sp_mu);
        if (h->sp_n == 0) { b2_encoder_close(h); return NULL; }
    }
    if (h->S > 1) {
        long ncpu = sysconf(_SC_NPROCESSORS_ONLN);
        int nw = ncpu > 2 ? (int)ncpu - 1 : 1;          /* frames, not GOPs, are the unit of work: use the cores there are */
        if (nw > B2_MAX_WORKERS) nw = B2_MAX_WORKERS;
        const char *e = getenv("B2ENC_ENTROPY_THREADS");
        if (e && atoi(e) > 0) nw = atoi(e) > B2_MAX_WORKERS ? B2_MAX_WORKERS : atoi(e);
        h->job_limit = 4 * nw > 64 ? 4 * nw : 64;
        /* frames in flight: N x S slots of L pictures + what waits for / sits in the entropy stage or for the caller */
        h->fifo_cap = (h->N * h->S + 2) * h->L + h->job_limit;
        h->job_cap = h->fifo_cap;
        h->fifo = (outframe_t *)calloc((size_t)h->fifo_cap, sizeof(outframe_t));
        h->jobs = (job_t *)calloc((size_t)h->job_cap, sizeof(job_t));
        if (!h->fifo || !h->jobs) { b2_encoder_close(h); return NULL; }
        for (int i = 0; i < nw; i++) {
            h->went[i] = b2h_entropy_create(h->mbw, h->mbh);
            h->wscratch[i] = (uint8_t *)malloc(h->scratch_cap);
            h->winfo[i] = (b2_mbinfo_t *)malloc((size_t)h->nmb * sizeof(b2_mbinfo_t));
            if (!h->went[i] || !h->wscratch[i] || !h->winfo[i]) { b2_encoder_close(h); return NULL; }
        }
        pthread_mutex_lock(&h->mu);                      /* workers look themselves up in h->workers[] under the lock */
        for (int i = 0; i < nw; i++) {
            if (pthread_create(&h->workers[i], NULL, worker_main, h)) break;
            h->nworkers++;
        }
        pthread_mutex_unlock(&h->mu);
        if (h->nworkers == 0) { b2_encoder_close(h); return NULL; }
        for (int d = 0; d < h->N; d++) {
            if (pthread_create(&h->dev[d].thread, NULL, dev_main, &h->dev[d])) { b2_encoder_close(h); return NULL; }
            h->dev[d].started = 1;
        }
    }
    return h;
}

void b2_encoder_close(b2_t *h)
{
    if (!h) return;
    pthread_mutex_lock(&h->mu);
    h->stop = 1;
    pthread_cond_broadcast(&h->cv_job); pthread_cond_broadcast(&h->cv_space); pthread_cond_broadcast(&h->cv_out);
    for (int d = 0; d < h->N; d++)
        if (h->dev[d].started) pthread_cond_broadcast(&h->dev[d].cv);
    pthread_mutex_unlock(&h->mu);
    for (int d = 0; d < h->N; d++)
        if (h->dev[d].started) pthread_join(h->dev[d].thread, NULL);
    for (int i = 0; i < h->nworkers; i++) pthread_join(h->workers[i], NULL);
    if (h->sp_n) {
        pthread_mutex_lock(&h->sp_mu);
        h->sp_stop = 1;
        pthread_cond_broadcast(&h->sp_cv_go);
        pthread_mutex_unlock(&h->sp_mu);
        for (int i = 0; i < h->sp_n; i++) pthread_join(h->sp_thread[i], NULL);
    }
    for (int i = 0; i < B2_MAX_WORKERS; i++) b2h_entropy_destroy(h->sp_ent[i]);
    if (h->sp_buf)
        for (int k = 0; k < h->ns; k++) free(h->sp_buf[k]);
    free(h->sp_buf); free(h->sp_cap); free(h->sp_len);
    if (h->stats && h->S > 1) {
        const double wall = now_s() - h->st_open;
        fprintf(stderr, "b2enc stats: %lld frames, %.3f s since open | caller: %.3f s waiting for a GOP slot / the fifo, %.3f s handing pictures over | "
                        "%d entropy workers: %.3f s busy in total (%.2f ms per frame)\n", (long long)h->frames_in, wall, h->st_caller_slot_wait,
                h->st_caller_put, h->nworkers, h->st_worker_busy, h->frames_in ? 1e3 * h->st_worker_busy / (double)h->frames_in : 0.0);
        for (int d = 0; d < h->N; d++)
            fprintf(stderr, "b2enc stats: GPU thread %d: %.3f s CPU, of it %.3f s copying result sets out of pinned memory; asleep %.3f s on a result set, "
                            "%.3f s without work; %ld rounds\n", h->dev[d].device, h->st_dev_cpu[d], h->st_dev_copy[d], h->st_dev_gpu_wait[d],
                    h->st_dev_idle[d], h->st_dev_rounds[d]);
    }
    for (int i = 0; i < B2_MAX_WORKERS; i++) { b2h_entropy_destroy(h->went[i]); free(h->wscratch[i]); free(h->winfo[i]); }
    if (h->jobs)
        for (int i = 0; i < h->job_count; i++) free(h->jobs[(h->job_head + i) % h->job_cap].res);     /* queued, never coded */
    free(h->jobs);
    for (int i = 0; i < h->pool_n; i++) free(h->pool[i]);
    if (h->fifo)
        for (int i = 0; i < h->fifo_cap; i++) { free(h->fifo[i].data); free(h->fifo[i].nal); }
    free(h->fifo);
    free(h->zout.data); free(h->zout.nal); free(h->scratch); free(h->ret_buf); free(h->nals);
    b2h_entropy_destroy(h->ent);
    for (int d = 0; d < B2_MAX_DEVICES; d++) {
        if (h->dev[d].eng) { b2h_picture_forget_engine(h->dev[d].eng); b2_engine_destroy(h->dev[d].eng); }
        if (h->dev[d].slots) { free(h->dev[d].slots); pthread_cond_destroy(&h->dev[d].cv); }
    }
    pthread_mutex_destroy(&h->mu);
    pthread_cond_destroy(&h->cv_job); pthread_cond_destroy(&h->cv_space); pthread_cond_destroy(&h->cv_out);
    if (h->nals) {                                       /* initialised together with the table */
        pthread_mutex_destroy(&h->sp_mu);
        pthread_cond_destroy(&h->sp_cv_go); pthread_cond_destroy(&h->sp_cv_done);
    }
    free(h);
}

/* ---- result-copy buffers ------------------------------------------------------------------------------------------- */
/* smallest idle buffer that holds `need` bytes (P frames leave the few large ones to the I frames), else a new one */
static uint8_t *res_take(b2_t *h, size_t need, size_t *cap)
{
    uint8_t *buf = NULL;
    pthread_mutex_lock(&h->mu);
    int best = -1;
    for (int i = 0; i < h->pool_n; i++)
        if (h->pool_cap[i] >= need && (best < 0 || h->pool_cap[i] < h->pool_cap[best])) best = i;
    if (best >= 0) {
        buf = h->pool[best]; *cap = h->pool_cap[best];
        h->pool_n--;
        h->pool[best] = h->pool[h->pool_n]; h->pool_cap[best] = h->pool_cap[h->pool_n];
    }
    pthread_mutex_unlock(&h->mu);
    if (!buf) {
        *cap = need + need / 4 + 4096;                    /* some slack: the next frame of the kind is rarely exactly as large */
        buf = (uint8_t *)malloc(*cap);
    }
    return buf;
}
/* call with h->mu held.  A full pool drops its smallest buffer. */
static void res_give_locked(b2_t *h, uint8_t *buf, size_t cap)
{
    if (!buf) return;
    if (h->pool_n < B2_RES_POOL) { h->pool[h->pool_n] = buf; h->pool_cap[h->pool_n] = cap; h->pool_n++; return; }
    int small = 0;
    for (int i = 1; i < h->pool_n; i++)
        if (h->pool_cap[i] < h->pool_cap[small]) small = i;
    if (h->pool_cap[small] < cap) { free(h->pool[small]); h->pool[small] = buf; h->pool_cap[small] = cap; }
    else free(buf);
}

/* ---- entropy stage ------------------------------------------------------------------------------------------------- */
static void put_prefix(uint8_t *d, int annexb, size_t nal_size)
{
    if (annexb) { d[0] = 0; d[1] = 0; d[2] = 0; d[3] = 1; }
    else { d[0] = (uint8_t)(nal_size >> 24); d[1] = (uint8_t)(nal_size >> 16); d[2] = (uint8_t)(nal_size >> 8); d[3] = (uint8_t)nal_size; }
}

static void add_nal(b2_t *h, outframe_t *o, uint8_t *at, size_t pos, size_t n, int type, int ref)
{
    put_prefix(at, h->p.b_annexb, n);
    o->nal[o->nal_count].off = (int)pos; o->nal[o->nal_count].size = (int)n + 4;
    o->nal[o->nal_count].type = type; o->nal[o->nal_count].ref = ref;
    o->nal_count++;
}

/* slice k of the picture (macroblock rows b2_slice_row(k) .. b2_slice_row(k + 1)) as one NAL into out[0..cap) */
static size_t write_slice_k(b2_t *h, b2h_entropy_t *ent, int k, const b2_mbinfo_t *info, const uint8_t *packed, size_t packed_bytes,
                            int t, int64_t gop_index, uint8_t *out, size_t cap)
{
    const int r0 = b2_slice_row(k, h->ns, h->mbh), r1 = b2_slice_row(k + 1, h->ns, h->mbh);
    return b2h_write_slice_rows_packed(ent, &h->seq, t == 0 ? B2_FRAME_I : B2_FRAME_P, t, (int)(gop_index & 0xffff), r0, r1 - r0, info,
                                       packed, packed_bytes, out, cap);
}

/* zero-delay slice pool: one thread of it */
static void *slice_main(void *arg)
{
    b2_t *h = (b2_t *)arg;
    b2h_entropy_t *ent = NULL;
    long seen = 0;
    pthread_mutex_lock(&h->sp_mu);
    for (int i = 0; i < h->sp_n; i++)
        if (pthread_equal(h->sp_thread[i], pthread_self())) ent = h->sp_ent[i];
    for (;;) {
        while (!h->sp_stop && h->sp_gen == seen) pthread_cond_wait(&h->sp_cv_go, &h->sp_mu);
        if (h->sp_stop) break;
        seen = h->sp_gen;
        while (h->sp_next < h->ns) {
            const int k = h->sp_next++;
            const b2_mbinfo_t *info = h->sp_info; const uint8_t *packed = h->sp_packed;
            const size_t packed_bytes = h->sp_packed_bytes; const int t = h->sp_t; const int64_t gi = h->sp_gop_index;
            pthread_mutex_unlock(&h->sp_mu);
            const size_t n = ent ? write_slice_k(h, ent, k, info, packed, packed_bytes, t, gi, h->sp_buf[k] + 4, h->sp_cap[k] - 4) : 0;
            pthread_mutex_lock(&h->sp_mu);
            h->sp_len[k] = n;
            if (++h->sp_done == h->ns) pthread_cond_signal(&h->sp_cv_done);
        }
    }
    pthread_mutex_unlock(&h->sp_mu);
    return NULL;
}

/* entropy-code one frame's results into *o (data, size, NAL table, key) */
static int finish_frame(b2_t *h, b2h_entropy_t *ent, uint8_t *s, const b2_mbinfo_t *info, const uint8_t *packed, size_t packed_bytes,
                        int t, int64_t gop_index, outframe_t *o)
{
    size_t pos = 0;
    o->nal_count = 0;
    free(o->nal);
    o->nal = (nalrec_t *)malloc(sizeof(nalrec_t) * ((size_t)h->ns + 2));
    if (!o->nal) return -1;
    const int is_idr = t == 0;
    if (is_idr) {
        for (int k = 0; k < 2; k++) {
            size_t n = k == 0 ? b2h_write_sps(&h->seq, s + pos + 4, h->scratch_cap - pos - 4)
                              : b2h_write_pps(&h->seq, s + pos + 4, h->scratch_cap - pos - 4);
            if (!n) return -1;
            add_nal(h, o, s + pos, pos, n, k == 0 ? B2_NAL_SPS : B2_NAL_PPS, 3);
            pos += n + 4;
        }
    }
    if (!info || !packed) return -1;
    if (h->sp_n) {                                        /* zero delay, several slices: the pool writes them at the same time */
        pthread_mutex_lock(&h->sp_mu);
        h->sp_info = info; h->sp_packed = packed; h->sp_packed_bytes = packed_bytes; h->sp_t = t; h->sp_gop_index = gop_index;
        h->sp_next = 0; h->sp_done = 0; h->sp_gen++;
        pthread_cond_broadcast(&h->sp_cv_go);
        while (h->sp_done < h->ns) pthread_cond_wait(&h->sp_cv_done, &h->sp_mu);
        pthread_mutex_unlock(&h->sp_mu);
    }
    for (int k = 0; k < h->ns; k++) {
        size_t n;
        if (h->sp_n) {
            n = h->sp_len[k];
            if (n && n + 4 <= h->scratch_cap - pos) memcpy(s + pos + 4, h->sp_buf[k] + 4, n);
            else n = 0;
        } else {
            n = write_slice_k(h, ent, k, info, packed, packed_bytes, t, gop_index, s + pos + 4, h->scratch_cap - pos - 4);
        }
        if (!n) { fprintf(stderr, "b2enc: slice buffer overflow\n"); return -1; }
        add_nal(h, o, s + pos, pos, n, is_idr ? B2_NAL_SLICE_IDR : B2_NAL_SLICE, is_idr ? 3 : 2);
        pos += n + 4;
    }
    free(o->data);
    o->data = (uint8_t *)malloc(pos);
    if (!o->data) return -1;
    memcpy(o->data, s, pos);
    o->size = (int)pos;
    o->key = is_idr;
    return 0;
}

static void *worker_main(void *arg)
{
    b2_t *h = (b2_t *)arg;
    int me = -1;
    /* The entropy workers are the bulk of the CPU time but not the critical path: the caller's thread, its staging-copy helpers
     * and the per-GPU threads each serialise a whole stream or GPU, and on a host whose cores are all busy a just-woken helper
     * that waits for a time slice stalls the caller.  The workers therefore run at a lower priority (Linux: the nice value is
     * per thread; raising it needs no privilege).  B2ENC_WORKER_NICE=0 turns it off. */
    {
        const char *ev = getenv("B2ENC_WORKER_NICE");
        const int nice_by = ev ? atoi(ev) : 10;
#ifdef SYS_gettid
        if (nice_by > 0) setpriority(PRIO_PROCESS, (id_t)syscall(SYS_gettid), nice_by > 19 ? 19 : nice_by);
#endif
    }
    pthread_mutex_lock(&h->mu);
    for (int i = 0; i < h->nworkers; i++)
        if (pthread_equal(h->workers[i], pthread_self())) me = i;
    for (;;) {
        while (!h->stop && h->job_count == 0) pthread_cond_wait(&h->cv_job, &h->mu);
        if (h->stop) break;
        job_t j = h->jobs[h->job_head];
        h->job_head = (h->job_head + 1) % h->job_cap;
        h->job_count--;
        pthread_cond_signal(&h->cv_space);
        pthread_mutex_unlock(&h->mu);
        outframe_t o;
        memset(&o, 0, sizeof(o));
        const double w0 = h->stats ? now_s() : 0.0;
        b2h_info_unpack((const b2_mbinfo_packed_t *)j.res, h->winfo[me], h->nmb);
        int rc = finish_frame(h, h->went[me], h->wscratch[me], h->winfo[me], j.res + (size_t)h->nmb * sizeof(b2_mbinfo_packed_t),
                              j.packed_bytes, j.t, j.gop_index, &o);
        const double w1 = h->stats ? now_s() : 0.0;
        pthread_mutex_lock(&h->mu);
        h->st_worker_busy += w1 - w0;
        res_give_locked(h, j.res, j.res_cap);
        if (rc) { h->error = 1; free(o.data); free(o.nal); }
        else {
            outframe_t *dst = &h->fifo[j.frame % h->fifo_cap];
            o.pts = dst->pts;                              /* written by the caller's thread when the picture came in */
            free(dst->data); free(dst->nal);
            *dst = o;
            dst->ready = 1;
        }
        pthread_cond_broadcast(&h->cv_out);
    }
    pthread_mutex_unlock(&h->mu);
    return NULL;
}

/* ---- per-GPU thread ------------------------------------------------------------------------------------------------ */
static void fail(b2_t *h)
{
    pthread_mutex_lock(&h->mu);
    h->error = 1;
    pthread_cond_broadcast(&h->cv_out);
    pthread_mutex_unlock(&h->mu);
}

/* copy step t's result set of slot s out of the pinned buffers and queue it for the entropy workers */
static int fetch_step(gpu_t *dv, int s, int t, int set)
{
    b2_t *h = dv->h;
    slot_t *sl = &dv->slots[s];
    const b2_mbinfo_packed_t *info = b2_engine_info_packed_set(dv->eng, set, s);
    size_t packed_bytes = 0;
    const uint8_t *packed = b2_engine_packed_set(dv->eng, set, s, &packed_bytes);
    if (!info || !packed) return -1;
    const size_t ni = (size_t)h->nmb * sizeof(b2_mbinfo_packed_t);
    job_t j = {sl->frame0 + t, t, sl->gop_index, NULL, 0, packed_bytes};
    j.res = res_take(h, ni + packed_bytes + 1, &j.res_cap);
    if (!j.res) return -1;
    const double c0 = h->stats ? now_s() : 0.0;
    memcpy(j.res, info, ni);
    memcpy(j.res + ni, packed, packed_bytes);
    if (h->stats) h->st_dev_copy[dv - h->dev] += now_s() - c0;
    pthread_mutex_lock(&h->mu);
    while (!h->stop && h->job_count >= h->job_limit) pthread_cond_wait(&h->cv_space, &h->mu);   /* entropy stage is behind: let the GPU wait */
    if (h->stop) { pthread_mutex_unlock(&h->mu); free(j.res); return 0; }
    h->jobs[(h->job_head + h->job_count) % h->job_cap] = j;
    h->job_count++;
    pthread_cond_signal(&h->cv_job);
    pthread_mutex_unlock(&h->mu);
    return 0;
}

static int slot_runnable(const slot_t *sl)
{
    return sl->state != SLOT_FREE && (sl->issued < sl->n || sl->fetched < sl->issued || sl->state == SLOT_CLOSED);
}

static void *dev_main(void *arg)
{
    gpu_t *dv = (gpu_t *)arg;
    b2_t *h = dv->h;
    const int S = h->S;
    int *n_snap = (int *)calloc((size_t)S, sizeof(int)), *st_snap = (int *)calloc((size_t)S, sizeof(int));
    if (!n_snap || !st_snap) { fail(h); free(n_snap); free(st_snap); return NULL; }
    int rr = 0;                                               /* which outstanding result set to sleep on: round robin */
    for (;;) {
        pthread_mutex_lock(&h->mu);
        for (;;) {
            int any = 0;
            for (int s = 0; s < S; s++) any |= slot_runnable(&dv->slots[s]);
            if (h->stop || h->error || any) break;
            const double i0 = h->stats ? now_s() : 0.0;
            pthread_cond_wait(&dv->cv, &h->mu);
            if (h->stats) h->st_dev_idle[dv - h->dev] += now_s() - i0;
        }
        if (h->stop || h->error) { pthread_mutex_unlock(&h->mu); break; }
        for (int s = 0; s < S; s++) { n_snap[s] = dv->slots[s].n; st_snap[s] = dv->slots[s].state; }
        pthread_mutex_unlock(&h->mu);
        int progress = 0, err = 0;
        h->st_dev_rounds[dv - h->dev]++;
        for (int s = 0; s < S && !err; s++) {
            slot_t *sl = &dv->slots[s];
            if (st_snap[s] == SLOT_FREE) continue;
            const int n = n_snap[s];
            for (;;) {
                if (sl->fetched < sl->issued) {               /* has the oldest step in flight landed? */
                    const int set = sl->set[sl->fetched & 1];
                    const int r = b2_engine_group_done(dv->eng, s, set);
                    if (r < 0) { err = 1; break; }
                    if (r == 1) {
                        if (fetch_step(dv, s, sl->fetched, set)) { err = 1; break; }
                        sl->fetched++; progress = 1;
                        continue;
                    }
                }
                if (sl->issued < n && sl->issued - sl->fetched < 2) {      /* two steps in flight per slot (two result sets) */
                    const int t = sl->issued;
                    if (b2_engine_encode_group(dv->eng, s, t == 0 ? B2_FRAME_I : B2_FRAME_P, t) || b2_engine_d2h_group(dv->eng, s)) { err = 1; break; }
                    sl->set[t & 1] = b2_engine_group_result_set(dv->eng, s);
                    sl->issued++; progress = 1;
                    continue;
                }
                break;
            }
            if (!err && st_snap[s] == SLOT_CLOSED && sl->fetched == n) {  /* the GOP has left the GPU: the slot is free again */
                pthread_mutex_lock(&h->mu);
                sl->state = SLOT_FREE;
                pthread_cond_broadcast(&h->cv_out);
                pthread_mutex_unlock(&h->mu);
                progress = 1;
            }
        }
        if (err) { fail(h); break; }
        if (!progress) {                                      /* everything issued, nothing landed: sleep on a result set */
            int waited = 0;
            for (int k = 0; k < S && !waited; k++) {
                const int s = (rr + k) % S;
                slot_t *sl = &dv->slots[s];
                if (st_snap[s] != SLOT_FREE && sl->fetched < sl->issued) {
                    const double g0 = h->stats ? now_s() : 0.0;
                    if (b2_engine_group_wait(dv->eng, s, sl->set[sl->fetched & 1])) { fail(h); free(n_snap); free(st_snap); return NULL; }
                    if (h->stats) h->st_dev_gpu_wait[dv - h->dev] += now_s() - g0;
                    rr = s + 1; waited = 1;
                }
            }
            if (!waited) {                                    /* open slots waiting for their next picture */
                pthread_mutex_lock(&h->mu);
                int changed = 0;
                for (int s = 0; s < S; s++) changed |= dv->slots[s].n != n_snap[s] || dv->slots[s].state != st_snap[s];
                const double i0 = h->stats ? now_s() : 0.0;
                if (!changed && !h->stop && !h->error) pthread_cond_wait(&dv->cv, &h->mu);
                if (h->stats) h->st_dev_idle[dv - h->dev] += now_s() - i0;
                pthread_mutex_unlock(&h->mu);
            }
        }
    }
    h->st_dev_cpu[dv - h->dev] = thread_cpu_s();
    free(n_snap); free(st_snap);
    return NULL;
}

/* ---- the calls of the reference's loops ------------------------------------------------------------------------------ */
int b2_encoder_delayed_frames(b2_t *h)
{
    if (!h || h->S == 1) return 0;
    pthread_mutex_lock(&h->mu);
    const int n = (int)(h->frames_in - h->frames_out);
    pthread_mutex_unlock(&h->mu);
    return n;
}

static int return_frame(b2_t *h, outframe_t *o, b2_nal_t **pp_nal, int *pi_nal, b2_picture_t *pic_out)
{
    free(h->ret_buf);
    h->ret_buf = o->data; o->data = NULL;                           /* hand the payload over; valid until the next call */
    for (int i = 0; i < o->nal_count; i++) {
        h->nals[i].i_ref_idc = o->nal[i].ref; h->nals[i].i_type = o->nal[i].type;
        h->nals[i].i_payload = o->nal[i].size; h->nals[i].p_payload = h->ret_buf + o->nal[i].off;
    }
    *pp_nal = h->nals; *pi_nal = o->nal_count;
    if (pic_out) {
        memset(pic_out, 0, sizeof(*pic_out));
        pic_out->i_pts = o->pts; pic_out->i_dts = o->pts; pic_out->b_keyframe = o->key;
        pic_out->i_type = o->key ? B2_TYPE_IDR : B2_TYPE_P;
    }
    return o->size;
}

/* where the picture's pixels are and in which layout: the I420 planes, or -- when b2_sws_scale deferred the conversion into
 * this picture -- the staged raw source (b2h_picture.h) */
static int picture_source(b2_t *h, b2_picture_t *pic, const uint8_t *src[4], int stride[4], int *fmt, b2h_picrec_t **staged)
{
    b2h_picrec_t *r = b2h_picture_find(pic->img.plane[0]);
    *staged = NULL;
    if (r && r->deferred) {
        int rb[3], rows[3];
        const int np = b2_fmt_layout(r->fmt, h->p.i_width, h->p.i_height, rb, rows);
        if (!np || r->width != h->p.i_width || r->height != h->p.i_height) return -1;
        const uint8_t *q = r->stage[r->cur];
        *staged = r;
        for (int k = 0; k < 4; k++) { src[k] = NULL; stride[k] = 0; }
        for (int k = 0; k < np; k++) { src[k] = q; stride[k] = rb[k]; q += (size_t)rb[k] * rows[k]; }
        *fmt = r->fmt;
        r->deferred = 0;
        return 0;
    }
    for (int k = 0; k < 4; k++) { src[k] = pic->img.plane[k]; stride[k] = pic->img.i_stride[k]; }
    *fmt = r ? B2_FMT_YUV420P : h->p.i_csp_in;              /* b2_picture_alloc pictures are I420 by construction */
    return 0;
}

/* the raw layout of the incoming pictures changed (first deferred picture, normally): drain, then re-shape the device rings */
static int switch_format(b2_t *h, int fmt)
{
    if (h->S > 1) {
        pthread_mutex_lock(&h->mu);
        if (h->g_slot >= 0) {                                 /* close the GOP being gathered: it stays in the old layout */
            h->dev[h->g_dev].slots[h->g_slot].state = SLOT_CLOSED;
            pthread_cond_broadcast(&h->dev[h->g_dev].cv);
            h->g_slot = -1; h->cur_gop++;
        }
        for (;;) {
            int busy = 0;
            for (int d = 0; d < h->N; d++)
                for (int s = 0; s < h->S; s++) busy |= h->dev[d].slots[s].state != SLOT_FREE;
            if (!busy || h->error) break;
            pthread_cond_wait(&h->cv_out, &h->mu);
        }
        pthread_mutex_unlock(&h->mu);
    }
    for (int d = 0; d < h->N; d++)
        if (b2_engine_set_input_format(h->dev[d].eng, fmt)) return -1;
    h->fmt = fmt;
    return 0;
}

static int encode_zero_delay(b2_t *h, b2_nal_t **pp_nal, int *pi_nal, const uint8_t *src[4], const int stride[4], int64_t pts,
                             b2_picture_t *pic_out)
{
    b2_engine_t *eng = h->dev[0].eng;
    const int t = h->gop_pos;
    if (b2_engine_put_picture(eng, 0, 0, src, stride)) return -1;
    if (b2_engine_encode_group(eng, 0, t == 0 ? B2_FRAME_I : B2_FRAME_P, 0) || b2_engine_d2h_group(eng, 0)) return -1;
    const int set = b2_engine_group_result_set(eng, 0);
    if (b2_engine_group_wait(eng, 0, set)) return -1;
    size_t packed_bytes = 0;
    const uint8_t *packed = b2_engine_packed_set(eng, set, 0, &packed_bytes);
    if (finish_frame(h, h->ent, h->scratch, b2_engine_info_set(eng, set, 0), packed, packed_bytes, t, h->gops_done, &h->zout)) return -1;
    h->zout.pts = pts;
    h->gop_pos = t + 1;
    if (h->gop_pos == h->L) { h->gop_pos = 0; h->gops_done++; }
    return return_frame(h, &h->zout, pp_nal, pi_nal, pic_out);
}

int b2_encoder_encode(b2_t *h, b2_nal_t **pp_nal, int *pi_nal, b2_picture_t *pic_in, b2_picture_t *pic_out)
{
    if (!h || !pp_nal || !pi_nal) return -1;
    *pi_nal = 0; *pp_nal = NULL;
    const uint8_t *src[4]; int stride[4], fmt = h->fmt;
    b2h_picrec_t *staged = NULL;                              /* the picture's pixels sit in library-owned staging (deferred sws_scale) */
    if (pic_in) {
        if (picture_source(h, pic_in, src, stride, &fmt, &staged)) { fprintf(stderr, "b2enc: picture does not match the encoder's size\n"); return -1; }
        if (fmt != h->fmt && switch_format(h, fmt)) return -1;
    }
    if (h->S == 1) return pic_in ? encode_zero_delay(h, pp_nal, pi_nal, src, stride, pic_in->i_pts, pic_out) : 0;

    pthread_mutex_lock(&h->mu);
    if (pic_in) {
        /* never more than fifo_cap - 1 frames delayed: when the caller is that far ahead, this call waits for the oldest frame
         * (returned below), like x264 blocks on its oldest frame thread */
        const double q0 = h->stats ? now_s() : 0.0;
        while (!h->error && h->frames_in - h->frames_out >= h->fifo_cap - 1 && !h->fifo[h->frames_out % h->fifo_cap].ready)
            pthread_cond_wait(&h->cv_out, &h->mu);
        if (h->g_slot < 0) {                                  /* a new closed GOP: GPU k % N, any free slot there */
            gpu_t *dv = &h->dev[h->cur_gop % h->N];
            int s = -1;
            while (!h->error) {
                for (int i = 0; i < h->S && s < 0; i++)
                    if (dv->slots[i].state == SLOT_FREE) s = i;
                if (s >= 0) break;
                pthread_cond_wait(&h->cv_out, &h->mu);
            }
            if (s >= 0) {
                slot_t *sl = &dv->slots[s];
                sl->n = 0; sl->issued = 0; sl->fetched = 0; sl->gop_index = h->cur_gop; sl->frame0 = h->frames_in;
                sl->state = SLOT_OPEN;
                h->g_dev = (int)(h->cur_gop % h->N); h->g_slot = s;
            }
        }
        if (h->stats) h->st_caller_slot_wait += now_s() - q0;
        if (h->error) { pthread_mutex_unlock(&h->mu); fprintf(stderr, "b2enc: encode pipeline failed\n"); return -1; }
        gpu_t *dv = &h->dev[h->g_dev];
        slot_t *sl = &dv->slots[h->g_slot];
        const int t = sl->n;
        pthread_mutex_unlock(&h->mu);
        const double p0 = h->stats ? now_s() : 0.0;
        /* picture -> ring entry t of the slot; returns when the picture has been read (av_encode.c:415, :545: it is refilled).
         * Staging the library owns is double buffered: its DMA is only waited for when that buffer comes round again. */
        if (staged) {
            const long ticket = b2_engine_put_picture_async(dv->eng, h->g_slot, t, src, stride);
            if (ticket < 0) { fail(h); return -1; }
            staged->busy_eng[staged->cur] = ticket > 0 ? (void *)dv->eng : NULL;
            staged->busy_ticket[staged->cur] = ticket;
        } else if (b2_engine_put_picture(dv->eng, h->g_slot, t, src, stride)) { fail(h); return -1; }
        if (h->stats) h->st_caller_put += now_s() - p0;
        pthread_mutex_lock(&h->mu);
        outframe_t *f = &h->fifo[h->frames_in % h->fifo_cap];
        f->pts = pic_in->i_pts; f->ready = 0;
        sl->n = t + 1;
        h->frames_in++;
        if (sl->n == h->L) { sl->state = SLOT_CLOSED; h->g_slot = -1; h->cur_gop++; }
        pthread_cond_signal(&dv->cv);
    } else {
        if (h->g_slot >= 0) {                                 /* flush: the GOP being gathered ends here */
            h->dev[h->g_dev].slots[h->g_slot].state = SLOT_CLOSED;
            pthread_cond_signal(&h->dev[h->g_dev].cv);
            h->g_slot = -1; h->cur_gop++;
        }
        /* a flush call waits for its frame (av_encode.c:1076-1083) */
        while (!h->error && h->frames_out < h->frames_in && !h->fifo[h->frames_out % h->fifo_cap].ready) pthread_cond_wait(&h->cv_out, &h->mu);
    }
    if (h->error) { pthread_mutex_unlock(&h->mu); fprintf(stderr, "b2enc: encode pipeline failed\n"); return -1; }
    outframe_t *head = &h->fifo[h->frames_out % h->fifo_cap];
    if (h->frames_out == h->frames_in || !head->ready) { pthread_mutex_unlock(&h->mu); return 0; }
    outframe_t o = *head;
    head->data = NULL; head->nal = NULL; head->ready = 0;
    h->frames_out++;
    pthread_mutex_unlock(&h->mu);
    const int n = return_frame(h, &o, pp_nal, pi_nal, pic_out);
    free(o.nal);
    return n;
}
