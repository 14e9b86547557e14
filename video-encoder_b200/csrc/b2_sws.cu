// b2_sws.cu -- GPU side of the libswscale drop-in (include/b2enc.h: b2_sws_*; host half in host/b2h_sws.c): the
// synchronous host -> GPU -> host conversion through kernel K0 that b2_sws_scale runs when the destination is plain
// host memory -- sws_scale's own host-in / host-out contract (av_encode.c:545-547) -- and the page-locked allocator
// behind b2_picture_alloc.  (Destinations that are encoder input pictures never come here: their conversion is deferred
// into b2_encoder_encode, see host/b2h_sws.c.)
#include <string.h>
#include "b2_common.cuh"
#include "b2_internal.h"
#include "../host/b2h_picture.h"

struct b2_sws_rt {
    int w, h, fmt, w16, h16, pitch, rows, pitchc, rowsc, device;
    size_t in_bytes;
    uint8_t *h_in = nullptr, *d_in = nullptr, *d_y = nullptr, *d_u = nullptr, *d_v = nullptr;
    cudaStream_t st = nullptr;
};

extern "C" void *b2_pinned_alloc(size_t n)
{
    void *p = nullptr;
    // portable: one stream may be spread over several GPUs (b2_param_t.i_devices), every one of them DMAs from the picture
    if (cudaHostAlloc(&p, n, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
extern "C" void b2_pinned_free(void *p) { if (p) cudaFreeHost(p); }

// NULL (with a message) when no CUDA device is visible: the conversion has no CPU fallback
extern "C" void *b2_sws_rt_create(int w, int h, int fmt)
{
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
        cudaGetLastError();
        fprintf(stderr, "b2enc: no CUDA device; conversion has no CPU fallback\n");
        return nullptr;
    }
    int rb[3], rws[3];
    if (!b2_fmt_layout(fmt, w, h, rb, rws)) return nullptr;
    b2_sws_rt *c = new b2_sws_rt();
    c->w = w; c->h = h; c->fmt = fmt;
    c->device = 0;
    cudaGetDevice(&c->device);                          // the device current at creation owns the buffers and runs K0
    c->w16 = (w + 15) & ~15; c->h16 = (h + 15) & ~15;
    b2_padded_layout(c->w16, c->h16, &c->pitch, &c->rows, &c->pitchc, &c->rowsc);
    c->in_bytes = 0;
    for (int p = 0; p < 3; p++) c->in_bytes += (size_t)rb[p] * rws[p];
    return c;                                           // buffers are allocated on first use
}

extern "C" void b2_sws_rt_free(void *rt)
{
    b2_sws_rt *c = (b2_sws_rt *)rt;
    if (!c) return;
    int prev = 0;
    cudaGetDevice(&prev);
    cudaSetDevice(c->device);
    cudaFreeHost(c->h_in); cudaFree(c->d_in); cudaFree(c->d_y); cudaFree(c->d_u); cudaFree(c->d_v);
    if (c->st) cudaStreamDestroy(c->st);
    cudaSetDevice(prev);
    delete c;
}

static int rt_alloc(b2_sws_rt *c)
{
    if (c->st) return 0;
    bool ok = cudaHostAlloc(&c->h_in, c->in_bytes, cudaHostAllocDefault) == cudaSuccess &&
              cudaMalloc(&c->d_in, c->in_bytes) == cudaSuccess && cudaMalloc(&c->d_y, (size_t)c->pitch * c->rows) == cudaSuccess &&
              cudaMalloc(&c->d_u, (size_t)c->pitchc * c->rowsc) == cudaSuccess &&
              cudaMalloc(&c->d_v, (size_t)c->pitchc * c->rowsc) == cudaSuccess && cudaStreamCreate(&c->st) == cudaSuccess;
    if (!ok) { cudaGetLastError(); fprintf(stderr, "b2enc: b2_sws_scale: allocation failed\n"); return -1; }
    return 0;
}

// whole frame: strided source planes -> pinned staging -> device -> K0 -> strided destination planes; returns h or < 0
extern "C" int b2_sws_rt_scale(void *rt, const uint8_t *const src[], const int srcStride[], uint8_t *const dst[], const int dstStride[])
{
    b2_sws_rt *c = (b2_sws_rt *)rt;
    const int w = c->w, h = c->h, cw = (w + 1) / 2, ch = (h + 1) / 2;
    int prev = 0;
    cudaGetDevice(&prev);
    B2_CUDA_OK(cudaSetDevice(c->device));
    if (rt_alloc(c)) { cudaSetDevice(prev); return -1; }
    int rb[3], rws[3];
    const int np = b2_fmt_layout(c->fmt, w, h, rb, rws);
    uint8_t *p = c->h_in;
    for (int k = 0; k < np; k++) {
        for (int y = 0; y < rws[k]; y++) memcpy(p + (size_t)y * rb[k], src[k] + (size_t)y * srcStride[k], rb[k]);
        p += (size_t)rb[k] * rws[k];
    }
    int rc = -1;
    do {
        if (cudaMemcpyAsync(c->d_in, c->h_in, c->in_bytes, cudaMemcpyHostToDevice, c->st) != cudaSuccess) break;
        if (b2_launch_convert(c->fmt, c->d_in, c->in_bytes, c->d_y, c->d_u, c->d_v, c->pitch, c->pitchc, (size_t)c->pitch * c->rows,
                              (size_t)c->pitchc * c->rowsc, w, h, 1, c->st))
            break;
        if (cudaMemcpy2DAsync(dst[0], dstStride[0], c->d_y + (size_t)B2_PAD * c->pitch + B2_PAD, c->pitch, w, h,
                              cudaMemcpyDeviceToHost, c->st) != cudaSuccess) break;
        if (cudaMemcpy2DAsync(dst[1], dstStride[1], c->d_u + (size_t)B2_PADC * c->pitchc + B2_PADC, c->pitchc, cw, ch,
                              cudaMemcpyDeviceToHost, c->st) != cudaSuccess) break;
        if (cudaMemcpy2DAsync(dst[2], dstStride[2], c->d_v + (size_t)B2_PADC * c->pitchc + B2_PADC, c->pitchc, cw, ch,
                              cudaMemcpyDeviceToHost, c->st) != cudaSuccess) break;
        if (cudaStreamSynchronize(c->st) != cudaSuccess) break;
        rc = h;
    } while (0);
    if (rc < 0) fprintf(stderr, "b2enc: b2_sws_scale: CUDA error %s\n", cudaGetErrorName(cudaGetLastError()));
    cudaSetDevice(prev);
    return rc;
}
