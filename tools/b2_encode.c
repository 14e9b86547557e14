/*
 * b2_encode.c -- host driver in C for the drop-in boundary (include/b2enc.h): the video half of the
 * reference's main() (av_encode.c:840-1128) with its command line (--preset --tune --quality --profile,
 * --silent, --frame-limit; av_encode.c:110-124), fed by raw I420 / YUV4MPEG2 instead of libavformat
 * (demux, decoders, filters, AAC and MP4 muxing are out of scope: SURVEY.md 2) and writing an
 * Annex-B .h264 elementary stream.  The call sequence is the reference's:
 *   param_default_preset -> field writes -> apply_profile -> encoder_open -> picture_alloc ->
 *   sws_getContext                                            (enc_x264_open,  av_encode.c:378-438)
 *   per frame: sws_scale into pic_in, encoder_encode          (av_encode.c:545-547, :970)
 *   drain: while delayed_frames() encode(NULL)                (av_encode.c:1076-1083)
 *   sws_freeContext, picture_clean, encoder_close             (enc_x264_close, av_encode.c:440-444)
 * Like the reference it takes --filters (av_encode.c:116): "hqdn3d", "yadif" or "hqdn3d,yadif" run on the GPU pre-filter stage
 * (include/b2enc_filters.h); and when the output name ends in ".mp4" it writes an MP4 with one AVC track from the encoder's
 * b_annexb = 0 payloads (tools/b2_mp4.h + b2_avcc_write), the video half of enc_mp4_write_video_sample (:683-744).
 * Extensions (not in the reference): --size WxH --fps N[/D] for raw input, --merange, --gop, --slots, --device, --devices N (one
 * stream over N GPUs by closed GOP), --8x8dct, --partitions, --slices N (row-aligned slices per picture, x264's --slices).
 * Regular input files are mmap'ed: the "decoded picture" the reference gets from libavcodec is then a pointer into the page
 * cache and b2_sws_scale's staging copy is the only time the host touches the pixels (pipes fall back to fread).
 */
#define _DEFAULT_SOURCE
#define _POSIX_C_SOURCE 200809L
#include <fcntl.h>
#include <getopt.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <time.h>
#include <unistd.h>
#include "b2enc.h"
#include "b2enc_filters.h"
#include "b2_mp4.h"

typedef struct {
    int silent, width, height, fps_num, fps_den, merange, gop, slots, device, devices, dct8, partitions, slices;
    long frame_limit;
    const char *input_file, *output_file, *preset, *tune, *profile, *video_filter;
    float quality;
} cli_options_t;

static int parse_cli_options(cli_options_t *o, int argc, char **argv)
{
    cli_options_t d = {.silent = 0, .width = 0, .height = 0, .fps_num = 25, .fps_den = 1, .merange = 0, .gop = 0, .slots = 0,
                       .device = 0, .devices = 0, .dct8 = 0, .partitions = 0, .slices = 0, .video_filter = NULL, .frame_limit = -1, .input_file = NULL, .output_file = NULL,
                       .preset = "medium", .tune = "film", .profile = NULL, .quality = 20.0f};   /* av_encode.c:91-106 */
    *o = d;
    struct option long_opts[] = {
        {"silent", no_argument, NULL, 's'}, {"frame-limit", required_argument, NULL, 'l'},
        {"preset", required_argument, NULL, 1}, {"tune", required_argument, NULL, 2},
        {"quality", required_argument, NULL, 3}, {"profile", required_argument, NULL, 4},
        {"size", required_argument, NULL, 5}, {"fps", required_argument, NULL, 6}, {"merange", required_argument, NULL, 7},
        {"gop", required_argument, NULL, 8}, {"slots", required_argument, NULL, 9}, {"device", required_argument, NULL, 10},
        {"filters", required_argument, NULL, 'f'}, {"8x8dct", no_argument, NULL, 11}, {"partitions", required_argument, NULL, 12},
        {"devices", required_argument, NULL, 13}, {"slices", required_argument, NULL, 14},
        {NULL, 0, NULL, 0}};
    int c, idx = 0;
    while ((c = getopt_long(argc, argv, "sl:f:", long_opts, &idx)) != -1) {
        switch (c) {
        case 's': o->silent = 1; break;
        case 'l': o->frame_limit = strtol(optarg, NULL, 10); break;
        case 1: o->preset = optarg; break;
        case 2: o->tune = optarg; break;
        case 3: o->quality = (float)strtod(optarg, NULL); break;
        case 4: o->profile = optarg; break;
        case 5: if (sscanf(optarg, "%dx%d", &o->width, &o->height) != 2) return 0; break;
        case 6: o->fps_den = 1; if (sscanf(optarg, "%d/%d", &o->fps_num, &o->fps_den) < 1) return 0; break;
        case 7: o->merange = atoi(optarg); break;
        case 8: o->gop = atoi(optarg); break;
        case 9: o->slots = atoi(optarg); break;
        case 10: o->device = atoi(optarg); break;
        case 'f': o->video_filter = optarg; break;                       /* av_encode.c:148-149 */
        case 11: o->dct8 = 1; break;
        case 12: o->partitions = atoi(optarg); break;
        case 13: o->devices = atoi(optarg); break;
        case 14: o->slices = atoi(optarg); break;
        default: return 0;
        }
    }
    if (optind + 2 != argc) return 0;
    o->input_file = argv[optind]; o->output_file = argv[optind + 1];
    return 1;
}

/* YUV4MPEG2 stream header: "YUV4MPEG2 W<w> H<h> F<n>:<d> ... \n" */
static int read_y4m_header(FILE *f, cli_options_t *o)
{
    char line[256];
    if (!fgets(line, sizeof(line), f) || strncmp(line, "YUV4MPEG2", 9)) return 0;
    for (char *tok = strtok(line + 9, " \n"); tok; tok = strtok(NULL, " \n")) {
        if (tok[0] == 'W') o->width = atoi(tok + 1);
        else if (tok[0] == 'H') o->height = atoi(tok + 1);
        else if (tok[0] == 'F') sscanf(tok + 1, "%d:%d", &o->fps_num, &o->fps_den);
        else if (tok[0] == 'C' && strncmp(tok + 1, "420", 3)) { fprintf(stderr, "y4m: only 4:2:0 input is supported\n"); return 0; }
    }
    return o->width > 0 && o->height > 0;
}

int main(int argc, char **argv)
{
    cli_options_t opts;
    if (!parse_cli_options(&opts, argc, argv)) {
        fprintf(stderr, "usage: %s [--preset p] [--tune t] [--quality q] [--profile p] [--frame-limit n] [--silent]\n"
                        "          [--size WxH --fps N[/D]] [--merange 16|32] [--gop n] [--slots n] [--device n] [--devices n]\n"
                        "          [--slices n]"
                        "          [--filters hqdn3d,yadif] [--8x8dct] [--partitions 0|1|2] input.{y4m,yuv} output.{h264,mp4}\n", argv[0]);
        return 1;
    }
    FILE *in = fopen(opts.input_file, "rb");
    if (!in) { perror(opts.input_file); return 2; }
    size_t n = strlen(opts.input_file);
    int is_y4m = n > 4 && !strcmp(opts.input_file + n - 4, ".y4m");
    if (is_y4m && !read_y4m_header(in, &opts)) { fprintf(stderr, "bad y4m header\n"); return 2; }
    if (opts.width <= 0 || opts.height <= 0) { fprintf(stderr, "raw input needs --size WxH\n"); return 2; }

    struct timespec t_start;
    clock_gettime(CLOCK_MONOTONIC, &t_start);
    /* enc_x264_open(), av_encode.c:378-438 */
    b2_param_t params;
    if (b2_param_default_preset(&params, opts.preset, opts.tune) != 0) {
        fprintf(stderr, "b2enc: failed to set preset %s and tune %s\n", opts.preset, opts.tune);
        return 8;
    }
    params.i_width = opts.width; params.i_height = opts.height;
    const size_t on = strlen(opts.output_file);
    const int to_mp4 = on > 4 && !strcmp(opts.output_file + on - 4, ".mp4");
    params.b_annexb = to_mp4 ? 0 : 1;                      /* MP4: 4-byte NAL lengths like the reference (av_encode.c:392); else Annex-B */
    params.b_transform_8x8 = opts.dct8; params.b_partitions = opts.partitions;
    params.i_fps_num = opts.fps_num; params.i_fps_den = opts.fps_den;
    params.vui.i_sar_width = 1; params.vui.i_sar_height = 1;
    params.rc.i_rc_method = B2_RC_CRF; params.rc.f_rf_constant = opts.quality;
    if (opts.merange) params.i_merange = opts.merange;
    if (opts.gop) params.i_keyint_max = opts.gop;
    if (opts.slots) params.i_gop_slots = opts.slots;
    params.i_device = opts.device; params.i_devices = opts.devices;
    params.i_slice_count = opts.slices;
    if (b2_param_apply_profile(&params, opts.profile) != 0) { fprintf(stderr, "b2enc: failed to apply profile %s\n", opts.profile); return 8; }
    b2_t *enc = b2_encoder_open(&params);
    if (!enc) { fprintf(stderr, "b2enc: failed to initialize encoder\n"); return 8; }
    b2_picture_t pic_in, pic_out;
    if (b2_picture_alloc(&pic_in, B2_CSP_I420, opts.width, opts.height) != 0) { fprintf(stderr, "b2enc: could not allocate input picture\n"); return 8; }
    pic_out.i_pts = 0;
    b2_sws_context_t *scaler = b2_sws_getContext(opts.width, opts.height, B2_FMT_YUV420P, opts.width, opts.height, B2_FMT_YUV420P,
                                                 B2_SWS_FAST_BILINEAR, NULL, NULL, NULL);
    if (!scaler) { fprintf(stderr, "failed to create software scaler to copy frames to the encoder\n"); return 8; }

    /* enc_avfilter_build_graph(), av_encode.c:451-517 */
    b2_filter_graph_t *graph = NULL;
    if (opts.video_filter && opts.video_filter[0]) {
        graph = b2_filter_graph_create(opts.width, opts.height, B2_FMT_YUV420P, opts.video_filter, opts.device);
        if (!graph) { fprintf(stderr, "failed to build the filter graph '%s'\n", opts.video_filter); return 8; }
    }
    FILE *out = NULL;
    b2_mp4_t mp4;
    if (to_mp4) { if (b2_mp4_open(&mp4, opts.output_file, opts.width, opts.height, opts.fps_num, opts.fps_den)) { perror(opts.output_file); return 9; } }
    else { out = fopen(opts.output_file, "wb"); if (!out) { perror(opts.output_file); return 9; } }
    const int cw = (opts.width + 1) / 2, ch = (opts.height + 1) / 2;
    const size_t frame_bytes = (size_t)opts.width * opts.height + 2 * (size_t)cw * ch;
    uint8_t *raw_buf = (uint8_t *)malloc(frame_bytes), *filt = (uint8_t *)malloc(frame_bytes);
    if (!raw_buf || !filt) { fprintf(stderr, "out of memory\n"); return 8; }
    /* regular file: map it, pictures are pointers into the page cache */
    const uint8_t *map = NULL; size_t map_size = 0, map_pos = (size_t)ftell(in);
    {
        struct stat st;
        if (fstat(fileno(in), &st) == 0 && S_ISREG(st.st_mode) && st.st_size > 0) {
            /* pre-faulted (no page faults inside the frame loop) unless the file is larger than what one would want resident at once */
            void *m = mmap(NULL, (size_t)st.st_size, PROT_READ, MAP_SHARED | (st.st_size <= ((off_t)16 << 30) ? MAP_POPULATE : 0), fileno(in), 0);
            if (m != MAP_FAILED) { map = (const uint8_t *)m; map_size = (size_t)st.st_size; madvise(m, map_size, MADV_SEQUENTIAL); }
        }
    }
    int write_error = 0;
    struct timespec t0, t1;
    clock_gettime(CLOCK_MONOTONIC, &t0);
    long frames_in = 0, frames_out = 0;
    size_t bytes_out = 0;
    b2_nal_t *nals; int nal_count;
#define EMIT(payload)                                                                                              \
    do {                                                                                                           \
        if ((payload) > 0) {                                                                                       \
            if (to_mp4) write_error |= b2_mp4_write_frame(&mp4, nals, nal_count, (payload), pic_out.b_keyframe) != 0; \
            else write_error |= fwrite(nals[0].p_payload, 1, (size_t)(payload), out) != (size_t)(payload);         \
            bytes_out += (size_t)(payload); frames_out++;                                                          \
        } else if ((payload) < 0) fprintf(stderr, "b2enc: encoder error\n");                                       \
    } while (0)
    int eof = 0;
    while (!eof) {
        if ((opts.frame_limit >= 0 && frames_in >= opts.frame_limit)) eof = 1;
        const uint8_t *raw = raw_buf;
        if (!eof && map) {
            if (is_y4m) {                                  /* "FRAME[ params]\n" */
                if (map_pos + 6 > map_size || memcmp(map + map_pos, "FRAME", 5)) eof = 1;
                else { const uint8_t *nl = (const uint8_t *)memchr(map + map_pos, '\n', map_size - map_pos); if (!nl) eof = 1; else map_pos = (size_t)(nl - map) + 1; }
            }
            if (!eof && map_pos + frame_bytes > map_size) eof = 1;
            if (!eof) { raw = map + map_pos; map_pos += frame_bytes; }
        } else {
            if (!eof && is_y4m) { char fl[64]; if (!fgets(fl, sizeof(fl), in) || strncmp(fl, "FRAME", 5)) eof = 1; }
            if (!eof && fread(raw_buf, 1, frame_bytes, in) != frame_bytes) eof = 1;
        }
        const uint8_t *src[4] = {raw, raw + (size_t)opts.width * opts.height, raw + (size_t)opts.width * opts.height + (size_t)cw * ch, NULL};
        const int stride[4] = {opts.width, cw, cw, 0};
        if (graph) {                                          /* av_vsrc_buffer_add_frame, av_encode.c:962 (flush at end of input) */
            if (!eof) { if (b2_filter_add_frame(graph, src, stride, frames_in, 1)) { fprintf(stderr, "b2enc: filter error\n"); return 10; } frames_in++; }
            else b2_filter_flush(graph);
        } else if (eof) break;
        /* pull all finished frames and encode them, av_encode.c:967-975 */
        for (;;) {
            const uint8_t *fsrc[4] = {src[0], src[1], src[2], NULL};
            int64_t pts = frames_in;
            if (graph) {
                uint8_t *fdst[3] = {filt, filt + (size_t)opts.width * opts.height, filt + (size_t)opts.width * opts.height + (size_t)cw * ch};
                if (b2_filter_get_frame(graph, fdst, stride, &pts) != 1) break;
                fsrc[0] = fdst[0]; fsrc[1] = fdst[1]; fsrc[2] = fdst[2];
            } else {
                pts = frames_in++;
            }
            /* enc_avfilter_pull_to_x264_context(), av_encode.c:543-547 */
            pic_in.i_type = B2_TYPE_AUTO; pic_in.i_pts = pts;
            if (b2_sws_scale(scaler, fsrc, stride, 0, opts.height, pic_in.img.plane, pic_in.img.i_stride) != opts.height) { fprintf(stderr, "b2enc: conversion failed\n"); return 10; }
            int payload = b2_encoder_encode(enc, &nals, &nal_count, &pic_in, &pic_out);            /* av_encode.c:970 */
            EMIT(payload);
            if (!graph) break;
        }
    }
    while (b2_encoder_delayed_frames(enc) > 0) {                                               /* av_encode.c:1076-1083 */
        int payload = b2_encoder_encode(enc, &nals, &nal_count, NULL, &pic_out);
        EMIT(payload);
        if (payload < 0) break;
    }
    clock_gettime(CLOCK_MONOTONIC, &t1);
    double dt = (double)(t1.tv_sec - t0.tv_sec) + 1e-9 * (double)(t1.tv_nsec - t0.tv_nsec);
    if (!opts.silent)
        printf("%ld frames in, %ld frames out, %zu bytes, %.2f s, %.1f fps (host entropy coding included); encoder start-up %.2f s\n",
               frames_in, frames_out, bytes_out, dt, dt > 0 ? frames_out / dt : 0.0,
               (double)(t0.tv_sec - t_start.tv_sec) + 1e-9 * (double)(t0.tv_nsec - t_start.tv_nsec));
    free(raw_buf); free(filt);
    if (map) munmap((void *)map, map_size);
    fclose(in);
    if (to_mp4) { if (b2_mp4_close(&mp4)) write_error = 1; }                                    /* MP4Close, av_encode.c:1110-1116 */
    else if (fclose(out) != 0) write_error = 1;
    if (write_error) fprintf(stderr, "b2enc: writing %s failed\n", opts.output_file);
    b2_filter_graph_free(graph);
    b2_sws_freeContext(scaler);                                                                /* enc_x264_close(), av_encode.c:440-444 */
    b2_picture_clean(&pic_in);
    b2_encoder_close(enc);
    return write_error ? 11 : 0;
}
