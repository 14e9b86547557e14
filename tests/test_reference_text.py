"""Compile-level proof of the drop-in (SURVEY.md 8b): the reference's OWN TEXT -- x264_context_t (av_encode.c:369-376),
enc_x264_open (:378-438), enc_x264_close (:440-444), enc_avfilter_pull_to_x264_context (:525-560), the encode loop (:968-975)
and the drain loop (:1076-1083) -- is read at test time from the av_encode.c that B2ENC_AV_ENCODE_C names (never copied into
the repository), compiled unchanged through include/b2enc_compat.h with stub libavcodec / libavfilter types, and
  * linked against the real libb2enc.so (every symbol the text needs resolves), and
  * linked against the host sources + the oracle-backed mock engine (tests/mock) and RUN on the CPU: the stream it muxes is
    byte-identical to the oracle encoder's at the reference's defaults (preset medium, tune film, CRF 20, profile NULL;
    av_encode.c:102-105).
Skipped when B2ENC_AV_ENCODE_C is not set."""
import ctypes as C
import glob
import os
import subprocess
import numpy as np
import pytest
from test_oracle_decode import smooth_seq

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("B2ENC_AV_ENCODE_C", "")                 # the reference program's av_encode.c

HARNESS_HEAD = r"""
#include <stdbool.h>
#include <stdio.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
/* ---- stub libav types: only the members the reference's text touches (FFmpeg 0.8 era names) ---- */
enum PixelFormat { PIX_FMT_NONE = -1, PIX_FMT_YUV420P, PIX_FMT_YUYV422, PIX_FMT_RGB24, PIX_FMT_BGR24, PIX_FMT_YUV422P, PIX_FMT_YUV444P,
                   PIX_FMT_YUV410P, PIX_FMT_YUV411P, PIX_FMT_GRAY8, PIX_FMT_UYVY422 = 17, PIX_FMT_NV12 = 25 };
typedef struct { int num, den; } AVRational;
typedef struct { int width, height; enum PixelFormat pix_fmt; AVRational time_base; } AVCodecContext;
typedef struct { uint8_t *data[4]; int linesize[4]; int64_t pts, pkt_pts, pkt_dts; int height; } AVFrame;
typedef struct AVFilterLink AVFilterLink;
typedef struct { AVFilterLink **inputs; } AVFilterContext;
typedef struct AVFilterBufferRef AVFilterBufferRef;
/* a one-picture "filter pipeline" fed by main() */
static int h_pending; static AVFrame h_pic;
static int avfilter_poll_frame(AVFilterLink *l) { (void)l; return h_pending; }
static int av_vsink_buffer_get_video_buffer_ref(AVFilterContext *c, AVFilterBufferRef **r, int flags) { (void)c; (void)flags; *r = NULL; h_pending = 0; return 0; }
static int avfilter_fill_frame_from_video_buffer_ref(AVFrame *f, AVFilterBufferRef *r) { (void)r; *f = h_pic; return 0; }
static void avfilter_unref_buffer(AVFilterBufferRef *r) { (void)r; }
static void enc_av_perror(const char *what, int e) { fprintf(stderr, "%s: %d\n", what, e); }
#define debug(...) do { } while (0)
#define format_pts(x) ((long)(x))
/* ---- the binding a maintainer adds ---- */
#include "b2enc_compat.h"
/* ---- the reference's text, verbatim ---- */
"""

HARNESS_TAIL = r"""
/* the muxer side of the hand-off: all NALs of a frame are contiguous from nals[0].p_payload, payload_size bytes in total
 * (av_encode.c:802, :808-812); every NAL starts with its 4-byte big-endian length (:722) */
static FILE *h_out; static long h_frames;
static void enc_mp4_mux_video(void *container, int track, x264_context_t *x)
{
    (void)container; (void)track;
    int total = 0;
    for (int i = 0; i < x->nal_count; i++) {
        const uint8_t *p = x->nals[i].p_payload;
        if (p != x->nals[0].p_payload + total) { fprintf(stderr, "NALs not contiguous\n"); exit(3); }
        if ((int)((p[0] << 24) | (p[1] << 16) | (p[2] << 8) | p[3]) != x->nals[i].i_payload - 4) { fprintf(stderr, "bad length prefix\n"); exit(3); }
        total += x->nals[i].i_payload;
    }
    if (total != x->payload_size) { fprintf(stderr, "payload size mismatch\n"); exit(3); }
    fwrite(x->nals[0].p_payload, 1, (size_t)x->payload_size, h_out);
    fwrite(&x->pic_out.i_pts, 8, 1, h_out);
    h_frames++;
}

int main(int argc, char **argv)
{
    if (argc != 7) return 1;
    const int w = atoi(argv[1]), h = atoi(argv[2]), fmt = atoi(argv[3]), nframes = atoi(argv[4]);
    FILE *in = fopen(argv[5], "rb"); h_out = fopen(argv[6], "wb");
    if (!in || !h_out) return 1;
    struct { const char *preset, *tune, *profile; float quality; bool silent; } opts = {"medium", "film", NULL, 20.0, true};   /* :102-105 */
    AVCodecContext vcc = {w, h, (enum PixelFormat)fmt, {1, 30}};
    AVCodecContext *video_codec_context_ptr = &vcc;
    AVRational sar = {1, 1};
    x264_context_t x264;
    if (!enc_x264_open(video_codec_context_ptr, sar, opts.preset, opts.tune, opts.quality, opts.profile, &x264)) return 2;   /* :897 */
    AVFilterLink *links[1] = {NULL};
    AVFilterContext sink = {links}, *sink_filter_context_ptr = &sink;
    AVFrame frame, *decoded_frame_ptr = &frame;
    void *mp4_container = NULL; int mp4_video_track = 0; int64_t encoded_video_pts = 0;
    const size_t bytes = fmt == PIX_FMT_YUV420P ? (size_t)w * h * 3 / 2 : (size_t)w * h * 2;
    uint8_t *buf = malloc(bytes);
    for (int t = 0; t < nframes; t++) {
        if (fread(buf, 1, bytes, in) != bytes) return 4;
        memset(&h_pic, 0, sizeof(h_pic));
        h_pic.height = h; h_pic.pts = 100 + t;
        if (fmt == PIX_FMT_YUV420P) {
            h_pic.data[0] = buf; h_pic.data[1] = buf + (size_t)w * h; h_pic.data[2] = buf + (size_t)w * h * 5 / 4;
            h_pic.linesize[0] = w; h_pic.linesize[1] = h_pic.linesize[2] = w / 2;
        } else { h_pic.data[0] = buf; h_pic.linesize[0] = 2 * w; }
        h_pending = 1;
        memset(&frame, 0, sizeof(frame));
"""

LOOP_GLUE = r"""
        memset(buf, 0xAA, bytes);          /* the reference frees / reuses the decoded picture right away (:550) */
        (void)encoded_video_pts;
    }
"""

END = r"""
    enc_x264_close(&x264);
    fclose(h_out);
    return h_frames == nframes ? 0 : 5;
}
"""


def ref_lines(a, b):
    lines = open(REF).read().split("\n")
    return "\n".join(lines[a - 1:b]) + "\n"


def build_harness(tmp_path):
    src = (HARNESS_HEAD + ref_lines(369, 376) + ref_lines(378, 438) + ref_lines(440, 444) + ref_lines(525, 560) + HARNESS_TAIL
           + ref_lines(968, 975) + "\n\t\t\tencoded_video_pts = x264.pic_out.i_pts;\n" + LOOP_GLUE + ref_lines(1076, 1083) + END)
    c = tmp_path / "ref_text_harness.c"
    c.write_text(src)
    return c


@pytest.fixture(scope="module")
def mock_so():
    if not os.path.exists(REF):
        pytest.skip("B2ENC_AV_ENCODE_C does not name the reference's av_encode.c")
    out = os.path.join(ROOT, "tests", "mock", "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libb2enc_mock.so")
    srcs = ([os.path.join(ROOT, "tests", "mock", "mock_engine.c")] + sorted(glob.glob(os.path.join(ROOT, "video-encoder_b200", "host", "*.c")))
            + sorted(glob.glob(os.path.join(ROOT, "oracle", "b2o_*.c"))))
    subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-std=c99", "-Wall", "-I" + os.path.join(ROOT, "include"),
                           "-I" + os.path.join(ROOT, "video-encoder_b200", "host"), "-o", so] + srcs + ["-lm", "-lpthread"])
    return so


def test_reference_text_links_against_libb2enc(b2, tmp_path):
    if not os.path.exists(REF):
        pytest.skip("B2ENC_AV_ENCODE_C does not name the reference's av_encode.c")
    c = build_harness(tmp_path)
    libdir = os.path.dirname(b2.so_path())
    r = subprocess.run(["gcc", "-std=gnu99", "-O1", "-I" + os.path.join(ROOT, "include"), "-o", str(tmp_path / "harness_real"), str(c),
                        "-L" + libdir, "-lb2enc", "-Wl,-rpath," + libdir], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


@pytest.mark.parametrize("fmt,avfmt", [("yuv420p", 0), ("yuyv422", 1)])
def test_reference_text_runs_and_matches_oracle(oracle, mock_so, tmp_path, fmt, avfmt):
    w, h, n = 64, 48, 40
    frames = smooth_seq(w, h, n, seed=23, cut=17)
    raw = tmp_path / "in.raw"
    conv = []
    with open(raw, "wb") as f:
        for y, u, v in frames:
            if fmt == "yuv420p":
                f.write(y.tobytes() + u.tobytes() + v.tobytes()); conv.append((y, u, v))
            else:
                p = np.empty((h, 2 * w), np.uint8); p[:, 0::2] = y
                p[:, 1::4] = np.repeat(u, 2, axis=0); p[:, 3::4] = np.repeat(v, 2, axis=0)
                f.write(p.tobytes()); conv.append(oracle.convert_to_i420("yuyv422", w, h, [p]))
    c = build_harness(tmp_path)
    exe = tmp_path / "harness_mock"
    r = subprocess.run(["gcc", "-std=gnu99", "-O1", "-I" + os.path.join(ROOT, "include"), "-o", str(exe), str(c), mock_so,
                        "-Wl,-rpath," + os.path.dirname(mock_so), "-lm", "-lpthread"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    out = tmp_path / "out.bin"
    r = subprocess.run([str(exe), str(w), str(h), str(avfmt), str(n), str(raw), str(out)], capture_output=True, text=True,
                       env=dict(os.environ, B2_MOCK_DEVICES="1"))
    assert r.returncode == 0, (r.returncode, r.stderr)
    # de-frame: payload (length-prefixed NALs) + 8-byte pts per frame; walk the NALs to find each frame's end
    data = open(out, "rb").read()
    ref, *_ = oracle.encode_sequence(conv, w, h, qp=20, merange=16, gop=32, fps=(30, 1), deblock=1, cabac=1, deblock_offsets=(-1, -1))
    pos, bs, pts = 0, b"", []
    while pos < len(data):
        while True:
            ln = int.from_bytes(data[pos:pos + 4], "big"); nal_type = data[pos + 4] & 31
            bs += b"\x00\x00\x00\x01" + data[pos + 4:pos + 4 + ln]; pos += 4 + ln
            if nal_type in (1, 5): break
        pts.append(int.from_bytes(data[pos:pos + 8], "little")); pos += 8
    assert pts == [100 + t for t in range(n)]                      # display order, pts passed through (av_encode.c:979)
    assert bs == ref
