"""What several slices per picture (i_slice_count) buy and cost, on the GPU the command runs on:
  1. K7 and the whole dependency chain of one frame (engine profile mode, CUDA events per kernel, one slot), I and P frames,
     1080p and 2160p, slices 1 / 2 / 4 / 8;
  2. per-picture wall time of b2_encoder_encode with tune zerolatency (one picture at a time, CABAC), 1080p and 2160p, slices
     1 / 4 / 8 -- the GPU chain plus the host slice writers, which run on min(n, cores - 1) threads;
  3. GOP-streaming throughput of the drop-in at its default settings (32 GOP slots), 1080p, slices 1 and 4 -- the cost of one
     K7 CTA per (frame, slice) in P frames.
Usage: slice_latency_probe.py [frames for part 3]"""
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "video-encoder_b200")); sys.path.insert(0, os.path.join(ROOT, "oracle"))
import numpy as np  # noqa: E402
import b2enc  # noqa: E402
import b2oracle as o  # noqa: E402

NSTREAM = int(sys.argv[1]) if len(sys.argv) > 1 else 960
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True).stdout.strip())
print("host cores: %d" % os.cpu_count(), flush=True)


def chain(W, H, slices):
    eng = b2enc.Engine(W, H, slots=1, ring=8, merange=16, qp=26, streams=1, deblock=1, pack_levels=1, profile=1, deblock_offsets=(-1, -1),
                       slices=slices)
    n_y = W * H
    for r in range(8):
        y, u, v = o.synth_frame(W, H, r, 0)
        if r >= 4:                                           # a scene cut: P frames after it hold many intra macroblocks
            y, u, v = 255 - y, 255 - u, 255 - v
        buf = eng.host_input(0, r); buf[:n_y] = y.ravel(); buf[n_y:n_y + u.size] = u.ravel(); buf[n_y + u.size:] = v.ravel()
    for r in range(8):
        eng.h2d(ring=r)
    def per_frame(ms):
        return ms["K7 intra recon"][0] / max(ms["K7 intra recon"][1], 1), sum(v[0] / max(v[1], 1) for v in ms.values())

    res = {}
    eng.profile_reset()                                      # I frames: 8 in a row
    for _ in range(8):
        eng.encode(b2enc.FRAME_I, ring=0)
    eng.sync(); res["I"] = [per_frame(eng.kernel_ms())]
    eng.encode(b2enc.FRAME_I, ring=0); eng.encode(b2enc.FRAME_P, ring=1); eng.sync(); eng.profile_reset()
    for r in (2, 3, 1, 2, 3, 1, 2, 3):                       # P frames of a pan: few intra macroblocks
        eng.encode(b2enc.FRAME_P, ring=r)
    eng.sync(); res["P"] = [per_frame(eng.kernel_ms())]
    res["P-cut"] = []
    for _ in range(4):                                       # the P frame right after the scene cut: mostly intra
        eng.encode(b2enc.FRAME_I, ring=0); eng.encode(b2enc.FRAME_P, ring=3); eng.sync(); eng.profile_reset()
        eng.encode(b2enc.FRAME_P, ring=4); eng.sync()
        res["P-cut"].append(per_frame(eng.kernel_ms()))
    eng.close()
    for kind, runs in res.items():
        print("%dx%d slices %d, %-5s frame: K7 %.3f ms, chain %.3f ms" % (W, H, slices, kind, np.mean([r[0] for r in runs]),
                                                                        np.mean([r[1] for r in runs])), flush=True)


def zerolatency(W, H, slices, n=40):
    frames = [o.synth_frame(W, H, t, 0) for t in range(8)]
    enc = b2enc.DropInEncoder(W, H, tune="zerolatency", quality=26, annexb=1, i_keyint_max=32, i_slice_count=slices)
    ts, kinds = [], []
    for t in range(n + 8):
        t0 = time.perf_counter()
        size, nals, *_ = enc.encode(frames[t % 8], t)
        dt = time.perf_counter() - t0
        if t >= 8:
            ts.append(dt); kinds.append(t % 32 == 0)
        assert size > 0 and sum(k in (1, 5) for k, _ in nals) == min(slices, (H + 15) // 16)
    enc.close()
    ts = np.array(ts) * 1e3
    print("zerolatency %dx%d slices %d: per picture median %.2f ms, p90 %.2f ms (P frames; %d pictures)"
          % (W, H, slices, np.median(ts[~np.array(kinds)]), np.percentile(ts[~np.array(kinds)], 90), len(ts)), flush=True)
    # the I frame on its own: open a fresh encoder so that every picture is an IDR
    enc = b2enc.DropInEncoder(W, H, tune="zerolatency", quality=26, annexb=1, i_keyint_max=1, i_slice_count=slices)
    ti = []
    for t in range(16):
        t0 = time.perf_counter()
        enc.encode(frames[t % 8], t)
        ti.append(time.perf_counter() - t0)
    enc.close()
    print("zerolatency %dx%d slices %d: per IDR picture median %.2f ms" % (W, H, slices, 1e3 * np.median(ti[4:])), flush=True)


def streaming(W, H, slices, n):
    frames = [o.synth_frame(W, H, t, 0) for t in range(8)]
    enc = b2enc.DropInEncoder(W, H, quality=26, annexb=1, i_slice_count=slices)
    for t in range(64):                                       # warm-up: two GOPs in
        enc.encode(frames[t % 8], t)
    while enc.delayed() > 0:
        enc.encode(None, 0)
    t0 = time.perf_counter()
    for t in range(n):
        enc.encode(frames[t % 8], t)
    while enc.delayed() > 0:
        enc.encode(None, 0)
    dt = time.perf_counter() - t0
    enc.close()
    print("GOP streaming %dx%d default settings, slices %d: %d frames in %.2f s = %.0f frames/s" % (W, H, slices, n, dt, n / dt), flush=True)


for W, H in ((1920, 1080), (3840, 2160)):
    for s in (1, 2, 4, 8):
        chain(W, H, s)
for W, H in ((1920, 1080), (3840, 2160)):
    for s in (1, 4, 8):
        zerolatency(W, H, s)
for rep in range(2):
    for s in (1, 4):
        streaming(1920, 1080, s, NSTREAM)
