"""Latency chain of ONE frame: every kernel of a step timed alone (CUDA events, engine profile mode) with a single slot, i.e. the
dependent chain a closed GOP's next frame waits for.  Usage: frame_latency_probe.py [W H MERANGE] [deblock]"""
import sys, os
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "video-encoder_b200")); sys.path.insert(0, os.path.join(ROOT, "oracle"))
import numpy as np, b2enc, b2oracle as o
W, H, R = (int(sys.argv[1]), int(sys.argv[2]), int(sys.argv[3])) if len(sys.argv) > 3 else (1920, 1080, 32)
deblock = int(sys.argv[4]) if len(sys.argv) > 4 else 1
for slots in (1, 4):
    eng = b2enc.Engine(W, H, slots=slots, ring=8, merange=R, qp=26, streams=1, deblock=deblock, pack_levels=1, profile=1, deblock_offsets=(-1, -1))
    n_y = W * H
    for s in range(slots):
        for r in range(8):
            y, u, v = o.synth_frame(W, H, r, s)
            buf = eng.host_input(s, r); buf[:n_y] = y.ravel(); buf[n_y:n_y + u.size] = u.ravel(); buf[n_y + u.size:] = v.ravel()
    for r in range(8):
        eng.h2d(ring=r)
    for kind, types in (("I", [b2enc.FRAME_I] * 4), ("P", [b2enc.FRAME_P] * 8)):
        eng.encode(b2enc.FRAME_I, ring=0); eng.encode(b2enc.FRAME_P, ring=1); eng.sync(); eng.profile_reset()
        for i, ft in enumerate(types):
            eng.encode(ft, ring=(2 + i) % 8)
        eng.sync()
        ms = eng.kernel_ms()
        tot = sum(v[0] / max(v[1], 1) for v in ms.values())
        print("%dx%d +-%d deblock %d, %d slot(s), %s frame: chain %.3f ms | " % (W, H, R, deblock, slots, kind, tot)
              + "  ".join("%s %.3f" % (k.split()[0], v[0] / max(v[1], 1)) for k, v in ms.items() if v[1]), flush=True)
    eng.close()
