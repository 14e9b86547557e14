"""GPU-side throughput of the drop-in's execution shape: SLOTS closed GOPs on one GPU, each stream group advanced on its own
(encode_group + d2h_group, two steps in flight per group, results fetched like b2h_encoder.c's per-GPU thread does), pictures
resident in the device ring.  Usage: slot_stream_probe.py SLOTS GROUPS DEBLOCK [STEPS] [ME_PRUNE]"""
import sys, os, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "video-encoder_b200")); sys.path.insert(0, os.path.join(ROOT, "oracle"))
import numpy as np, b2enc, b2oracle as o
W, H = 1920, 1080
slots, groups, deblock = int(sys.argv[1]), int(sys.argv[2]), int(sys.argv[3])
steps = int(sys.argv[4]) if len(sys.argv) > 4 else 64
prune = int(sys.argv[5]) if len(sys.argv) > 5 else 0
GOP, RING = 32, 8
eng = b2enc.Engine(W, H, slots=slots, ring=RING, merange=32, qp=26, streams=groups, deblock=deblock, pack_levels=1, deblock_offsets=(-1, -1), me_prune=prune)
n_y = W * H
for s in range(slots):
    for r in range(RING):
        y, u, v = o.synth_frame(W, H, r, s)
        buf = eng.host_input(s, r); buf[:n_y] = y.ravel(); buf[n_y:n_y + u.size] = u.ravel(); buf[n_y + u.size:] = v.ravel()
for r in range(RING):
    eng.h2d(ring=r)
eng.sync()
G = len(eng.groups())
phase = [g * GOP // G for g in range(G)]
issued = [0] * G; fetched = [0] * G; sets = [[0, 0] for _ in range(G)]


def run(total):
    t0 = time.perf_counter()
    done = 0
    while done < total * G:
        progress = False
        for g in range(G):
            while True:
                if fetched[g] < issued[g] and eng.group_done(g, sets[g][fetched[g] & 1]) == 1:
                    fetched[g] += 1; done += 1; progress = True
                    continue
                if issued[g] < total and issued[g] - fetched[g] < 2:
                    t = issued[g]
                    eng.encode_group(g, b2enc.FRAME_I if (t + phase[g]) % GOP == 0 or t == 0 else b2enc.FRAME_P, ring=t % RING)
                    eng.d2h_group(g)
                    sets[g][t & 1] = eng.group_result_set(g)
                    issued[g] += 1; progress = True
                    continue
                break
        if not progress:
            for g in range(G):
                if fetched[g] < issued[g]:
                    eng.group_wait(g, sets[g][fetched[g] & 1]); break
    eng.sync()
    return time.perf_counter() - t0


run(6)
for g in range(G):
    issued[g] = fetched[g] = 0
dt = run(steps)
print("slots %2d groups %2d deblock %d me_prune %d: %d frames in %.3f s = %.0f frames/s" %
      (slots, G, deblock, prune, slots * steps, dt, slots * steps / dt), flush=True)
eng.close()
