"""K1 exhaustive vs pruned (K1a block sums + successive elimination), kernel alone: the bench's synthetic sequence (uniform pan,
predictor = the previous frame's vector = exact) and a smooth 'natural-like' field with a differently moving object and a
predictor that is right only for the background; +-32 at 1080p, +-16 at 720p; 16 frames per launch.  Results are compared."""
import os, sys, json
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "video-encoder_b200")); sys.path.insert(0, os.path.join(ROOT, "oracle"))
import numpy as np, b2enc, b2oracle
import scipy.ndimage as ndi

peak, _ = b2enc.vabsdiff4_peak(0, 512, 5)


def natural(w, h, n):
    rng = np.random.default_rng(1)
    base = rng.normal(size=(h // 8 + 40, w // 8 + 40))
    big = ndi.zoom(ndi.gaussian_filter(base, 2.0), 8, order=1)
    big = (big - big.min()) / (big.max() - big.min()) * 200 + 20 + ndi.gaussian_filter(rng.normal(size=big.shape), 1.0) * 25
    out = []
    for t in range(n + 1):
        y = big[100 + 2 * t:100 + 2 * t + h, 100 + 5 * t:100 + 5 * t + w].copy()
        y[h // 4:h // 4 + 160, w // 4 + 9 * t:w // 4 + 320 + 9 * t] = big[400:560, 600:920]
        out.append(np.clip(y + rng.normal(size=y.shape) * 2.0, 0, 255).astype(np.uint8))
    return out


for (w, h, R, n) in ((1920, 1088, 32, 16), (1280, 720, 16, 16)):
    nmb = (w // 16) * (h // 16)
    for name in ("synthetic pan", "natural-like"):
        if name == "synthetic pan":
            fr = [b2oracle.synth_frame(w, h, t, 0)[0] for t in range(n + 1)]
            pm = (12, 8)
        else:
            fr = natural(w, h, n); pm = (20, 8)
        cur = np.stack(fr[1:]); ref = np.stack(fr[:-1])
        pmv = np.zeros((n, nmb), b2enc.MV); pmv["x"] = pm[0]; pmv["y"] = pm[1]
        mv_a, cost_a, ms_a = b2enc.me_fullpel(cur, ref, R, pmv, 5, iters=10)
        mv_b, cost_b, st = b2enc.me_fullpel_pruned(cur, ref, R, pmv, 5, iters=10)
        same = bool(np.array_equal(mv_a, mv_b) and np.array_equal(cost_a, cost_b))
        work = n * nmb * (2 * R + 1) ** 2 * 256
        print(json.dumps({"case": "%dx%d +-%d %s" % (w, h, R, name), "rows_per_lane_task": b2enc.k1_prune_rows(R), "identical": same, "exhaustive_ms": round(ms_a, 4),
                          "exhaustive_frac_of_peak": round(work / (ms_a * 1e-3) / (peak * 4), 4),
                          "pruned_ms": round(st["kernel_ms"], 4), "block_sums_ms": round(st["sums_ms"], 4),
                          "speedup_incl_sums": round(ms_a / (st["kernel_ms"] + st["sums_ms"]), 3),
                          "executed_fraction": round(st["swept"] / st["all"], 4)}), flush=True)
