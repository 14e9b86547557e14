"""K2 alone (b2k_me_subpel) at the bench's shape: 64 frames of 1080p in one launch, the synthetic panning sequence with the
vectors K1 finds for it.  Prints one JSON line with the mean launch time (CUDA events) for partitions 0 and 1.  Point
B2ENC_LIB at another libb2enc.so to compare builds (e.g. one compiled with -DB2_K2_MBS=N)."""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "video-encoder_b200"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import b2enc  # noqa: E402
import b2oracle  # noqa: E402

W, H, N = 1920, 1088, 64
ys = [b2oracle.synth_frame(W, H, t)[0] for t in range(N + 1)]
cur, ref = np.stack(ys[1:]), np.stack(ys[:-1])
mvf, _, _ = b2enc.me_fullpel(cur, ref, 32)
pmv = np.zeros_like(mvf); pmv["x"] = 12; pmv["y"] = 8
out = {"lib": b2enc.so_path(), "frames": N, "size": [W, H]}
for parts in (0, 1):
    ms = [b2enc.me_subpel(cur, ref, mvf, pmv, 5, 1, parts, iters=50)[-1] for _ in range(3)]
    out["k2_ms_partitions%d" % parts] = [round(m, 4) for m in ms]
print(json.dumps(out))
