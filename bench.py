#!/usr/bin/env python
"""bench.py -- encode-stage throughput of the B200 engine on BASELINE.json's 1080p configuration.

Workload (config C3 of BASELINE.json): 1920x1080 synthetic frames (moving gradient + panning texture +
sensor noise, oracle/b2o_frame.c), yuv420p in, exhaustive +-32 full-pel SAD search + half/quarter-pel
SATD refinement, intra 16x16/4x4 + inter mode decision, 4x4 DCT/quant/dequant/recon, constant QP 26.
One GPU encodes SLOTS (64) closed GOPs of GOP frames in lock-step; a *step* advances every GOP by one frame
(step i is an I frame when i % GOP == 0, else a P frame), i.e. one pass of the hot path over a batch of
SLOTS frames.  With N GPUs every rank encodes its own SLOTS GOPs (closed-GOP sharding, no collective,
weak scaling); time = max over ranks.

  value : frames/s with the raw input pictures already resident in HBM (CUDA events on the engine stream)
  e2e   : frames/s through the C-ABI engine with HOST buffers: pinned-host -> device copy of every step's
          pictures and device -> host copy of every step's per-MB decisions + quantised levels inside the
          timed region (copy-in / compute / copy-out streams overlapped)
  roofline      : K1 (exhaustive SAD search, the dominant kernel): algorithmic pixel-SADs per launch /
                  mean launch time (CUDA events, live) against the chip's VABSDIFF4 rate measured live by
                  a microbenchmark in the same process (MEASURED_PEAKS.json has no integer-ALU number);
                  plus the HBM fraction of K0 (conversion) against MEASURED_PEAKS.json
  cpu_baseline  : the C oracle of the same stage on the host cores (one closed GOP per thread)
  dropin        : the same pictures through the x264-mirror call sequence (b2_encoder_encode, one picture per call,
                  host CABAC included) -- what an unmodified av_encode.c main loop would see (N=1 only)
  pruned        : value / e2e of the same workload with the engine's lossless search pruning on (me_prune: successive
                  elimination + partial-distortion exit in front of the same sweep; identical vectors and costs, oracle-verified),
                  the fraction of candidate vectors that was evaluated and K1's time alone with and without it (any N: whole-job figures).
                  Reported BESIDE the figures above, which are always the exhaustive search; never part of `roofline`

`--impl reference` times that CPU implementation alone (the reference's own libx264/libswscale path
cannot be built in this image: no headers, no libraries -- see DESIGN.md), all host threads.

`--dump-outputs DIR` writes what the last step of the timed `e2e` leg handed its caller, plus the reconstruction that step left
on the GPU (read back after timing), to DIR/*.npy (see dump_outputs).
The inputs depend on the arguments alone, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
# one hardware queue per stream group; must be in the environment before the first CUDA context exists (torch creates it under torchrun)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
sys.path.insert(0, os.path.join(ROOT, "video-encoder_b200"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))

W, H, MERANGE, QP, GOP = 1920, 1080, 32, 26, 32
# 64 GOPs x 8 stream groups: swept on the B200 (B2_BENCH_SLOTS): 32 -> 4,645, 48 -> 4,766, 64 -> 4,876, 96/128 -> 4,879 frames/s
SLOTS, RING, STREAMS = int(os.environ.get("B2_BENCH_SLOTS", "64")), 8, int(os.environ.get("B2_BENCH_STREAMS", "8"))
METRIC, UNIT = "1080p encode-stage frames/s", "frames/s"
WORKLOAD = ("C3: 1920x1080 synthetic yuv420p, +-32 exhaustive SAD + qpel SATD refine, intra16x16/4x4+inter decision, "
            "4x4 DCT/quant/recon, QP 26, closed GOP 32, %d GOPs in lock-step per GPU" % SLOTS)

# BASELINE.json's other GPU configurations (parity-test cases; `--workload` times them with the same harness).
# The default run is c3, the configuration the headline metric is quoted on.
WORKLOADS = {
    "c2": dict(W=1280, H=720, MERANGE=16, SLOTS=64, STREAMS=8, METRIC="720p encode-stage frames/s",
               WORKLOAD="C2: 1280x720 synthetic, P-frames, +-16 full-pel search (+ qpel, intra/inter as in C3), QP 26, GOP 32, 64 GOPs in lock-step per GPU"),
    "c3": None,
    "c4": dict(W=3840, H=2160, MERANGE=32, SLOTS=16, STREAMS=8, METRIC="2160p encode-stage frames/s",
               WORKLOAD="C4: 3840x2160 synthetic, closed-GOP sharding, +-32 + qpel + intra/inter, QP 26, GOP 32, 16 GOPs in lock-step per GPU"),
    "c5": dict(W=1280, H=720, MERANGE=16, SLOTS=8, STREAMS=4, METRIC="720p live-stream encode-stage frames/s",
               WORKLOAD="C5: 64 concurrent 720p live streams over 8 GPUs = 8 streams in lock-step per GPU (one frame of latency), +-16 + qpel + intra/inter, QP 26, GOP 32"),
}


def select_workload(name):
    global W, H, MERANGE, SLOTS, STREAMS, METRIC, WORKLOAD
    wl = WORKLOADS.get(name)
    if wl:
        W, H, MERANGE, SLOTS, STREAMS, METRIC, WORKLOAD = (wl["W"], wl["H"], wl["MERANGE"], wl["SLOTS"], wl["STREAMS"],
                                                             wl["METRIC"], wl["WORKLOAD"])
        STREAMS = int(os.environ.get("B2_BENCH_STREAMS", STREAMS))          # tuning sweeps only


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback"


class ClockSampler:
    """samples nvidia-smi clocks / throttle reasons during the timed region"""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(device), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def mark(self):
        return len(self.rows)

    def stop(self, start=0):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r.split(", ") for r in self.rows[start:] if r] or [r.split(", ") for r in self.rows if r]
        mhz = sorted(int(r[0]) for r in rows if r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in rows for n, v in zip(names, r[3:7]) if v.strip() == "Active"})
        return {"sm_mhz": mhz[len(mhz) // 2] if mhz else None, "sm_max_mhz": int(rows[0][1]) if rows and rows[0][1].isdigit() else None,
                "power_w_max": max((float(r[2]) for r in rows if r[2].replace(".", "").isdigit()), default=None),
                "samples": len(rows), "reasons": reasons}


_PICTURES = {}                                                  # (frame index, stream) -> packed I420 picture: several engines get the same input


def fill_inputs(eng, b2oracle, rank):
    import numpy as np
    import sharding
    streams = sharding.slot_streams(rank, eng.slots)            # disjoint synthetic streams per rank
    for s in range(eng.slots):
        for r in range(eng.ring):
            key = (W, H, r, streams[s])
            pic = _PICTURES.get(key)
            if pic is None:
                y, u, v = b2oracle.synth_frame(W, H, r, streams[s])
                pic = _PICTURES[key] = np.concatenate([y.ravel(), u.ravel(), v.ravel()])
            eng.host_input(s, r)[:pic.size] = pic


def dropin_leg(b2enc, b2oracle, deblock, transform8x8, partitions, frames=2048, gop_slots=None):
    """The same pictures through the x264-mirror call sequence of the reference (b2_encoder_encode, include/b2enc.h;
    av_encode.c:968-975, :1076-1083): one picture per call from host memory, host entropy coding (CABAC) included.
    deblock=None: the mirror's defaults, i.e. what an unmodified av_encode.c gets (x264's: loop filter on, tune film -1:-1)."""
    src = [b2oracle.synth_frame(W, H, t, 0) for t in range(16)]
    ext = dict(i_keyint_max=GOP, b_transform_8x8=transform8x8, b_partitions=partitions)
    if gop_slots: ext["i_gop_slots"] = gop_slots
    if deblock is not None: ext["b_deblocking_filter"] = deblock
    def open_encoder():
        return b2enc.DropInEncoder(W, H, preset="slow" if MERANGE == 32 else "medium", tune="film", quality=QP, fps=(60, 1), annexb=0, **ext)
    # untimed warm-up with a throw-away encoder (two GOPs in, flush, close): one-time costs of the process -- CUDA module loading of
    # kernels this configuration uses first, page-locking of the staging buffers, thread start-up -- stay out of the timed encoder,
    # like the warm-up steps of the engine legs; the timed encoder still pays its own open, pipeline fill and drain
    warm = open_encoder()
    for t in range(2 * GOP):
        warm.encode_via_sws("yuv420p", src[t % 16], t)
    while warm.delayed() > 0 and warm.encode(None, 0)[0] > 0:
        pass
    warm.close()
    enc = open_encoder()
    t0 = time.perf_counter(); nout = 0; nbytes = 0; first = None; first_ms = None
    for t in range(frames):
        # the reference's per-frame pair: sws_scale(decoded picture -> pic_in), x264_encoder_encode(pic_in) (av_encode.c:545-547, :970)
        size = enc.encode_via_sws("yuv420p", src[t % 16], t)[0]
        if size > 0:
            nout += 1; nbytes += size
            if first is None: first = t + 1; first_ms = (time.perf_counter() - t0) * 1e3
    while enc.delayed() > 0:
        size = enc.encode(None, 0)[0]
        if size <= 0: break
        nout += 1; nbytes += size
    dt = time.perf_counter() - t0
    slots = enc.param.i_gop_slots
    enc.close()
    return {"value": round(nout / dt, 1), "unit": UNIT, "frames": nout, "gop_slots_per_gpu": slots, "bytes_per_frame": int(nbytes / max(nout, 1)),
            "deblocking_filter": "x264 default (on, tune film -1:-1)" if deblock is None else bool(deblock),
            "first_output_after_pictures": first, "first_output_after_ms": round(first_ms, 1) if first_ms else None,
            "first_output_note": "one GOP fill is not needed: a GOP starts with its first picture; the first frame is an IDR whose host CABAC takes "
                                 "tens of ms at 1080p, during which this producer keeps handing pictures in",
            "host_cores": os.cpu_count(),
            "api": "b2_param_default_preset / b2_encoder_open / b2_picture_alloc / b2_encoder_encode / b2_encoder_delayed_frames "
                   "(x264 mirror, include/b2enc.h) with b2_sws_scale(decoder picture -> pic_in) in front of every encode call, as av_encode.c:545-547/:970 does; driven from Python: one picture per call, pipeline fill and drain inside the timed region",
            "note": "entropy coding (CABAC) on the host cores is part of this call sequence; the encode stage itself is `e2e`"}


def verify_final_state(eng, b2enc, b2oracle, rank, groups, ftype, last_step, args):
    """After the timed regions (outside every timing): the first slot of every stream group is replayed on the CPU oracle from
    the group's last I step to the last issued step, and its final per-MB decisions, packed levels and reconstruction on the
    GPU must equal the oracle's bit for bit -- the state left behind by the exact pipelined path that was timed."""
    import numpy as np
    import sharding
    from concurrent.futures import ThreadPoolExecutor
    streams = sharding.slot_streams(rank, eng.slots)
    prm = b2oracle.Params(QP, MERANGE, 1, 1, args.deblock, args.transform8x8, args.partitions)

    def chain(g):
        slot = groups[g][0]
        s0 = max(s for s in range(last_step + 1) if ftype(s, g) == b2enc.FRAME_I)
        prev = None; pmv = None
        for s in range(s0, last_step + 1):
            cur = b2oracle.OFrame(W, H).load(*b2oracle.synth_frame(W, H, s % RING, streams[slot])); rec = b2oracle.OFrame(W, H)
            info, coef = b2oracle.encode_frame(prm, 0 if s == s0 else 1, cur, prev, rec, pmv)
            pmv = np.zeros(info.size, b2oracle.MV); pmv["x"] = info["mvx"]; pmv["y"] = info["mvy"]
            prev = rec
        return slot, last_step + 1 - s0, info, coef, rec

    t0 = time.perf_counter()
    with ThreadPoolExecutor(min(len(groups), os.cpu_count() or 1)) as ex:
        res = list(ex.map(chain, range(len(groups))))
    bad = []
    for slot, n, info_o, coef_o, rec in res:
        info_g, _ = eng.results(slot)
        want = b2enc.shipped_info(info_o) if args.pack_levels else info_o
        ok = all(np.array_equal(info_g[f], want[f]) for f in info_o.dtype.names)
        if args.pack_levels:
            ok = ok and np.array_equal(eng.packed(slot), b2enc.pack_levels(info_o, coef_o))
        else:
            ok = ok and np.array_equal(eng.results(slot)[1]["blk"], coef_o["blk"])
        ry, ru, rv = eng.recon(slot)
        ok = ok and np.array_equal(ry, rec.y) and np.array_equal(ru, rec.u) and np.array_equal(rv, rec.v)
        if not ok:
            bad.append(slot)
    return {"verified": not bad, "slots_checked": [r[0] for r in res], "frames_replayed_on_oracle": int(sum(r[1] for r in res)),
            "mismatching_slots": bad, "seconds": round(time.perf_counter() - t0, 1),
            "what": "final per-MB decisions, packed levels and reconstruction of the first slot of every stream group after the timed "
                    "regions == CPU oracle replay from the group's last I step (bit-exact)"}


DUMP_MBS = 16384                                                # --dump-outputs sample: ~57 MB of .npy files, under 64 MB


def dump_outputs(eng, out_dir):
    """--dump-outputs: the results of the engine's last step for a fixed sample of DUMP_MBS macroblocks drawn over all slots
    (numpy seed 0, sorted by slot and macroblock; every macroblock when there are fewer):
      mb_info.npy  float64 (n, 33): the per-MB decisions the caller receives, MBINFO fields in order, subarrays flattened
      levels.npy   float32 (n, 26, 16): the quantised levels the caller receives (unpacked when they leave the GPU packed)
      recon.npy    float32 (n, 384): the reconstructed macroblock, 16x16 luma then 8x8 Cb and 8x8 Cr, row by row.  The caller
                   does not receive it: it is the reference state of the next step, read back from the GPU after timing
    Every value is exact in its type."""
    import numpy as np
    from numpy.lib import recfunctions
    n = min(DUMP_MBS, eng.slots * eng.nmb)
    pick = np.sort(np.random.default_rng(0).choice(eng.slots * eng.nmb, n, replace=False))
    info, levels, recon = [], [], []
    for s in np.unique(pick // eng.nmb):
        mbs = pick[pick // eng.nmb == s] % eng.nmb
        i, coef = eng.results(int(s))
        info.append(recfunctions.structured_to_unstructured(i[mbs], np.float64))
        levels.append(coef["blk"][mbs].astype(np.float32))
        blocks = [p.reshape(eng.mbh, b, eng.mbw, b).transpose(0, 2, 1, 3).reshape(eng.nmb, b * b)[mbs]
                  for p, b in zip(eng.recon(int(s)), (16, 8, 8))]
        recon.append(np.concatenate(blocks, axis=1).astype(np.float32))
    os.makedirs(out_dir, exist_ok=True)
    for name, parts in (("mb_info", info), ("levels", levels), ("recon", recon)):
        np.save(os.path.join(out_dir, name + ".npy"), np.concatenate(parts))


def cpu_encode_gop(b2oracle, np, stream, n_p, times):
    """one closed GOP on one host thread: 1 I + n_p P frames through the oracle encode stage"""
    prm = b2oracle.Params(QP, MERANGE, 1, 1)
    prev = None; pmv = None
    for t in range(1 + n_p):
        y, u, v = b2oracle.synth_frame(W, H, t, stream)
        src = (y, u, v)
        t0 = time.perf_counter()
        # conversion (a1) + load into the padded frame, then the frame-level stage
        cy, cu, cv = b2oracle.convert_to_i420("yuv420p", W, H, list(src))
        cur = b2oracle.OFrame(W, H).load(cy, cu, cv); rec = b2oracle.OFrame(W, H)
        info, coef = b2oracle.encode_frame(prm, 0 if t == 0 else 1, cur, prev, rec, pmv)
        times.append((t == 0, time.perf_counter() - t0))
        pmv = np.zeros(info.size, b2oracle.MV); pmv["x"] = info["mvx"]; pmv["y"] = info["mvy"]
        prev = rec


def cpu_baseline(n_p=6):
    import numpy as np
    import b2oracle
    from concurrent.futures import ThreadPoolExecutor
    b2oracle.lib()
    threads = os.cpu_count() or 1
    times = [[] for _ in range(threads)]
    t0 = time.perf_counter()
    with ThreadPoolExecutor(threads) as ex:
        list(ex.map(lambda i: cpu_encode_gop(b2oracle, np, i, n_p, times[i]), range(threads)))
    wall = time.perf_counter() - t0
    t_i = sum(t for ts in times for is_i, t in ts if is_i) / threads
    t_p = sum(t for ts in times for is_i, t in ts if not is_i) / (threads * n_p)
    fps = threads * GOP / (t_i + (GOP - 1) * t_p)          # GOP-32 equivalent, all threads busy
    return {"value": round(fps, 3), "unit": UNIT, "cores": threads, "kind": "port",
            "sample": "C oracle (oracle/b2o_*.c, gcc -O3 -march=native), %d threads x (1 I + %d P) 1080p frames, one closed GOP "
                      "per thread, %.1f s wall; value = GOP-%d equivalent from mean I (%.3f s) and P (%.3f s) frame times"
                      % (threads, n_p, wall, GOP, t_i, t_p)}


def run_reference(args):
    """--impl reference: the CPU implementation of the path (oracle port; libx264/libswscale absent)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import numpy as np
    import b2oracle
    from concurrent.futures import ThreadPoolExecutor
    b2oracle.lib()
    threads = os.cpu_count() or 1
    prm = b2oracle.Params(QP, MERANGE, 1, 1)
    state = []
    for i in range(threads):                                   # untimed: frame 0 (I) of every thread's GOP
        cur = b2oracle.OFrame(W, H).load(*b2oracle.synth_frame(W, H, 0, i)); rec = b2oracle.OFrame(W, H)
        info, _ = b2oracle.encode_frame(prm, 0, cur, None, rec, None)
        state.append([rec, None, 1])

    # GOP phases staggered over the threads like the GPU arm staggers its stream groups: over the run the I : P mix is the
    # workload's 1 : GOP-1 (an I frame costs the CPU ~6x less than a P frame, so P-only steps would under-state it)
    phase = [i * GOP // threads for i in range(threads)]

    def step(i):
        rec_prev, pmv, t = state[i]
        is_i = (phase[i] + t) % GOP == 0
        cur = b2oracle.OFrame(W, H).load(*b2oracle.convert_to_i420("yuv420p", W, H, list(b2oracle.synth_frame(W, H, t % RING, i))))
        rec = b2oracle.OFrame(W, H)
        info, _ = b2oracle.encode_frame(prm, 0 if is_i else 1, cur, None if is_i else rec_prev, rec, None if is_i else pmv)
        pmv = np.zeros(info.size, b2oracle.MV); pmv["x"] = info["mvx"]; pmv["y"] = info["mvy"]
        state[i] = [rec, pmv, t + 1]

    with ThreadPoolExecutor(threads) as ex:
        for _ in range(args.warmup):
            list(ex.map(step, range(threads)))
        t0 = time.perf_counter()
        for _ in range(args.steps):
            list(ex.map(step, range(threads)))
        dt = time.perf_counter() - t0
    fps = threads * args.steps / dt
    sample = ("each step = one %dx%d frame per host thread (%d threads = all host CPUs, one closed GOP of %d each, GOP phases staggered so "
              "that I frames occur at the workload's 1 : %d rate) through the C oracle port of the stage, scalar C built -O3 "
              "-march=native (libx264/libswscale are not buildable here: this is NOT x264's speed)" % (W, H, threads, GOP, GOP - 1))
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": round(fps, 3), "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(dt / args.steps * 1e3, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": sample},
        "cpu_baseline": {"value": round(fps, 3), "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": round(fps, 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-dropin", action="store_true", help="skip the x264-mirror call-sequence leg (key `dropin`)")
    ap.add_argument("--no-verify", action="store_true", help="skip the post-run oracle check of the engine's final state (key `verified`)")
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--deblock", type=int, default=0, help="1: also run the in-loop deblocking filter K8 (row N2, outside the named path)")
    ap.add_argument("--pack-levels", type=int, default=1, help="1: levels leave the GPU packed (K9: only blocks with a non-zero level); "
                    "0: dense 832 B/MB array")
    ap.add_argument("--partitions", type=int, default=0, help="1: inter partitions 16x8/8x16/8x8 (row N1, outside the named path)")
    ap.add_argument("--me-prune", type=int, default=0, help="1: run the MAIN legs with the lossless search pruning on (default 0: exhaustive; the "
                    "pruned figures are reported beside them under `pruned`)")
    ap.add_argument("--no-pruned-leg", action="store_true", help="skip the `pruned` leg")
    ap.add_argument("--transform8x8", type=int, default=0, help="1: adaptive 8x8 transform for inter MBs (row N1, outside the named path)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last `e2e` step, and the reconstruction "
                    "read back from the GPU after timing, for a fixed sample of macroblocks (rank 0) to DIR/*.npy")
    args = ap.parse_args()
    select_workload(args.workload)
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs applies to --impl b200")
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    import numpy as np  # noqa: F401
    import b2enc
    import b2oracle
    b2enc.require_gpu()
    numa_cpus = b2enc.bind_to_gpu_numa(local)                  # pinned staging next to the GPU's PCIe root

    def barrier():
        if dist is not None:
            import torch
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def make_engine(me_prune, profile=0, streams=STREAMS, ring=RING):
        e = b2enc.Engine(W, H, slots=SLOTS, fmt="yuv420p", ring=ring, merange=MERANGE, qp=QP, subpel=1, intra_in_p=1,
                         device=local, profile=profile, streams=streams, deblock=args.deblock, transform8x8=args.transform8x8,
                         pack_levels=args.pack_levels, partitions=args.partitions, me_prune=me_prune)
        fill_inputs(e, b2oracle, rank)
        for r in range(ring):
            e.h2d(ring=r)
        e.sync()
        return e

    eng = make_engine(args.me_prune)
    int_rate, _ = b2enc.vabsdiff4_peak(local, 512, 5)           # VABSDIFF4 lane-instructions / s, live

    groups = eng.groups()
    NG = len(groups)
    phase = [g * GOP // NG for g in range(NG)]                  # staggered GOP phases: one group in an I frame at a time

    def ftype(step, g):
        """frame type of group g at global step `step` (step 0 = every group's first IDR)"""
        return b2enc.FRAME_I if step == 0 or (step + phase[g]) % GOP == 0 else b2enc.FRAME_P

    def issue(step, with_copies, eng=eng):
        ring = step % RING
        if with_copies:
            eng.h2d(ring=ring)                                   # this step's pictures: pinned host -> device ring
        for g in range(NG):
            eng.encode_group(g, ftype(step, g), ring=ring)
            if with_copies:
                eng.d2h_group(g)                                 # decisions + levels -> pinned host

    # ---- device-resident throughput ------------------------------------------------------------------
    step = 0
    for _ in range(args.warmup):
        issue(step, False); step += 1
    eng.sync()
    clocks = ClockSampler(local)
    time.sleep(0.3)
    barrier()
    mark = clocks.mark()
    l0 = eng.launch_count()
    eng.timer_start()
    for _ in range(args.steps):
        issue(step, False); step += 1
    ms = eng.timer_stop()
    eng.sync()
    barrier()
    launches = eng.launch_count() - l0
    ms = max_over_ranks(ms)
    value = world * SLOTS * args.steps / (ms * 1e-3)

    # ---- end to end through the C-ABI with host buffers ----------------------------------------------
    n_e2e = args.steps
    for _ in range(2):                                             # warm the copy paths
        issue(step, True); step += 1
    eng.sync()
    packed0 = eng.packed_bytes_total() if args.pack_levels else 0
    barrier()
    t0 = time.perf_counter()
    for _ in range(n_e2e):
        issue(step, True); step += 1
    eng.sync()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    packed_per_step = (eng.packed_bytes_total() - packed0) / n_e2e if args.pack_levels else 0
    barrier()
    clk = clocks.stop(mark)
    e2e = world * SLOTS * n_e2e / e2e_s
    if rank == 0 and args.dump_outputs:
        dump_outputs(eng, args.dump_outputs)                     # the e2e leg's last step: its results are in the host buffers

    # ---- after the timed legs: verification of the state they left (rank 0), then the same legs with the search pruning on ------
    iso = None
    verify = None
    pruned = None
    if rank == 0 and not args.no_verify:
        verify = verify_final_state(eng, b2enc, b2oracle, rank, groups, ftype, step - 1, args)
    eng.close()

    # the same workload with the lossless search pruning on (engine option me_prune; reported beside, never instead).  Every rank
    # runs it, timed like the legs above (device events / wall clock, barrier on both sides, max over ranks)
    run_pruned = not args.no_pruned_leg and not args.me_prune and args.partitions != 2 and MERANGE == 32     # the engine prunes at +-32 only
    if run_pruned:
        engp = make_engine(1)
        sp = 0
        for _ in range(args.warmup):
            issue(sp, False, engp); sp += 1
        engp.sync()
        sw0, al0 = engp.k1_stats()
        barrier()
        engp.timer_start()
        for _ in range(args.steps):
            issue(sp, False, engp); sp += 1
        msp = engp.timer_stop()
        engp.sync()
        barrier()
        msp = max_over_ranks(msp)
        sw1, al1 = engp.k1_stats()
        for _ in range(2):
            issue(sp, True, engp); sp += 1
        engp.sync()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            issue(sp, True, engp); sp += 1
        engp.sync()
        e2ep = max_over_ranks(time.perf_counter() - t0)
        barrier()
        vp = None
        if rank == 0 and not args.no_verify:
            vp = verify_final_state(engp, b2enc, b2oracle, rank, groups, ftype, sp - 1, args)
        engp.close()

    # ---- K1/K0 alone (one stream, nothing overlapping): the roofline numerator --------------------------
    if rank == 0:
        def kernels_alone(me_prune):
            # the same picture sequence as the timed legs (ring of RING pictures): the pruned search depends on the content
            e1 = make_engine(me_prune, profile=1, streams=1, ring=RING)
            e1.encode(b2enc.FRAME_I, ring=0)
            for i in range(2):
                e1.encode(b2enc.FRAME_P, ring=(i + 1) % RING)
            e1.sync(); e1.profile_reset()
            for i in range(8):
                e1.encode(b2enc.FRAME_P, ring=(i + 3) % RING)
            r = e1.kernel_ms(), e1.nmb, e1.in_bytes, e1.w16, e1.h16
            e1.close()
            return r

        # the roofline kernel is ALWAYS the exhaustive one, whatever --me-prune says
        iso, mbs, in_bytes, w16, h16 = kernels_alone(0)
        if run_pruned:
            isop = kernels_alone(1)[0]
            pruned = {"value": round(world * SLOTS * args.steps / (msp * 1e-3), 2), "unit": UNIT, "n_gpus": world, "ms_per_step": round(msp / args.steps, 4),
                      "e2e": round(world * SLOTS * args.steps / e2ep, 2),
                      "verified": vp["verified"] if vp else None, "verify_seconds": vp["seconds"] if vp else None,
                      "k1_candidates_evaluated": int(sw1 - sw0), "k1_candidates_algorithmic": int(al1 - al0),
                      "k1_executed_fraction": round((sw1 - sw0) / max(al1 - al0, 1), 4),
                      "k1_rows_per_lane_task": b2enc.k1_prune_rows(MERANGE),
                      "k1_ms_per_step_alone": round(isop["K1 full-pel SAD"][0] / 8, 4),
                      "k1_ms_per_step_alone_exhaustive": round(iso["K1 full-pel SAD"][0] / 8, 4),
                      "what": "engine option me_prune=1: K1a (min | max of the reference's 16x16 block sums over the rows of a lane-task, once per P step) + "
                              "successive elimination in K1 -- a candidate whose |sum(cur) - sum(ref)| + mvcost exceeds the exact cost of the zero vector / "
                              "the rounded predictor cannot be the minimum, and a lane-task (k1_rows_per_lane_task consecutive dy at one dx) is skipped when "
                              "that holds for all of its candidates -- plus a partial-distortion exit inside the sweep; vectors, costs and tie-break are those "
                              "of the exhaustive scan (tests/test_me_fullpel.py, the oracle replay of this leg's final state), only the time changes, and it "
                              "depends on the content (this synthetic sequence pans uniformly, so the predictor is exact except where the 8-picture ring "
                              "wraps; k1_executed_fraction = candidates evaluated / candidates of the exhaustive search, rank 0).  Whole-job figures at "
                              "n_gpus, timed like `value` / `e2e`.  Not part of `value`, `e2e` or `roofline`: those are the exhaustive search"}

    if rank == 0:
        peaks, peak_src = measured_peaks()
        k1_ms, k1_n = iso["K1 full-pel SAD"]
        k0_ms, k0_n = iso["K0 convert"]
        sads_per_launch = SLOTS * mbs * (2 * MERANGE + 1) ** 2 * 256
        k1_rate = sads_per_launch / (k1_ms / max(k1_n, 1) * 1e-3) if k1_n else 0.0
        k0_bytes = SLOTS * (in_bytes + 1.5 * w16 * h16)
        k0_gbs = k0_bytes / (k0_ms / max(k0_n, 1) * 1e-3) / 1e9 if k0_n else 0.0
        total_k = sum(v[0] for v in iso.values())
        out = {
            "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(ms / args.steps, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": {"workload": WORKLOAD, "frames_per_step": SLOTS * world, "gop": GOP, "input_ring_frames": RING,
                       "l2": "no flush needed: per-step working set (cur+ref+recon planes of %d frames ~ %d MB + raw ring) exceeds the 126 MB L2"
                             % (SLOTS, int(SLOTS * 3 * 1.5 * w16 * h16 / 1e6)),
                       "host_cpus_bound_to_gpu_numa_node": len(numa_cpus) if numa_cpus else None, "stream_groups": NG, "gop_phase_per_group": phase, "deblocking_filter": bool(args.deblock),
                       "deblocking_note": "the named path (BASELINE.json C3) has no loop filter, so K8 is off here (--deblock 1 adds it); an av_encode.c user of the x264 mirror gets x264's default: filter ON, tune film offsets -1:-1 -- that configuration is the `dropin` leg", "transform8x8": bool(args.transform8x8), "partitions": bool(args.partitions),
                       "parallelism": "closed-GOP sharding, %d GPUs x %d GOPs, no collective" % (world, SLOTS)},
            "e2e": {"value": round(e2e, 2), "unit": UNIT, "h2d_bytes_per_step": int(world * SLOTS * in_bytes),
                    "d2h_bytes_per_step": int(world * (SLOTS * mbs * 24 + packed_per_step)) if args.pack_levels else int(world * SLOTS * mbs * (48 + 832)),
                    "d2h_note": ("per-MB decisions (24-byte records, b2_mbinfo_packed_t) + packed levels (K9: blocks with a non-zero level only; mean over the timed steps, rank 0 x n_gpus)"
                                 if args.pack_levels else "per-MB decisions (48 B) + dense levels (832 B)"), "api": "b2_engine_h2d/encode/d2h (include/b2enc_engine.h), pinned host buffers",
                    "timing": "host wall clock around %d pipelined steps, synchronised on both sides" % n_e2e},
            "gpu_launches": int(launches),
            "verified": verify["verified"] if verify else None, "verify": verify,
            "clocks": clk,
            "roofline": {"bound": "int_alu", "kernel": "k1_me_fullpel_kernel<%d,256>" % MERANGE, "achieved": round(k1_rate / 1e12, 3),
                         "peak": round(int_rate * 4 / 1e12, 3), "unit": "Tpixel-SAD/s", "frac": round(k1_rate / (int_rate * 4), 4),
                         "peak_source": "live VABSDIFF4.U8.ACC microbenchmark (b2_bench_vabsdiff4_peak), x4 pixels per lane-instruction",
                         "algorithmic_per_launch": sads_per_launch, "ms_per_launch": round(k1_ms / max(k1_n, 1), 4),
                         "how": "launch covering all %d frames timed alone on one stream (8 launches, CUDA events) right after the timed region; inside the timed region %d stream groups overlap, so per-kernel times there are not separable" % (SLOTS, NG),
                         "share_of_step": round(k1_ms / total_k, 3) if total_k else None,
                         "share_note": "K1 time / sum of all kernel times of a P step, each timed alone on one stream",
                         "executed_note": "no pruning: the ncu capture in profiles/ counts 275.8 M VABSDIFF4 warp-instructions for a 4-frame 1080p +-32 launch = the algorithmic 4 x 8160 x 4225 x 64 / 32",
                         "traffic": 18.5e6 * SLOTS / 4, "traffic_note": "dram bytes of one launch from the ncu --set full capture in profiles/ (4-frame launch: 18.5 MB), scaled to %d frames" % SLOTS,
                         "hbm": {"kernel": "k0_convert_kernel", "bound": "hbm", "achieved": round(k0_gbs, 1), "peak": peaks.get("hbm_gbs"),
                                 "unit": "GB/s", "frac": round(k0_gbs / peaks.get("hbm_gbs", 6650.0), 4), "peak_source": peak_src,
                                 "algorithmic_bytes_per_launch": int(k0_bytes)}},
            "kernel_ms_per_step_alone": {k: round(v[0] / 8, 4) for k, v in iso.items()},
        }
        out["config"]["me_prune"] = bool(args.me_prune)
        if pruned:
            out["pruned"] = pruned
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline()
        if world == 1 and not args.no_dropin and args.workload in ("c2", "c3"):
            out["dropin"] = dropin_leg(b2enc, b2oracle, None, args.transform8x8, args.partitions)          # what av_encode.c gets
            out["dropin_named_path"] = dropin_leg(b2enc, b2oracle, 0, args.transform8x8, args.partitions)   # loop filter off like `value`
        print(json.dumps(out))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
