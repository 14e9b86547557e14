"""Whole encode stage on the GPU (through the C-ABI engine, include/b2enc_engine.h) against the C
oracle, frame by frame: converted/padded current planes (K0/K6), full-pel MVs and costs (K1), sub-pel
MVs and costs (K2), intra costs and modes (K3), decisions, quantised levels, cbp (K5/K7) and the
reconstructed planes must all be bit-identical."""
import numpy as np
import pytest
from test_oracle_decode import smooth_seq, coarse_seq, shear_seq

pytestmark = pytest.mark.gpu

INFO_FIELDS = ["mb_type", "mvx", "mvy", "i16_mode", "chroma_mode", "cbp", "i4_mode", "cost", "nnz_mask", "mv8", "part", "transform8x8", "i8_modes"]


def run_and_compare(oracle, b2, seqs, w, h, qp, R, subpel=1, intra_in_p=1, fmt="yuv420p", deblock=0, transform8x8=0, pack_levels=0,
                    partitions=0, deblock_offsets=(0, 0), me_prune=0, streams=0):
    """seqs: list (one per slot) of lists of (y,u,v) frames; streams: stream groups (0: the engine's default)"""
    S, T = len(seqs), len(seqs[0])
    eng = b2.Engine(w, h, slots=S, fmt=fmt, ring=2, merange=R, qp=qp, subpel=subpel, intra_in_p=intra_in_p, deblock=deblock,
                    transform8x8=transform8x8, pack_levels=pack_levels, partitions=partitions, deblock_offsets=deblock_offsets,
                    me_prune=me_prune, streams=streams)
    prm = oracle.Params(qp, R, subpel, intra_in_p, deblock, transform8x8, partitions, deblock_offsets[0], deblock_offsets[1])
    stats = {"t8": 0, "coded4": 0, "i8": 0, "parts": np.zeros(4, int), "mvx_mod4": np.zeros(4, int)}
    prev = [None] * S; prev_mv = [None] * S
    for t in range(T):
        for s in range(S):
            eng.put_frame(s, t % 2, list(seqs[s][t]))
        eng.h2d(ring=t % 2)
        ft = b2.FRAME_I if t == 0 else b2.FRAME_P
        eng.encode(ft, ring=t % 2)
        eng.d2h()
        eng.sync()
        for s in range(S):
            cur = oracle.OFrame(w, h).load(*seqs[s][t]); rec = oracle.OFrame(w, h)
            info_o, coef_o = oracle.encode_frame(prm, ft, cur, prev[s], rec, prev_mv[s])
            cy, cu, cv = eng.cur(s)
            assert np.array_equal(cy, cur.y) and np.array_equal(cu, cur.u) and np.array_equal(cv, cur.v), f"cur planes t={t} s={s}"
            info_g, coef_g = eng.results(s)
            if pack_levels:                            # K9's stream is exactly the host-side packing of the oracle's levels
                assert np.array_equal(eng.packed(s), b2.pack_levels(info_o, coef_o)), f"packed stream t={t} s={s}"
            if ft == b2.FRAME_P:
                mvf_o, cf_o = oracle.me_fullpel(cur, prev[s], R, prev_mv[s], oracle.lib().b2o_lambda(qp))
                assert np.array_equal(eng.stage(s, 0), mvf_o), f"K1 mv t={t} s={s}"
                assert np.array_equal(eng.stage(s, 1), cf_o), f"K1 cost t={t} s={s}"
                stats["mvx_mod4"] += np.bincount(mvf_o["x"].astype(int) & 3, minlength=4)
            want = b2.shipped_info(info_o) if pack_levels else info_o      # packed copy-out: 24-byte decision records
            for f in INFO_FIELDS:
                assert np.array_equal(info_g[f], want[f]), f"info.{f} t={t} s={s}: {np.argwhere(info_g[f] != want[f])[:5].tolist()}"
            assert np.array_equal(coef_g["blk"], coef_o["blk"]), f"levels t={t} s={s}"
            ry, ru, rv = eng.recon(s)
            assert np.array_equal(ry, rec.y), f"recon Y t={t} s={s}"
            assert np.array_equal(ru, rec.u) and np.array_equal(rv, rec.v), f"recon UV t={t} s={s}"
            stats["parts"] += np.bincount(info_o["part"][info_o["mb_type"] == 0], minlength=4)
            stats["t8"] += int(info_o["transform8x8"].sum()); stats["i8"] += int((info_o["mb_type"] == 3).sum())
            stats["coded4"] += int(((info_o["mb_type"] == 0) & (info_o["transform8x8"] == 0) & ((info_o["cbp"] & 15) != 0)).sum())
            prev[s] = rec
            prev_mv[s] = np.zeros(info_o.size, oracle.MV); prev_mv[s]["x"] = info_o["mvx"]; prev_mv[s]["y"] = info_o["mvy"]
    if me_prune and partitions != 2 and T > 1 and R == 32:          # +-16 and the wide partition search keep the exhaustive kernel
        swept, every = eng.k1_stats()
        assert 0 < swept <= every
        stats["k1_swept"] = swept / every
    elif me_prune:
        assert eng.k1_stats() is None
    eng.close()
    return stats


@pytest.mark.parametrize("w,h,qp,R,cut", [(176, 144, 26, 16, None), (320, 240, 32, 32, 2), (208, 160, 18, 16, 1),
                                          (318, 242, 28, 16, 3), (64, 48, 45, 32, 1)])
def test_engine_matches_oracle(oracle, b2, w, h, qp, R, cut):
    seqs = [smooth_seq(w, h, 5, seed=qp, cut=cut)]
    run_and_compare(oracle, b2, seqs, w, h, qp, R)


@pytest.mark.parametrize("w,h,qp,R,cut", [(176, 144, 26, 32, None), (320, 240, 32, 32, 2), (318, 242, 28, 16, 3), (64, 48, 45, 32, 1), (208, 160, 18, 32, 3)])
def test_engine_pruned_search_matches_oracle(oracle, b2, w, h, qp, R, cut):
    """engine option me_prune (K1a block sums + successive elimination in K1): every stage output still equals the oracle's, whose
    full-pel search is the plain exhaustive scan; several slots, scene cuts (predictors that point nowhere), packed and all tools on"""
    seqs = [smooth_seq(w, h, 5, seed=qp, cut=cut), smooth_seq(w, h, 5, seed=qp + 1), [oracle.synth_frame(w, h, t, 1) for t in range(5)]]
    st = run_and_compare(oracle, b2, seqs, w, h, qp, R, me_prune=1)
    if R == 32:
        assert st["k1_swept"] < 1.0
    run_and_compare(oracle, b2, seqs[:2], w, h, qp, R, me_prune=1, deblock=1, transform8x8=1, partitions=1, pack_levels=1)


def test_k2_patch_alignments(oracle, b2):
    """K2 stages its 22x22 reference patch as aligned words and keeps the byte alignment (mv.x - 3) mod 4 in shared memory:
    bands that pan by different whole-pixel amounts make every alignment occur, and everything stays oracle-exact"""
    w, h, n = 256, 256, 3
    rng = np.random.default_rng(77)
    import cv2
    base = cv2.resize(rng.integers(0, 256, (h // 4 + 8, (w + 128) // 4 + 8)).astype(np.float32), (w + 128, h), interpolation=cv2.INTER_CUBIC)
    pans = [0, 1, 2, 3, -1, -2, -3, 6]                                   # whole pixels per frame, one per 32-row band
    frames = []
    for t in range(n):
        img = np.empty((h, w), np.uint8)
        for b, px in enumerate(pans):
            x0 = 64 + px * t
            img[32 * b:32 * b + 32] = np.clip(base[32 * b:32 * b + 32, x0:x0 + w] + rng.normal(0, 1.0, (32, w)), 0, 255).astype(np.uint8)
        frames.append((img, (img[::2, ::2] // 2 + 60).astype(np.uint8), (200 - img[::2, ::2] // 2).astype(np.uint8)))
    stats = run_and_compare(oracle, b2, [frames], w, h, 28, 16)
    assert (stats["mvx_mod4"] > 8).all(), stats["mvx_mod4"]


def test_put_frame_direct(oracle, b2):
    """b2_engine_put_frame_direct: a picture in page-locked memory (strided, as b2_picture_alloc hands it out) goes to the
    device ring without the host copy and h2d skips it; pageable sources are refused with 1; results equal the staged path"""
    import ctypes as C
    w, h = 208, 112
    L = b2.lib()
    L.b2_pinned_alloc.restype = C.c_void_p; L.b2_pinned_alloc.argtypes = [C.c_size_t]; L.b2_pinned_free.argtypes = [C.c_void_p]
    stride = w + 48
    nbytes = stride * h + 2 * (stride // 2) * (h // 2)
    buf = L.b2_pinned_alloc(nbytes)
    assert buf
    try:
        mem = np.frombuffer((C.c_uint8 * nbytes).from_address(buf), np.uint8)
        py = mem[:stride * h].reshape(h, stride)[:, :w]
        pu = mem[stride * h:stride * h + (stride // 2) * (h // 2)].reshape(h // 2, stride // 2)[:, :w // 2]
        pv = mem[stride * h + (stride // 2) * (h // 2):].reshape(h // 2, stride // 2)[:, :w // 2]
        frames = smooth_seq(w, h, 3, seed=5)
        eng_a = b2.Engine(w, h, slots=2, ring=2, merange=16, qp=28)
        eng_b = b2.Engine(w, h, slots=2, ring=2, merange=16, qp=28)
        assert eng_a.put_frame_direct(0, 0, [np.ascontiguousarray(p) for p in frames[0]]) == 1      # pageable: refused
        for t, f in enumerate(frames):
            for s in range(2):
                g = frames[(t + s) % 3] if t == 0 else (frames[t] if s == 0 else frames[(t + 1) % 3])
                py[:] = g[0]; pu[:] = g[1]; pv[:] = g[2]
                if s == 0:
                    assert eng_a.put_frame_direct(s, t % 2, [py, pu, pv]) == 0
                else:
                    eng_a.put_frame(s, t % 2, list(g))               # mixed: one entry direct, one staged
                eng_b.put_frame(s, t % 2, list(g))
            mem[:] = 0                                               # the source may be reused as soon as the call returns
            ft = b2.FRAME_I if t == 0 else b2.FRAME_P
            for e in (eng_a, eng_b):
                e.h2d(ring=t % 2); e.encode(ft, ring=t % 2); e.d2h(); e.sync()
            for s in range(2):
                ia, ca = eng_a.results(s); ib, cb = eng_b.results(s)
                assert np.array_equal(ia, ib) and np.array_equal(ca["blk"], cb["blk"]), f"t={t} s={s}"
                for pa, pb in zip(eng_a.recon(s), eng_b.recon(s)):
                    assert np.array_equal(pa, pb)
        eng_a.close(); eng_b.close()
    finally:
        L.b2_pinned_free(buf)


def test_engine_lockstep_slots(oracle, b2):
    """several GOPs/streams in lock-step, different content per slot"""
    w, h = 192, 112
    seqs = [smooth_seq(w, h, 4, seed=s, cut=(2 if s == 1 else None)) for s in range(3)]
    seqs.append([oracle.synth_frame(w, h, t, 3) for t in range(4)])
    run_and_compare(oracle, b2, seqs, w, h, 30, 16)


def test_engine_fullpel_only_no_intra(oracle, b2):
    w, h = 160, 96
    seqs = [smooth_seq(w, h, 4, seed=9)]
    run_and_compare(oracle, b2, seqs, w, h, 26, 16, subpel=0, intra_in_p=0)


def test_engine_extreme_content(oracle, b2):
    w, h = 64, 64
    rng = np.random.default_rng(3)
    noise = [((rng.integers(0, 2, (h, w)) * 255).astype(np.uint8), (rng.integers(0, 2, (h // 2, w // 2)) * 255).astype(np.uint8),
              (rng.integers(0, 2, (h // 2, w // 2)) * 255).astype(np.uint8)) for _ in range(3)]
    flat = [(np.full((h, w), 90, np.uint8), np.full((h // 2, w // 2), 128, np.uint8), np.full((h // 2, w // 2), 128, np.uint8))] * 3
    for qp in (10, 51):
        run_and_compare(oracle, b2, [noise, flat], w, h, qp, 16)


@pytest.mark.parametrize("w,h,qp,R,cut", [(176, 144, 30, 16, None), (320, 240, 38, 32, 2), (208, 160, 20, 16, 1), (318, 242, 28, 16, 3),
                                          (64, 48, 51, 16, 1), (96, 80, 12, 16, 2)])
def test_engine_with_deblocking(oracle, b2, w, h, qp, R, cut):
    """K8 in-loop deblocking (SURVEY.md 8f N2): reconstruction and everything downstream stay bit-exact"""
    seqs = [smooth_seq(w, h, 5, seed=qp + 1, cut=cut), smooth_seq(w, h, 5, seed=qp + 2)]
    run_and_compare(oracle, b2, seqs, w, h, qp, R, deblock=1)


def test_engine_deblocking_wavefront(oracle, b2):
    """K8 takes its anti-diagonal wavefront when a launch covers 4 frames or more (bench.py's shape: 8 slots per stream group); the
    other deblocking tests put at most 3 slots in a group and so reach only the row pipeline.  Here 4 slots share one stream group.
    At 576x320 a diagonal holds up to 18 macroblocks, so each frame is a cluster of two CTAs with a cluster barrier per diagonal.
    The second run adds the 8x8 transform and 8x8 partitions, whose edge rules the wavefront derives on its own."""
    w, h = 576, 320
    seqs = [smooth_seq(w, h, 4, seed=41 + s, cut=(2 if s == 1 else None)) for s in range(3)] + [[oracle.synth_frame(w, h, t, 3) for t in range(4)]]
    run_and_compare(oracle, b2, seqs, w, h, 30, 16, deblock=1, streams=1)
    run_and_compare(oracle, b2, seqs, w, h, 26, 16, deblock=1, transform8x8=1, partitions=1, streams=1)


@pytest.mark.parametrize("offs", [(-1, -1), (3, -2), (-6, 6)])
def test_engine_deblocking_offsets(oracle, b2, offs):
    """tune film & co: loop-filter offsets (indexA = qp + 2a, indexB = qp + 2b) in K8 == oracle"""
    w, h, qp = 208, 160, 30
    seqs = [smooth_seq(w, h, 4, seed=31, cut=2), smooth_seq(w, h, 4, seed=32)]
    run_and_compare(oracle, b2, seqs, w, h, qp, 16, deblock=1, transform8x8=1, deblock_offsets=offs)


@pytest.mark.parametrize("w,h,qp,R,cut,deblock", [(176, 144, 26, 16, None, 1), (320, 240, 33, 32, 2, 1), (208, 160, 18, 16, 1, 0),
                                                  (318, 242, 28, 16, 3, 1), (64, 48, 12, 16, 1, 0), (96, 80, 44, 16, 2, 1)])
def test_engine_adaptive_8x8_transform(oracle, b2, w, h, qp, R, cut, deblock):
    """row N1: SA8D/SATD transform-size decision, 8x8 DCT/quant/dequant/IDCT in K5, transform-aware edges in K8"""
    seqs = [smooth_seq(w, h, 5, seed=qp + 3, cut=cut), smooth_seq(w, h, 5, seed=qp + 4)]
    stats = run_and_compare(oracle, b2, seqs, w, h, qp, R, deblock=deblock, transform8x8=1)
    assert stats["t8"] > 0
    if qp < 40:
        assert stats["coded4"] > 0


@pytest.mark.parametrize("w,h,qp,t8", [(176, 144, 26, 0), (320, 240, 34, 1), (64, 48, 12, 1), (318, 242, 45, 0)])
def test_engine_packed_levels(oracle, b2, w, h, qp, t8):
    """K9: only blocks with a non-zero level leave the GPU; stream == host packing of the oracle levels, several slots"""
    seqs = [smooth_seq(w, h, 4, seed=qp + 5, cut=2), smooth_seq(w, h, 4, seed=qp + 6), [oracle.synth_frame(w, h, t, 2) for t in range(4)]]
    run_and_compare(oracle, b2, seqs, w, h, qp, 16, deblock=1, transform8x8=t8, pack_levels=1)


@pytest.mark.parametrize("w,h,qp,scale,deblock,pack", [(96, 80, 40, 10, 1, 0), (176, 144, 44, 12, 0, 1), (208, 160, 36, 16, 1, 0),
                                                       (70, 54, 46, 8, 1, 1), (320, 240, 30, 14, 1, 0)])
def test_engine_intra8x8(oracle, b2, w, h, qp, scale, deblock, pack):
    """row N1, intra 8x8: K3 analysis (edge tables, SA8D), K5 decision, K7 serial 8x8 reconstruction; I and P frames"""
    seqs = [coarse_seq(w, h, 4, seed=qp, scale=scale), coarse_seq(w, h, 4, seed=qp + 1, scale=scale + 2)]
    for s in seqs:                       # scene change in every sequence -> intra macroblocks inside the P frames too
        s[2] = coarse_seq(w, h, 1, seed=qp + 9, scale=scale)[0]
    stats = run_and_compare(oracle, b2, seqs, w, h, qp, 16, deblock=deblock, transform8x8=1, pack_levels=pack)
    if qp >= 36:
        assert stats["i8"] >= 8


@pytest.mark.parametrize("w,h,qp,deblock,t8,pack", [(176, 144, 26, 1, 0, 0), (320, 240, 30, 1, 1, 1), (208, 160, 20, 0, 1, 0), (96, 80, 36, 1, 0, 1),
                                                    (70, 54, 30, 1, 0, 0)])
def test_engine_inter_partitions(oracle, b2, w, h, qp, deblock, t8, pack):
    """row N1: K2 per-quadrant refinement + shape decision, K5 per-quadrant chroma MC, K8 vector-aware boundary strengths"""
    seqs = [shear_seq(w, h, 4, seed=qp), shear_seq(w, h, 4, seed=qp + 1, stripe=40, band=16)]
    stats = run_and_compare(oracle, b2, seqs, w, h, qp, 16, deblock=deblock, transform8x8=t8, pack_levels=pack, partitions=1)
    assert np.all(stats["parts"][1:] > 0), stats["parts"]


@pytest.mark.parametrize("w,h,qp,R,amp,t8,pack", [(176, 144, 26, 16, 5, 0, 0), (320, 240, 30, 32, 9, 1, 1), (208, 160, 22, 16, 3, 1, 0), (96, 80, 34, 32, 7, 0, 1)])
def test_engine_wide_partition_search(oracle, b2, w, h, qp, R, amp, t8, pack):
    """row N1, partitions = 2: K1<PART> (quadrant SADs -> nine part vectors), shape on full-pel costs and per-part refinement in
    k2_me_subpel_wide_kernel; shears of several pixels per frame so that the parts really move apart"""
    seqs = [shear_seq(w, h, 4, seed=qp, amp=amp), shear_seq(w, h, 4, seed=qp + 1, stripe=40, band=16, amp=amp)]
    stats = run_and_compare(oracle, b2, seqs, w, h, qp, R, deblock=1, transform8x8=t8, pack_levels=pack, partitions=2)
    assert np.all(stats["parts"][1:] > 0), stats["parts"]


@pytest.mark.parametrize("pm", [1, 2])
def test_engine_all_features_extremes(oracle, b2, pm):
    """rows N1-N2 together on the edge cases the reference's domain has: one-macroblock pictures, saturated noise and flat
    content, QP 10 and 51, odd sizes -- deblocking + 8x8 transform / intra 8x8 + partitions + packed levels"""
    rng = np.random.default_rng(17)
    for (w, h) in ((16, 16), (32, 16), (16, 48), (70, 38)):
        cw, ch = (w + 1) // 2, (h + 1) // 2
        noise = [((rng.integers(0, 2, (h, w)) * 255).astype(np.uint8), (rng.integers(0, 2, (ch, cw)) * 255).astype(np.uint8),
                  (rng.integers(0, 2, (ch, cw)) * 255).astype(np.uint8)) for _ in range(3)]
        flat = [(np.full((h, w), 90, np.uint8), np.full((ch, cw), 128, np.uint8), np.full((ch, cw), 128, np.uint8))] * 3
        ramp = [((np.add.outer(np.arange(h) * 3, np.arange(w) * 2) + 5 * t).astype(np.uint8), np.full((ch, cw), 100 + t, np.uint8),
                 np.full((ch, cw), 140 - t, np.uint8)) for t in range(3)]
        for qp in (10, 51):
            run_and_compare(oracle, b2, [noise, flat, ramp], w, h, qp, 16, deblock=1, transform8x8=1, partitions=pm, pack_levels=1)


def _to_fmt(fmt, y, u, v):
    """repack an I420 picture into the raw layout `fmt` (exact inverse for the formats whose conversion is a copy;
    for packed 4:2:2 the chroma is duplicated on both lines so that the vertical average returns it)"""
    h, w = y.shape
    if fmt == "yuv420p":
        return [y, u, v]
    if fmt == "nv12":
        uv = np.empty((u.shape[0], 2 * u.shape[1]), np.uint8); uv[:, 0::2] = u; uv[:, 1::2] = v
        return [y, uv]
    p = np.empty((h, 2 * w), np.uint8)
    yo, uo, vo = (0, 1, 3) if fmt == "yuyv422" else (1, 0, 2)
    p[:, yo::2] = y
    p[:, uo::4] = np.repeat(u, 2, axis=0); p[:, vo::4] = np.repeat(v, 2, axis=0)
    return [p]


def _raw_planes(fmt, w, h, seed):
    """raw picture of the row-N4 layouts (band-limited content per plane)"""
    def plane(hh, ww, k):
        y = smooth_seq(max(ww, 16), max(hh, 16), 1, seed=seed + k)[0][0]
        return np.ascontiguousarray(y[:hh, :ww])
    if fmt in ("bgr24", "rgb24"):
        return [np.ascontiguousarray(np.stack([plane(h, w, 0), plane(h, w, 1), plane(h, w, 2)], axis=2).reshape(h, 3 * w))]
    scw = (w + 1) // 2 if fmt == "yuv422p" else (w + 3) // 4
    return [plane(h, w, 0), plane(h, scw, 1), plane(h, scw, 2)]


@pytest.mark.parametrize("fmt,w,h", [("nv12", 150, 98), ("yuyv422", 158, 82), ("uyvy422", 176, 144), ("yuv420p", 161, 99),
                                     ("nv12", 64, 48), ("bgr24", 150, 99), ("rgb24", 158, 82), ("yuv422p", 161, 98), ("yuv411p", 176, 144),
                                     ("yuv411p", 100, 50)])
def test_engine_input_formats_and_odd_sizes(oracle, b2, fmt, w, h):
    """K0 inside the engine: every supported raw layout, widths/heights that are not multiples of 16 (or even odd),
    checked against oracle conversion (pinned by live libswscale) + oracle frame encoder"""
    S, T, qp, R = 2, 3, 29, 16
    eng = b2.Engine(w, h, slots=S, fmt=fmt, ring=1, merange=R, qp=qp, subpel=1, intra_in_p=1, deblock=1)
    prm = oracle.Params(qp, R, 1, 1, 1)
    prev = [None] * S; prev_mv = [None] * S
    seqs = [smooth_seq(w, h, T, seed=7 + s) for s in range(S)]
    for t in range(T):
        raws = []
        for s in range(S):
            if fmt in ("bgr24", "rgb24", "yuv422p", "yuv411p"):
                raws.append(_raw_planes(fmt, w, h, 100 * s + 10 * t))
            else:
                y, u, v = seqs[s][t]
                u = u[:(h + 1) // 2, :(w + 1) // 2]; v = v[:(h + 1) // 2, :(w + 1) // 2]
                raws.append(_to_fmt(fmt, y, u, v))
            eng.put_frame(s, 0, raws[-1])
        ft = b2.FRAME_I if t == 0 else b2.FRAME_P
        eng.h2d(); eng.encode(ft); eng.d2h(); eng.sync()
        for s in range(S):
            cy, cu, cv = oracle.convert_to_i420(fmt, w, h, raws[s])
            cur = oracle.OFrame(w, h).load(cy, cu, cv); rec = oracle.OFrame(w, h)
            info_o, coef_o = oracle.encode_frame(prm, ft, cur, prev[s], rec, prev_mv[s])
            gy, gu, gv = eng.cur(s)
            assert np.array_equal(gy, cur.y) and np.array_equal(gu, cur.u) and np.array_equal(gv, cur.v), f"K0 {fmt} t={t}"
            info_g, coef_g = eng.results(s)
            assert np.array_equal(info_g, info_o) and np.array_equal(coef_g["blk"], coef_o["blk"])
            ry, ru, rv = eng.recon(s)
            assert np.array_equal(ry, rec.y) and np.array_equal(ru, rec.u) and np.array_equal(rv, rec.v)
            prev[s] = rec
            prev_mv[s] = np.zeros(info_o.size, oracle.MV); prev_mv[s]["x"] = info_o["mvx"]; prev_mv[s]["y"] = info_o["mvy"]
    eng.close()
