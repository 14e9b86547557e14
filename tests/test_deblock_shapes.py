"""K8, the in-loop deblocking filter (H.264 8.7), at every launch shape of its two schedules: on its own (b2k_deblock) against
the oracle's normative filter (b2o_deblock_frame, pinned to libavcodec by test_oracle_decode.py), and inside the engine at the
picture sizes users run.

The schedule and the cluster size depend on the picture size and on the number of frames in a launch (b2_deblock_shape):
- row pipeline (fewer than 4 frames): one warp per macroblock row, 8 warps per CTA, the ceil(mbh / 8) CTAs of a frame form a
  cluster (non-portable size above 8, at most 16).  Beyond 128 rows a warp takes several rows, and the last warp of the last
  CTA hands its bottom rows to warp 0 of CTA 0 through distributed shared memory for that warp's next round.
- anti-diagonal wavefront (4 frames or more): 16 warps per CTA, a cluster of 1, 2, 4 or 8 CTAs chosen from the longest
  diagonal min(mbh, ceil(mbw / 2)), a CTA barrier (1 CTA) or cluster barrier between diagonals; beyond 128 macroblocks per
  diagonal a warp takes several.  It derives the boundary strengths with its own code.
A mistake in a cross-CTA hand-off, a round counter or the per-diagonal work split only shows at those sizes, and silently:
the filtered picture is the next frame's reference.  Every case asserts the (wavefront, CTAs per frame, rounds per warp) it
reaches, so that a retuned threshold cannot leave a case testing nothing new.

Not covered: the row pipeline's 8-CTA fallback for a device that refuses the non-portable cluster size.  A B200 never refuses
it, and it cannot be forced without changing the launcher."""
import numpy as np
import pytest
from b2oracle import MBINFO, PAD, PADC
from test_full_size import _encode_and_check

# alpha(indexA) and beta(indexB), Table 8-16
ALPHA = [0] * 16 + [4, 4, 5, 6, 7, 8, 9, 10, 12, 13, 15, 17, 20, 22, 25, 28, 32, 36, 40, 45, 50, 56, 63, 71, 80, 90, 101, 113, 127,
                    144, 162, 182, 203, 226, 255, 255]
BETA = [0] * 16 + [2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13, 14, 14, 15, 15, 16, 16, 17, 17,
                   18, 18]
# (qp, slice_alpha_c0_offset_div2, slice_beta_offset_div2) taken in turn by the cases: QP 10..51, offsets -6..6, indexA clipped
# to 51 (51 + 12) and to 0 (10 - 12: nothing is filtered)
QPS = [(26, 0, 0), (51, 6, 6), (30, -1, -1), (10, -6, -6), (38, 3, -2), (45, -6, 6), (18, 6, 1), (24, 3, -2), (34, -3, 3),
       (42, 1, -1), (14, 6, 6), (49, -2, 4), (33, 0, -3)]
# centres of the motion vectors of a 4x4-macroblock tile: around zero (components of both signs, int16 sign handling), and
# far out in the int16 range
MV_CENTRES = np.array([0, -1000, -32760, 32760])


def clip_index(qp, off):
    """indexA / indexB (8.7.2.2)"""
    return min(51, max(0, qp + 2 * off))


def make_info(rng, n, mbw, mbh):
    """random decisions for n frames, covering every input of the boundary-strength rule"""
    nmb = mbw * mbh
    info = np.zeros((n, nmb), MBINFO)
    t = rng.choice(4, (n, nmb), p=[0.55, 0.15, 0.15, 0.15])
    info["mb_type"] = t
    info["part"] = rng.integers(0, 4, (n, nmb))
    info["transform8x8"] = np.where(t == 3, 1, rng.integers(0, 2, (n, nmb)))
    info["nnz_mask"] = ((rng.random((n, nmb, 27)) < 0.3) * (1 << np.arange(27, dtype=np.int64))).sum(-1).astype(np.uint32)
    tiles = rng.choice(len(MV_CENTRES), (n, (mbh + 3) // 4, (mbw + 3) // 4), p=[0.6, 0.15, 0.15, 0.1])
    centre = MV_CENTRES[tiles].repeat(4, 1).repeat(4, 2)[:, :mbh, :mbw].reshape(n, nmb)
    # components spread by -3..3 around the centre: neighbouring vectors differ by 0..6, i.e. by 3, 4 and 5 too
    mv = centre[:, :, None] + rng.integers(-3, 4, (n, nmb, 8))
    info["mvx"], info["mvy"] = mv[..., 0], mv[..., 1]
    info["mv8"] = mv[..., 2:].reshape(n, nmb, 3, 2)
    return info


def make_planes(rng, w, h, n, alpha):
    """n frames of padded planes in the engine's layout: random border bytes (which K8 must leave alone) around a picture of
    smooth fields with per-4x4-block steps of up to alpha (a quarter of that in half the blocks), flat macroblocks (strong
    filter) and macroblocks near 0 and 255 (clipping)"""
    import b2enc
    pitch, rows, pitchc, rowsc = b2enc.padded_layout(w, h)
    amp = max(alpha, 8)
    planes = []
    for (pw, ph, pp, pr, pad, mb) in ((w, h, pitch, rows, PAD, 16), (w // 2, h // 2, pitchc, rowsc, PADC, 8), (w // 2, h // 2, pitchc, rowsc, PADC, 8)):
        out = rng.integers(0, 256, (n, pr, pp), dtype=np.uint8)
        for f in range(n):
            phase = rng.random(2) * 6.3
            field = ((128 + 50 * np.sin(np.arange(pw) / 23 + phase[0]))[None, :] + (40 * np.cos(np.arange(ph) / 31 + phase[1]))[:, None])
            field = field.astype(np.int16) + rng.integers(-1, 2, (ph, pw), dtype=np.int16)
            # per macroblock: the field (55 %), flat (25 %), near 0 (10 %), near 255 (10 %)
            mode = rng.choice(4, (ph // mb, pw // mb), p=[0.55, 0.25, 0.1, 0.1])
            level = np.select([mode == 1, mode == 2, mode == 3], [rng.integers(90, 170, mode.shape), 3, 252], -1)
            level = level.astype(np.int16).repeat(mb, 0).repeat(mb, 1)
            pic = np.where(level >= 0, level, field)
            step = rng.integers(-amp, amp + 1, (ph // 4, pw // 4), dtype=np.int16)
            step = np.where(rng.random(step.shape) < 0.5, step // 4, step)
            pic = (pic.reshape(ph // 4, 4, pw // 4, 4) + step[:, None, :, None]).reshape(ph, pw)
            out[f, pad:pad + ph, pad:pad + pw] = np.clip(pic, 0, 255)
        planes.append(out)
    return planes


def bs_histogram(info, mbw, mbh):
    """boundary strengths (8.7.2.1) of all luma edge segments the filter visits: counts [internal edges | MB edges][bS 0..4]"""
    info = info.reshape(-1, mbh, mbw)
    typ, t8, nnz = info["mb_type"].astype(int), info["transform8x8"] != 0, info["nnz_mask"].astype(np.int64)
    mvq = np.concatenate([np.stack([info["mvx"], info["mvy"]], -1)[..., None, :], info["mv8"]], -2).astype(np.int64)
    mvq[..., 1:, :] = np.where((info["part"] == 0)[..., None, None], mvq[..., :1, :], mvq[..., 1:, :])

    def coded(sl, bx, by):
        z = (bx & 1) | ((by & 1) << 1) | ((bx >> 1) << 2) | ((by >> 1) << 3)
        return np.where(t8[sl], ((nnz[sl] >> (4 * ((bx >> 1) | ((by >> 1) << 1)))) & 15) != 0, ((nnz[sl] >> z) & 1) != 0)

    hist = np.zeros((2, 5), int)
    full = np.s_[:, :, :]
    for d in (0, 1):
        for e in range(4):
            if e == 0:
                qs, ps = (np.s_[:, :, 1:], np.s_[:, :, :-1]) if d == 0 else (np.s_[:, 1:, :], np.s_[:, :-1, :])
            else:
                qs = ps = full
            for k in range(4):
                pbx, pby = ((3 if e == 0 else e - 1), k) if d == 0 else (k, (3 if e == 0 else e - 1))
                qbx, qby = (e, k) if d == 0 else (k, e)
                intra = (typ[ps] != 0) | (typ[qs] != 0)
                a = mvq[ps][..., (pbx >> 1) | ((pby >> 1) << 1), :]
                b = mvq[qs][..., (qbx >> 1) | ((qby >> 1) << 1), :]
                bs = np.where(intra, 4 if e == 0 else 3,
                              np.where(coded(ps, pbx, pby) | coded(qs, qbx, qby), 2, (np.abs(a - b) >= 4).any(-1).astype(int)))
                if e & 1:
                    bs = bs[~t8[qs]]
                hist[int(e == 0)] += np.bincount(bs.ravel(), minlength=5)
    return hist


def _first_diff(got, want, pad, pw, ph, what):
    """where two stacks of padded planes of pictures pw x ph differ, in picture coordinates (or 'border')"""
    f, r, c = (int(i) for i in np.argwhere(got != want)[0])
    y, x = r - pad, c - pad
    inside = 0 <= y < ph and 0 <= x < pw
    return "%s frame %d (%s) sample (x=%d, y=%d): K8 %d, oracle %d; %d samples differ" % (
        what, f, "picture" if inside else "border", x, y, got[f, r, c], want[f, r, c], int((got != want).sum()))


def check_case(oracle, b2, w, h, n, qp, a, b, seed, expect, single_frames=False):
    """K8 on n frames in one launch == oracle frame by frame; the border is left alone; the launch has the shape `expect`.
    single_frames: also run every frame in a launch of its own (row pipeline), which must give the same pictures."""
    rng = np.random.default_rng(seed)
    mbw, mbh = w // 16, h // 16
    alpha, beta = ALPHA[clip_index(qp, a)], BETA[clip_index(qp, b)]
    y, u, v = make_planes(rng, w, h, n, alpha)
    info = make_info(rng, n, mbw, mbh)
    gy, gu, gv, shape = b2.deblock(y, u, v, info, qp, a, b)
    assert shape == expect, "%dx%d x%d: launch shape %s, expected %s" % (w, h, n, shape, expect)
    oy, ou, ov = y.copy(), u.copy(), v.copy()
    for f in range(n):
        oracle.deblock_frame(oy[f], ou[f], ov[f], info[f], qp, a, b)
    for got, want, pad, s, what in ((gy, oy, PAD, 1, "Y"), (gu, ou, PADC, 2, "U"), (gv, ov, PADC, 2, "V")):
        assert np.array_equal(got, want), _first_diff(got, want, pad, w // s, h // s, what)
    if single_frames:
        for f in range(n):
            sy, su, sv, sshape = b2.deblock(y[f:f + 1], u[f:f + 1], v[f:f + 1], info[f:f + 1], qp, a, b)
            assert sshape[0] == 0
            assert np.array_equal(sy, gy[f:f + 1]) and np.array_equal(su, gu[f:f + 1]) and np.array_equal(sv, gv[f:f + 1]), \
                "frame %d alone (row pipeline) != frame %d of the %d-frame launch" % (f, f, n)
    # the generator reaches what the case claims: the filters fire in luma and chroma (with alpha or beta 0: nothing at all),
    # and where there are enough macroblocks, every boundary strength occurs at internal and at macroblock edges
    changed = float((oy[:, PAD:PAD + h, PAD:PAD + w] != y[:, PAD:PAD + h, PAD:PAD + w]).mean())
    changed_c = float((ou[:, PADC:PADC + h // 2, PADC:PADC + w // 2] != u[:, PADC:PADC + h // 2, PADC:PADC + w // 2]).mean())
    if alpha == 0 or beta == 0:
        assert changed == 0.0 and changed_c == 0.0
    elif n * mbw * mbh >= 64:
        assert changed > 0.2 and changed_c > 0.005, "only %.3f / %.3f of the luma / U samples filtered" % (changed, changed_c)
    if n * mbw * mbh >= 200 and mbw > 1 and mbh > 1:
        hist = bs_histogram(info, mbw, mbh)
        assert (hist[0, :4] > 0).all() and (hist[1, [0, 1, 2, 4]] > 0).all(), hist


def rows_shape(mbh):
    ncta = min(16, -(-mbh // 8))
    return (0, ncta, -(-mbh // (8 * ncta)))


# row pipeline: macroblock rows around the CTA boundaries (8, 9), the portable cluster limit (64, 65), 15 and 16 CTAs (120, 128),
# two and three rounds per warp (129, 135, 257, 270); widths around the 8-entry ring of bottom rows (K8_RING); 1-3 frames
ROW_GRID = [(16 * mbw, 16 * mbh, 1 + i % 3, QPS[i % len(QPS)], rows_shape(mbh))
            for i, (mbh, mbw) in enumerate((mbh, mbw) for mbh in (1, 8, 9, 64, 65, 120, 128, 129, 135, 257, 270) for mbw in (1, 7, 8, 9))]
# the sizes users run: 2160p (16 CTAs, 2 rounds), 4320p (3 rounds), portrait 1080x1920 (15 CTAs), 1080p (9 CTAs)
ROW_SIZES = [(3840, 2160, 1, (30, -1, -1), (0, 16, 2)), (3840, 2160, 3, (26, 0, 0), (0, 16, 2)), (7680, 4320, 1, (32, -1, -1), (0, 16, 3)),
             (1088, 1920, 2, (30, -1, -1), (0, 15, 1)), (1920, 1088, 3, (36, 2, 0), (0, 9, 1))]
# wavefront: longest diagonal 1 (a single row, a single column), 16, 17, 32, 33, 64, 65, 129 -> 1 / 1 / 2 / 2 / 4 / 4 / 8 / 8 CTAs,
# two macroblocks per warp and diagonal at 129; 1080p (4 CTAs: bench.py --deblock 1), 2160p (8), 4320p (8 CTAs, 2 rounds)
WAVE_CASES = [(4096, 16, 4, (1, 1, 1)), (16, 2048, 5, (1, 1, 1)), (512, 256, 8, (1, 1, 1)), (544, 272, 4, (1, 2, 1)),
              (1024, 512, 5, (1, 2, 1)), (1056, 528, 8, (1, 4, 1)), (2048, 1024, 4, (1, 4, 1)), (2080, 1040, 5, (1, 8, 1)),
              (4128, 2064, 8, (1, 8, 2)), (1920, 1088, 8, (1, 4, 1)), (3840, 2160, 4, (1, 8, 1)), (7680, 4320, 4, (1, 8, 2))]


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,n,q,expect", [pytest.param(*c, id="%dx%d-n%d" % c[:3]) for c in ROW_GRID + ROW_SIZES])
def test_deblock_rows_matches_oracle(oracle, b2, w, h, n, q, expect):
    check_case(oracle, b2, w, h, n, *q, seed=w * 7 + h * 3 + n, expect=expect)


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,n,expect", [pytest.param(*c, id="%dx%d-n%d" % c[:3]) for c in WAVE_CASES])
def test_deblock_wavefront_matches_oracle(oracle, b2, w, h, n, expect):
    """also every frame in a launch of its own (row pipeline): the two schedules agree directly"""
    qp, a, b = QPS[(w // 16 + h // 16) % len(QPS)] if w * h < 1920 * 1080 else (28, 0, 0)
    check_case(oracle, b2, w, h, n, qp, a, b, seed=w * 5 + h * 11 + n, expect=expect, single_frames=True)


@pytest.mark.gpu
@pytest.mark.parametrize("qp,a,b", [(51, 6, 6), (10, -6, -6), (10, 6, 6), (26, -6, 6), (40, 6, -6)])
@pytest.mark.parametrize("n,expect", [(1, (0, 5, 1)), (4, (1, 2, 1))])
def test_deblock_qp_and_offset_ends(oracle, b2, qp, a, b, n, expect):
    """both schedules at the ends of indexA / indexB: clipped to 51, clipped to 0 (nothing filtered), opposite offsets"""
    check_case(oracle, b2, 704, 576, n, qp, a, b, seed=3000 + qp + 7 * a + n, expect=expect)


def test_deblock_matrix_reaches_every_boundary_strength():
    """CPU: the decision generator gives every bS class at internal and at macroblock edges even on a small picture"""
    hist = bs_histogram(make_info(np.random.default_rng(5), 1, 22, 18), 22, 18)
    assert (hist[0, :4] > 0).all() and hist[0, 4] == 0 and (hist[1, [0, 1, 2, 4]] > 0).all() and hist[1, 3] == 0, hist


# ---- the engine at the sizes users run: oracle-exact on one slot, libavcodec-exact on every slot --------------------------------
def _cut_frames(oracle, w, h):
    """synthetic frames with a scene cut at t = 2 (inverted picture): intra macroblocks inside a P frame"""
    def fn(t, s):
        f = oracle.synth_frame(w, h, t, s)
        return f if t < 2 else tuple(255 - p for p in f)
    return fn


def _engine_case(oracle, b2, w, h, nslots, expect, offsets=(0, 0), t8=0, partitions=0, frame_fn=None):
    w16, h16 = (w + 15) & ~15, (h + 15) & ~15
    assert b2.deblock_shape(w16, h16, nslots) == expect
    _encode_and_check(oracle, b2, w, h, 16, 30, nslots=nslots, nframes=3, oracle_slots=[0], deblock=1, t8=t8, partitions=partitions,
                      frame_fn=frame_fn or _cut_frames(oracle, w, h), deblock_offsets=offsets, streams=1,
                      expect_groups=[(0, nslots)])


@pytest.mark.gpu
def test_engine_2160p_one_slot_rows_16_ctas(oracle, b2):
    """the drop-in's shape at 4K with x264's default loop filter and tune film: 16-CTA row pipeline, two rounds per warp"""
    _engine_case(oracle, b2, 3840, 2160, 1, (0, 16, 2), offsets=(-1, -1))


@pytest.mark.gpu
def test_engine_2160p_four_slots_wavefront(oracle, b2):
    _engine_case(oracle, b2, 3840, 2160, 4, (1, 8, 1))


@pytest.mark.gpu
def test_engine_1080p_eight_slots_wavefront(oracle, b2):
    """bench.py --deblock 1: 8 frames per stream group at 1080p, a 4-CTA wavefront; with the 8x8 transform and partitions"""
    from test_oracle_decode import shear_seq
    w, h = 1920, 1080
    seq = shear_seq(w, h, 3, seed=51, stripe=72, band=56)
    cut = _cut_frames(oracle, w, h)
    _engine_case(oracle, b2, w, h, 8, (1, 4, 1), t8=1, partitions=1, frame_fn=lambda t, s: seq[t] if s == 0 else cut(t, s))


@pytest.mark.gpu
def test_engine_portrait_1080x1920_rows_15_ctas(oracle, b2):
    _engine_case(oracle, b2, 1080, 1920, 1, (0, 15, 1), offsets=(-1, -1))
