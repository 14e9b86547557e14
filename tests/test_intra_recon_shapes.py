"""K7, the reconstruction of intra macroblocks on reconstructed neighbours, at every launch shape of its two schedules: on its own
(b2k_intra_recon) against the oracle (b2o_recon_intra_frame, which runs b2o_recon_intra_mb in raster order), and inside the engine.

The launch shape depends on the picture size and on the frame type (b2_intra_recon_shape):
- I frames: one cluster of 1, 2, 4 or 8 CTAs of 16 warps per frame, sized from the longest anti-diagonal
  maxdiag = min(mbh, ceil(mbw / 2)); a cluster barrier between diagonals; every macroblock is two tasks (luma, chroma), and a warp
  takes ceil(2 * maxdiag / (16 * ncta)) of them per diagonal (2 at 2160p, 4 at 4320p).
- P frames: one CTA of 16 warps per frame walking the ballot-compacted list of the diagonals that hold intra macroblocks,
  ceil(maxdiag / 8) tasks per warp (15 at 2160p).
Every case asserts the (CTAs, rounds) it reaches, so that a retuned threshold cannot leave a case testing nothing new.

The decisions are random but obey the engine's contract: every mode is legal for the neighbours its block has (K7 does not
check), intra records are zero apart from mb_type, the modes and cost (nnz_mask == 0: K7 ORs its masks in), while inter records,
every level (the engine never clears coef) and the padding and inter pixels of the reconstruction hold random bytes.  K7 must
rewrite all 26 x 16 levels of an intra macroblock and nothing outside it.

Mode rules (H.264 8.3; what b2o_intra_analyse and K3 obey):
- I4x4 / I8x8: b2o_i4_mode_ok on the block's availability (b2o_blk_avail / b2o_blk8_avail): V, DDL, VL need the top, H and HU
  the left, DDR, VR and HD left, top and top-left; DC always.  A missing top-right is replaced by the last top sample.
- I16x16: b2o_i16_mode_ok on the macroblock's availability; chroma: DC always, H needs the left, V the top, plane left, top and
  top-left (the same as I16x16 with the chroma numbering)."""
import functools

import numpy as np
import pytest
from b2oracle import MBCOEF, MBINFO, PAD, PADC

I16, I4, I8 = 1, 2, 3
IC_DC, IC_H, IC_V, IC_PLANE = 0, 1, 2, 3
I16_OF_CHROMA = {IC_DC: 2, IC_H: 1, IC_V: 0, IC_PLANE: 3}        # B2_IC_* -> the B2_I16_* mode with the same neighbour needs


@functools.lru_cache(None)
def rules():
    """legality and availability tables from the oracle: blk4 [mba][b], blk8 [mba][q], ok4 [avail][mode], ok16 / okc [mba][mode]"""
    import b2oracle
    L = b2oracle.lib()
    blk4 = np.array([[L.b2o_blk_avail(b, a) for b in range(16)] for a in range(16)])
    blk8 = np.array([[L.b2o_blk8_avail(q, a) for q in range(4)] for a in range(16)])
    ok4 = np.array([[L.b2o_i4_mode_ok(m, a) != 0 for m in range(9)] for a in range(16)])
    ok16 = np.array([[L.b2o_i16_mode_ok(m, a) != 0 for m in range(4)] for a in range(16)])
    okc = np.array([[chroma_mode_ok(m, a) for m in range(4)] for a in range(16)])
    return blk4, blk8, ok4, ok16, okc


def chroma_mode_ok(mode, avail):
    return mode == IC_DC or (mode == IC_H and avail & 1 != 0) or (mode == IC_V and avail & 2 != 0) or (mode == IC_PLANE and avail & 7 == 7)


def mb_avail(mbw, mbh):
    """b2o_mb_avail of every macroblock, [mbh, mbw]: L 1, T 2, TL 4, TR 8"""
    x, y = np.arange(mbw)[None, :], np.arange(mbh)[:, None]
    return ((x > 0) * 1 + (y > 0) * 2 + ((x > 0) & (y > 0)) * 4 + ((y > 0) & (x < mbw - 1)) * 8).astype(np.int64)


def _pick(rng, legal):
    """a uniformly random legal mode along the last axis of the boolean array `legal`"""
    key = rng.random(legal.shape)
    return np.argmax(np.where(legal, key, -1.0), -1)


def make_decisions(rng, n, mbw, mbh, intra):
    """info / coef for n frames; intra [n, mbs] bool marks the intra macroblocks (each I16x16, I4x4 or I8x8 with equal odds)"""
    blk4, blk8, ok4, ok16, okc = rules()
    nmb = mbw * mbh
    mba = np.broadcast_to(mb_avail(mbw, mbh).reshape(nmb), (n, nmb))
    info = rng.integers(0, 256, (n, nmb, MBINFO.itemsize), dtype=np.uint8).view(MBINFO)[..., 0]      # inter records: garbage
    rec = np.zeros((n, nmb), MBINFO)                                                                  # intra records: as K5 leaves them
    rec["mb_type"] = rng.integers(I16, I8 + 1, (n, nmb))
    rec["mb_type"][:, 0] = I16 + (np.arange(n) + rng.integers(3)) % 3     # the only blocks without neighbours: each type in 3 frames
    rec["i16_mode"] = _pick(rng, ok16[mba])
    rec["chroma_mode"] = _pick(rng, okc[mba])
    rec["i4_mode"] = _pick(rng, ok4[blk4[mba]])
    m8 = _pick(rng, ok4[blk8[mba]])
    rec["i8_modes"] = (m8 << (4 * np.arange(4))).sum(-1)
    rec["cost"] = rng.integers(0, 1 << 32, (n, nmb), dtype=np.uint64)
    info = np.where(intra, rec, info)
    info["mb_type"] = np.where(intra, info["mb_type"], 0)
    coef = rng.integers(-32768, 32768, (n, nmb, 26 * 16), dtype=np.int16).view(MBCOEF)[..., 0]       # never cleared by the engine
    return info, coef


def make_planes(rng, w, h, n):
    """(cur, rec) padded planes for n frames.  cur: per macroblock noise over the whole range (large levels, DC included), a
    smooth field, a flat area or noise near 0 or 255 (clipping); rec: random bytes everywhere -- the padding and the inter
    macroblocks, which K7 reads as neighbours and must leave alone"""
    import b2enc
    pitch, rows, pitchc, rowsc = b2enc.padded_layout(w, h)
    mbw, mbh = w // 16, h // 16
    cur, rec = [], []
    for pw, ph, pp, pr, pad, mb in ((w, h, pitch, rows, PAD, 16), (w // 2, h // 2, pitchc, rowsc, PADC, 8),
                                    (w // 2, h // 2, pitchc, rowsc, PADC, 8)):
        c = rng.integers(0, 256, (n, pr, pp), dtype=np.uint8)
        for f in range(n):
            kind = rng.choice(5, (mbh, mbw), p=[0.25, 0.35, 0.15, 0.125, 0.125]).repeat(mb, 0).repeat(mb, 1)
            level = rng.integers(40, 216, (mbh, mbw)).repeat(mb, 0).repeat(mb, 1)
            phase = rng.random(2) * 6.3
            field = ((128 + 60 * np.sin(np.arange(pw) / (9 * mb / 16) + phase[0]))[None, :]
                     + (50 * np.cos(np.arange(ph) / (13 * mb / 16) + phase[1]))[:, None])
            noise = rng.integers(0, 256, (ph, pw))
            low, high = rng.integers(0, 8, (ph, pw)), rng.integers(248, 256, (ph, pw))
            pic = np.select([kind == 0, kind == 1, kind == 2, kind == 3], [noise, field, level, low], high)
            c[f, pad:pad + ph, pad:pad + pw] = np.clip(pic, 0, 255)
        cur.append(c)
        rec.append(rng.integers(0, 256, (n, pr, pp), dtype=np.uint8))
    return tuple(cur), tuple(rec)


def oracle_recon(oracle, cur, rec, info, coef, qp):
    """the oracle's result of one launch: (rec y, u, v, info, coef), frame by frame"""
    ry, ru, rv = (p.copy() for p in rec)
    oinfo, ocoef = info.copy(), coef.copy()
    for f in range(ry.shape[0]):
        oracle.recon_intra_frame((cur[0][f], cur[1][f], cur[2][f]), (ry[f], ru[f], rv[f]), oinfo[f], ocoef[f], qp)
    return ry, ru, rv, oinfo, ocoef


def _first_diff(got, want, pad, pw, ph, what):
    f, r, c = (int(i) for i in np.argwhere(got != want)[0])
    y, x = r - pad, c - pad
    mb = 16 if pad == PAD else 8
    where = "MB (%d, %d)" % (x // mb, y // mb) if 0 <= y < ph and 0 <= x < pw else "border"
    return "%s frame %d %s sample (x=%d, y=%d): K7 %d, oracle %d; %d samples differ" % (
        what, f, where, x, y, got[f, r, c], want[f, r, c], int((got != want).sum()))


def _first_record_diff(got, want, what):
    g, o = got.view(np.uint8).reshape(got.shape + (-1,)), want.view(np.uint8).reshape(want.shape + (-1,))
    f, i = (int(k) for k in np.argwhere((g != o).any(-1))[0])
    fields = [nm for nm in got.dtype.names if not np.array_equal(got[f, i][nm], want[f, i][nm])]
    return "%s differ: frame %d MB %d (type %d), fields %s; %d records differ" % (
        what, f, i, int(want[f, i]["mb_type"]) if "mb_type" in want.dtype.names else -1, fields, int((g != o).any(-1).sum()))


def coverage(info_in, mbw, mbh):
    """what the decisions of a launch exercise: {("i4" | "i8", block availability, mode), ("i16" | "chroma", mba & 7, mode)}"""
    blk4, blk8 = rules()[:2]
    n = info_in.shape[0]
    mba = np.broadcast_to(mb_avail(mbw, mbh).reshape(-1), (n, mbw * mbh))
    t = info_in["mb_type"]
    out = set()
    for name, sel, cls, mode in (("i16", t == I16, mba & 7, info_in["i16_mode"]), ("chroma", t != 0, mba & 7, info_in["chroma_mode"])):
        out |= {(name, int(a), int(m)) for a, m in set(zip(cls[sel].tolist(), mode[sel].tolist()))}
    sel = t == I4
    a4, m4 = blk4[mba[sel]], info_in["i4_mode"][sel].astype(np.int64)
    out |= {("i4", int(a), int(m)) for a, m in set(zip(a4.ravel().tolist(), m4.ravel().tolist()))}
    sel = t == I8
    a8 = blk8[mba[sel]]
    m8 = (info_in["i8_modes"][sel].astype(np.int64)[:, None] >> (4 * np.arange(4))) & 15
    out |= {("i8", int(a), int(m)) for a, m in set(zip(a8.ravel().tolist(), m8.ravel().tolist()))}
    return out


def coverage_target(mbw, mbh):
    """every legal (kind, availability class, mode) that a picture of mbw x mbh macroblocks admits"""
    blk4, blk8, ok4, ok16, okc = rules()
    mbas = set(mb_avail(mbw, mbh).ravel().tolist())
    out = set()
    for a in mbas:
        out |= {("i16", a & 7, m) for m in range(4) if ok16[a, m]} | {("chroma", a & 7, m) for m in range(4) if okc[a, m]}
        out |= {("i4", int(b), m) for b in blk4[a] for m in range(9) if ok4[b, m]}
        out |= {("i8", int(b), m) for b in blk8[a] for m in range(9) if ok4[b, m]}
    return out


def level_and_clip_reach(info_in, ocoef, ry, ru, w, h):
    """(luma DC, chroma DC, chroma AC levels non-zero, a reconstructed intra sample at 0, one at 255) of the oracle's result"""
    intra = info_in["mb_type"] != 0
    blk = ocoef["blk"]
    n, mbw, mbh = intra.shape[0], w // 16, h // 16
    ymask = intra.reshape(n, mbh, mbw).repeat(16, 1).repeat(16, 2)
    pic = ry[:, PAD:PAD + h, PAD:PAD + w][ymask]
    return ((blk[info_in["mb_type"] == I16][:, 24] != 0).any(), (blk[intra][:, 25, :8] != 0).any(), (blk[intra][:, 16:24] != 0).any(),
            bool((pic == 0).any()), bool((pic == 255).any()))


def check_case(oracle, b2, w, h, intra, qp, all_intra, seed, expect):
    """K7 on the frames of one launch == the oracle frame by frame, padding, inter macroblocks, records and levels included; the
    launch has the shape `expect` = (CTAs per frame, rounds)"""
    rng = np.random.default_rng(seed)
    n, mbw, mbh = intra.shape[0], w // 16, h // 16
    info, coef = make_decisions(rng, n, mbw, mbh, intra)
    cur, rec = make_planes(rng, w, h, n)
    gy, gu, gv, ginfo, gcoef, shape = b2.intra_recon(cur, rec, info, coef, qp, all_intra)
    assert shape[:2] == expect, "%dx%d all_intra=%d: launch shape %s, expected %s" % (w, h, all_intra, shape[:2], expect)
    oy, ou, ov, oinfo, ocoef = oracle_recon(oracle, cur, rec, info, coef, qp)
    for got, want, pad, s, what in ((gy, oy, PAD, 1, "Y"), (gu, ou, PADC, 2, "U"), (gv, ov, PADC, 2, "V")):
        assert np.array_equal(got, want), _first_diff(got, want, pad, w // s, h // s, what)
    inter = ~intra
    assert np.array_equal(ginfo[inter].view(np.uint8), info[inter].view(np.uint8)), "K7 changed an inter record"
    assert np.array_equal(gcoef[inter].view(np.uint8), coef[inter].view(np.uint8)), "K7 changed the levels of an inter macroblock"
    assert np.array_equal(ginfo.view(np.uint8), oinfo.view(np.uint8)), _first_record_diff(ginfo, oinfo, "records")
    assert np.array_equal(gcoef.view(np.uint8), ocoef.view(np.uint8)), _first_record_diff(gcoef, ocoef, "levels")
    if intra.sum() >= 1000:                                    # a case of that size reaches every kind of level and both clips
        assert all(level_and_clip_reach(info, ocoef, oy, ou, w, h))
    return (gy, gu, gv, ginfo, gcoef), (cur, rec, info, coef)


def i_shape(w, h):
    maxdiag = min(h // 16, (w // 16 + 1) // 2)
    ncta = 1
    while ncta < 8 and 16 * ncta < 2 * maxdiag:
        ncta *= 2
    return ncta, -(-2 * maxdiag // (16 * ncta))


def p_shape(w, h):
    return 1, -(-min(h // 16, (w // 16 + 1) // 2) // 8)


# ---- I schedule: (w, h, frames per launch, qp, (CTAs, rounds)) -----------------------------------------------------------------------
# single macroblock, single row, single column; longest diagonal 8 / 9 / 16 / 17 / 32 / 33 / 64 / 65 / 129 (1 / 2 / 2 / 4 / 4 / 8 /
# 8 / 8 CTAs, 2 and 3 rounds beyond 64 macroblocks per diagonal), landscape and portrait 1080p, 2160p, 4320p and the tallest
# diagonal table within level 6.2
I_CASES = [(16, 16, 3, 26, (1, 1)), (4096, 16, 2, 10, (1, 1)), (16, 4096, 2, 51, (1, 1)), (256, 128, 3, 30, (1, 1)),
           (288, 144, 2, 22, (2, 1)), (512, 256, 3, 40, (2, 1)), (544, 272, 2, 14, (4, 1)), (1024, 512, 1, 34, (4, 1)),
           (1056, 528, 2, 46, (8, 1)), (2048, 1024, 1, 18, (8, 1)), (2080, 1040, 1, 28, (8, 2)), (4128, 2064, 1, 36, (8, 3)),
           (1920, 1088, 2, 51, (8, 1)), (1088, 1920, 1, 10, (8, 1)), (3840, 2160, 1, 26, (8, 2)), (7680, 4320, 1, 32, (8, 4)),
           (2112, 16880, 1, 24, (8, 2))]
# ---- P schedule: (w, h, intra pattern per frame, qp) -------------------------------------------------------------------------------
# ndiag 31, 32, 33, 64, 65 (ballot boundaries of the diagonal list); the sizes of the I grid with 2 % scattered intra, only the
# first and last diagonals, a single intra macroblock in the bottom-right corner, all intra; one launch of none | sparse | all
P_CASES = [(496, 16, ("sparse30",), 26), (512, 16, ("sparse30",), 51), (528, 16, ("ends",), 10), (1024, 16, ("sparse30", "corner"), 33),
           (1040, 16, ("sparse30",), 20), (16, 4096, ("sparse2",), 44), (256, 128, ("all",), 12), (288, 144, ("ends", "all"), 38),
           (1056, 528, ("sparse2",), 26), (2048, 1024, ("corner", "all"), 30), (1920, 1088, ("none", "sparse2", "all"), 28),
           (3840, 2160, ("all",), 26), (3840, 2160, ("sparse2", "ends"), 51), (7680, 4320, ("all",), 32), (2112, 16880, ("sparse2",), 22)]


def intra_pattern(rng, kind, mbw, mbh):
    d = (np.arange(mbw)[None, :] + 2 * np.arange(mbh)[:, None]).ravel()
    ndiag = mbw + 2 * (mbh - 1)
    if kind == "all":
        return np.ones(mbw * mbh, bool)
    if kind == "none":
        return np.zeros(mbw * mbh, bool)
    if kind == "ends":
        return (d == 0) | (d == ndiag - 1)
    if kind == "corner":
        return d == ndiag - 1
    m = rng.random(mbw * mbh) < {"sparse2": 0.02, "sparse30": 0.3}[kind]
    m[-1] = True                                             # the last diagonal always holds one
    return m


def i_launch(w, h, n):
    return np.ones((n, (w // 16) * (h // 16)), bool)


def p_launch(w, h, kinds, seed):
    rng = np.random.default_rng(seed)
    return np.stack([intra_pattern(rng, k, w // 16, h // 16) for k in kinds])


def _id(c):
    return "%dx%d-%s" % (c[0], c[1], c[2] if isinstance(c[2], int) else "-".join(c[2]))


def test_shape_table():
    """CPU: the launch shapes the cases name are the ones b2_intra_recon_shape picks; the diagonal table is 8 bytes a diagonal"""
    import b2enc
    for w, h, n, qp, expect in I_CASES:
        ncta, rounds, dyn = b2enc.intra_recon_shape(w, h, 1)
        assert (ncta, rounds) == expect == i_shape(w, h), (w, h)
        assert dyn == 8 * (w // 16 + 2 * (h // 16 - 1))
    for w, h, kinds, qp in P_CASES:
        assert b2enc.intra_recon_shape(w, h, 0)[:2] == p_shape(w, h)
    assert {1, 2, 8, 15, 30} <= {p_shape(w, h)[1] for w, h, kinds, qp in P_CASES}
    assert b2enc.intra_recon_shape(2112, 16880, 1)[2] == 8 * 2240


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,n,qp,expect", [pytest.param(*c, id=_id(c)) for c in I_CASES])
def test_intra_recon_i_schedule(oracle, b2, w, h, n, qp, expect):
    """also every frame again through the P schedule (one CTA): the two schedules agree"""
    (gy, gu, gv, ginfo, gcoef), (cur, rec, info, coef) = check_case(oracle, b2, w, h, i_launch(w, h, n), qp, 1, seed=w * 7 + h * 3 + n,
                                                                    expect=expect)
    for f in range(n):
        sl = slice(f, f + 1)
        py, pu, pv, pinfo, pcoef, shape = b2.intra_recon(tuple(p[sl] for p in cur), tuple(p[sl] for p in rec), info[sl], coef[sl], qp, 0)
        assert shape[:2] == p_shape(w, h)
        assert np.array_equal(py, gy[sl]) and np.array_equal(pu, gu[sl]) and np.array_equal(pv, gv[sl]), \
            "frame %d through the P schedule != the I schedule" % f
        assert np.array_equal(pinfo.view(np.uint8), ginfo[sl].view(np.uint8)) and np.array_equal(pcoef.view(np.uint8), gcoef[sl].view(np.uint8))


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,kinds,qp", [pytest.param(*c, id=_id(c)) for c in P_CASES])
def test_intra_recon_p_schedule(oracle, b2, w, h, kinds, qp):
    seed = w * 5 + h * 11 + len(kinds)
    check_case(oracle, b2, w, h, p_launch(w, h, kinds, seed), qp, 0, seed=seed, expect=p_shape(w, h))


@pytest.mark.gpu
def test_intra_recon_i_schedule_16_frames_1080p(oracle, b2):
    """16 clusters of 8 CTAs in one launch: more than the GPU holds at once"""
    check_case(oracle, b2, 1920, 1088, i_launch(1920, 1088, 16), 30, 1, seed=1616, expect=(8, 1))


@pytest.mark.gpu
def test_intra_recon_refuses_diagonal_table_beyond_shared_memory(oracle, b2):
    """the last picture height whose diagonal table fits (ndiag 3134) is reconstructed; one macroblock row more is refused"""
    w = 32
    for h, ok in ((16 * 1567, True), (16 * 1568, False)):
        assert b2.intra_recon_shape(w, h, 1)[2] == 8 * (w // 16 + 2 * (h // 16 - 1))
        if ok:
            check_case(oracle, b2, w, h, i_launch(w, h, 1), 26, 1, seed=h, expect=(1, 1))
        else:
            rng = np.random.default_rng(h)
            info, coef = make_decisions(rng, 1, w // 16, h // 16, i_launch(w, h, 1))
            cur, rec = make_planes(rng, w, h, 1)
            with pytest.raises(RuntimeError):
                b2.intra_recon(cur, rec, info, coef, 26, 1)


# ---- the generator reaches what the cases claim (CPU) -------------------------------------------------------------------------------
def test_generator_alone_reaches_every_mode_level_and_clip(oracle):
    """on one small picture: every legal I4 / I8 mode at every block availability (top-right missing included), every legal
    I16 / chroma mode at the top row, the left column and the interior, non-zero luma DC, chroma DC and chroma AC levels, and
    reconstructed samples at 0 and 255 -- at the lowest and the highest QP"""
    w, h, n = 352, 288, 3
    for qp in (10, 51):
        rng = np.random.default_rng(qp)
        intra = i_launch(w, h, n)
        info, coef = make_decisions(rng, n, w // 16, h // 16, intra)
        cur, rec = make_planes(rng, w, h, n)
        target = coverage_target(w // 16, h // 16)
        assert coverage(info, w // 16, h // 16) == target
        assert {("i4", 7, m) for m in range(9)} <= target and {("i8", 7, m) for m in range(9)} <= target   # top-right missing
        oy, ou, ov, oinfo, ocoef = oracle_recon(oracle, cur, rec, info, coef, qp)
        assert all(level_and_clip_reach(info, ocoef, oy, ou, w, h))


def test_cases_together_reach_every_mode_at_every_availability():
    """the decisions of the GPU cases (regenerated here) cover every legal mode of every kind at every availability class"""
    reached, target = set(), set()
    for w, h, n, qp, expect in I_CASES:
        rng = np.random.default_rng(w * 7 + h * 3 + n)
        info, _ = make_decisions(rng, n, w // 16, h // 16, i_launch(w, h, n))
        reached |= coverage(info, w // 16, h // 16)
        target |= coverage_target(w // 16, h // 16)
    assert reached == target, sorted(target - reached)


def test_mode_rules():
    """the generator's rules: chroma as I16x16 with the chroma numbering; I8x8 with the I4x4 rule on b2o_blk8_avail; a missing
    top-right never restricts a mode (it is substituted)"""
    blk4, blk8, ok4, ok16, okc = rules()
    for a in range(16):
        for m in range(4):
            assert okc[a, m] == ok16[a, I16_OF_CHROMA[m]]
        for m in range(9):
            assert ok4[a, m] == ok4[a & 7, m]
    # top-right of the blocks on the MB's top edge comes from the MB to the top-right: missing in the right column (mba 7)
    assert blk8[15][1] == 15 and blk8[7][1] == 7 and blk8[15][3] == 7
    assert blk4[15][5] == 15 and blk4[7][5] == 7


# ---- the oracle against libavcodec (CPU): random legal modes of every kind, not only the ones the analysis picks -----------------
@pytest.mark.parametrize("qp,cabac", [(10, 0), (28, 1), (51, 0), (36, 1)])
def test_oracle_recon_decodes_exactly(oracle, qp, cabac):
    w, h = 352, 288
    rng = np.random.default_rng(400 + qp)
    intra = i_launch(w, h, 1)
    info, coef = make_decisions(rng, 1, w // 16, h // 16, intra)
    cur, rec = make_planes(rng, w, h, 1)
    oy, ou, ov, oinfo, ocoef = oracle_recon(oracle, cur, rec, info, coef, qp)
    assert set(oinfo["mb_type"].ravel().tolist()) == {I16, I4, I8}
    ent = oracle.Entropy(w, h, qp, cabac=cabac, transform8x8=1)
    sc = b"\x00\x00\x00\x01"
    au = sc + ent.sps() + sc + ent.pps() + sc + ent.slice(0, 0, 0, oinfo[0], ocoef[0])
    (dy, du, dv), = oracle.decode_yuv([au])
    assert np.array_equal(dy, oy[0, PAD:PAD + h, PAD:PAD + w])
    assert np.array_equal(du, ou[0, PADC:PADC + h // 2, PADC:PADC + w // 2]) and np.array_equal(dv, ov[0, PADC:PADC + h // 2, PADC:PADC + w // 2])


# ---- the engine: oracle-exact on slot 0, decoder-exact on every slot; scene cut at t = 2 for a dense P frame -------------------------
def _engine_case(oracle, b2, w, h, expect_i):
    from test_deblock_shapes import _cut_frames
    from test_full_size import _encode_and_check
    assert b2.intra_recon_shape((w + 15) & ~15, (h + 15) & ~15, 1)[:2] == expect_i
    infos = []
    _encode_and_check(oracle, b2, w, h, 16, 30, nslots=1, nframes=3, oracle_slots=[0], t8=1, frame_fn=_cut_frames(oracle, w, h),
                      infos=infos)
    types = {t: np.bincount(info["mb_type"].ravel(), minlength=4) for t, s, info in infos}
    assert (types[0][1:] > 0).all(), types[0]                  # the I frame holds all three intra types, I8x8 included
    assert types[2][1:].sum() > types[2].sum() // 2, types[2]  # after the cut the P frame is mostly intra


@pytest.mark.gpu
def test_engine_2160p_intra8x8_two_rounds(oracle, b2):
    _engine_case(oracle, b2, 3840, 2160, (8, 2))


@pytest.mark.gpu
def test_engine_portrait_1080x1920_intra8x8(oracle, b2):
    _engine_case(oracle, b2, 1080, 1920, (8, 1))
