"""Several slices per picture (x264 i_slice_count): the row split, slice-aware neighbour availability in the oracle, the host slice
writers, K3 / K7 and the drop-in encoder.

The slice-aware reference is the oracle run slice by slice (tests/slice_ref.py, tests/mock/slices_ref.c).

Definition (include/b2enc_types.h): n = min(max(i_slice_count, 1), mbh) row-aligned slices; slice k covers macroblock rows
[(k mbh + n/2) / n, ((k+1) mbh + n/2) / n).  The left neighbour is always in the same slice; the top, top-left and top-right
neighbours are unavailable exactly on the first row of a slice.  The loop filter runs across slice boundaries
(disable_deblocking_filter_idc 0).

The decoder pin (libavcodec decodes every oracle stream to the oracle's reconstruction, slices parsed from the NALs) is what fixes
availability and context selection normatively; the kernel and engine cases then hold the GPU to the oracle bit for bit."""
import os

import numpy as np
import pytest
from b2oracle import MBCOEF, MBINFO, PAD, PADC
import slice_ref as ref
from test_host_pipeline import annexb, b2mod, drive  # noqa: F401  (fixture)
from test_intra_recon_shapes import I16, I8, _first_diff, _first_record_diff, _pick, make_planes, rules
from test_oracle_decode import smooth_seq

SC = b"\x00\x00\x00\x01"


# ---- helpers -------------------------------------------------------------------------------------------------------------------
def row0_of_rows(oracle, mbh, slices):
    """first row of the slice of every macroblock row, [mbh]"""
    first = ref.slice_rows(mbh, slices)
    out = np.zeros(mbh, np.int64)
    for r0, r1 in zip(first[:-1], first[1:]):
        out[r0:r1] = r0
    return out


def slice_mb_avail(oracle, mbw, mbh, slices):
    """b2o_mb_avail of every macroblock with `slices` slices, [mbh, mbw]: L 1, T 2, TL 4, TR 8"""
    x = np.arange(mbw)[None, :]
    top = (np.arange(mbh) > row0_of_rows(oracle, mbh, slices))[:, None]
    return ((x > 0) * 1 + top * 2 + ((x > 0) & top) * 4 + (top & (x < mbw - 1)) * 8).astype(np.int64)


def read_ue(data, bitpos):
    """exp-Golomb ue(v) at bit `bitpos` of `data` (no emulation prevention in the first bytes of a slice header)"""
    zeros = 0
    while not (data[(bitpos + zeros) >> 3] >> (7 - ((bitpos + zeros) & 7))) & 1:
        zeros += 1
    v = 0
    for i in range(zeros + 1):
        p = bitpos + zeros + i
        v = (v << 1) | ((data[p >> 3] >> (7 - (p & 7))) & 1)
    return v - 1, bitpos + 2 * zeros + 1


def slice_starts(au):
    """first_mb_in_slice of every slice NAL of an Annex-B access unit"""
    return [read_ue(p[1:], 0)[0] for p in au.split(SC)[1:] if p[0] & 31 in (1, 5)]


def check_split_in_stream(oracle, bs, mbw, mbh, slices, nframes):
    aus = ref.split_access_units(bs)
    assert len(aus) == nframes
    want = [r * mbw for r in ref.slice_rows(mbh, slices)[:-1]]
    for t, au in enumerate(aus):
        assert slice_starts(au) == want, "picture %d: first_mb_in_slice %s, split %s" % (t, slice_starts(au), want)
    return aus


# ---- 1. the split (CPU) --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mbh,n", [(68, 8), (135, 8), (3, 2), (5, 5), (4, 9), (1, 3), (270, 17), (45, 1), (45, 0), (9, 7)])
def test_split_table(oracle, mbh, n):
    first = ref.slice_rows(mbh, n)
    ns = min(max(n, 1), mbh)
    assert len(first) == ns + 1 and first[0] == 0 and first[-1] == mbh
    assert first == [(k * mbh + ns // 2) // ns for k in range(ns + 1)]
    sizes = np.diff(first)
    assert (sizes >= 1).all() and sizes.max() - sizes.min() <= 1                 # every row in exactly one slice, balanced
    r0 = row0_of_rows(oracle, mbh, n)
    assert sorted(set(r0.tolist())) == first[:-1]


# ---- 2. the oracle's analysis (CPU) --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("w,h,slices", [(352, 288, 4), (176, 144, 9), (640, 368, 7)])
def test_oracle_analysis_sees_no_neighbour_in_another_slice(oracle, w, h, slices):
    """off the first rows of the slices the analysis is the unsliced one; on them every chosen mode is legal without the
    neighbours above; and some first-row macroblocks do choose differently (the rule is exercised)"""
    y, u, v = smooth_seq(w, h, 1, seed=w + slices)[0]
    f = oracle.OFrame(w, h).load(y, u, v)
    mbw, mbh = w // 16, h // 16
    one, c1 = ref.intra_analyse(f, 1, 28)
    sl, cs = ref.intra_analyse(f, slices, 28)
    first_row = (np.arange(mbh) == row0_of_rows(oracle, mbh, slices)).repeat(mbw)
    inner = ~first_row
    inner[:mbw] = False                                                            # row 0 is a first row either way
    for name in ("i16_mode", "chroma_mode", "i4_mode", "i8_modes"):
        assert np.array_equal(one[name][inner], sl[name][inner]), name
    for a, b in zip(c1, cs):
        assert np.array_equal(a[inner], b[inner])
    blk4, blk8, ok4, ok16, okc = rules()
    mba = slice_mb_avail(oracle, mbw, mbh, slices).ravel()
    assert (mba[first_row] & 14 == 0).all()
    assert ok16[mba, sl["i16_mode"]].all() and okc[mba, sl["chroma_mode"]].all()
    assert ok4[blk4[mba], sl["i4_mode"].astype(np.int64)].all()
    m8 = (sl["i8_modes"].astype(np.int64)[:, None] >> (4 * np.arange(4))) & 15
    assert ok4[blk8[mba], m8].all()
    moved = first_row.copy(); moved[:mbw] = False
    differ = np.zeros(mbw * mbh, bool)
    for name in ("i16_mode", "chroma_mode"):
        differ |= one[name] != sl[name]
    differ |= (one["i4_mode"] != sl["i4_mode"]).any(-1) | (one["i8_modes"] != sl["i8_modes"])
    assert differ[moved].sum() > mbw, "only %d first-row macroblocks changed their modes" % differ[moved].sum()
    assert not differ[~first_row].any()


# ---- 3. the decoder pin (CPU) --------------------------------------------------------------------------------------------------
# (w, h, slices, cabac, transform8x8, partitions, deblock offsets); slices None = one slice per macroblock row
PIN_CASES = [(64, 48, 2, 0, 0, 0, (0, 0)), (80, 64, 3, 1, 1, 1, (-1, -1)), (112, 112, 7, 1, 1, 2, (2, -3)), (100, 90, None, 0, 1, 2, (0, 0)),
             (176, 144, 7, 0, 0, 1, (1, 1)), (200, 120, 3, 1, 1, 0, (-2, 2)), (96, 80, None, 1, 0, 0, (0, 0)), (48, 144, 2, 0, 1, 1, (0, 0))]


@pytest.mark.parametrize("w,h,slices,cabac,t8,parts,offs", PIN_CASES)
def test_oracle_streams_with_slices_decode_exactly(oracle, w, h, slices, cabac, t8, parts, offs):
    """every picture: n slice NALs at the split, decoded by libavcodec to the oracle's reconstruction; a scene cut at t = 2 puts
    intra macroblocks into P frames next to slice boundaries"""
    mbw, mbh = (w + 15) // 16, (h + 15) // 16
    n = mbh if slices is None else slices
    frames = smooth_seq(w, h, 6, seed=w * 3 + h, cut=2)
    bs, recons, infos, _ = ref.encode_sequence(frames, w, h, qp=30, gop=4, deblock=1, cabac=cabac, transform8x8=t8, partitions=parts,
                                                   deblock_offsets=offs, slices=n)
    aus = check_split_in_stream(oracle, bs, mbw, mbh, n, len(frames))
    assert sum(((i["mb_type"] != 0) & (np.arange(mbw * mbh) // mbw > 0)).sum() for i in infos[2:4]) > 0   # intra in P frames
    dec = oracle.decode_yuv(aus)
    assert len(dec) == len(frames)
    for t, ((dy, du, dv), rec) in enumerate(zip(dec, recons)):
        assert np.array_equal(dy, rec.y[:h, :w]), "luma of frame %d" % t
        assert np.array_equal(du, rec.u[:(h + 1) // 2, :(w + 1) // 2]) and np.array_equal(dv, rec.v[:(h + 1) // 2, :(w + 1) // 2]), t
    one, *_ = oracle.encode_sequence(frames, w, h, qp=30, gop=4, deblock=1, cabac=cabac, transform8x8=t8, partitions=parts,
                                     deblock_offsets=offs)
    assert ref.encode_sequence(frames, w, h, qp=30, gop=4, deblock=1, cabac=cabac, transform8x8=t8, partitions=parts,
                                  deblock_offsets=offs, slices=1)[0] == one


def test_packed_writer_finds_each_slice(oracle):
    """the packed level stream of the whole picture: each slice finds its first macroblock's blocks behind the ones in front"""
    w, h = 160, 112
    frames = smooth_seq(w, h, 3, seed=8, cut=1)
    _, _, infos, coefs = ref.encode_sequence(frames, w, h, qp=24, gop=8, deblock=1, cabac=1, transform8x8=1, slices=5)
    for cabac in (0, 1):
        ent = ref.Entropy(w, h, 24, 5, deblock=1, cabac=cabac, transform8x8=1)
        for t, (info, coef) in enumerate(zip(infos, coefs)):
            packed = _pack(info, coef)
            assert ent.slice_packed(int(t > 0), t, 0, info, packed) == ent.slice(int(t > 0), t, 0, info, coef)


def _pack(info, coef):
    """the packed level stream (b2_coef_present blocks of every macroblock, in raster order)"""
    out = []
    for m, c in zip(info, coef):
        nnz, t8 = int(m["nnz_mask"]), int(m["transform8x8"])
        luma = nnz & 0xFFFF
        if t8:
            for q in range(4):
                if (luma >> (4 * q)) & 15:
                    luma |= 15 << (4 * q)
        present = luma | (nnz & 0x01FF0000) | ((1 << 25) if nnz & 0x06000000 else 0)
        out += [c["blk"][b].tobytes() for b in range(26) if present >> b & 1]
    return np.frombuffer(b"".join(out), np.uint8)


# ---- 4. the host pipeline on the mock engine (CPU) -----------------------------------------------------------------------------
@pytest.fixture(scope="module")
def mock_slices():
    return ref.mock_lib()


@pytest.mark.parametrize("slices,cabac", [(2, 1), (3, 0), (5, 1)])
def test_dropin_slices_on_mock_engine(oracle, b2mod, mock_slices, slices, cabac):
    """zero delay (one GOP slot: the slices of a picture are written concurrently by the slice pool) and GOP streaming on 1, 2
    and 3 pretend GPUs: the oracle encoder's bytes with the same slices"""
    w, h, qp, gop, n = 80, 80, 30, 3, 8
    frames = smooth_seq(w, h, n, seed=slices, cut=4)
    want, *_ = ref.encode_sequence(frames, w, h, qp=qp, merange=16, gop=gop, deblock=1, cabac=cabac, deblock_offsets=(-1, -1), slices=slices)
    prof = None if cabac else "baseline"
    out = drive(b2mod, mock_slices, frames, w, h, tune="film,zerolatency", quality=qp, profile=prof, annexb=1, i_keyint_max=gop, i_slice_count=slices)
    assert all(sum(t in (1, 5) for t, _ in nals) == slices for nals, *_ in out)
    assert annexb(out) == want
    for devices in (1, 2, 3):
        out = drive(b2mod, mock_slices, frames, w, h, devices=devices, tune="film", quality=qp, profile=prof, annexb=1, i_keyint_max=gop,
                    i_gop_slots=2, i_slice_count=slices)
        assert annexb(out) == want, devices


def test_dropin_slices_from_environment(oracle, b2mod, mock_slices):
    """an unmodified av_encode.c cannot set i_slice_count: B2ENC_SLICES does; more slices than rows are clamped to the rows"""
    w, h, qp = 48, 48, 32
    frames = smooth_seq(w, h, 4, seed=21)
    os.environ["B2ENC_SLICES"] = "7"
    try:
        out = drive(b2mod, mock_slices, frames, w, h, tune="film,zerolatency", quality=qp, annexb=1, i_keyint_max=2)
    finally:
        del os.environ["B2ENC_SLICES"]
    want, *_ = ref.encode_sequence(frames, w, h, qp=qp, gop=2, deblock=1, cabac=1, deblock_offsets=(-1, -1), slices=3)
    assert annexb(out) == want


# ---- 5. K7 alone (GPU) ---------------------------------------------------------------------------------------------------------
def make_decisions_sliced(oracle, rng, n, mbw, mbh, intra, slices):
    """test_intra_recon_shapes.make_decisions with the availability of `slices` slices"""
    blk4, blk8, ok4, ok16, okc = rules()
    nmb = mbw * mbh
    mba = np.broadcast_to(slice_mb_avail(oracle, mbw, mbh, slices).reshape(nmb), (n, nmb))
    info = rng.integers(0, 256, (n, nmb, MBINFO.itemsize), dtype=np.uint8).view(MBINFO)[..., 0]
    rec = np.zeros((n, nmb), MBINFO)
    rec["mb_type"] = rng.integers(I16, I8 + 1, (n, nmb))
    rec["i16_mode"] = _pick(rng, ok16[mba])
    rec["chroma_mode"] = _pick(rng, okc[mba])
    rec["i4_mode"] = _pick(rng, ok4[blk4[mba]])
    m8 = _pick(rng, ok4[blk8[mba]])
    rec["i8_modes"] = (m8 << (4 * np.arange(4))).sum(-1)
    rec["cost"] = rng.integers(0, 1 << 32, (n, nmb), dtype=np.uint64)
    info = np.where(intra, rec, info)
    info["mb_type"] = np.where(intra, info["mb_type"], 0)
    coef = rng.integers(-32768, 32768, (n, nmb, 26 * 16), dtype=np.int16).view(MBCOEF)[..., 0]
    return info, coef


def tallest(oracle, mbh, slices):
    return int(np.diff(ref.slice_rows(mbh, slices)).max())


def i_shape_rows(mbw, rows):
    maxdiag = min(rows, (mbw + 1) // 2)
    ncta = 1
    while ncta < 8 and 16 * ncta < 2 * maxdiag:
        ncta *= 2
    return ncta, -(-2 * maxdiag // (16 * ncta))


def check_sliced_case(oracle, b2, w, h, slices, intra, qp, all_intra, seed, expect):
    rng = np.random.default_rng(seed)
    n, mbw, mbh = intra.shape[0], w // 16, h // 16
    info, coef = make_decisions_sliced(oracle, rng, n, mbw, mbh, intra, slices)
    cur, rec = make_planes(rng, w, h, n)
    gy, gu, gv, ginfo, gcoef, shape = b2.intra_recon(cur, rec, info, coef, qp, all_intra, slices=slices)
    assert shape[:2] == expect, "%dx%d, %d slices, all_intra=%d: launch shape %s, expected %s" % (w, h, slices, all_intra, shape[:2], expect)
    assert shape[2] == 8 * (mbw + 2 * (tallest(oracle, mbh, slices) - 1))
    oy, ou, ov = (p.copy() for p in rec)
    oinfo, ocoef = info.copy(), coef.copy()
    for f in range(n):
        ref.recon_intra_frame((cur[0][f], cur[1][f], cur[2][f]), (oy[f], ou[f], ov[f]), oinfo[f], ocoef[f], qp, slices)
    for got, want, pad, s, what in ((gy, oy, PAD, 1, "Y"), (gu, ou, PADC, 2, "U"), (gv, ov, PADC, 2, "V")):
        assert np.array_equal(got, want), _first_diff(got, want, pad, w // s, h // s, what)
    assert np.array_equal(ginfo.view(np.uint8), oinfo.view(np.uint8)), _first_record_diff(ginfo, oinfo, "records")
    assert np.array_equal(gcoef.view(np.uint8), ocoef.view(np.uint8)), _first_record_diff(gcoef, ocoef, "levels")


# (w, h, frames, slices, qp, (CTAs, rounds) of the tallest slice): every I-schedule shape a sliced launch takes
I_SLICED = [(16, 64, 2, 4, 26, (1, 1)), (256, 128, 2, 8, 30, (1, 1)), (352, 288, 3, 7, 51, (1, 1)), (1920, 1088, 2, 8, 22, (2, 1)),
            (1024, 512, 1, 2, 34, (2, 1)), (3840, 2160, 1, 8, 26, (4, 1)), (2048, 1024, 1, 3, 18, (4, 1)), (1088, 1920, 1, 5, 10, (4, 1)),
            (2048, 2048, 1, 2, 40, (8, 1)), (4128, 2080, 1, 2, 28, (8, 2)), (4128, 4128, 1, 2, 36, (8, 3)), (7680, 6208, 1, 2, 32, (8, 4))]
# (w, h, slices, intra pattern per frame, qp): the P schedule, one CTA per (frame, slice)
P_SLICED = [(1920, 1088, 8, ("none", "sparse2", "all"), 28), (3840, 2160, 8, ("boundary",), 26), (352, 288, 18, ("sparse30", "boundary"), 40),
            (1024, 512, 3, ("all",), 12), (16, 4096, 7, ("sparse30",), 44), (3840, 2160, 135, ("sparse2", "all"), 33)]


def sliced_pattern(oracle, rng, kind, mbw, mbh, slices):
    rows = np.arange(mbh).repeat(mbw)
    first = np.array(ref.slice_rows(mbh, slices))
    if kind == "all":
        return np.ones(mbw * mbh, bool)
    if kind == "none":
        return np.zeros(mbw * mbh, bool)
    if kind == "boundary":                                   # first and last row of every slice
        return np.isin(rows, first[:-1]) | np.isin(rows, first[1:] - 1)
    return rng.random(mbw * mbh) < {"sparse2": 0.02, "sparse30": 0.3}[kind]


def test_sliced_shape_table(oracle):
    """CPU: the shapes the cases name are b2_intra_recon_shape's for the tallest slice; one slice is exactly the old shape"""
    import b2enc
    for w, h, n, slices, qp, expect in I_SLICED:
        rows = tallest(oracle, h // 16, slices)
        assert b2enc.intra_recon_shape(w, h, 1, slices=slices)[:2] == expect == i_shape_rows(w // 16, rows), (w, h, slices)
        assert b2enc.intra_recon_shape(w, h, 1, slices=slices) == b2enc.intra_recon_shape(w, 16 * rows, 1)
    assert {e for *_, e in I_SLICED} == {(1, 1), (2, 1), (4, 1), (8, 1), (8, 2), (8, 3), (8, 4)}
    for w, h, slices, kinds, qp in P_SLICED:
        rows = tallest(oracle, h // 16, slices)
        assert b2enc.intra_recon_shape(w, h, 0, slices=slices)[:2] == (1, -(-min(rows, (w // 16 + 1) // 2) // 8))
    for w, h in ((1920, 1088), (16, 4096), (7680, 4320)):
        for a in (0, 1):
            assert b2enc.intra_recon_shape(w, h, a, slices=1) == b2enc.intra_recon_shape(w, h, a, slices=0) == b2enc.intra_recon_shape(w, h, a)


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,n,slices,qp,expect", I_SLICED, ids=["%dx%d-%d-s%d" % c[:4] for c in I_SLICED])
def test_k7_sliced_i_schedule(oracle, b2, w, h, n, slices, qp, expect):
    check_sliced_case(oracle, b2, w, h, slices, np.ones((n, (w // 16) * (h // 16)), bool), qp, 1, w * 7 + h * 3 + slices, expect)


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,slices,kinds,qp", P_SLICED, ids=["%dx%d-s%d-%s" % (c[0], c[1], c[2], "-".join(c[3])) for c in P_SLICED])
def test_k7_sliced_p_schedule(oracle, b2, w, h, slices, kinds, qp):
    rng = np.random.default_rng(w + h + slices)
    intra = np.stack([sliced_pattern(oracle, rng, k, w // 16, h // 16, slices) for k in kinds])
    rows = tallest(oracle, h // 16, slices)
    check_sliced_case(oracle, b2, w, h, slices, intra, qp, 0, w * 5 + slices, (1, -(-min(rows, (w // 16 + 1) // 2) // 8)))


# ---- 6. the engine against the oracle (GPU) ------------------------------------------------------------------------------------
def _cut_frames(oracle, w, h):
    def fn(t, s):
        f = oracle.synth_frame(w, h, t, s)
        return f if t < 2 else tuple(255 - p for p in f)
    return fn


def engine_case(oracle, b2, w, h, slices, nslots=1, qp=30, t8=0, partitions=0, offsets=(0, 0), cabac=1, pack=0, streams=0, nframes=3):
    """the engine with `slices` slices, I and P frames (scene cut at t = 2): every record field, the levels (dense, or packed) and
    the reconstruction equal the oracle's on slot 0; every slot's stream has the slices at the split and decodes exactly"""
    eng = b2.Engine(w, h, slots=nslots, ring=1, merange=16, qp=qp, deblock=1, transform8x8=t8, partitions=partitions, pack_levels=pack,
                    deblock_offsets=offsets, streams=streams, slices=slices)
    prm = oracle.Params(qp, 16, 1, 1, 1, t8, partitions, offsets[0], offsets[1])
    ents = [ref.Entropy(w, h, qp, slices, deblock=1, cabac=cabac, transform8x8=t8, deblock_offsets=offsets) for _ in range(nslots)]
    frame_fn = _cut_frames(oracle, w, h)
    bs = [bytearray() for _ in range(nslots)]
    recons = [[] for _ in range(nslots)]
    prev = pmv = None
    for t in range(nframes):
        frames = [frame_fn(t, s) for s in range(nslots)]
        for s in range(nslots):
            eng.put_frame(s, 0, list(frames[s]))
        ft = b2.FRAME_I if t == 0 else b2.FRAME_P
        eng.h2d(); eng.encode(ft); eng.d2h(); eng.sync()
        for s in range(nslots):
            info, coef = eng.results(s)
            if t == 0:
                bs[s] += SC + ents[s].sps() + SC + ents[s].pps()
            bs[s] += SC + ents[s].slice(ft, t, 0, info, coef)
            recons[s].append(eng.recon(s))
        cur = oracle.OFrame(w, h).load(*frames[0]); rec = oracle.OFrame(w, h)
        info_o, coef_o = ref.encode_frame(prm, ft, cur, prev, rec, pmv, slices)
        info, coef = eng.results(0)
        want = b2.shipped_info(info_o) if pack else info_o
        assert np.array_equal(info.view(np.uint8), want.view(np.uint8)), _first_record_diff(info[None], want[None], "records t=%d" % t)
        assert np.array_equal(coef["blk"], coef_o["blk"]), "levels t=%d" % t
        ry, ru, rv = recons[0][-1]
        assert np.array_equal(ry, rec.y) and np.array_equal(ru, rec.u) and np.array_equal(rv, rec.v), "recon t=%d" % t
        if t == 2:
            assert (info_o["mb_type"] != 0).sum() > info_o.size // 4, "the cut gives a P frame with intra macroblocks"
        prev = rec
        pmv = np.zeros(info_o.size, oracle.MV); pmv["x"] = info_o["mvx"]; pmv["y"] = info_o["mvy"]
    eng.close()
    mbw, mbh = (w + 15) // 16, (h + 15) // 16
    for s in range(nslots):
        aus = check_split_in_stream(oracle, bytes(bs[s]), mbw, mbh, slices, nframes)
        for t, (dy, du, dv) in enumerate(oracle.decode_yuv(aus)):
            ry, ru, rv = recons[s][t]
            assert np.array_equal(dy, ry[:h, :w]), "decoded luma != engine recon, slot %d frame %d" % (s, t)
            assert np.array_equal(du, ru[:(h + 1) // 2, :(w + 1) // 2]) and np.array_equal(dv, rv[:(h + 1) // 2, :(w + 1) // 2])


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,slices,kw", [
    (1920, 1080, 8, {}), (3840, 2160, 8, {"t8": 1}), (1080, 1920, 8, {"cabac": 0}), (1000, 600, 5, {"t8": 1, "partitions": 2}),
    (176, 144, 9, {"pack": 1, "partitions": 1}),
    (1920, 1080, 4, {"nslots": 4, "streams": 1, "t8": 1, "partitions": 1, "offsets": (-2, 1)})],
    ids=["1080p-s8", "2160p-s8", "portrait-s8", "odd-s5", "every-row", "4slots-wavefront"])
def test_engine_slices_match_oracle(oracle, b2, w, h, slices, kw):
    if kw.get("nslots", 1) == 4:
        assert b2.deblock_shape(1920, 1088, 4)[0] == 1                   # the K8 wavefront schedule
    engine_case(oracle, b2, w, h, slices, **kw)


# ---- 7. the drop-in encoder (GPU) ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["zerolatency", "4slots", "2devices"])
def test_dropin_slices_gpu(oracle, b2, mode):
    import b2enc
    if mode == "2devices" and b2enc.lib().b2_device_count() < 2:
        pytest.skip("one GPU visible")
    w, h, qp, gop, n, slices = 640, 368, 28, 4, 10, 6
    frames = smooth_seq(w, h, n, seed=77, cut=6)
    kw = {"tune": "film,zerolatency"} if mode == "zerolatency" else {"tune": "film", "i_gop_slots": 4}
    out = drive(b2enc, None, frames, w, h, devices=2 if mode == "2devices" else 1, quality=qp, annexb=1, i_keyint_max=gop,
                i_slice_count=slices, **kw)
    bs = annexb(out)
    want, recons, *_ = ref.encode_sequence(frames, w, h, qp=qp, merange=16, gop=gop, deblock=1, cabac=1, deblock_offsets=(-1, -1),
                                             slices=slices)
    assert bs == want
    aus = check_split_in_stream(oracle, bs, w // 16, (h + 15) // 16, slices, n)
    for t, (dy, du, dv) in enumerate(oracle.decode_yuv(aus)):
        assert np.array_equal(dy, recons[t].y[:h, :w]), t
