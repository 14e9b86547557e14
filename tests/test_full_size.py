"""BASELINE.json's named configurations at FULL size on the GPU (C2 720p +-16, C3 1080p +-32 + qpel + intra/inter,
C4 2160p, C5 many 720p streams): bit-exact against the oracle where the oracle finishes in seconds, and through the
size-independent decoder-drift property (entropy-code the engine's output, decode with libavcodec, compare with the
engine's own reconstruction) for every stream."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _encode_and_check(oracle, b2, w, h, R, qp, nslots, nframes, oracle_slots, subpel=1, intra_in_p=1, deblock=0, cabac=0, t8=0,
                      partitions=0, pack=0, frame_fn=None, deblock_offsets=(0, 0), streams=0, expect_groups=None, infos=None):
    """expect_groups: the engine's stream groups as (first slot, slots) -- the frames of a group share every launch;
    infos: a list that receives (t, slot, the engine's info) of every frame"""
    eng = b2.Engine(w, h, slots=nslots, ring=1, merange=R, qp=qp, subpel=subpel, intra_in_p=intra_in_p, deblock=deblock,
                    transform8x8=t8, partitions=partitions, pack_levels=pack, deblock_offsets=deblock_offsets, streams=streams)
    if expect_groups is not None:
        assert eng.groups() == expect_groups
    prm = oracle.Params(qp, R, subpel, intra_in_p, deblock, t8, partitions, *deblock_offsets)
    ents = [oracle.Entropy(w, h, qp, deblock=deblock, cabac=cabac, transform8x8=t8, deblock_offsets=deblock_offsets) for _ in range(nslots)]
    frame_fn = frame_fn or (lambda t, s: oracle.synth_frame(w, h, t, s))
    streams = [bytearray() for _ in range(nslots)]
    recons = [[] for _ in range(nslots)]
    prev = {s: None for s in oracle_slots}; pmv = {s: None for s in oracle_slots}
    sc = b"\x00\x00\x00\x01"
    for t in range(nframes):
        frames = [frame_fn(t, s) for s in range(nslots)]
        for s in range(nslots):
            eng.put_frame(s, 0, list(frames[s]))
        ft = b2.FRAME_I if t == 0 else b2.FRAME_P
        eng.h2d(); eng.encode(ft); eng.d2h(); eng.sync()
        for s in range(nslots):
            info, coef = eng.results(s)
            if infos is not None:
                infos.append((t, s, info.copy()))
            if t == 0:
                streams[s] += sc + ents[s].sps() + sc + ents[s].pps()
            streams[s] += sc + ents[s].slice(ft, t, 0, info, coef)
            recons[s].append(eng.recon(s))
            if s in oracle_slots:
                cur = oracle.OFrame(w, h).load(*frames[s]); rec = oracle.OFrame(w, h)
                info_o, coef_o = oracle.encode_frame(prm, ft, cur, prev[s], rec, pmv[s])
                assert np.array_equal(info, b2.shipped_info(info_o) if pack else info_o), f"decisions differ t={t} s={s}"
                assert np.array_equal(coef["blk"], coef_o["blk"]), f"levels differ t={t} s={s}"
                ry, ru, rv = recons[s][-1]
                assert np.array_equal(ry, rec.y) and np.array_equal(ru, rec.u) and np.array_equal(rv, rec.v), f"recon t={t} s={s}"
                prev[s] = rec
                pmv[s] = np.zeros(info_o.size, oracle.MV); pmv[s]["x"] = info_o["mvx"]; pmv[s]["y"] = info_o["mvy"]
    eng.close()
    # decoder drift: every stream decodes to exactly the engine's reconstruction
    for s in range(nslots):
        dec = oracle.decode_yuv(oracle.split_access_units(bytes(streams[s])))
        assert len(dec) == nframes
        for t, (dy, du, dv) in enumerate(dec):
            ry, ru, rv = recons[s][t]
            assert np.array_equal(dy, ry[:h, :w]), f"decoded luma != engine recon, stream {s} frame {t}"
            assert np.array_equal(du, ru[:(h + 1) // 2, :(w + 1) // 2]) and np.array_equal(dv, rv[:(h + 1) // 2, :(w + 1) // 2])
    return streams


def test_c2_720p_merange16(oracle, b2):
    _encode_and_check(oracle, b2, 1280, 720, 16, 26, nslots=2, nframes=4, oracle_slots=[0, 1])


def test_c3_1080p_merange32_qpel_intra(oracle, b2):
    _encode_and_check(oracle, b2, 1920, 1080, 32, 26, nslots=2, nframes=3, oracle_slots=[0])


def test_c4_2160p(oracle, b2):
    _encode_and_check(oracle, b2, 3840, 2160, 32, 30, nslots=1, nframes=2, oracle_slots=[0])


def test_c5_many_720p_streams(oracle, b2):
    """one GPU's share of the 64-stream configuration: 8 live streams in lock-step, each with its own pan vector"""
    streams = _encode_and_check(oracle, b2, 1280, 720, 16, 28, nslots=8, nframes=3, oracle_slots=[3])
    assert len({bytes(s) for s in streams}) == 8            # different content -> different streams


def test_c3_1080p_with_deblocking(oracle, b2):
    _encode_and_check(oracle, b2, 1920, 1080, 32, 32, nslots=2, nframes=3, oracle_slots=[0], deblock=1)


def test_c3_1080p_all_features(oracle, b2):
    """rows N1-N3 together at full size: CABAC, adaptive 8x8 transform + intra 8x8, inter partitions, deblocking, packed
    levels -- oracle-exact on one stream and decoder-exact on both (content: sheared motion so that partitions occur)"""
    from test_oracle_decode import shear_seq
    w, h = 1920, 1080
    seqs = [shear_seq(w, h, 3, seed=31, stripe=72, band=56), shear_seq(w, h, 3, seed=32, stripe=40, band=88)]
    _encode_and_check(oracle, b2, w, h, 32, 30, nslots=2, nframes=3, oracle_slots=[0], deblock=1, cabac=1, t8=1, partitions=1, pack=1,
                      frame_fn=lambda t, s: seqs[s][t])
