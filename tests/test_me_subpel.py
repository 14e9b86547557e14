"""K2 parity: CUDA half- then quarter-pel SATD refinement (through the C-ABI b2k_me_subpel) vs the C oracle b2o_me_subpel /
b2o_me_subpel_part -- bit-exact vectors, costs, partition shapes, quadrant vectors and the motion-compensated 16x16 prediction
K2 hands to K5, at every launch shape: frame counts 1, 2, 7 and 64, picture widths that are and are not a multiple of the
macroblocks per CTA, 720p and 1080p."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _oframes(oracle, cur, ref):
    h, w = cur.shape
    z = np.zeros((h // 2, w // 2), np.uint8)
    return oracle.OFrame(w, h).load(cur, z, z), oracle.OFrame(w, h).load(ref, z, z)


def _mc(oracle, r, x, y, mvx, mvy, bw, bh, dst):
    """b2o_mc_luma into the uint8 view dst (row pitch 16)"""
    L = oracle.lib()
    L.b2o_mc_luma.argtypes = [C.c_void_p, C.c_int] + [C.c_int] * 6 + [C.c_void_p, C.c_int]
    L.b2o_mc_luma(r.f.y, r.f.pitch, x, y, mvx, mvy, bw, bh, dst.ctypes.data, 16)


def oracle_subpel(oracle, cur, ref, mvf, pmv, lam, subpel, partitions):
    """oracle results of one frame: (mv, cost, pred [mbs,16,16], part, mv8 [mbs,3])"""
    L = oracle.lib()
    c, r = _oframes(oracle, cur, ref)
    mbw, mbh = c.f.mbw, c.f.mbh
    n = mbw * mbh
    mvf = np.ascontiguousarray(mvf, oracle.MV)
    pm = np.zeros(n, oracle.MV) if pmv is None else np.ascontiguousarray(pmv, oracle.MV)
    mv = np.zeros(n, oracle.MV); cost = np.zeros(n, np.uint32)
    part = np.zeros(n, np.uint8); mv8 = np.zeros((n, 3), oracle.MV)
    if subpel and partitions:
        mv4 = np.zeros((n, 4), oracle.MV)
        L.b2o_me_subpel_part(C.byref(c.f), C.byref(r.f), oracle._p(mvf), oracle._p(pm), lam, oracle._p(part), oracle._p(mv4), oracle._p(cost))
        mv[:] = mv4[:, 0]; mv8[:] = mv4[:, 1:]
    elif subpel:
        L.b2o_me_subpel(C.byref(c.f), C.byref(r.f), oracle._p(mvf), oracle._p(pm), lam, oracle._p(mv), oracle._p(cost))
    else:                                    # the full-pel vector priced in the SATD domain (b2o_encode_frame without sub-pel)
        L.b2o_satd16x16.restype = C.c_uint32
        L.b2o_satd16x16.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int]
        mv["x"] = mvf["x"] * 4; mv["y"] = mvf["y"] * 4
        for i in range(n):
            mbx, mby = i % mbw, i // mbw
            a = c.f.y + mby * 16 * c.f.pitch + mbx * 16
            b = r.f.y + (mby * 16 + int(mvf["y"][i])) * r.f.pitch + mbx * 16 + int(mvf["x"][i])
            cost[i] = L.b2o_satd16x16(a, c.f.pitch, b, r.f.pitch) + lam * (L.b2o_mvbits(int(mv["x"][i]) - int(pm["x"][i])) +
                                                                          L.b2o_mvbits(int(mv["y"][i]) - int(pm["y"][i])))
    pred = np.zeros((n, 16, 16), np.uint8)
    for i in range(n):
        mbx, mby = i % mbw, i // mbw
        if part[i] == 0:
            _mc(oracle, r, mbx * 16, mby * 16, int(mv["x"][i]), int(mv["y"][i]), 16, 16, pred[i])
            continue
        for q in range(4):
            v = mv[i] if q == 0 else mv8[i, q - 1]
            qx, qy = (q & 1) * 8, (q >> 1) * 8
            _mc(oracle, r, mbx * 16 + qx, mby * 16 + qy, int(v["x"]), int(v["y"]), 8, 8, pred[i, qy:, qx:])
    return mv, cost, pred, part, mv8


def check(oracle, b2, cur, ref, mvf, pmv=None, lam=0, subpel=1, partitions=0):
    """runs the kernel on all frames in one launch and compares every output with the oracle, frame by frame; returns the
    kernel's vectors"""
    n = cur.shape[0]
    mv_g, cost_g, pred_g, part_g, mv8_g, _ = b2.me_subpel(cur, ref, mvf, pmv, lam, subpel, partitions)
    for f in range(n):
        mv_o, cost_o, pred_o, part_o, mv8_o = oracle_subpel(oracle, cur[f], ref[f], mvf[f], None if pmv is None else pmv[f], lam,
                                                             subpel, partitions)
        bad = np.flatnonzero((mv_g[f] != mv_o) | (cost_g[f] != cost_o))
        assert bad.size == 0, f"frame {f}: vector/cost differ at MBs {bad[:6].tolist()}: " \
                              f"gpu {mv_g[f][bad[:3]].tolist()} {cost_g[f][bad[:3]].tolist()} oracle {mv_o[bad[:3]].tolist()} {cost_o[bad[:3]].tolist()}"
        assert np.array_equal(part_g[f], part_o), f"frame {f}: partition shapes differ"
        assert np.array_equal(mv8_g[f], mv8_o), f"frame {f}: quadrant vectors differ"
        bad = np.flatnonzero((pred_g[f] != pred_o).any(axis=(1, 2)))
        assert bad.size == 0, f"frame {f}: prediction differs at MBs {bad[:6].tolist()}"
    return mv_g


def random_vectors(rng, n, nmb, R=32):
    mvf = np.zeros((n, nmb), np.dtype([("x", "<i2"), ("y", "<i2")]))
    mvf["x"] = rng.integers(-R, R + 1, mvf.shape); mvf["y"] = rng.integers(-R, R + 1, mvf.shape)
    return mvf


def edge_vectors(n, w, h, R=32):
    """every MB on the picture's border points its patch as far out as the range allows, the others alternate +-R"""
    mbw, mbh = w // 16, h // 16
    mvf = np.zeros((n, mbh, mbw), np.dtype([("x", "<i2"), ("y", "<i2")]))
    yy, xx = np.mgrid[0:mbh, 0:mbw]
    mvf["x"][:] = np.where(xx == 0, -R, np.where(xx == mbw - 1, R, np.where((xx + yy) % 2, R, -R)))
    mvf["y"][:] = np.where(yy == 0, -R, np.where(yy == mbh - 1, R, np.where(xx % 2, -R, R)))
    return mvf.reshape(n, mbw * mbh)


def smooth_planes(rng, n, w, h, sigma=2.5):
    import scipy.ndimage as ndi
    out = []
    for _ in range(n):
        p = ndi.gaussian_filter(rng.normal(size=(h, w)), sigma)
        out.append(np.clip((p - p.min()) / (p.max() - p.min()) * 235 + 10, 0, 255).astype(np.uint8))
    return np.stack(out)


def quarter_shifted(oracle, ref, mvf):
    """a current frame whose MB i is the reference interpolated at 4*mvf + d_i, d_i running through every offset of [-3,3]^2:
    with lambda 0 that offset is (nearly always) the winner, so every quarter-pel fraction wins somewhere"""
    n, h, w = ref.shape
    mbw = w // 16
    cur = np.zeros_like(ref)
    for f in range(n):
        _, r = _oframes(oracle, ref[f], ref[f])
        for i in range(mvf.shape[1]):
            mbx, mby = i % mbw, i // mbw
            d = (i + 11 * f) % 49
            dx, dy = d % 7 - 3, d // 7 - 3
            blk = np.zeros((16, 16), np.uint8)
            _mc(oracle, r, mbx * 16, mby * 16, 4 * int(mvf["x"][f, i]) + dx, 4 * int(mvf["y"][f, i]) + dy, 16, 16, blk)
            cur[f, mby * 16:mby * 16 + 16, mbx * 16:mbx * 16 + 16] = blk
    return cur


MODES = [(1, 0), (1, 1), (0, 0), (0, 1)]          # (subpel, partitions)


@pytest.mark.parametrize("subpel,partitions", MODES)
@pytest.mark.parametrize("n", [1, 2, 7, 64])
def test_random_content_frame_counts(oracle, b2, n, subpel, partitions):
    """white noise, random vectors over the whole +-32 range and random predictors; 11 x 9 MBs: 11 is not a multiple of the MBs
    per CTA, so every launch has a partial tail CTA in every row"""
    w, h = 176, 144
    rng = np.random.default_rng(1000 * n + 10 * subpel + partitions)
    cur = rng.integers(0, 256, (n, h, w), dtype=np.uint8); ref = rng.integers(0, 256, (n, h, w), dtype=np.uint8)
    nmb = (w // 16) * (h // 16)
    mvf = random_vectors(rng, n, nmb)
    pmv = np.zeros((n, nmb), b2.MV); pmv["x"] = rng.integers(-150, 150, pmv.shape); pmv["y"] = rng.integers(-150, 150, pmv.shape)
    check(oracle, b2, cur, ref, mvf, pmv, 4, subpel, partitions)


@pytest.mark.parametrize("subpel,partitions", MODES)
@pytest.mark.parametrize("wh", [(16, 16), (48, 32), (208, 48), (256, 64)])
def test_patches_reach_the_padding(oracle, b2, wh, subpel, partitions):
    """full-pel vectors at +-32 on every border MB: the 22 x 22 patches (and the aligned words around them) reach into the
    replicated padding at all four edges and corners"""
    w, h = wh
    rng = np.random.default_rng(w + h)
    n = 2
    cur = rng.integers(0, 256, (n, h, w), dtype=np.uint8); ref = rng.integers(0, 256, (n, h, w), dtype=np.uint8)
    ref[1] = smooth_planes(rng, 1, w, h)[0]
    check(oracle, b2, cur, ref, edge_vectors(n, w, h), None, 0, subpel, partitions)


@pytest.mark.parametrize("partitions", [0, 1])
def test_every_quarter_fraction_wins(oracle, b2, partitions):
    """smooth content, each MB a quarter-pel shift of the reference: all 16 fractions of the vector occur among the winners"""
    w, h, n = 208, 112, 2
    rng = np.random.default_rng(5)
    ref = smooth_planes(rng, n, w, h)
    nmb = (w // 16) * (h // 16)
    mvf = random_vectors(rng, n, nmb, 24)
    cur = quarter_shifted(oracle, ref, mvf)
    mv = check(oracle, b2, cur, ref, mvf, None, 0, 1, partitions)
    frac = set(zip((mv["x"] & 3).ravel().tolist(), (mv["y"] & 3).ravel().tolist()))
    assert len(frac) == 16, sorted(frac)


@pytest.mark.parametrize("subpel,partitions", MODES)
def test_exact_ties(oracle, b2, subpel, partitions):
    """flat, saturated, periodic and stepped content: many candidates cost exactly the same and the lower index must win"""
    w, h = 96, 64
    yy, xx = np.mgrid[0:h, 0:w]
    planes = [np.full((h, w), 77, np.uint8), np.where(xx > w // 2, 255, 0).astype(np.uint8),
              (((xx // 2) + (yy // 2)) % 2 * 255).astype(np.uint8), ((xx % 8) * 32).astype(np.uint8),
              np.where(yy % 16 < 8, 0, 255).astype(np.uint8)]
    cur = np.stack(planes + [np.full((h, w), 200, np.uint8)])
    ref = np.stack(planes + [np.full((h, w), 199, np.uint8)])
    n, nmb = cur.shape[0], (w // 16) * (h // 16)
    rng = np.random.default_rng(3)
    for mvf in (np.zeros((n, nmb), b2.MV), random_vectors(rng, n, nmb, 8)):
        mv = check(oracle, b2, cur, ref, mvf, None, 0, subpel, partitions)
    assert (mv[0]["x"] == 4 * mvf[0]["x"]).all() and (mv[0]["y"] == 4 * mvf[0]["y"]).all()       # flat: every candidate ties, the centre wins


@pytest.mark.parametrize("subpel,partitions", MODES)
def test_far_predictors_large_lambda(oracle, b2, subpel, partitions):
    """predictors far from the vector and large lambdas: the vector cost dominates the choice"""
    w, h, n = 128, 80, 3
    rng = np.random.default_rng(17)
    ref = smooth_planes(rng, n, w, h, 1.5)
    nmb = (w // 16) * (h // 16)
    mvf = random_vectors(rng, n, nmb)
    cur = quarter_shifted(oracle, ref, mvf)
    pmv = np.zeros((n, nmb), b2.MV); pmv["x"] = rng.choice([-2000, 2000, 3, -5], pmv.shape); pmv["y"] = rng.choice([-1500, 1700, 1], pmv.shape)
    for lam in (91, 4000):
        check(oracle, b2, cur, ref, mvf, pmv, lam, subpel, partitions)


@pytest.mark.parametrize("subpel,partitions", MODES)
@pytest.mark.parametrize("wh", [(1280, 720), (1920, 1088)])
def test_full_sizes(oracle, b2, wh, subpel, partitions):
    """720p and 1080p: the bench's synthetic panning sequence with the vectors K1 finds for it, and noise with random vectors"""
    w, h = wh
    y0, _, _ = oracle.synth_frame(w, h, 4)
    y1, _, _ = oracle.synth_frame(w, h, 5)
    mvf, _, _ = b2.me_fullpel(y1, y0, 32)
    pmv = np.zeros_like(mvf); pmv["x"] = 12; pmv["y"] = 8
    check(oracle, b2, y1[None], y0[None], mvf, pmv, 5, subpel, partitions)
    rng = np.random.default_rng(w)
    cur = rng.integers(0, 256, (1, h, w), dtype=np.uint8); ref = rng.integers(0, 256, (1, h, w), dtype=np.uint8)
    check(oracle, b2, cur, ref, random_vectors(rng, 1, (w // 16) * (h // 16)), None, 5, subpel, partitions)
