"""K1 parity: CUDA exhaustive full-pel SAD search (through the C-ABI b2k_me_fullpel) vs the C
oracle b2o_me_fullpel -- bit-exact MVs and costs, identical tie-breaking (T1/T2 of SURVEY.md 4)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _oracle_me(oracle, cur, ref, R, pmv=None, lam=0):
    h, w = cur.shape
    z = np.zeros((h // 2, w // 2), np.uint8)
    c = oracle.OFrame(w, h).load(cur, z, z)
    r = oracle.OFrame(w, h).load(ref, z, z)
    return oracle.me_fullpel(c, r, R, pmv, lam)


def _check(oracle, b2, cur, ref, R, pmv=None, lam=0):
    mv_g, cost_g, _ = b2.me_fullpel(cur, ref, R, pmv, lam)
    for i in range(cur.shape[0]):
        mv_o, cost_o = _oracle_me(oracle, cur[i], ref[i], R, None if pmv is None else pmv[i], lam)
        assert np.array_equal(cost_g[i], cost_o), f"cost mismatch frame {i}"
        assert np.array_equal(mv_g[i]["x"], mv_o["x"]) and np.array_equal(mv_g[i]["y"], mv_o["y"]), f"mv mismatch frame {i}"


@pytest.mark.parametrize("R", [16, 32])
@pytest.mark.parametrize("wh", [(128, 64), (80, 48), (176, 144), (16, 16)])
def test_random_frames(oracle, b2, R, wh):
    w, h = wh
    rng = np.random.default_rng(R * 1000 + w)
    cur = rng.integers(0, 256, (2, h, w), dtype=np.uint8)
    ref = rng.integers(0, 256, (2, h, w), dtype=np.uint8)
    _check(oracle, b2, cur, ref, R)


@pytest.mark.parametrize("R", [16, 32])
def test_adversarial_ties(oracle, b2, R):
    """flat, periodic and saturated content: many candidates tie, the lowest scan index must win."""
    w, h = 192, 96
    flat = np.full((h, w), 77, np.uint8)
    yy, xx = np.mgrid[0:h, 0:w]
    periodic = (((xx // 4) + (yy // 4)) % 2 * 255).astype(np.uint8)
    stripes = ((xx % 8) * 32).astype(np.uint8)
    sat = np.where(xx > w // 2, 255, 0).astype(np.uint8)
    cur = np.stack([flat, periodic, stripes, sat, flat])
    ref = np.stack([flat, periodic, stripes, sat, np.full((h, w), 80, np.uint8)])
    _check(oracle, b2, cur, ref, R)
    mv, cost, _ = b2.me_fullpel(cur[:1], ref[:1], R)
    assert (mv["x"] == -R).all() and (mv["y"] == -R).all() and (cost == 0).all()


@pytest.mark.parametrize("R", [16, 32])
def test_lambda_and_predictors(oracle, b2, R):
    w, h = 256, 80
    rng = np.random.default_rng(7 + R)
    base = rng.integers(0, 256, (h + 80, w + 80), dtype=np.uint8)
    ref = base[40:40 + h, 40:40 + w][None].copy()
    cur = base[43:43 + h, 35:35 + w][None].copy()          # true motion (-5,+3)
    pmv = np.zeros((1, (w // 16) * (h // 16)), b2.MV)
    pmv["x"] = rng.integers(-140, 140, pmv.shape); pmv["y"] = rng.integers(-140, 140, pmv.shape)
    for lam in (0, 4, 91):
        _check(oracle, b2, cur, ref, R, pmv, lam)


def test_synth_known_answer_1080p(oracle, b2):
    """full C3 size: interior MBs of the panning synthetic sequence have the known MV (+3,+2);
    a random sample of MBs is checked against the oracle (size-independent spot check)."""
    w, h = 1920, 1088
    y0, _, _ = oracle.synth_frame(w, h, 4)
    y1, _, _ = oracle.synth_frame(w, h, 5)
    mv, cost, _ = b2.me_fullpel(y1, y0, 32)
    mbw, mbh = w // 16, h // 16
    mvx = mv["x"].reshape(mbh, mbw); mvy = mv["y"].reshape(mbh, mbw)
    assert (mvx[:-1, :-1] == 3).all() and (mvy[:-1, :-1] == 2).all()
    z = np.zeros((h // 2, w // 2), np.uint8)
    c = oracle.OFrame(w, h).load(y1, z, z); r = oracle.OFrame(w, h).load(y0, z, z)
    rng = np.random.default_rng(1)
    for _ in range(40):
        mbx, mby = int(rng.integers(0, mbw)), int(rng.integers(0, mbh))
        (ox, oy), oc = oracle.me_fullpel_mb(c, r, 32, mbx, mby)
        i = mby * mbw + mbx
        assert (int(mv["x"][0, i]), int(mv["y"][0, i]), int(cost[0, i])) == (ox, oy, oc)


# ---- K1 partition variant (row N1, partitions = 2): best vector of each of the nine shape parts -------------------------
def _check_parts(oracle, b2, cur, ref, R, pmv=None, lam=0):
    mv_g, cost_g, _ = b2.me_fullpel_parts(cur, ref, R, pmv, lam)
    for i in range(cur.shape[0]):
        h, w = cur[i].shape
        z = np.zeros((h // 2, w // 2), np.uint8)
        c = oracle.OFrame(w, h).load(cur[i], z, z); r = oracle.OFrame(w, h).load(ref[i], z, z)
        mv_o, cost_o = oracle.me_fullpel_parts(c, r, R, None if pmv is None else pmv[i], lam)
        assert np.array_equal(cost_g[i], cost_o), f"part costs differ, frame {i}: {np.argwhere(cost_g[i] != cost_o)[:4].tolist()}"
        assert np.array_equal(mv_g[i], mv_o), f"part vectors differ, frame {i}"
        # part 0 is the plain 16x16 search
        mv16, c16 = oracle.me_fullpel(c, r, R, None if pmv is None else pmv[i], lam)
        assert np.array_equal(mv_g[i][:, 0], mv16) and np.array_equal(cost_g[i][:, 0], c16)


@pytest.mark.parametrize("R", [16, 32])
@pytest.mark.parametrize("wh", [(128, 64), (80, 48), (176, 144), (16, 16)])
def test_parts_random_frames(oracle, b2, R, wh):
    w, h = wh
    rng = np.random.default_rng(R * 77 + w)
    cur = rng.integers(0, 256, (2, h, w), dtype=np.uint8); ref = rng.integers(0, 256, (2, h, w), dtype=np.uint8)
    _check_parts(oracle, b2, cur, ref, R)


@pytest.mark.parametrize("R", [16, 32])
def test_parts_ties_lambda_and_predictors(oracle, b2, R):
    w, h = 192, 96
    yy, xx = np.mgrid[0:h, 0:w]
    flat = np.full((h, w), 77, np.uint8)
    periodic = (((xx // 4) + (yy // 4)) % 2 * 255).astype(np.uint8)
    sat = np.where(xx > w // 2, 255, 0).astype(np.uint8)
    cur = np.stack([flat, periodic, sat]); ref = np.stack([flat, periodic, sat])
    _check_parts(oracle, b2, cur, ref, R)
    rng = np.random.default_rng(11 + R)
    base = rng.integers(0, 256, (h + 80, w + 80), dtype=np.uint8)
    ref = base[40:40 + h, 40:40 + w][None].copy(); cur = base[43:43 + h, 35:35 + w][None].copy()
    cur[0, :, w // 2:] = base[38:38 + h, 44 + w // 2:44 + w]                       # right half moves differently
    pmv = np.zeros((1, (w // 16) * (h // 16)), b2.MV)
    pmv["x"] = rng.integers(-140, 140, pmv.shape); pmv["y"] = rng.integers(-140, 140, pmv.shape)
    for lam in (0, 4, 91):
        _check_parts(oracle, b2, cur, ref, R, pmv, lam)


# ---- K1 with lossless pruning (engine option me_prune): K1a block sums + successive elimination ---------------------------
def _check_pruned(oracle, b2, cur, ref, R, pmv=None, lam=0):
    """vectors and costs equal the oracle's exhaustive scan (and hence the un-pruned kernel's); returns evaluated / all candidates"""
    mv_g, cost_g, st = b2.me_fullpel_pruned(cur, ref, R, pmv, lam)
    for i in range(cur.shape[0]):
        mv_o, cost_o = _oracle_me(oracle, cur[i], ref[i], R, None if pmv is None else pmv[i], lam)
        assert np.array_equal(cost_g[i], cost_o), f"cost mismatch frame {i}: {np.argwhere(cost_g[i] != cost_o)[:4].tolist()}"
        assert np.array_equal(mv_g[i]["x"], mv_o["x"]) and np.array_equal(mv_g[i]["y"], mv_o["y"]), f"mv mismatch frame {i}"
    assert 0 < st["swept"] <= st["all"]
    return st["swept"] / st["all"]


@pytest.mark.parametrize("ks", [1, 3, 5])
def test_block_sums_kernel(b2, ks):
    """K1a against numpy: minimum and maximum over ks rows of the 16x16 block sums of the padded plane"""
    rng = np.random.default_rng(5 + ks)
    for (w, h) in ((176, 144), (16, 16), (400, 48)):
        y = rng.integers(0, 256, (2, h, w), dtype=np.uint8)
        y[1, : h // 2] = 255                                        # the largest sums: 65,280 must not wrap
        lo, hi = b2.block_sums(y, ks)
        n, rows, pitch = lo.shape
        assert (rows, pitch) == (h + 128, w + 128)
        for i in range(n):
            ext = np.pad(y[i], 64, mode="edge").astype(np.int64)    # the padded plane as the kernels see it
            ii = np.zeros((rows + 1, pitch + 1), np.int64); ii[1:, 1:] = ext.cumsum(0).cumsum(1)
            S = ii[16:, 16:] - ii[:-16, 16:] - ii[16:, :-16] + ii[:-16, :-16]            # [rows-15, pitch-15]
            nv = rows - 15 - (ks - 1)                                                      # rows whose whole window is inside
            win = np.stack([S[j:j + nv] for j in range(ks)])
            assert np.array_equal(lo[i, :nv, :pitch - 15], win.min(0).astype(np.uint16)), (w, h, i, "min")
            assert np.array_equal(hi[i, :nv, :pitch - 15], win.max(0).astype(np.uint16)), (w, h, i, "max")
            # outside: the never-prune interval
            assert (lo[i, nv:, :] == 0).all() and (hi[i, nv:, :] == 0xffff).all()
            assert (lo[i, :, pitch - 15:] == 0).all() and (hi[i, :, pitch - 15:] == 0xffff).all()


@pytest.mark.parametrize("R", [16, 32])
@pytest.mark.parametrize("wh", [(128, 64), (80, 48), (176, 144), (16, 16), (208, 32)])
def test_pruned_random_frames(oracle, b2, R, wh):
    """white noise: the bound prunes next to nothing, every path of the survivor list (full words, ragged strips) is exercised"""
    w, h = wh
    rng = np.random.default_rng(R * 1000 + w)
    cur = rng.integers(0, 256, (2, h, w), dtype=np.uint8)
    ref = rng.integers(0, 256, (2, h, w), dtype=np.uint8)
    _check_pruned(oracle, b2, cur, ref, R)


@pytest.mark.parametrize("R", [16, 32])
def test_pruned_adversarial_ties(oracle, b2, R):
    """flat / periodic / saturated content: candidates tie at the minimum, all of them have to survive the bound and the lowest
    scan index has to win exactly as in the exhaustive scan"""
    w, h = 192, 96
    flat = np.full((h, w), 77, np.uint8)
    yy, xx = np.mgrid[0:h, 0:w]
    periodic = (((xx // 4) + (yy // 4)) % 2 * 255).astype(np.uint8)
    stripes = ((xx % 8) * 32).astype(np.uint8)
    sat = np.where(xx > w // 2, 255, 0).astype(np.uint8)
    cur = np.stack([flat, periodic, stripes, sat, flat])
    ref = np.stack([flat, periodic, stripes, sat, np.full((h, w), 80, np.uint8)])
    _check_pruned(oracle, b2, cur, ref, R)
    mv, cost, _ = b2.me_fullpel_pruned(cur[:1], ref[:1], R)
    assert (mv["x"] == -R).all() and (mv["y"] == -R).all() and (cost == 0).all()


@pytest.mark.parametrize("R", [16, 32])
def test_pruned_lambda_and_predictors(oracle, b2, R):
    """true motion + random (mostly wrong, partly out-of-range) predictors and three lambdas: the threshold candidates are poor,
    the vector costs large; results still equal the exhaustive scan"""
    w, h = 256, 80
    rng = np.random.default_rng(7 + R)
    base = rng.integers(0, 256, (h + 80, w + 80), dtype=np.uint8)
    ref = base[40:40 + h, 40:40 + w][None].copy()
    cur = base[43:43 + h, 35:35 + w][None].copy()
    pmv = np.zeros((1, (w // 16) * (h // 16)), b2.MV)
    pmv["x"] = rng.integers(-140, 140, pmv.shape); pmv["y"] = rng.integers(-140, 140, pmv.shape)
    for lam in (0, 4, 91):
        _check_pruned(oracle, b2, cur, ref, R, pmv, lam)
    good = np.zeros_like(pmv); good["x"] = -20; good["y"] = 12                            # the true motion in quarter-pels
    frac = _check_pruned(oracle, b2, cur, ref, R, good, 4)
    assert frac < 0.9                                                                      # a good predictor does prune


@pytest.mark.parametrize("R", [16, 32])
def test_pruned_smooth_content_matches_exhaustive_kernel(b2, R):
    """smooth moving content (where the bound bites): pruned == un-pruned kernel on every macroblock, several frames per launch"""
    import scipy.ndimage as ndi
    rng = np.random.default_rng(11)
    w, h, n = 352, 288, 3
    big = ndi.gaussian_filter(rng.normal(size=(h + 64, w + 64)), 6.0)
    big = (big - big.min()) / (big.max() - big.min()) * 220 + 16 + rng.normal(size=big.shape) * 2
    frames = [np.clip(big[20 + 3 * t:20 + 3 * t + h, 20 + 5 * t:20 + 5 * t + w], 0, 255).astype(np.uint8) for t in range(n + 1)]
    cur = np.stack(frames[1:]); ref = np.stack(frames[:-1])
    pmv = np.zeros((n, (w // 16) * (h // 16)), b2.MV); pmv["x"] = -20; pmv["y"] = -12
    for lam in (0, 5):
        mv_a, cost_a, _ = b2.me_fullpel(cur, ref, R, pmv, lam)
        mv_b, cost_b, st = b2.me_fullpel_pruned(cur, ref, R, pmv, lam)
        assert np.array_equal(mv_a, mv_b) and np.array_equal(cost_a, cost_b)
        assert st["swept"] < 0.9 * st["all"], st


def test_pruned_synth_1080p(oracle, b2):
    """C3 size, the bench's synthetic sequence: identical to the exhaustive kernel on all 8,160 macroblocks"""
    w, h = 1920, 1088
    y0, _, _ = oracle.synth_frame(w, h, 4)
    y1, _, _ = oracle.synth_frame(w, h, 5)
    pmv = np.zeros((1, (w // 16) * (h // 16)), b2.MV); pmv["x"] = 12; pmv["y"] = 8
    mv_a, cost_a, _ = b2.me_fullpel(y1, y0, 32, pmv, 5)
    mv_b, cost_b, st = b2.me_fullpel_pruned(y1, y0, 32, pmv, 5)
    assert np.array_equal(mv_a, mv_b) and np.array_equal(cost_a, cost_b)
    assert st["swept"] < 0.6 * st["all"], st

