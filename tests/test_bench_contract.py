"""bench.py's reference arm runs on the CPU (oracle port of the stage): one tiny run checks the contract of the JSON result line
(keys, units, impl marker, zero copy bytes) without a GPU.  On the GPU: the outputs --dump-outputs writes."""
import json
import os
import subprocess
import sys
import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_contract():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c5", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-500:]
    line = r.stdout.strip().splitlines()[-1]
    d = json.loads(line)
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "frames/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["vs_baseline"] is None


def test_default_arm_refuses_to_run_without_a_gpu():
    """no CPU fallback: on a box without a CUDA device the product arm must fail loudly, not fall back to the oracle"""
    sys.path.insert(0, os.path.join(ROOT, "video-encoder_b200"))
    import b2enc
    if b2enc.lib().b2_device_count() > 0:
        return
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True, timeout=600)
    assert r.returncode != 0
    assert "CUDA" in (r.stderr + r.stdout) or "GPU" in (r.stderr + r.stdout)


@pytest.mark.gpu
def test_dump_outputs_repeat_exactly(tmp_path):
    """--dump-outputs: the last timed step's decisions, levels and reconstruction as float .npy files of at most 64 MB together,
    taken from the state the oracle check passes, and identical from run to run with the same arguments"""
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c5", "--steps", "2", "--warmup", "3", "--no-cpu-baseline", "--no-dropin"]
    dumps = []
    for run in range(2):
        d = tmp_path / str(run)
        r = subprocess.run(cmd + ["--dump-outputs", str(d)], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        out = json.loads(r.stdout.strip().splitlines()[-1])
        assert out["steps"] == 2 and out["verified"] is True
        files = sorted(os.listdir(d))
        assert files == ["levels.npy", "mb_info.npy", "recon.npy"]
        assert sum(os.path.getsize(d / f) for f in files) <= 64 << 20
        arrays = {f: np.load(d / f) for f in files}
        assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
        assert arrays["recon.npy"].max() > 0 and np.abs(arrays["levels.npy"]).max() > 0
        dumps.append(arrays)
    for f in dumps[0]:
        assert np.array_equal(dumps[0][f], dumps[1][f]), f


@pytest.mark.gpu
def test_dump_outputs_rows_are_the_engines_results(oracle, b2, tmp_path, monkeypatch):
    """dump_outputs' layout: row k of each file is the k-th macroblock of the seed-0 sample (sorted by slot, then macroblock), and it
    holds that macroblock's decisions and levels from eng.results(slot) and its pixels from eng.recon(slot)"""
    # bench sets CUDA_DEVICE_MAX_CONNECTIONS when imported; monkeypatch restores the variable after the test
    monkeypatch.setenv("CUDA_DEVICE_MAX_CONNECTIONS", os.environ.get("CUDA_DEVICE_MAX_CONNECTIONS", "32"))
    import bench
    n = 50
    monkeypatch.setattr(bench, "DUMP_MBS", n)                      # fewer than the engine's 4 x 24 macroblocks: the sample is drawn
    w, h, slots = 96, 64, 4
    eng = b2.Engine(w, h, slots=slots, ring=1, merange=16, qp=20, pack_levels=1)
    for t in range(2):
        for s in range(slots):
            eng.put_frame(s, 0, list(oracle.synth_frame(w, h, t, s)))
        eng.h2d(); eng.encode(b2.FRAME_I if t == 0 else b2.FRAME_P); eng.d2h(); eng.sync()
    bench.dump_outputs(eng, str(tmp_path))
    info, levels, recon = (np.load(tmp_path / f) for f in ("mb_info.npy", "levels.npy", "recon.npy"))
    assert info.shape == (n, 33) and levels.shape == (n, 26, 16) and recon.shape == (n, 384)
    assert np.abs(levels).max() > 0
    results = {s: [a.copy() for a in eng.results(s)] for s in range(slots)}      # info is a view of the engine's host buffer
    planes = {s: eng.recon(s) for s in range(slots)}
    eng.close()
    pick = np.sort(np.random.default_rng(0).choice(slots * eng.nmb, n, replace=False))
    for k, p in enumerate(pick):
        s, m = divmod(int(p), eng.nmb)
        by, bx = divmod(m, eng.mbw)
        mbinfo, coef = results[s]
        y, u, v = planes[s]
        assert np.array_equal(info[k], np.concatenate([np.ravel(mbinfo[f][m]) for f in mbinfo.dtype.names]).astype(np.float64)), k
        assert np.array_equal(levels[k], coef["blk"][m]), k
        assert np.array_equal(recon[k], np.concatenate([y[16 * by:16 * by + 16, 16 * bx:16 * bx + 16].ravel(),
                                                        u[8 * by:8 * by + 8, 8 * bx:8 * bx + 8].ravel(),
                                                        v[8 * by:8 * by + 8, 8 * bx:8 * bx + 8].ravel()])), k
