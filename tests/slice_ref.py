"""The oracle with several row-aligned slices per picture (tests/mock/slices_ref.c, built here next to the mock engine), the host
slice writers on row ranges, and an access-unit splitter that keeps the slices of a picture together.  Test infrastructure."""
import ctypes as C
import glob
import os
import subprocess

import numpy as np
import b2oracle as oracle
from b2oracle import MBCOEF, MBINFO, MV, _p, _padded_frame

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BUILD = os.path.join(ROOT, "tests", "mock", "_build")
SC = b"\x00\x00\x00\x01"
_LIB = {}


def _sources(host="b2h_ca*.c"):
    """the oracle and the host sources (default: the two slice writers, as in oracle/Makefile)"""
    return sorted(glob.glob(os.path.join(ROOT, "oracle", "b2o_*.c"))) + sorted(glob.glob(os.path.join(ROOT, "video-encoder_b200", "host", host)))


def _stale(so, srcs):
    deps = srcs + glob.glob(os.path.join(ROOT, "include", "*.h")) + glob.glob(os.path.join(ROOT, "video-encoder_b200", "host", "*.h")) \
        + glob.glob(os.path.join(ROOT, "oracle", "*.h"))
    return not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in deps)


def _cc(args):
    subprocess.check_call(["gcc", "-O2", "-fPIC", "-std=gnu99", "-Wall", "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, "oracle"),
                           "-I" + os.path.join(ROOT, "video-encoder_b200", "host")] + args)


def lib():
    """the oracle, the host writers and the slice reference in one library"""
    if "ref" not in _LIB:
        os.makedirs(BUILD, exist_ok=True)
        so = os.path.join(BUILD, "libb2slices_ref.so")
        srcs = [os.path.join(ROOT, "tests", "mock", "slices_ref.c")] + _sources()
        if _stale(so, srcs):
            _cc(["-shared", "-o", so] + srcs + ["-lm", "-lpthread"])
        _LIB["ref"] = C.CDLL(so)
    return _LIB["ref"]


def mock_lib():
    """libb2enc's host side on the mock engine (tests/mock/mock_engine.c), with cfg.slices honoured through slices_ref.c"""
    if "mock" not in _LIB:
        os.makedirs(BUILD, exist_ok=True)
        so = os.path.join(BUILD, "libb2enc_mock_slices.so")
        mock = os.path.join(ROOT, "tests", "mock", "mock_engine.c")
        srcs = [mock, os.path.join(ROOT, "tests", "mock", "slices_ref.c")] + _sources("*.c")
        if _stale(so, srcs):
            obj = os.path.join(BUILD, "mock_engine_slices.o")
            _cc(["-c", "-o", obj, "-Db2o_encode_frame=b2s_mock_encode_frame", "-Db2_engine_create=b2s_mock_engine_create", mock])
            _cc(["-shared", "-DB2S_MOCK", "-o", so, obj] + srcs[1:] + ["-lm", "-lpthread"])
        _LIB["mock"] = C.CDLL(so)
    return _LIB["mock"]


def slice_rows(mbh, slices):
    """[first row of slice k, k = 0..n], the last entry being mbh (b2_slice_row)"""
    first = np.zeros(mbh + 1, np.int32)
    n = lib().b2s_slice_rows(slices, mbh, _p(first))
    return [int(r) for r in first[:n + 1]]


def intra_analyse(frame, slices, qp, i8=True):
    """the oracle's intra analysis of an OFrame with `slices` slices: (info, [cost I16, cost I4, cost I8])"""
    n = frame.f.mbw * frame.f.mbh
    info = np.zeros(n, MBINFO)
    costs = [np.zeros(n, np.uint32) for _ in range(3)]
    L = lib()
    L.b2s_intra_analyse(C.byref(frame.f), slices, L.b2o_lambda(qp), _p(info), _p(costs[0]), _p(costs[1]), _p(costs[2]) if i8 else None)
    return info, costs


def recon_intra_frame(cur, rec, info, coef, qp, slices):
    """oracle.recon_intra_frame with `slices` slices (same arguments; rec, info and coef updated in place)"""
    fc, fr = _padded_frame(*cur), _padded_frame(*rec)
    for a, dt in ((info, MBINFO), (coef, MBCOEF)):
        assert a.dtype == dt and a.flags.c_contiguous and a.flags.writeable and a.size == fc.mbw * fc.mbh
    lib().b2s_recon_intra_frame(qp, slices, C.byref(fc), C.byref(fr), _p(info), _p(coef))


def encode_frame(prm, frame_type, cur, ref, recon, prev_mv, slices):
    """oracle.encode_frame with `slices` slices"""
    n = cur.f.mbw * cur.f.mbh
    info = np.zeros(n, MBINFO); coef = np.zeros(n, MBCOEF)
    rc = lib().b2s_encode_frame(C.byref(prm), slices, frame_type, C.byref(cur.f), C.byref(ref.f) if ref is not None else None,
                                C.byref(recon.f), _p(prev_mv) if prev_mv is not None else None, _p(info), _p(coef))
    assert rc == 0
    return info, coef


class Entropy(oracle.Entropy):
    """oracle.Entropy writing each picture as the slices of `slices` (b2h_write_slice_rows / b2h_write_slice_rows_packed)"""

    def __init__(self, w, h, qp, slices=1, **kw):
        super().__init__(w, h, qp, **kw)
        self.rows = slice_rows(self.mbh, slices)

    def slice_nals(self, frame_type, frame_num, idr_id, info, coef=None, packed=None):
        L = oracle.lib()
        for fn in (L.b2h_write_slice_rows, L.b2h_write_slice_rows_packed):
            fn.restype = C.c_size_t
        L.b2h_write_slice_rows.argtypes = [C.c_void_p, C.c_void_p] + [C.c_int] * 5 + [C.c_void_p] * 3 + [C.c_size_t]
        L.b2h_write_slice_rows_packed.argtypes = [C.c_void_p, C.c_void_p] + [C.c_int] * 5 + [C.c_void_p] * 2 + [C.c_size_t, C.c_void_p, C.c_size_t]
        info = np.ascontiguousarray(info, MBINFO)
        if packed is not None:
            packed = np.ascontiguousarray(packed, np.uint8)
        else:
            coef = np.ascontiguousarray(coef, MBCOEF)
        nals = []
        for r0, r1 in zip(self.rows[:-1], self.rows[1:]):
            if packed is not None:
                n = L.b2h_write_slice_rows_packed(self.e, C.addressof(self.seq), frame_type, frame_num, idr_id, r0, r1 - r0, _p(info), _p(packed),
                                                  packed.size, _p(self.buf), self.buf.size)
            else:
                n = L.b2h_write_slice_rows(self.e, C.addressof(self.seq), frame_type, frame_num, idr_id, r0, r1 - r0, _p(info), _p(coef),
                                           _p(self.buf), self.buf.size)
            assert n > 0, "slice writer overflow"
            nals.append(self.buf[:n].tobytes())
        return nals

    def slice(self, frame_type, frame_num, idr_id, info, coef):
        """the picture's slice NALs joined by Annex-B start codes"""
        return SC.join(self.slice_nals(frame_type, frame_num, idr_id, info, coef))

    def slice_packed(self, frame_type, frame_num, idr_id, info, packed):
        return SC.join(self.slice_nals(frame_type, frame_num, idr_id, info, packed=packed))


def encode_sequence(frames, w, h, qp=26, merange=16, subpel=1, intra_in_p=1, gop=32, fps=(30, 1), deblock=0, cabac=0, transform8x8=0,
                    partitions=0, deblock_offsets=(0, 0), slices=1):
    """oracle.encode_sequence with `slices` slices per picture: (annexb_bytes, [recon OFrame], [info], [coef])"""
    prm = oracle.Params(qp, merange, subpel, intra_in_p, deblock, transform8x8, partitions, deblock_offsets[0], deblock_offsets[1])
    ent = Entropy(w, h, qp, slices, fps=fps, deblock=deblock, cabac=cabac, transform8x8=transform8x8, deblock_offsets=deblock_offsets)
    out = bytearray()
    recons, infos, coefs = [], [], []
    prev = None; prev_mv = None; idr = 0
    for t, (y, u, v) in enumerate(frames):
        cur = oracle.OFrame(w, h).load(y, u, v)
        rec = oracle.OFrame(w, h)
        if t % gop == 0:
            out += SC + ent.sps() + SC + ent.pps()
            info, coef = encode_frame(prm, 0, cur, None, rec, None, slices)
            out += SC + ent.slice(0, 0, idr, info, coef); idr += 1
        else:
            info, coef = encode_frame(prm, 1, cur, prev, rec, prev_mv, slices)
            out += SC + ent.slice(1, t % gop, 0, info, coef)
        prev_mv = np.zeros(info.size, MV); prev_mv["x"] = info["mvx"]; prev_mv["y"] = info["mvy"]
        prev = rec
        recons.append(rec); infos.append(info); coefs.append(coef)
    return bytes(out), recons, infos, coefs


def split_access_units(annexb):
    """Annex-B stream -> access units: the SEI / parameter sets in front of a picture and all its slice NALs.  Those NAL types (6-9),
    or a slice with first_mb_in_slice = 0 (top bit of the first byte after the NAL header: ue(0) = '1'), start a picture."""
    aus, cur, open_slices = [], b"", False
    for p in annexb.split(SC)[1:]:
        t = p[0] & 31
        if open_slices and (t in (6, 7, 8, 9) or (t in (1, 5) and p[1] & 0x80)):
            aus.append(cur); cur = b""; open_slices = False
        cur += SC + p
        open_slices = open_slices or t in (1, 5)
    if open_slices:
        aus.append(cur)
    return aus
