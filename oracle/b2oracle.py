"""ctypes loader for the CPU oracle (oracle/libb2oracle.so).  TEST INFRASTRUCTURE ONLY:
import from tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs.
The product (video-encoder_b200/) never imports this module."""
import ctypes as C
import os
import subprocess
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

PAD = 64
PADC = 32


class Frame(C.Structure):
    _fields_ = [("w", C.c_int), ("h", C.c_int), ("w16", C.c_int), ("h16", C.c_int),
                ("mbw", C.c_int), ("mbh", C.c_int), ("pitch", C.c_int), ("pitchc", C.c_int),
                ("buf", C.c_void_p * 3), ("y", C.c_void_p), ("u", C.c_void_p), ("v", C.c_void_p)]


class Params(C.Structure):
    _fields_ = [("qp", C.c_int), ("merange", C.c_int), ("subpel", C.c_int), ("intra_in_p", C.c_int), ("deblock", C.c_int), ("transform8x8", C.c_int), ("partitions", C.c_int),
                ("deblock_alpha", C.c_int), ("deblock_beta", C.c_int)]


MV = np.dtype([("x", "<i2"), ("y", "<i2")])
MBINFO = np.dtype([("mvx", "<i2"), ("mvy", "<i2"), ("mb_type", "u1"), ("i16_mode", "u1"),
                   ("chroma_mode", "u1"), ("cbp", "u1"), ("i4_mode", "u1", (16,)),
                   ("cost", "<u4"), ("nnz_mask", "<u4"), ("mv8", "<i2", (3, 2)), ("part", "u1"),
                   ("transform8x8", "u1"), ("i8_modes", "<u2")])
MBCOEF = np.dtype([("blk", "<i2", (26, 16))])
assert MBINFO.itemsize == 48 and MBCOEF.itemsize == 832


def build(force=False):
    so = os.path.join(_HERE, "libb2oracle.so")
    if force or not os.path.exists(so):
        subprocess.check_call(["make", "-C", _HERE, "-s"] + (["-B"] if force else []))
    return so


def lib():
    global _LIB
    if _LIB is None:
        _LIB = C.CDLL(build())
        _LIB.b2o_psnr_y.restype = C.c_double
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class OFrame:
    """A padded oracle frame (owns its memory)."""

    def __init__(self, w, h):
        self.f = Frame()
        if lib().b2o_frame_alloc(C.byref(self.f), w, h) != 0:
            raise MemoryError
        self.w, self.h = w, h

    def __del__(self):
        try:
            lib().b2o_frame_free(C.byref(self.f))
        except Exception:
            pass

    def load(self, y, u, v):
        y = np.ascontiguousarray(y, np.uint8); u = np.ascontiguousarray(u, np.uint8); v = np.ascontiguousarray(v, np.uint8)
        planes = (C.c_void_p * 3)(y.ctypes.data, u.ctypes.data, v.ctypes.data)
        strides = (C.c_int * 3)(y.shape[1], u.shape[1], v.shape[1])
        lib().b2o_frame_load(C.byref(self.f), planes, strides)
        return self

    def _plane(self, ptr, pitch, w, h):
        n = pitch * (h - 1) + w
        buf = (C.c_uint8 * n).from_address(ptr)
        a = np.frombuffer(buf, np.uint8)
        return np.lib.stride_tricks.as_strided(a, (h, w), (pitch, 1))

    @property
    def y(self):   # coded-size view
        return self._plane(self.f.y, self.f.pitch, self.f.w16, self.f.h16)

    @property
    def u(self):
        return self._plane(self.f.u, self.f.pitchc, self.f.w16 // 2, self.f.h16 // 2)

    @property
    def v(self):
        return self._plane(self.f.v, self.f.pitchc, self.f.w16 // 2, self.f.h16 // 2)


def synth_frame(w, h, t, stream=0):
    y = np.empty((h, w), np.uint8)
    u = np.empty(((h + 1) // 2, (w + 1) // 2), np.uint8)
    v = np.empty_like(u)
    lib().b2o_synth_frame(w, h, t, stream, _p(y), _p(u), _p(v))
    return y, u, v


def me_fullpel(cur: OFrame, ref: OFrame, R, pmv=None, lam=0):
    n = cur.f.mbw * cur.f.mbh
    mv = np.zeros(n, MV); cost = np.zeros(n, np.uint32)
    lib().b2o_me_fullpel(C.byref(cur.f), C.byref(ref.f), R, _p(pmv) if pmv is not None else None, lam, _p(mv), _p(cost))
    return mv, cost


def me_fullpel_mb(cur, ref, R, mbx, mby, pmv=(0, 0), lam=0):
    mv = np.zeros(1, MV); cost = np.zeros(1, np.uint32)
    p = np.zeros(1, MV); p["x"] = pmv[0]; p["y"] = pmv[1]
    lib().b2o_me_fullpel_mb.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p]
    packed = int(p.view(np.uint32)[0])
    lib().b2o_me_fullpel_mb(C.addressof(cur.f), C.addressof(ref.f), R, mbx, mby, packed, lam, _p(mv), _p(cost))
    return (int(mv["x"][0]), int(mv["y"][0])), int(cost[0])


def me_fullpel_parts(cur: OFrame, ref: OFrame, R, pmv=None, lam=0):
    """best full-pel vector / cost of the nine shape parts of every MB (b2o_me_fullpel_parts_mb): mv[mbs,9], cost[mbs,9]"""
    L = lib()
    L.b2o_me_fullpel_parts_mb.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p]
    mbw, mbh = cur.f.mbw, cur.f.mbh
    mv = np.zeros((mbw * mbh, 9), MV); cost = np.zeros((mbw * mbh, 9), np.uint32)
    for i in range(mbw * mbh):
        packed = int(np.ascontiguousarray(pmv[i:i + 1]).view(np.uint32)[0]) if pmv is not None else 0
        L.b2o_me_fullpel_parts_mb(C.addressof(cur.f), C.addressof(ref.f), R, i % mbw, i // mbw, packed, lam,
                                  mv[i].ctypes.data_as(C.c_void_p), cost[i].ctypes.data_as(C.c_void_p))
    return mv, cost


# ---- frame-level oracle encoder + host entropy coder (linked into libb2oracle.so) ---------------
def deblock_frame(y, u, v, info, qp, alpha_off=0, beta_off=0):
    """b2o_deblock_frame in place on one frame's padded planes: y [h16 + 2*PAD, w16 + 2*PAD], u/v [h16/2 + 2*PADC, pitchc]
    C-contiguous uint8 arrays (any chroma pitch); info MBINFO [mbs] in raster order"""
    assert all(p.flags.writeable for p in (y, u, v))
    f = _padded_frame(y, u, v)
    info = np.ascontiguousarray(info, MBINFO)
    assert info.size == f.mbw * f.mbh
    lib().b2o_deblock_frame(C.byref(f), _p(info), qp, alpha_off, beta_off)


def _padded_frame(y, u, v):
    """b2o_frame_t over one frame's padded planes (y [h16 + 2*PAD, w16 + 2*PAD], u/v [h16/2 + 2*PADC, pitchc])"""
    for p in (y, u, v):
        assert p.dtype == np.uint8 and p.flags.c_contiguous
    assert u.shape == v.shape
    f = Frame()
    f.w16 = f.w = y.shape[1] - 2 * PAD
    f.h16 = f.h = y.shape[0] - 2 * PAD
    f.mbw, f.mbh = f.w16 // 16, f.h16 // 16
    f.pitch, f.pitchc = y.strides[0], u.strides[0]
    f.y = y.ctypes.data + PAD * f.pitch + PAD
    f.u = u.ctypes.data + PADC * f.pitchc + PADC
    f.v = v.ctypes.data + PADC * f.pitchc + PADC
    return f


def recon_intra_frame(cur, rec, info, coef, qp):
    """b2o_recon_intra_frame on one frame: cur / rec = (y, u, v) padded planes as for deblock_frame; rec, info (MBINFO [mbs])
    and coef (MBCOEF [mbs]) are updated in place -- intra macroblocks only, in raster order"""
    fc, fr = _padded_frame(*cur), _padded_frame(*rec)
    assert all(p.flags.writeable for p in rec) and (fc.w16, fc.h16, fc.pitchc) == (fr.w16, fr.h16, fr.pitchc)
    for a, dt in ((info, MBINFO), (coef, MBCOEF)):
        assert a.dtype == dt and a.flags.c_contiguous and a.flags.writeable and a.size == fc.mbw * fc.mbh
    lib().b2o_recon_intra_frame(qp, C.byref(fc), C.byref(fr), _p(info), _p(coef))


class Seq(C.Structure):
    _fields_ = [("width", C.c_int), ("height", C.c_int), ("fps_num", C.c_int), ("fps_den", C.c_int),
                ("sar_w", C.c_int), ("sar_h", C.c_int), ("qp", C.c_int), ("deblock", C.c_int),
                ("cabac", C.c_int), ("transform8x8", C.c_int), ("deblock_alpha", C.c_int), ("deblock_beta", C.c_int)]


def encode_frame(prm: Params, frame_type, cur: OFrame, ref, recon: OFrame, prev_mv=None):
    n = cur.f.mbw * cur.f.mbh
    info = np.zeros(n, MBINFO); coef = np.zeros(n, MBCOEF)
    lib().b2o_encode_frame(C.byref(prm), frame_type, C.byref(cur.f), C.byref(ref.f) if ref is not None else None,
                           C.byref(recon.f), _p(prev_mv) if prev_mv is not None else None, _p(info), _p(coef))
    return info, coef


class Entropy:
    def __init__(self, w, h, qp, fps=(30, 1), sar=(1, 1), deblock=0, cabac=0, transform8x8=0, deblock_offsets=(0, 0)):
        L = lib()
        L.b2h_entropy_create.restype = C.c_void_p
        L.b2h_write_sps.restype = C.c_size_t; L.b2h_write_pps.restype = C.c_size_t; L.b2h_write_slice.restype = C.c_size_t
        L.b2h_write_slice.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
        L.b2h_entropy_destroy.argtypes = [C.c_void_p]
        self.seq = Seq(w, h, fps[0], fps[1], sar[0], sar[1], qp, deblock, cabac, transform8x8, deblock_offsets[0], deblock_offsets[1])
        self.mbw, self.mbh = (w + 15) // 16, (h + 15) // 16
        self.e = L.b2h_entropy_create(self.mbw, self.mbh)
        self.buf = np.zeros(self.mbw * self.mbh * 3072 + 65536, np.uint8)

    def __del__(self):
        try:
            lib().b2h_entropy_destroy(self.e)
        except Exception:
            pass

    def sps(self):
        n = lib().b2h_write_sps(C.byref(self.seq), _p(self.buf), self.buf.size)
        assert n > 0
        return self.buf[:n].tobytes()

    def pps(self):
        n = lib().b2h_write_pps(C.byref(self.seq), _p(self.buf), self.buf.size)
        assert n > 0
        return self.buf[:n].tobytes()

    def slice_packed(self, frame_type, frame_num, idr_id, info, packed):
        """same slice from the packed level stream (b2h_write_slice_packed)"""
        L = lib()
        L.b2h_write_slice_packed.restype = C.c_size_t
        L.b2h_write_slice_packed.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t,
                                             C.c_void_p, C.c_size_t]
        info = np.ascontiguousarray(info, MBINFO); packed = np.ascontiguousarray(packed, np.uint8)
        n = L.b2h_write_slice_packed(self.e, C.addressof(self.seq), frame_type, frame_num, idr_id, _p(info), _p(packed), packed.size,
                                     _p(self.buf), self.buf.size)
        assert n > 0, "slice writer overflow"
        return self.buf[:n].tobytes()

    def slice(self, frame_type, frame_num, idr_id, info, coef):
        info = np.ascontiguousarray(info, MBINFO); coef = np.ascontiguousarray(coef, MBCOEF)
        n = lib().b2h_write_slice(self.e, C.addressof(self.seq), frame_type, frame_num, idr_id, _p(info), _p(coef),
                                  _p(self.buf), self.buf.size)
        assert n > 0, "slice writer overflow"
        return self.buf[:n].tobytes()


def encode_sequence(frames, w, h, qp=26, merange=16, subpel=1, intra_in_p=1, gop=32, fps=(30, 1), deblock=0, cabac=0, transform8x8=0, partitions=0,
                    deblock_offsets=(0, 0)):
    """frames: iterable of (y,u,v).  Returns (annexb_bytes, [recon OFrame], [info], [coef])."""
    prm = Params(qp, merange, subpel, intra_in_p, deblock, transform8x8, partitions, deblock_offsets[0], deblock_offsets[1])
    ent = Entropy(w, h, qp, fps, deblock=deblock, cabac=cabac, transform8x8=transform8x8, deblock_offsets=deblock_offsets)
    out = bytearray()
    sc = b"\x00\x00\x00\x01"
    recons, infos, coefs = [], [], []
    prev = None; prev_mv = None; idr = 0
    for t, (y, u, v) in enumerate(frames):
        cur = OFrame(w, h).load(y, u, v)
        rec = OFrame(w, h)
        is_i = (t % gop) == 0
        if is_i:
            out += sc + ent.sps() + sc + ent.pps()
            info, coef = encode_frame(prm, 0, cur, None, rec, None)
            out += sc + ent.slice(0, 0, idr, info, coef); idr += 1
        else:
            info, coef = encode_frame(prm, 1, cur, prev, rec, prev_mv)
            out += sc + ent.slice(1, t % gop, 0, info, coef)
        prev_mv = np.zeros(info.size, MV); prev_mv["x"] = info["mvx"]; prev_mv["y"] = info["mvy"]
        prev = rec
        recons.append(rec); infos.append(info); coefs.append(coef)
    return bytes(out), recons, infos, coefs


def decode_luma(annexb: bytes, path="/tmp/b2_dec.h264"):
    """decode an Annex-B stream with libavcodec's H.264 decoder (through OpenCV); exact luma planes."""
    import cv2
    with open(path, "wb") as f:
        f.write(annexb)
    cap = cv2.VideoCapture(path, cv2.CAP_FFMPEG)
    cap.set(cv2.CAP_PROP_CONVERT_RGB, 0)
    out = []
    while True:
        ok, fr = cap.read()
        if not ok:
            break
        out.append(fr.copy())
    cap.release()
    return out


# ---- full YUV decode through libavcodec (ctypes), for chroma drift checks --------------------------
def _avlibs():
    import glob
    import cv2  # noqa: F401  (loads the bundled FFmpeg libs so that siblings resolve)
    d = os.path.join(os.path.dirname(cv2.__file__), "..", "opencv_python_headless.libs")
    avutil = C.CDLL(glob.glob(os.path.join(d, "libavutil-*.so*"))[0])
    avcodec = C.CDLL(glob.glob(os.path.join(d, "libavcodec-*.so*"))[0])
    return avutil, avcodec


def decode_yuv(access_units):
    """access_units: list of Annex-B byte strings (one picture each, SPS/PPS may be prepended).
    Returns a list of (y,u,v) uint8 arrays decoded by libavcodec's native H.264 decoder."""
    avutil, avc = _avlibs()
    avc.avcodec_find_decoder.restype = C.c_void_p
    avc.avcodec_alloc_context3.restype = C.c_void_p; avc.avcodec_alloc_context3.argtypes = [C.c_void_p]
    avc.avcodec_open2.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    avc.av_packet_alloc.restype = C.c_void_p
    avutil.av_frame_alloc.restype = C.c_void_p
    avc.avcodec_send_packet.argtypes = [C.c_void_p, C.c_void_p]
    avc.avcodec_receive_frame.argtypes = [C.c_void_p, C.c_void_p]
    avc.avcodec_free_context.argtypes = [C.c_void_p]
    codec = avc.avcodec_find_decoder(27)            # AV_CODEC_ID_H264
    assert codec
    ctx = avc.avcodec_alloc_context3(codec)
    assert avc.avcodec_open2(ctx, codec, None) == 0
    pkt = avc.av_packet_alloc(); frm = avutil.av_frame_alloc()
    out = []

    def drain():
        while avc.avcodec_receive_frame(ctx, frm) == 0:
            data = (C.c_void_p * 8).from_address(frm)
            ls = (C.c_int * 8).from_address(frm + 64)
            w = C.c_int.from_address(frm + 104).value; h = C.c_int.from_address(frm + 108).value
            planes = []
            for i, (pw, ph) in enumerate([(w, h), ((w + 1) // 2, (h + 1) // 2), ((w + 1) // 2, (h + 1) // 2)]):
                buf = (C.c_uint8 * (ls[i] * ph)).from_address(data[i])
                planes.append(np.frombuffer(buf, np.uint8).reshape(ph, ls[i])[:, :pw].copy())
            out.append(tuple(planes))

    keep = []
    for au in access_units:
        b = np.frombuffer(au + b"\0" * 64, np.uint8).copy(); keep.append(b)
        C.c_void_p.from_address(pkt + 24).value = b.ctypes.data      # AVPacket.data
        C.c_int.from_address(pkt + 32).value = len(au)               # AVPacket.size
        rc = avc.avcodec_send_packet(ctx, pkt)
        assert rc == 0, "avcodec_send_packet failed %d" % rc
        drain()
    avc.avcodec_send_packet(ctx, None)
    drain()
    ctxp = C.c_void_p(ctx)
    avc.avcodec_free_context(C.byref(ctxp))
    return out


def split_access_units(annexb: bytes):
    """split an Annex-B stream into access units (each ends with a slice NAL type 1 or 5)."""
    parts = annexb.split(b"\x00\x00\x00\x01")[1:]
    aus, cur = [], b""
    for p in parts:
        cur += b"\x00\x00\x00\x01" + p
        if (p[0] & 31) in (1, 5):
            aus.append(cur); cur = b""
    return aus


FMT = {"yuv420p": 0, "nv12": 1, "yuyv422": 2, "uyvy422": 3, "bgr24": 4, "rgb24": 5, "yuv422p": 6, "yuv411p": 7}


def convert_to_i420(fmt, w, h, planes):
    """planes: list of 2-D uint8 arrays (their row length is the stride).  Returns (y,u,v)."""
    cw, ch = (w + 1) // 2, (h + 1) // 2
    planes = [np.ascontiguousarray(p, np.uint8) for p in planes]
    y = np.zeros((h, w), np.uint8); u = np.zeros((ch, cw), np.uint8); v = np.zeros((ch, cw), np.uint8)
    sp = (C.c_void_p * 4)(*([p.ctypes.data for p in planes] + [None] * (4 - len(planes))))
    ss = (C.c_int * 4)(*([p.shape[1] for p in planes] + [0] * (4 - len(planes))))
    dp = (C.c_void_p * 3)(y.ctypes.data, u.ctypes.data, v.ctypes.data)
    ds = (C.c_int * 3)(w, cw, cw)
    rc = lib().b2o_convert_to_i420(FMT[fmt], w, h, sp, ss, dp, ds)
    if rc != 0:
        raise ValueError("unsupported conversion")
    return y, u, v


# ---- row N4: pre-filters (oracle/b2o_filters.c; parity unpinned, see there) ------------------------------------------------
def _plane_dims(fmt, w, h):
    if fmt == "yuv420p":
        return [(w, h), ((w + 1) // 2, (h + 1) // 2), ((w + 1) // 2, (h + 1) // 2)]
    if fmt == "yuv422p":
        return [(w, h), ((w + 1) // 2, h), ((w + 1) // 2, h)]
    return [(w, h), ((w + 3) // 4, h), ((w + 3) // 4, h)]


class Hqdn3d:
    """stateful denoiser over a sequence of (y,u,v) frames"""

    def __init__(self, w, h, fmt="yuv420p", ls=4.0, cs=None, lt=None, ct=None):
        cs = 3.0 * ls / 4.0 if cs is None else cs
        lt = 6.0 * ls / 4.0 if lt is None else lt
        ct = (lt * cs / ls if ls > 0 else 0.0) if ct is None else ct
        L = lib()
        L.b2o_hqdn3d_coefs.argtypes = [C.c_double, C.c_void_p]
        self.ct = []
        for s in (ls, lt, cs, ct):
            t = np.zeros(8192, np.int32); L.b2o_hqdn3d_coefs(float(s), _p(t)); self.ct.append(t)
        self.dims = _plane_dims(fmt, w, h)
        self.ant = [np.zeros(pw * ph, np.uint16) for pw, ph in self.dims]
        self.first = 1

    def __call__(self, frame):
        out = []
        for p, (pw, ph) in enumerate(self.dims):
            src = np.ascontiguousarray(frame[p], np.uint8); dst = np.zeros((ph, pw), np.uint8)
            lib().b2o_hqdn3d_plane(_p(src), pw, _p(dst), pw, pw, ph, _p(self.ant[p]), self.first, _p(self.ct[2 if p else 0]), _p(self.ct[3 if p else 1]))
            out.append(dst)
        self.first = 0
        return tuple(out)


def yadif_sequence(frames, w, h, fmt="yuv420p", tff=1):
    """yadif mode 0 over a whole sequence: first frame is its own predecessor, last frame its own successor"""
    dims = _plane_dims(fmt, w, h)
    out = []
    for t in range(len(frames)):
        prev, cur, nxt = frames[max(t - 1, 0)], frames[t], frames[min(t + 1, len(frames) - 1)]
        planes = []
        for p, (pw, ph) in enumerate(dims):
            a, b, c = [np.ascontiguousarray(f[p], np.uint8) for f in (prev, cur, nxt)]
            dst = np.zeros((ph, pw), np.uint8)
            lib().b2o_yadif_plane(_p(a), _p(b), _p(c), pw, _p(dst), pw, pw, ph, tff)
            planes.append(dst)
        out.append(tuple(planes))
    return out
