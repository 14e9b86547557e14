"""ctypes binding of libb2enc.so -- the Python-side harness over the C-ABI in include/*.h.
The library is CUDA-only: there is no CPU fallback, loading or calling fails loudly when the
shared object or a GPU is missing."""
import ctypes as C
import os
import subprocess
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

MV = np.dtype([("x", "<i2"), ("y", "<i2")])
MBINFO = np.dtype([("mvx", "<i2"), ("mvy", "<i2"), ("mb_type", "u1"), ("i16_mode", "u1"),
                   ("chroma_mode", "u1"), ("cbp", "u1"), ("i4_mode", "u1", (16,)),
                   ("cost", "<u4"), ("nnz_mask", "<u4"), ("mv8", "<i2", (3, 2)), ("part", "u1"),
                   ("transform8x8", "u1"), ("i8_modes", "<u2")])
MBCOEF = np.dtype([("blk", "<i2", (26, 16))])


def so_path():
    return os.environ.get("B2ENC_LIB") or os.path.join(_HERE, "libb2enc.so")      # B2ENC_LIB: a libb2enc.so built elsewhere


def build(force=False):
    if force or not os.path.exists(so_path()):
        subprocess.check_call(["make", "-C", _HERE, "-s"] + (["-B"] if force else []))
    return so_path()


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(so_path()):
            raise RuntimeError("libb2enc.so is not built (run `make -C video-encoder_b200`); "
                               "there is no CPU fallback for the encode stage")
        _LIB = C.CDLL(so_path())
        _LIB.b2_bench_vabsdiff4_peak.restype = C.c_double
        _LIB.b2_bench_vabsdiff4_peak.argtypes = [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double)]
    return _LIB


def require_gpu():
    if lib().b2_device_count() <= 0:
        raise RuntimeError("b2enc: no CUDA device visible; the encode stage has no CPU fallback")


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def me_fullpel(cur_y, ref_y, merange, pmv=None, lam=0, iters=0):
    """cur_y/ref_y: uint8 [n,h,w] (or [h,w]).  Returns (mv[n,mbs], cost[n,mbs], kernel_ms|None)."""
    require_gpu()
    cur_y = np.ascontiguousarray(cur_y, np.uint8); ref_y = np.ascontiguousarray(ref_y, np.uint8)
    if cur_y.ndim == 2:
        cur_y = cur_y[None]; ref_y = ref_y[None]
    n, h, w = cur_y.shape
    nmb = (w // 16) * (h // 16)
    mv = np.zeros((n, nmb), MV); cost = np.zeros((n, nmb), np.uint32)
    if pmv is not None:
        pmv = np.ascontiguousarray(pmv, MV).reshape(n, nmb)
    ms = C.c_float(0)
    rc = lib().b2k_me_fullpel(_p(cur_y), _p(ref_y), w, h, n, merange, _p(pmv), lam, _p(mv), _p(cost),
                              iters, C.byref(ms) if iters > 0 else None)
    if rc != 0:
        raise RuntimeError("b2k_me_fullpel failed (%d)" % rc)
    return mv, cost, (ms.value if iters > 0 else None)


def me_fullpel_pruned(cur_y, ref_y, merange, pmv=None, lam=0, iters=0):
    """K1 with lossless pruning (K1a block sums + successive elimination).  Returns (mv, cost, stats) with stats =
    {"kernel_ms", "sums_ms" (None without iters), "swept", "all"}: candidate vectors evaluated / of the exhaustive search."""
    require_gpu()
    cur_y = np.ascontiguousarray(cur_y, np.uint8); ref_y = np.ascontiguousarray(ref_y, np.uint8)
    if cur_y.ndim == 2:
        cur_y = cur_y[None]; ref_y = ref_y[None]
    n, h, w = cur_y.shape
    nmb = (w // 16) * (h // 16)
    mv = np.zeros((n, nmb), MV); cost = np.zeros((n, nmb), np.uint32)
    if pmv is not None:
        pmv = np.ascontiguousarray(pmv, MV).reshape(n, nmb)
    ms = C.c_float(0); sms = C.c_float(0); swept = C.c_ulonglong(0); every = C.c_ulonglong(0)
    L = lib()
    L.b2k_me_fullpel_pruned.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
                                        C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    rc = L.b2k_me_fullpel_pruned(_p(cur_y), _p(ref_y), w, h, n, merange, _p(pmv), lam, _p(mv), _p(cost), iters,
                                 C.addressof(ms) if iters > 0 else None, C.addressof(sms), C.addressof(swept), C.addressof(every))
    if rc != 0:
        raise RuntimeError("b2k_me_fullpel_pruned failed (%d)" % rc)
    return mv, cost, {"kernel_ms": ms.value if iters > 0 else None, "sums_ms": sms.value if iters > 0 else None,
                      "swept": swept.value, "all": every.value}


def block_sums(y, ks=1):
    """K1a alone: y uint8 [n,h,w] -> (min, max) u16 arrays [n,rows,pitch] over `ks` rows of the 16x16 block sums of the padded planes
    (see b2k_block_sums); ks=1: both are the plain block sums"""
    require_gpu()
    y = np.ascontiguousarray(y, np.uint8)
    if y.ndim == 2:
        y = y[None]
    n, h, w = y.shape
    pitch = C.c_int(0); rows = C.c_int(0)
    L = lib()
    L.b2k_block_sums.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    if L.b2k_block_sums(_p(y), w, h, n, ks, None, C.addressof(pitch), C.addressof(rows)) != 0:
        raise RuntimeError("b2k_block_sums failed")
    out = np.zeros((n, rows.value, pitch.value), np.uint32)
    if L.b2k_block_sums(_p(y), w, h, n, ks, _p(out), None, None) != 0:
        raise RuntimeError("b2k_block_sums failed")
    return (out & 0xffff).astype(np.uint16), (out >> 16).astype(np.uint16)


PAD, PADC = 64, 32                     # B2_PAD / B2_PADC (include/b2enc_types.h)


def padded_layout(w, h):
    """(pitch, rows, pitchc, rowsc) of the device planes of a coded size w x h (b2_padded_layout, csrc/b2_internal.h)"""
    return w + 2 * PAD, h + 2 * PAD, (w // 2 + 2 * PADC + 15) & ~15, h // 2 + 2 * PADC


def _deblock_lib():
    L = lib()
    L.b2k_deblock.argtypes = [C.c_void_p] * 3 + [C.c_int] * 6 + [C.c_void_p] * 4
    return L


def deblock_shape(w, h, nframes):
    """K8's launch shape for nframes frames of coded size w x h: (wavefront 0/1, CTAs per frame, rounds per warp)"""
    out = [C.c_int(0) for _ in range(3)]
    if _deblock_lib().b2k_deblock(None, None, None, w, h, nframes, 26, 0, 0, None, *[C.addressof(o) for o in out]) != 0:
        raise RuntimeError("b2k_deblock failed")
    return tuple(o.value for o in out)


def deblock(y, u, v, info, qp, alpha_off=0, beta_off=0):
    """K8 alone (b2k_deblock): y [n, h + 2*PAD, w + 2*PAD], u/v [n, h/2 + 2*PADC, pitchc] uint8 planes in the engine's padded
    layout (see padded_layout), info MBINFO [n, mbs].  Returns (filtered copies of y, u, v, (wavefront, ncta, rounds))."""
    require_gpu()
    y, u, v = (np.array(p, np.uint8, order="C", copy=True) for p in (y, u, v))
    n = y.shape[0]
    w, h = y.shape[2] - 2 * PAD, y.shape[1] - 2 * PAD
    pitch, rows, pitchc, rowsc = padded_layout(w, h)
    if y.shape != (n, rows, pitch) or u.shape != (n, rowsc, pitchc) or v.shape != u.shape:
        raise ValueError("planes are not in the padded layout of %dx%d" % (w, h))
    info = np.ascontiguousarray(info, MBINFO).reshape(n, (w // 16) * (h // 16))
    out = [C.c_int(0) for _ in range(3)]
    if _deblock_lib().b2k_deblock(_p(y), _p(u), _p(v), w, h, n, qp, alpha_off, beta_off, _p(info), *[C.addressof(o) for o in out]) != 0:
        raise RuntimeError("b2k_deblock failed")
    return y, u, v, tuple(o.value for o in out)


def _intra_recon_lib():
    L = lib()
    L.b2k_intra_recon.argtypes = [C.c_void_p] * 6 + [C.c_int] * 6 + [C.c_void_p] * 5
    return L


def intra_recon_shape(w, h, all_intra, slices=1):
    """K7's launch shape for frames of coded size w x h cut into `slices` row-aligned slices: (CTAs per (frame, slice), tasks of
    the longest diagonal per warp, dynamic shared memory bytes per CTA), for the tallest slice"""
    out = [C.c_int(0) for _ in range(3)]
    if _intra_recon_lib().b2k_intra_recon(None, None, None, None, None, None, w, h, 1, slices, 26, int(all_intra), None, None,
                                          *[C.addressof(o) for o in out]) != 0:
        raise RuntimeError("b2k_intra_recon failed")
    return tuple(o.value for o in out)


def intra_recon(cur, rec, info, coef, qp, all_intra, slices=1):
    """K7 alone (b2k_intra_recon): cur / rec = (y, u, v) uint8 planes [n, rows, pitch] in the engine's padded layout (see
    padded_layout), info MBINFO [n, mbs], coef MBCOEF [n, mbs], frames of `slices` row-aligned slices.  Returns (copies of rec y,
    u, v, info, coef after the launch, (ncta, rounds, dyn_smem))."""
    require_gpu()
    cy, cu, cv = (np.ascontiguousarray(p, np.uint8) for p in cur)
    ry, ru, rv = (np.array(p, np.uint8, order="C", copy=True) for p in rec)
    n = cy.shape[0]
    w, h = cy.shape[2] - 2 * PAD, cy.shape[1] - 2 * PAD
    pitch, rows, pitchc, rowsc = padded_layout(w, h)
    for p, shape in ((cy, (n, rows, pitch)), (ry, (n, rows, pitch)), (cu, (n, rowsc, pitchc)), (cv, (n, rowsc, pitchc)),
                     (ru, (n, rowsc, pitchc)), (rv, (n, rowsc, pitchc))):
        if p.shape != shape:
            raise ValueError("planes are not in the padded layout of %dx%d" % (w, h))
    nmb = (w // 16) * (h // 16)
    info = np.array(info, MBINFO, order="C", copy=True).reshape(n, nmb)
    coef = np.array(coef, MBCOEF, order="C", copy=True).reshape(n, nmb)
    out = [C.c_int(0) for _ in range(3)]
    if _intra_recon_lib().b2k_intra_recon(_p(cy), _p(cu), _p(cv), _p(ry), _p(ru), _p(rv), w, h, n, slices, qp, int(all_intra), _p(info), _p(coef),
                                          *[C.addressof(o) for o in out]) != 0:
        raise RuntimeError("b2k_intra_recon failed")
    return ry, ru, rv, info, coef, tuple(o.value for o in out)


def k1_prune_rows(merange):
    return lib().b2_k1_prune_rows(merange)


def me_fullpel_parts(cur_y, ref_y, merange, pmv=None, lam=0, iters=0):
    """K1 partition variant: returns (mv9[n,mbs,9], cost9[n,mbs,9], kernel_ms|None)"""
    require_gpu()
    cur_y = np.ascontiguousarray(cur_y, np.uint8); ref_y = np.ascontiguousarray(ref_y, np.uint8)
    if cur_y.ndim == 2:
        cur_y = cur_y[None]; ref_y = ref_y[None]
    n, h, w = cur_y.shape
    nmb = (w // 16) * (h // 16)
    mv = np.zeros((n, nmb, 9), MV); cost = np.zeros((n, nmb, 9), np.uint32)
    if pmv is not None:
        pmv = np.ascontiguousarray(pmv, MV).reshape(n, nmb)
    ms = C.c_float(0)
    rc = lib().b2k_me_fullpel_parts(_p(cur_y), _p(ref_y), w, h, n, merange, _p(pmv), lam, _p(mv), _p(cost),
                                    iters, C.byref(ms) if iters > 0 else None)
    if rc != 0:
        raise RuntimeError("b2k_me_fullpel_parts failed (%d)" % rc)
    return mv, cost, (ms.value if iters > 0 else None)


def vabsdiff4_peak(device=0, outer=256, reps=5):
    require_gpu()
    ms = C.c_double(0)
    rate = lib().b2_bench_vabsdiff4_peak(device, outer, reps, C.byref(ms))
    if rate <= 0:
        raise RuntimeError("vabsdiff4 microbenchmark failed")
    return rate, ms.value


# ---- engine binding (include/b2enc_engine.h) ----------------------------------------------------------
FMT = {"yuv420p": 0, "nv12": 1, "yuyv422": 2, "uyvy422": 3, "bgr24": 4, "rgb24": 5, "yuv422p": 6, "yuv411p": 7}
FRAME_I, FRAME_P = 0, 1
KERNEL_NAMES = ["K0 convert", "K6 border(cur)", "K1 full-pel SAD", "K2 sub-pel SATD", "K3 intra analyse",
                "K5 decide+inter recon", "K7 intra recon", "K6 border(recon)", "K8 deblock", "K9 pack levels"]


def bind_to_gpu_numa(device):
    """Pin this process to the CPUs of the NUMA node the GPU hangs off (sysfs local_cpulist of its PCI function), so that
    the pinned staging buffers are allocated next to the PCIe root the copies go through.  Returns the cpu list or None."""
    try:
        L = lib()
        buf = C.create_string_buffer(32)
        L.b2_device_pci_bus_id.argtypes = [C.c_int, C.c_char_p, C.c_int]
        if L.b2_device_pci_bus_id(device, buf, 32) != 0:
            return None
        bus = buf.value.decode().lower()
        path = "/sys/bus/pci/devices/%s/local_cpulist" % bus
        if not os.path.exists(path):
            path = "/sys/bus/pci/devices/%s/local_cpulist" % bus[4:] if len(bus) > 12 else path
        cpus = set()
        for part in open(path).read().strip().split(","):
            if "-" in part:
                a, b = part.split("-"); cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return sorted(cpus)
    except Exception:
        pass
    return None


def coef_present(info):
    """vectorised b2_coef_present (include/b2enc_types.h): 26-bit block-presence mask per macroblock"""
    m = info["nnz_mask"].astype(np.uint32)
    luma = m & 0xffff
    t8 = info["transform8x8"] != 0
    for q in range(4):
        quad = (luma >> (4 * q)) & 15
        luma = np.where(t8 & (quad != 0), luma | (15 << (4 * q)), luma)
    return (luma | (m & 0x01ff0000) | np.where((m & 0x06000000) != 0, 1 << 25, 0)).astype(np.uint32)


def shipped_info(info):
    """test helper: what is left of an MBINFO array after the 24-byte records of the packed copy-out (b2_mbinfo_packed_t,
    include/b2enc_types.h): `cost`, `i8_modes` and the intra analysis modes of inter macroblocks are not shipped"""
    out = np.array(info, copy=True)
    out["cost"] = 0; out["i8_modes"] = 0
    inter = out["mb_type"] == 0
    out["i4_mode"][inter] = 0; out["i16_mode"][inter] = 0; out["chroma_mode"][inter] = 0
    out["mv8"][~inter] = 0
    out["transform8x8"] = (out["transform8x8"] != 0).astype(np.uint8)
    return out


def pack_levels(info, coef):
    """test helper: the packed stream K9 produces, built on the host from a dense MBCOEF array"""
    pm = coef_present(info)
    bits = ((pm[:, None] >> np.arange(26, dtype=np.uint32)[None, :]) & 1).astype(bool)
    return np.frombuffer(np.ascontiguousarray(coef["blk"][bits]).tobytes(), np.uint8)


def unpack_levels(info, packed):
    """test helper: dense MBCOEF array from the packed stream (harness only; the product's host stage reads it in place)"""
    coef = np.zeros(info.size, MBCOEF)
    pm = coef_present(info)
    bits = ((pm[:, None] >> np.arange(26, dtype=np.uint32)[None, :]) & 1).astype(bool)
    blocks = np.frombuffer(packed.tobytes(), "<i2").reshape(-1, 16)
    assert blocks.shape[0] == int(bits.sum()), "packed stream size does not match the presence masks"
    coef["blk"][bits] = blocks
    return coef


class EngineCfg(C.Structure):
    _fields_ = [("device", C.c_int), ("width", C.c_int), ("height", C.c_int), ("slots", C.c_int), ("in_fmt", C.c_int),
                ("in_ring", C.c_int), ("merange", C.c_int), ("qp", C.c_int), ("subpel", C.c_int), ("intra_in_p", C.c_int),
                ("profile", C.c_int), ("streams", C.c_int), ("deblock", C.c_int), ("transform8x8", C.c_int), ("partitions", C.c_int), ("pack_levels", C.c_int),
                ("deblock_alpha", C.c_int), ("deblock_beta", C.c_int), ("me_prune", C.c_int), ("slices", C.c_int)]


class Engine:
    """One GPU's encode-stage engine: `slots` closed GOPs / streams advanced in lock-step."""

    def __init__(self, width, height, slots=1, fmt="yuv420p", ring=1, merange=16, qp=26, subpel=1, intra_in_p=1,
                 device=0, profile=0, streams=0, deblock=0, transform8x8=0, pack_levels=0, partitions=0, deblock_offsets=(0, 0),
                 me_prune=0, slices=1):
        require_gpu()
        L = lib()
        L.b2_engine_create.restype = C.c_void_p
        L.b2_engine_host_input.restype = C.c_void_p
        L.b2_engine_info.restype = C.c_void_p; L.b2_engine_coef.restype = C.c_void_p
        L.b2_engine_input_bytes.restype = C.c_size_t; L.b2_engine_result_bytes.restype = C.c_size_t
        L.b2_engine_launch_count.restype = C.c_long
        for fn in ("b2_engine_destroy", "b2_engine_input_bytes", "b2_engine_result_bytes", "b2_engine_sync",
                   "b2_engine_timer_start", "b2_engine_profile_reset", "b2_engine_launch_count"):
            getattr(L, fn).argtypes = [C.c_void_p]
        L.b2_engine_host_input.argtypes = [C.c_void_p, C.c_int, C.c_int]
        L.b2_engine_put_frame.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        L.b2_engine_put_frame_direct.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        L.b2_engine_h2d.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
        L.b2_engine_encode.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
        L.b2_engine_d2h.argtypes = [C.c_void_p, C.c_int]
        L.b2_engine_groups.argtypes = [C.c_void_p]
        L.b2_engine_group_range.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.b2_engine_encode_group.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
        L.b2_engine_d2h_group.argtypes = [C.c_void_p, C.c_int]
        L.b2_engine_group_result_set.argtypes = [C.c_void_p, C.c_int]
        L.b2_engine_group_done.argtypes = [C.c_void_p, C.c_int, C.c_int]
        L.b2_engine_group_wait.argtypes = [C.c_void_p, C.c_int, C.c_int]
        L.b2_engine_info_set.restype = C.c_void_p; L.b2_engine_info_set.argtypes = [C.c_void_p, C.c_int, C.c_int]
        L.b2_engine_packed_set.restype = C.c_void_p; L.b2_engine_packed_set.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_size_t)]
        L.b2_engine_put_picture.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        L.b2_engine_set_input_format.argtypes = [C.c_void_p, C.c_int]
        L.b2_engine_info.argtypes = [C.c_void_p, C.c_int]; L.b2_engine_coef.argtypes = [C.c_void_p, C.c_int]
        L.b2_engine_packed.restype = C.c_void_p; L.b2_engine_packed.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_size_t)]
        L.b2_engine_packed_bytes_total.restype = C.c_longlong; L.b2_engine_packed_bytes_total.argtypes = [C.c_void_p]
        L.b2_engine_get_recon.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.b2_engine_get_cur.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.b2_engine_get_stage.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        L.b2_engine_geometry.argtypes = [C.c_void_p] + [C.POINTER(C.c_int)] * 4
        L.b2_engine_timer_stop.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
        L.b2_engine_kernel_ms.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_long)]
        self.L = L
        self.cfg = EngineCfg(device, width, height, slots, FMT[fmt] if isinstance(fmt, str) else fmt, ring, merange, qp,
                             subpel, intra_in_p, profile, streams, deblock, transform8x8, partitions, pack_levels,
                             deblock_offsets[0], deblock_offsets[1], me_prune, slices)
        L.b2_engine_k1_stats.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        self.h = L.b2_engine_create(C.byref(self.cfg))
        if not self.h:
            raise RuntimeError("b2_engine_create failed")
        g = [C.c_int() for _ in range(4)]
        L.b2_engine_geometry(self.h, *[C.byref(x) for x in g])
        self.mbw, self.mbh, self.w16, self.h16 = [x.value for x in g]
        self.nmb = self.mbw * self.mbh
        self.width, self.height, self.slots, self.ring = width, height, slots, ring
        self.in_bytes = L.b2_engine_input_bytes(self.h)
        self.result_bytes = L.b2_engine_result_bytes(self.h)

    def k1_stats(self):
        """me_prune: (candidate vectors the pruned search evaluated, candidates of the exhaustive search) since creation; None when off"""
        a = C.c_ulonglong(0); b = C.c_ulonglong(0)
        if self.L.b2_engine_k1_stats(self.h, C.addressof(a), C.addressof(b)) != 0:
            return None
        return a.value, b.value

    def close(self):
        if self.h:
            self.L.b2_engine_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc, what):
        if rc != 0:
            raise RuntimeError("%s failed (%d)" % (what, rc))

    def host_input(self, slot, ring=0):
        """numpy view of the pinned staging buffer of (slot, ring)"""
        p = self.L.b2_engine_host_input(self.h, slot, ring)
        return np.frombuffer((C.c_uint8 * self.in_bytes).from_address(p), np.uint8)

    def put_frame(self, slot, ring, planes):
        planes = [np.ascontiguousarray(p, np.uint8) for p in planes]
        sp = (C.c_void_p * 4)(*([p.ctypes.data for p in planes] + [None] * (4 - len(planes))))
        ss = (C.c_int * 4)(*([p.shape[1] for p in planes] + [0] * (4 - len(planes))))
        self._ck(self.L.b2_engine_put_frame(self.h, slot, ring, sp, ss), "put_frame")

    def put_frame_direct(self, slot, ring, planes):
        """planes: uint8 arrays (any host memory); returns 0 when they were DMA'd straight into the device ring, 1 when the
        source is not page-locked (nothing copied: use put_frame)"""
        sp = (C.c_void_p * 4)(*([p.ctypes.data for p in planes] + [None] * (4 - len(planes))))
        ss = (C.c_int * 4)(*([p.strides[0] for p in planes] + [0] * (4 - len(planes))))
        rc = self.L.b2_engine_put_frame_direct(self.h, slot, ring, sp, ss)
        if rc < 0: self._ck(rc, "put_frame_direct")
        return rc

    def h2d(self, slot0=0, nslots=None, ring=0):
        self._ck(self.L.b2_engine_h2d(self.h, slot0, self.slots if nslots is None else nslots, ring), "h2d")

    def encode(self, frame_type, nslots=None, ring=0):
        self._ck(self.L.b2_engine_encode(self.h, frame_type, self.slots if nslots is None else nslots, ring), "encode")

    def groups(self):
        out = []
        for g in range(self.L.b2_engine_groups(self.h)):
            a, b = C.c_int(), C.c_int()
            self.L.b2_engine_group_range(self.h, g, C.byref(a), C.byref(b))
            out.append((a.value, b.value))
        return out

    def encode_group(self, group, frame_type, ring=0):
        self._ck(self.L.b2_engine_encode_group(self.h, group, frame_type, ring), "encode_group")

    def d2h_group(self, group):
        self._ck(self.L.b2_engine_d2h_group(self.h, group), "d2h_group")

    def d2h(self, nslots=None):
        self._ck(self.L.b2_engine_d2h(self.h, self.slots if nslots is None else nslots), "d2h")

    def put_picture(self, slot, ring, planes):
        """b2_engine_put_picture: planes = 2-D uint8 arrays (row length = stride) in any host memory"""
        sp = (C.c_void_p * 4)(*([p.ctypes.data for p in planes] + [None] * (4 - len(planes))))
        ss = (C.c_int * 4)(*([p.strides[0] for p in planes] + [0] * (4 - len(planes))))
        self._ck(self.L.b2_engine_put_picture(self.h, slot, ring, sp, ss), "put_picture")

    def group_result_set(self, group):
        return self.L.b2_engine_group_result_set(self.h, group)

    def group_done(self, group, rset):
        return self.L.b2_engine_group_done(self.h, group, rset)

    def group_wait(self, group, rset):
        self._ck(self.L.b2_engine_group_wait(self.h, group, rset), "group_wait")

    def results_set(self, rset, slot):
        """(info copy, packed level stream copy) of result set `rset` of `slot` (pack_levels engines)"""
        pi = self.L.b2_engine_info_set(self.h, rset, slot)
        info = np.frombuffer((C.c_uint8 * (self.nmb * MBINFO.itemsize)).from_address(pi), MBINFO).copy()
        n = C.c_size_t(0)
        pp = self.L.b2_engine_packed_set(self.h, rset, slot, C.byref(n))
        packed = np.frombuffer((C.c_uint8 * n.value).from_address(pp), np.uint8).copy() if n.value else np.zeros(0, np.uint8)
        return info, packed

    def sync(self):
        self._ck(self.L.b2_engine_sync(self.h), "sync")

    def results(self, slot):
        """(info, coef) numpy views of the last fetched results of `slot` (pack_levels: coef is unpacked from the stream)"""
        pi = self.L.b2_engine_info(self.h, slot)
        info = np.frombuffer((C.c_uint8 * (self.nmb * MBINFO.itemsize)).from_address(pi), MBINFO)
        if self.cfg.pack_levels:
            return info, unpack_levels(info, self.packed(slot))
        pc = self.L.b2_engine_coef(self.h, slot)
        coef = np.frombuffer((C.c_uint8 * (self.nmb * 832)).from_address(pc), MBCOEF)
        return info, coef

    def packed(self, slot):
        """the slot's packed level stream (cfg.pack_levels) as a uint8 array"""
        n = C.c_size_t(0)
        p = self.L.b2_engine_packed(self.h, slot, C.byref(n))
        if not p:
            raise RuntimeError("engine was not created with pack_levels")
        return np.frombuffer((C.c_uint8 * n.value).from_address(p), np.uint8).copy() if n.value else np.zeros(0, np.uint8)

    def packed_bytes_total(self):
        return int(self.L.b2_engine_packed_bytes_total(self.h))

    def _planes(self, fn, slot):
        y = np.zeros((self.h16, self.w16), np.uint8)
        u = np.zeros((self.h16 // 2, self.w16 // 2), np.uint8); v = np.zeros_like(u)
        self._ck(fn(self.h, slot, _p(y), _p(u), _p(v)), "get planes")
        return y, u, v

    def recon(self, slot=0):
        return self._planes(self.L.b2_engine_get_recon, slot)

    def cur(self, slot=0):
        return self._planes(self.L.b2_engine_get_cur, slot)

    def stage(self, slot, what):
        out = np.zeros(self.nmb, MV if what in (0, 2) else np.uint32)
        self._ck(self.L.b2_engine_get_stage(self.h, slot, what, _p(out)), "get_stage")
        return out

    def timer_start(self):
        self._ck(self.L.b2_engine_timer_start(self.h), "timer_start")

    def timer_stop(self):
        ms = C.c_float(0)
        self._ck(self.L.b2_engine_timer_stop(self.h, C.byref(ms)), "timer_stop")
        return ms.value

    def kernel_ms(self):
        out = {}
        for i, n in enumerate(KERNEL_NAMES):
            ms = C.c_double(0); cnt = C.c_long(0)
            self._ck(self.L.b2_engine_kernel_ms(self.h, i, C.byref(ms), C.byref(cnt)), "kernel_ms")
            out[n] = (ms.value, cnt.value)
        return out

    def profile_reset(self):
        self.L.b2_engine_profile_reset(self.h)

    def launch_count(self):
        return self.L.b2_engine_launch_count(self.h)


# ---- drop-in boundary binding (include/b2enc.h): the x264 / swscale call subset of av_encode.c -------
class Param(C.Structure):
    class _Vui(C.Structure):
        _fields_ = [("i_sar_width", C.c_int), ("i_sar_height", C.c_int)]

    class _Rc(C.Structure):
        _fields_ = [("i_rc_method", C.c_int), ("f_rf_constant", C.c_float), ("i_qp_constant", C.c_int)]
    _fields_ = [("i_width", C.c_int), ("i_height", C.c_int), ("b_annexb", C.c_int), ("i_fps_num", C.c_int), ("i_fps_den", C.c_int),
                ("vui", _Vui), ("rc", _Rc), ("i_keyint_max", C.c_int), ("i_gop_slots", C.c_int), ("i_merange", C.c_int),
                ("b_subpel", C.c_int), ("b_intra_in_p", C.c_int), ("i_device", C.c_int), ("i_csp_in", C.c_int),
                ("b_deblocking_filter", C.c_int), ("b_cabac", C.c_int), ("b_transform_8x8", C.c_int), ("b_partitions", C.c_int),
                ("i_deblocking_filter_alphac0", C.c_int), ("i_deblocking_filter_beta", C.c_int), ("i_devices", C.c_int),
                ("b_me_prune", C.c_int), ("i_slice_count", C.c_int)]


class Image(C.Structure):
    _fields_ = [("i_csp", C.c_int), ("i_plane", C.c_int), ("i_stride", C.c_int * 4), ("plane", C.c_void_p * 4)]


class Picture(C.Structure):
    _fields_ = [("i_type", C.c_int), ("i_pts", C.c_int64), ("i_dts", C.c_int64), ("b_keyframe", C.c_int), ("img", Image),
                ("opaque", C.c_void_p)]


class Nal(C.Structure):
    _fields_ = [("i_ref_idc", C.c_int), ("i_type", C.c_int), ("i_payload", C.c_int), ("p_payload", C.c_void_p)]


def _dropin_lib(L=None):
    """argtypes of the drop-in boundary on `L` (default: libb2enc.so; the CPU host-logic tests pass their mock build)"""
    L = L or lib()
    L.b2_encoder_open.restype = C.c_void_p; L.b2_encoder_open.argtypes = [C.POINTER(Param)]
    L.b2_encoder_encode.argtypes = [C.c_void_p, C.POINTER(C.POINTER(Nal)), C.POINTER(C.c_int), C.POINTER(Picture), C.POINTER(Picture)]
    L.b2_encoder_delayed_frames.argtypes = [C.c_void_p]; L.b2_encoder_close.argtypes = [C.c_void_p]
    L.b2_param_default_preset.argtypes = [C.POINTER(Param), C.c_char_p, C.c_char_p]
    L.b2_param_apply_profile.argtypes = [C.POINTER(Param), C.c_char_p]
    L.b2_picture_alloc.argtypes = [C.POINTER(Picture), C.c_int, C.c_int, C.c_int]; L.b2_picture_clean.argtypes = [C.POINTER(Picture)]
    L.b2_sws_getContext.restype = C.c_void_p
    L.b2_sws_getContext.argtypes = [C.c_int] * 7 + [C.c_void_p, C.c_void_p, C.c_void_p]
    L.b2_sws_scale.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.b2_sws_freeContext.argtypes = [C.c_void_p]
    return L


def sws_convert(fmt, w, h, planes, dst_pad=0):
    """b2_sws_getContext + b2_sws_scale + b2_sws_freeContext, the way av_encode.c:427-430/545-547 uses them"""
    require_gpu()
    L = _dropin_lib()
    ctx = L.b2_sws_getContext(w, h, FMT[fmt], w, h, FMT["yuv420p"], 1, None, None, None)
    if not ctx:
        raise RuntimeError("b2_sws_getContext failed")
    cw, ch = (w + 1) // 2, (h + 1) // 2
    planes = [np.ascontiguousarray(p, np.uint8) for p in planes]
    y = np.zeros((h, w + dst_pad), np.uint8); u = np.zeros((ch, cw + dst_pad), np.uint8); v = np.zeros((ch, cw + dst_pad), np.uint8)
    sp = (C.c_void_p * 4)(*([p.ctypes.data for p in planes] + [None] * (4 - len(planes))))
    ss = (C.c_int * 4)(*([p.shape[1] for p in planes] + [0] * (4 - len(planes))))
    dp = (C.c_void_p * 4)(y.ctypes.data, u.ctypes.data, v.ctypes.data, None)
    ds = (C.c_int * 4)(y.shape[1], u.shape[1], v.shape[1], 0)
    r = L.b2_sws_scale(ctx, sp, ss, 0, h, dp, ds)
    L.b2_sws_freeContext(ctx)
    if r != h:
        raise RuntimeError("b2_sws_scale failed (%d)" % r)
    return y[:, :w], u[:, :cw], v[:, :cw]


class DropInEncoder:
    """Drives the b2_* mirror of the x264 API exactly like av_encode.c does (open :378-438, loop :968-975,
    drain :1076-1083)."""

    def __init__(self, w, h, preset="medium", tune="film", quality=26, profile=None, fps=(30, 1), annexb=0, library=None, **ext):
        if library is None:
            require_gpu()
        self.L = L = _dropin_lib(library)
        self.sws = None
        self.w, self.h = w, h
        p = Param()
        if L.b2_param_default_preset(C.byref(p), preset.encode() if preset else None, tune.encode() if tune else None) != 0:
            raise ValueError("bad preset/tune")
        p.i_width, p.i_height, p.b_annexb = w, h, annexb
        p.i_fps_num, p.i_fps_den = fps
        p.vui.i_sar_width = p.vui.i_sar_height = 1
        p.rc.i_rc_method = 1; p.rc.f_rf_constant = float(quality)
        for k, v in ext.items():
            setattr(p, k, v)
        if L.b2_param_apply_profile(C.byref(p), profile.encode() if profile else None) != 0:
            raise ValueError("bad profile")
        self.h_enc = L.b2_encoder_open(C.byref(p))
        if not self.h_enc:
            raise RuntimeError("b2_encoder_open failed")
        self.pic_in = Picture(); self.pic_out = Picture()
        if L.b2_picture_alloc(C.byref(self.pic_in), 1, w, h) != 0:
            raise MemoryError
        self.param = p

    def _fill(self, y, u, v):
        cw, ch = (self.w + 1) // 2, (self.h + 1) // 2
        for i, (a, ww, hh) in enumerate(((y, self.w, self.h), (u, cw, ch), (v, cw, ch))):
            dst = np.frombuffer((C.c_uint8 * (ww * hh)).from_address(self.pic_in.img.plane[i]), np.uint8).reshape(hh, ww)
            dst[:] = a

    def encode(self, frame, pts):
        """frame: (y,u,v) or None to flush.  Returns (size, [(type, bytes)], pts, dts, keyframe)."""
        nal = C.POINTER(Nal)(); n = C.c_int(0)
        if frame is not None:
            self._fill(*frame)
            self.pic_in.i_type = 0; self.pic_in.i_pts = pts
            size = self.L.b2_encoder_encode(self.h_enc, C.byref(nal), C.byref(n), C.byref(self.pic_in), C.byref(self.pic_out))
        else:
            size = self.L.b2_encoder_encode(self.h_enc, C.byref(nal), C.byref(n), None, C.byref(self.pic_out))
        nals = []
        if size > 0:
            base = nal[0].p_payload
            whole = C.string_at(base, size)
            off = 0
            for i in range(n.value):
                assert nal[i].p_payload == base + off, "NAL payloads are not contiguous"
                nals.append((nal[i].i_type, whole[off:off + nal[i].i_payload]))
                off += nal[i].i_payload
            assert off == size
        return size, nals, self.pic_out.i_pts, self.pic_out.i_dts, self.pic_out.b_keyframe

    def encode_raw(self, planes, pts):
        """hand over a picture in the encoder's i_csp_in format straight from the caller's own (pageable) planes: 2-D uint8
        arrays whose row length is the stride, as a decoder would deliver them.  Returns like encode()."""
        planes = [np.ascontiguousarray(p, np.uint8) for p in planes]
        pic = Picture()
        pic.i_type = 0; pic.i_pts = pts
        pic.img.i_csp = 0; pic.img.i_plane = len(planes)
        for i, a in enumerate(planes):
            pic.img.plane[i] = a.ctypes.data; pic.img.i_stride[i] = a.shape[1]
        nal = C.POINTER(Nal)(); n = C.c_int(0)
        size = self.L.b2_encoder_encode(self.h_enc, C.byref(nal), C.byref(n), C.byref(pic), C.byref(self.pic_out))
        nals = []
        if size > 0:
            base = nal[0].p_payload; whole = C.string_at(base, size); off = 0
            for i in range(n.value):
                nals.append((nal[i].i_type, whole[off:off + nal[i].i_payload])); off += nal[i].i_payload
        return size, nals, self.pic_out.i_pts, self.pic_out.i_dts, self.pic_out.b_keyframe

    def encode_via_sws(self, fmt, planes, pts, flags=1):
        """the reference's per-frame sequence (av_encode.c:543-547, :970): sws_scale the decoder's picture (strided planes in
        format `fmt`) INTO pic_in, then encode pic_in.  Returns like encode()."""
        if self.sws is None or self.sws[0] != (fmt, flags):
            if self.sws is not None:
                self.L.b2_sws_freeContext(self.sws[1])
            ctx = self.L.b2_sws_getContext(self.w, self.h, FMT[fmt], self.w, self.h, FMT["yuv420p"], flags, None, None, None)
            if not ctx:
                raise RuntimeError("b2_sws_getContext failed")
            self.sws = ((fmt, flags), ctx)
        planes = [np.ascontiguousarray(p, np.uint8) for p in planes]
        sp = (C.c_void_p * 4)(*([p.ctypes.data for p in planes] + [None] * (4 - len(planes))))
        ss = (C.c_int * 4)(*([p.shape[1] for p in planes] + [0] * (4 - len(planes))))
        dp = (C.c_void_p * 4)(*[self.pic_in.img.plane[i] for i in range(4)])
        ds = (C.c_int * 4)(*[self.pic_in.img.i_stride[i] for i in range(4)])
        if self.L.b2_sws_scale(self.sws[1], sp, ss, 0, self.h, dp, ds) != self.h:
            raise RuntimeError("b2_sws_scale failed")
        self.pic_in.i_type = 0; self.pic_in.i_pts = pts
        nal = C.POINTER(Nal)(); n = C.c_int(0)
        size = self.L.b2_encoder_encode(self.h_enc, C.byref(nal), C.byref(n), C.byref(self.pic_in), C.byref(self.pic_out))
        nals = []
        if size > 0:
            base = nal[0].p_payload; whole = C.string_at(base, size); off = 0
            for i in range(n.value):
                nals.append((nal[i].i_type, whole[off:off + nal[i].i_payload])); off += nal[i].i_payload
        return size, nals, self.pic_out.i_pts, self.pic_out.i_dts, self.pic_out.b_keyframe

    def delayed(self):
        return self.L.b2_encoder_delayed_frames(self.h_enc)

    def close(self):
        if self.sws is not None:
            self.L.b2_sws_freeContext(self.sws[1]); self.sws = None
        if self.h_enc:
            self.L.b2_picture_clean(C.byref(self.pic_in))
            self.L.b2_encoder_close(self.h_enc)
            self.h_enc = None


# ---- pre-filter stage binding (include/b2enc_filters.h) ---------------------------------------------------------------------
class FilterGraph:
    """push / poll / pull like the reference drives its libavfilter graph (av_encode.c:962, :525-560)"""

    def __init__(self, w, h, filters, fmt="yuv420p", device=0):
        require_gpu()
        L = self.L = lib()
        L.b2_filter_graph_create.restype = C.c_void_p
        L.b2_filter_graph_create.argtypes = [C.c_int, C.c_int, C.c_int, C.c_char_p, C.c_int]
        L.b2_filter_add_frame.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int]
        L.b2_filter_poll_frame.argtypes = [C.c_void_p]
        L.b2_filter_get_frame.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int64)]
        L.b2_filter_flush.argtypes = [C.c_void_p]; L.b2_filter_graph_free.argtypes = [C.c_void_p]
        self.g = L.b2_filter_graph_create(w, h, FMT[fmt], filters.encode() if filters is not None else None, device)
        if not self.g:
            raise RuntimeError("b2_filter_graph_create failed")
        cw = (w + 1) // 2 if fmt != "yuv411p" else (w + 3) // 4
        ch = (h + 1) // 2 if fmt == "yuv420p" else h
        self.dims = [(w, h), (cw, ch), (cw, ch)]

    def add(self, frame, pts=0, tff=1):
        planes = [np.ascontiguousarray(p, np.uint8) for p in frame]
        sp = (C.c_void_p * 3)(*[p.ctypes.data for p in planes]); ss = (C.c_int * 3)(*[p.shape[1] for p in planes])
        if self.L.b2_filter_add_frame(self.g, sp, ss, pts, tff) != 0:
            raise RuntimeError("b2_filter_add_frame failed")

    def poll(self):
        return self.L.b2_filter_poll_frame(self.g)

    def get(self, pad=0):
        out = [np.zeros((ph, pw + pad), np.uint8) for pw, ph in self.dims]
        dp = (C.c_void_p * 3)(*[p.ctypes.data for p in out]); ds = (C.c_int * 3)(*[p.shape[1] for p in out])
        pts = C.c_int64(0)
        r = self.L.b2_filter_get_frame(self.g, dp, ds, C.byref(pts))
        if r < 0:
            raise RuntimeError("b2_filter_get_frame failed")
        if r == 0:
            return None
        return tuple(o[:, :pw] for o, (pw, ph) in zip(out, self.dims)), pts.value

    def flush(self):
        if self.L.b2_filter_flush(self.g) != 0:
            raise RuntimeError("b2_filter_flush failed")

    def run(self, frames, tff=1):
        """whole sequence in, whole sequence out (frames in display order)"""
        out = []
        for t, f in enumerate(frames):
            self.add(f, pts=100 + t, tff=tff)
            while self.poll() > 0:
                out.append(self.get(pad=3))
        self.flush()
        while self.poll() > 0:
            out.append(self.get(pad=3))
        return out

    def close(self):
        if self.g:
            self.L.b2_filter_graph_free(self.g); self.g = None
