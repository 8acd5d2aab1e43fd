"""ctypes binding of libx265cu.so (include/x265_b200.h).  Host-side plumbing only: the arithmetic is
all in the CUDA library.  Raises CudaUnavailable instead of falling back when no GPU is present."""
import ctypes as C
import os

import numpy as np

from . import build as _build

P = C.c_void_p
I = C.c_int
I64 = C.c_int64
IP = C.c_ssize_t


class CudaUnavailable(RuntimeError):
    pass


class MeChroma(C.Structure):
    """x265cu_me_chroma (include/x265_b200.h)"""
    _fields_ = [("fencCb_dev", C.c_void_p), ("fencCr_dev", C.c_void_p), ("refCb_dev", C.c_void_p), ("refCr_dev", C.c_void_p),
                ("cstride", C.c_int)]


# job record layouts (must match include/x265_b200.h)
CMP_JOB = np.dtype([("a_off", "<i8"), ("b_off", "<i8"), ("a_stride", "<i4"), ("b_stride", "<i4"),
                    ("w", "<i2"), ("h", "<i2"), ("pad", "<i4")], align=True)
BLK_JOB = np.dtype([("d_off", "<i8"), ("a_off", "<i8"), ("b_off", "<i8"), ("d_stride", "<i4"), ("a_stride", "<i4"),
                    ("b_stride", "<i4"), ("w", "<i2"), ("h", "<i2"), ("p0", "<i4"), ("p1", "<i4"), ("p2", "<i4"), ("p3", "<i4")], align=True)
INTERP_JOB = np.dtype([("s_off", "<i8"), ("d_off", "<i8"), ("s_stride", "<i4"), ("d_stride", "<i4"), ("w", "<i2"), ("h", "<i2"),
                       ("idxX", "i1"), ("idxY", "i1"), ("rowExt", "i1"), ("ntaps", "i1")], align=True)
INTRA_JOB = np.dtype([("mode", "<i4"), ("bFilter", "<i4")], align=True)
PRED_JOB = np.dtype([("offset", "<i4"), ("pw", "<i2"), ("ph", "<i2"), ("ref0", "i1"), ("ref1", "i1"), ("cost", "u1"), ("flags", "u1"),
                     ("mv0", "<i2", 2), ("mv1", "<i2", 2)])
PRED_SAD, PRED_SATD, PRED_CHROMA, PRED_AVG_PP = 0, 1, 1, 2
ME_JOB = np.dtype([("offset", "<i4"), ("ref", "<i2"), ("pw", "i1"), ("ph", "i1"), ("mvmin", "<i2", 2), ("mvmax", "<i2", 2),
                   ("qmvp", "<i2", 2), ("mvc", "<i2", 8), ("numCand", "i1"), ("method", "i1"), ("subme", "i1"), ("merange", "i1")], align=True)
assert CMP_JOB.itemsize == 32 and BLK_JOB.itemsize == 56 and INTERP_JOB.itemsize == 32 and ME_JOB.itemsize == 40

OPS_CMP = dict(sad=0, satd=1, sa8d=2, sse_pp=3, sse_ss=4, ssd_s=5, var=6, psy=7)
OPS_BLK = dict(copy_pp=0, copy_ss=1, copy_sp=2, copy_ps=3, sub_ps=4, add_ps=5, pixelavg_pp=6, addAvg=7, p2s=8, transpose=9,
               blockfill_s=10, cpy2Dto1D_shl=11, cpy2Dto1D_shr=12, cpy1Dto2D_shl=13, cpy1Dto2D_shr=14, weight_pp=15,
               weight_sp=16, scale2D_64to32=17, dequant_normal=18)
OPS_INTERP = dict(hpp=0, hps=1, vpp=2, vps=3, vsp=4, vss=5, hvpp=6)
OPS_TR = dict(dct=0, idct=1, dst4=2, idst4=3)

_PROTOS = {
    "x265cu_device_count": (I, []),
    "x265cu_create": (P, [I]),
    "x265cu_destroy": (None, [P]),
    "x265cu_last_error": (C.c_char_p, []),
    "x265cu_sync": (I, [P]),
    "x265cu_stream": (P, [P]),
    "x265cu_malloc": (P, [P, C.c_size_t]),
    "x265cu_free": (None, [P, P]),
    "x265cu_host_alloc": (P, [C.c_size_t]),
    "x265cu_host_free": (None, [P]),
    "x265cu_h2d": (I, [P, P, P, C.c_size_t]),
    "x265cu_d2h": (I, [P, P, P, C.c_size_t]),
    "x265cu_memset": (I, [P, P, I, C.c_size_t]),
    "x265cu_copy2d": (I, [P, P, C.c_size_t, P, C.c_size_t, C.c_size_t, C.c_size_t, I]),
    "x265cu_timer_begin": (I, [P]),
    "x265cu_timer_end": (C.c_float, [P]),
    "x265cu_launch_count": (C.c_uint64, [P]),
    "x265cu_me_phase_ms": (I, [P, C.POINTER(C.c_float)]),
    "x265cu_get_primitive": (P, [I, C.c_char_p, I, I, I]),
    "x265cu_primitive_error": (I, []),
    "x265cu_primitive_error_string": (C.c_char_p, []),
    "x265cu_primitive_error_clear": (None, []),
    "x265cu_primitive_calls": (C.c_uint64, []),
    "x265cu_pixelcmp_batch": (I, [P, I, I, P, P, P, I, P]),
    "x265cu_pixelcmp_grid": (I, [P, I, I, P, I64, P, I64, I, I, I, I, P]),
    "x265cu_blockop_batch": (I, [P, I, I, P, P, P, P, I]),
    "x265cu_interp_batch": (I, [P, I, I, P, P, P, I]),
    "x265cu_transform_batch": (I, [P, I, I, I, P, P, I, I64, I]),
    "x265cu_quant_batch": (I, [P, P, P, P, P, I, I, I, I, I, P]),
    "x265cu_dequant_normal_batch": (I, [P, P, P, I64, I, I]),
    "x265cu_dequant_scaling_batch": (I, [P, P, P, P, I, I, I, I]),
    "x265cu_intra_pred_batch": (I, [P, I, I, P, I64, P, I64, I, P, I]),
    "x265cu_intra_filter_batch": (I, [P, I, I, P, P, I64, I]),
    "x265cu_intra_allangs_batch": (I, [P, I, I, P, P, I64, P, I, I]),
    "x265cu_frame_init_lowres": (I, [P, I, P, I, P, P, P, P, I, I, I, I, I]),
    "x265cu_extend_border": (I, [P, I, P, I, I, I, I, I]),
    "x265cu_mvcost_table": (None, [C.c_double, I, P]),
    "x265cu_me_batch": (I, [P, I, P, I, P, I, I, P, I, P, I, P]),
    "x265cu_me_batch_chroma": (I, [P, I, P, I, P, I, P, P, I, P, I, P]),
    "x265cu_pred_cost_batch": (I, [P, I, P, I, P, I, P, P, I, P]),
}


class DeviceBuffer:
    """A device allocation owned by the Lib context."""

    def __init__(self, lib, nbytes):
        self.lib = lib
        self.nbytes = int(nbytes)
        self.ptr = lib.L.x265cu_malloc(lib.ctx, max(self.nbytes, 16))
        if not self.ptr:
            raise MemoryError("x265cu_malloc(%d) failed: %s" % (nbytes, lib.last_error()))

    def upload(self, arr, offset=0):
        arr = np.ascontiguousarray(arr)
        assert offset + arr.nbytes <= self.nbytes
        self.lib.check(self.lib.L.x265cu_h2d(self.lib.ctx, self.ptr + offset, arr.ctypes.data, arr.nbytes))
        self.lib.sync()          # pageable source: make the copy complete before numpy may free it
        return self

    def download(self, dtype, count=None, offset=0):
        dt = np.dtype(dtype)
        if count is None:
            count = (self.nbytes - offset) // dt.itemsize
        out = np.empty(count, dt)
        self.lib.check(self.lib.L.x265cu_d2h(self.lib.ctx, out.ctypes.data, self.ptr + offset, out.nbytes))
        self.lib.sync()
        return out

    def free(self):
        if self.ptr:
            self.lib.L.x265cu_free(self.lib.ctx, self.ptr)
            self.ptr = None


class Lib:
    def __init__(self, device=0, need_gpu=True):
        path = _build.build()
        self.path = path
        self.L = C.CDLL(path)
        for name, (res, args) in _PROTOS.items():
            f = getattr(self.L, name)       # AttributeError if the ABI lost a symbol
            f.restype = res
            f.argtypes = args
        self.ctx = None
        if need_gpu:
            if self.L.x265cu_device_count() <= 0:
                raise CudaUnavailable("libx265cu.so loaded but no CUDA device is visible; there is no CPU fallback")
            self.ctx = self.L.x265cu_create(device)
            if not self.ctx:
                raise CudaUnavailable("x265cu_create(%d) failed: %s" % (device, self.last_error()))

    # ---- plumbing ----
    def last_error(self):
        e = self.L.x265cu_last_error()
        return e.decode() if e else ""

    def check(self, rc):
        if rc != 0:
            raise RuntimeError("x265cu call failed: " + self.last_error())

    def sync(self):
        self.check(self.L.x265cu_sync(self.ctx))

    def alloc(self, nbytes):
        return DeviceBuffer(self, nbytes)

    def to_device(self, arr):
        arr = np.ascontiguousarray(arr)
        return DeviceBuffer(self, arr.nbytes).upload(arr)

    def timer_begin(self):
        self.check(self.L.x265cu_timer_begin(self.ctx))

    def timer_end(self):
        ms = self.L.x265cu_timer_end(self.ctx)
        if ms < 0:
            raise RuntimeError("timer failed: " + self.last_error())
        return ms

    def me_phase_ms(self):
        ms = (C.c_float * 3)()
        self.check(self.L.x265cu_me_phase_ms(self.ctx, ms))
        return [float(x) for x in ms]

    def launch_count(self):
        return int(self.L.x265cu_launch_count(self.ctx))

    def close(self):
        if self.ctx:
            self.L.x265cu_destroy(self.ctx)
            self.ctx = None

    # ---- per-call table ----
    def primitive(self, depth, name, restype, argtypes, i=0, j=0, k=0):
        p = self.L.x265cu_get_primitive(depth, name.encode(), i, j, k)
        if not p:
            return None
        return C.CFUNCTYPE(restype, *argtypes)(p)

    # ---- batched API (device buffers in, device buffers out) ----
    def pixelcmp_batch(self, depth, op, A, B, jobs_dev, n, out_dev):
        self.check(self.L.x265cu_pixelcmp_batch(self.ctx, depth, OPS_CMP[op], A.ptr, B.ptr, jobs_dev.ptr, n, out_dev.ptr))

    def pixelcmp_grid(self, depth, op, a_ptr, a_stride, b_ptr, b_stride, bw, bh, nbx, nby, out_dev):
        """a_ptr / b_ptr: device addresses of block (0,0) in each plane (ints); strides in pixels."""
        self.check(self.L.x265cu_pixelcmp_grid(self.ctx, depth, OPS_CMP[op], a_ptr, a_stride, b_ptr, b_stride, bw, bh, nbx, nby, out_dev.ptr))

    def blockop_batch(self, depth, op, D, A, B, jobs_dev, n):
        self.check(self.L.x265cu_blockop_batch(self.ctx, depth, OPS_BLK[op], D.ptr, A.ptr if A else None, B.ptr if B else None, jobs_dev.ptr, n))

    def interp_batch(self, depth, op, S, D, jobs_dev, n):
        self.check(self.L.x265cu_interp_batch(self.ctx, depth, OPS_INTERP[op], S.ptr, D.ptr, jobs_dev.ptr, n))

    def transform_batch(self, depth, op, size, S, D, stride, tu_pitch, n):
        self.check(self.L.x265cu_transform_batch(self.ctx, depth, OPS_TR[op], size, S.ptr, D.ptr, stride, tu_pitch, n))

    def me_batch(self, depth, fenc, fstride, refs_ptr_table, rstride, lowres, mvcost_dev, mvcost_range, jobs_dev, n, out_dev):
        centre = mvcost_dev.ptr + 2 * mvcost_range
        self.check(self.L.x265cu_me_batch(self.ctx, depth, fenc.ptr, fstride, refs_ptr_table.ptr, rstride, lowres, centre,
                                          mvcost_range, jobs_dev.ptr, n, out_dev.ptr))

    def me_batch_chroma(self, depth, fenc, fstride, refs_ptr_table, rstride, fenc_cb, fenc_cr, ref_cb_table, ref_cr_table, cstride,
                        mvcost_dev, mvcost_range, jobs_dev, n, out_dev):
        """x265cu_me_batch with the chroma-SATD term of subpelCompare (4:2:0 planes at half resolution)."""
        ch = MeChroma(fenc_cb.ptr, fenc_cr.ptr, ref_cb_table.ptr, ref_cr_table.ptr, cstride)
        self.check(self.L.x265cu_me_batch_chroma(self.ctx, depth, fenc.ptr, fstride, refs_ptr_table.ptr, rstride, C.byref(ch),
                                                 mvcost_dev.ptr + 2 * mvcost_range, mvcost_range, jobs_dev.ptr, n, out_dev.ptr))

    def pred_cost_batch(self, depth, fenc, fstride, refs_ptr_table, rstride, chroma, jobs_dev, n, out_dev):
        """x265cu_pred_cost_batch: AMVP candidate SADs, merge candidate / bidir SATDs (search.cpp:1901-2023, 2474-2607).
        chroma: None or (fenc_cb, fenc_cr, ref_cb_table, ref_cr_table, cstride) device buffers."""
        ch = MeChroma(chroma[0].ptr, chroma[1].ptr, chroma[2].ptr, chroma[3].ptr, chroma[4]) if chroma else None
        self.check(self.L.x265cu_pred_cost_batch(self.ctx, depth, fenc.ptr, fstride, refs_ptr_table.ptr, rstride,
                                                 C.byref(ch) if ch else None, jobs_dev.ptr, n, out_dev.ptr))

    def lookahead_weights_analyse(self, depth, fenc_buf, ref_bufs, wbuf, planesize, stride, width, lines, padoffset, intra_cost, stats):
        """x265cu_lookahead_weights_analyse: returns (isWeighted, scale, log2denom, offset); wbuf then holds the 4 weighted planes."""
        refs = (C.c_void_p * 4)(*[b.ptr for b in ref_bufs])
        intra = np.ascontiguousarray(intra_cost, np.int32)
        st = np.ascontiguousarray(stats, np.uint64)
        wp = np.zeros(4, np.int32)
        self.check(self.L.x265cu_lookahead_weights_analyse(self.ctx, depth, fenc_buf.ptr, refs, wbuf.ptr, planesize, stride, width, lines,
                                                           padoffset, intra.ctypes.data, st.ctypes.data, wp.ctypes.data))
        return tuple(int(x) for x in wp)

    def mvcost_table(self, lam, rng):
        t = np.zeros(2 * rng + 1, np.uint16)
        self.L.x265cu_mvcost_table(C.c_double(lam), rng, t.ctypes.data)
        return t


_cached = {}


def load(device=0, need_gpu=True):
    key = (device, need_gpu)
    if key not in _cached:
        _cached[key] = Lib(device, need_gpu)
    return _cached[key]


LA_INTRA_JOB = np.dtype([("plane0", "<u8"), ("invQscale", "<u8"), ("intraCost", "<u8"), ("intraMode", "<u8"), ("lowresCosts", "<u8"),
                         ("rowSatds", "<u8"), ("out", "<u8")], align=True)
LA_JOB = np.dtype([("fenc", "<u8", 4), ("ref0", "<u8", 4), ("ref1", "<u8", 4), ("mvs", "<u8", 2), ("mvcosts", "<u8", 2), ("intraCost", "<u8"),
                   ("invQscale", "<u8"), ("lowresCosts", "<u8"), ("rowSatds", "<u8"), ("out", "<u8"), ("bidir", "<i4"), ("doSearch0", "<i4"),
                   ("doSearch1", "<i4"), ("rows", "<i4")], align=True)
assert LA_INTRA_JOB.itemsize == 56 and LA_JOB.itemsize == 184


# ---------------- frame-level analyser (x265cu_analyser_*) ----------------
class AnalysisParams(C.Structure):
    _fields_ = [("width", I), ("height", I), ("depth", I), ("numRefs", I), ("method", I), ("subme", I), ("merange", I),
                ("rect", I), ("qp", I), ("lam", C.c_double), ("amp", I)]


class AnalysisOut(C.Structure):
    _fields_ = [("me_packed", P), ("cu_sse", P), ("cu_numsig", P), ("cu_ref", P), ("intra_cost", P)]


_AN_PROTOS = {
    "x265cu_analyser_create": (P, [P, C.POINTER(AnalysisParams)]),
    "x265cu_analyser_destroy": (None, [P]),
    "x265cu_analyser_counts": (I, [P, C.POINTER(I), C.POINTER(I), C.POINTER(I), C.POINTER(I64), C.POINTER(I)]),
    "x265cu_analyser_set_ref": (I, [P, I, P, I]),
    "x265cu_analyser_load_inputs": (I, [P, P, I, P]),
    "x265cu_analyser_run_resident": (I, [P, I]),
    "x265cu_analyser_analyse": (I, [P, P, I, P, I, C.POINTER(AnalysisOut)]),
    "x265cu_analyser_fetch": (I, [P, I, P]),
    "x265cu_analyser_stage_ms": (I, [P, C.POINTER(C.c_float)]),
    "x265cu_analyser_ref_plane": (P, [P, I, C.POINTER(I)]),
    "x265cu_analyser_ref_updated": (I, [P, I]),
    "x265cu_analyser_ctu_rows": (I, [P]),
    "x265cu_analyser_row_range": (I, [P, I, I, C.POINTER(I), C.POINTER(I), C.POINTER(I), C.POINTER(I)]),
    "x265cu_analyser_run_rows": (I, [P, I, I, I]),
    "x265cu_analyser_analyse_rows": (I, [P, P, I, P, I, I, I, C.POINTER(AnalysisOut)]),
    "x265cu_analyser_recon_plane": (P, [P, I, C.POINTER(I)]),
    "x265cu_analyser_recon_to_ref": (I, [P, I, I, I, I]),
    "x265cu_analyser_enable_chroma": (I, [P]),
    "x265cu_analyser_set_ref_chroma": (I, [P, I, P, P, I]),
    "x265cu_analyser_load_chroma": (I, [P, P, P, I]),
    "x265cu_analyser_phase_planes_ms": (I, [P, C.POINTER(C.c_float)]),
    "x265cu_analyser_ref_plane_phase": (P, [P, I, I]),
    "x265cu_analyser_phase_region": (I, [P, I, C.POINTER(I)]),
}
_AN_PROTOS["x265cu_propagate_cost_batch"] = (I, [P, P, P, P, P, P, C.c_double, I64])
_AN_PROTOS["x265cu_lowres_intra_batch"] = (I, [P, I, P, I, I, I, I, I])
_AN_PROTOS["x265cu_lookahead_cost_batch"] = (I, [P, I, P, I, I, I, I, P])
_AN_PROTOS["x265cu_lookahead_weights_analyse"] = (I, [P, I, P, P, P, I64, I, I, I, I64, P, P, P])
_PROTOS.update(_AN_PROTOS)


class Analyser:
    """Host mirror of x265cu_analyser: the public call a user makes for one frame is analyse()."""

    def __init__(self, lib, width, height, depth=8, numRefs=4, method=3, subme=3, merange=57, rect=1, qp=30, lam=None, amp=0):
        self.lib = lib
        if lam is None:
            lam = round(2.0 ** (qp / 6.0 - 2.0) * (1 << (depth - 8)), 4)      # x265_lambda_tab (constants.cpp:33-50)
        self.params = AnalysisParams(width, height, depth, numRefs, method, subme, merange, rect, qp, lam, amp)
        self.h = lib.L.x265cu_analyser_create(lib.ctx, C.byref(self.params))
        if not self.h:
            raise RuntimeError("x265cu_analyser_create failed: " + lib.last_error())
        nj, nc, nt, st = I(), I(), I(), I()
        ncoef = I64()
        lib.L.x265cu_analyser_counts(self.h, C.byref(nj), C.byref(nc), C.byref(nt), C.byref(ncoef), C.byref(st))
        self.njobs, self.ncu, self.ntu, self.ncoef, self.stride = nj.value, nc.value, nt.value, ncoef.value, st.value
        self.depth, self.width, self.height, self.numRefs = depth, width, height, numRefs
        self.dtype = np.uint8 if depth == 8 else np.uint16
        # host result buffers (pinned so D2H is real DMA)
        self._pinned = []
        self.me_packed = self._pin((self.njobs, 2), np.int32)
        self.cu_sse = self._pin((self.ncu,), np.uint64)
        self.cu_numsig = self._pin((self.ncu,), np.uint32)
        self.cu_ref = self._pin((self.ncu,), np.int32)
        self.intra_cost = self._pin((self.ncu, 36), np.uint32)
        self.out = AnalysisOut(self.me_packed.ctypes.data, self.cu_sse.ctypes.data, self.cu_numsig.ctypes.data,
                               self.cu_ref.ctypes.data, self.intra_cost.ctypes.data)

    def _pin(self, shape, dtype):
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        p = self.lib.L.x265cu_host_alloc(max(n, 16))
        if not p:
            raise MemoryError("pinned alloc failed")
        self._pinned.append(p)
        buf = (C.c_uint8 * n).from_address(p)
        return np.frombuffer(buf, dtype=dtype).reshape(shape)

    def set_ref(self, idx, img):
        img = np.ascontiguousarray(img, self.dtype)
        assert img.shape == (self.height, self.width)
        self.lib.check(self.lib.L.x265cu_analyser_set_ref(self.h, idx, img.ctypes.data, self.width))

    def load_inputs(self, fenc, field):
        fenc = np.ascontiguousarray(fenc, self.dtype)
        field = np.ascontiguousarray(field, np.int16)
        self.lib.check(self.lib.L.x265cu_analyser_load_inputs(self.h, fenc.ctypes.data, self.width, field.ctypes.data))

    def run_resident(self, stages=7):
        self.lib.check(self.lib.L.x265cu_analyser_run_resident(self.h, stages))

    def analyse(self, fenc, field, stages=7):
        """e2e: host frame + predictor field in, host results out (synchronous)."""
        self.lib.check(self.lib.L.x265cu_analyser_analyse(self.h, fenc.ctypes.data, self.width, field.ctypes.data, stages, C.byref(self.out)))
        return self

    # ---- CTU-row shards (x265cu_analyser_*_rows): rows [r0, r1) are one contiguous slice of every result array ----
    @property
    def ctu_rows(self):
        return int(self.lib.L.x265cu_analyser_ctu_rows(self.h))

    def row_range(self, r0, r1):
        """(job0, njobs, cu0, ncu) of the CTU rows [r0, r1)."""
        v = [I(), I(), I(), I()]
        self.lib.check(self.lib.L.x265cu_analyser_row_range(self.h, r0, r1, *[C.byref(x) for x in v]))
        return tuple(x.value for x in v)

    def run_rows(self, r0, r1, stages=7):
        self.lib.check(self.lib.L.x265cu_analyser_run_rows(self.h, stages, r0, r1))

    def analyse_rows(self, fenc, field, r0, r1, stages=7):
        """e2e for a row shard: host frame + field in, the shard's slice of the host result arrays out."""
        self.lib.check(self.lib.L.x265cu_analyser_analyse_rows(self.h, fenc.ctypes.data, self.width, field.ctypes.data, stages, r0, r1, C.byref(self.out)))
        return self

    def d2h_bytes_rows(self, r0, r1):
        _, nj, _, nc = self.row_range(r0, r1)
        return nj * 8 + nc * (8 + 4 + 4 + 36 * 4)

    def recon_plane_ptr(self, depth_idx):
        st = I()
        return self.lib.L.x265cu_analyser_recon_plane(self.h, depth_idx, C.byref(st)), st.value

    def recon_to_ref(self, depth_idx, ref_idx, r0, r1):
        self.lib.check(self.lib.L.x265cu_analyser_recon_to_ref(self.h, depth_idx, ref_idx, r0, r1))

    # ---- 4:2:0 chroma for the chroma-SATD term of subpelCompare ----
    def enable_chroma(self):
        self.lib.check(self.lib.L.x265cu_analyser_enable_chroma(self.h))

    def set_ref_chroma(self, idx, cb, cr):
        cb = np.ascontiguousarray(cb, self.dtype); cr = np.ascontiguousarray(cr, self.dtype)
        assert cb.shape == cr.shape == (self.height // 2, self.width // 2)
        self.lib.check(self.lib.L.x265cu_analyser_set_ref_chroma(self.h, idx, cb.ctypes.data, cr.ctypes.data, self.width // 2))

    def load_chroma(self, cb, cr):
        """Source chroma of the next analyse() / run_*() (pass pinned arrays for true async DMA)."""
        assert cb.shape == cr.shape == (self.height // 2, self.width // 2) and cb.dtype == self.dtype and cb.flags.c_contiguous and cr.flags.c_contiguous
        self.lib.check(self.lib.L.x265cu_analyser_load_chroma(self.h, cb.ctypes.data, cr.ctypes.data, self.width // 2))

    def h2d_bytes(self, field):
        return self.width * self.height * np.dtype(self.dtype).itemsize + field.nbytes

    def d2h_bytes(self):
        return self.me_packed.nbytes + self.cu_sse.nbytes + self.cu_numsig.nbytes + self.cu_ref.nbytes + self.intra_cost.nbytes

    def stage_ms(self):
        ms = (C.c_float * 4)()
        self.lib.check(self.lib.L.x265cu_analyser_stage_ms(self.h, ms))
        return [float(x) for x in ms]

    def ref_plane_ptr(self, idx):
        st = I()
        return self.lib.L.x265cu_analyser_ref_plane(self.h, idx, C.byref(st)), st.value

    def ref_updated(self, idx):
        self.lib.check(self.lib.L.x265cu_analyser_ref_updated(self.h, idx))

    # ---- quarter-pel phase planes of the references (X265CU_ME_PHASEPLANES) ----
    def phase_planes_ms(self):
        """Device ms of the last run's phase-plane build (0.0 when it built none)."""
        ms = C.c_float()
        self.lib.check(self.lib.L.x265cu_analyser_phase_planes_ms(self.h, C.byref(ms)))
        return float(ms.value)

    def phase_region(self, idx):
        """(x0, x1, y0, y1): the picture rectangle of reference idx's phase planes that the last run built."""
        box = (I * 4)()
        self.lib.check(self.lib.L.x265cu_analyser_phase_region(self.h, idx, box))
        return tuple(int(v) for v in box)

    def fetch_phase_plane(self, idx, phase):
        """Phase plane (yFrac << 2) | xFrac of reference idx, margins included: (height + 160) x stride, pixel (0, 0) at
        row 80, column 96."""
        ptr = self.lib.L.x265cu_analyser_ref_plane_phase(self.h, idx, phase)
        if not ptr:
            raise RuntimeError("no phase plane %d of reference %d" % (phase, idx))
        es = np.dtype(self.dtype).itemsize
        out = np.zeros((self.height + 160, self.stride), self.dtype)
        self.lib.check(self.lib.L.x265cu_d2h(self.lib.ctx, out.ctypes.data, ptr - (80 * self.stride + 96) * es, out.nbytes))
        self.lib.sync()
        return out

    def fetch(self, what):
        es = np.dtype(self.dtype).itemsize
        rows = self.height + 160
        spec = {"jobs": (0, ME_JOB, self.njobs), "me_out": (1, np.int32, self.njobs * 4), "coef": (2, np.int16, self.ncoef),
                "recon0": (3, self.dtype, self.stride * rows), "recon1": (4, self.dtype, self.stride * rows),
                "recon2": (5, self.dtype, self.stride * rows), "recon3": (6, self.dtype, self.stride * rows),
                "cu_jobs": (7, np.int32, self.ncu * self.numRefs), "fenc": (8, self.dtype, self.stride * rows)}[what]
        out = np.zeros(spec[2], spec[1])
        self.lib.check(self.lib.L.x265cu_analyser_fetch(self.h, spec[0], out.ctypes.data))
        return out

    def close(self):
        if self.h:
            self.lib.L.x265cu_analyser_destroy(self.h)
            self.h = None
        for p in self._pinned:
            self.lib.L.x265cu_host_free(p)
        self._pinned = []
