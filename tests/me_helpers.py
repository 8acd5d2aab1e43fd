"""Helpers that run one motionEstimate job through the real reference MotionEstimate
(oracle/_ref, motion.cpp:739) and through the oracle restatement (oracle/oracle_me.c)."""
import ctypes as C
import numpy as np
from common import P, I, IP, ptr, pixel_dtype, make_plane, same

MVRANGE = 65536  # +-2*BC_MAX_MV like bitcost.h:77


class OrcMeJob(C.Structure):
    _fields_ = [("fenc", P), ("fencStride", IP), ("offset", IP), ("ref", P * 4), ("refStride", IP),
                ("lowres", I), ("pw", I), ("ph", I), ("method", I), ("subme", I),
                ("mvmin", I * 2), ("mvmax", I * 2), ("qmvp", I * 2), ("numCand", I), ("mvc", P),
                ("merange", I), ("mvcost", P),
                ("chroma", I), ("fencC", P * 2), ("refC", P * 2), ("cstride", IP), ("integral", P)]


_tables = {}


def mvcost_table(O, lam):
    key = (id(O), lam)
    if key not in _tables:
        t = np.zeros(2 * MVRANGE + 1, np.uint16)
        O.orc_mvcost_table(C.c_double(lam), MVRANGE, ptr(t))
        _tables[key] = t
    return _tables[key]


def lowres_planes(O, depth, full, fw, fh, margin=32):
    """4 hpel planes with replicated margins from a full-res image (lowres.cpp:259-302 layout)."""
    dt = pixel_dtype(depth)
    lw, lh = fw // 2, fh // 2
    stride = (lw + 2 * margin + 31) // 32 * 32
    planes = [np.zeros((lh + 2 * margin, stride), dt) for _ in range(4)]
    org = margin * stride + margin
    src = np.zeros((fh + 2, fw + 2), dt)
    src[:fh, :fw] = full
    src[fh:, :fw] = full[-1:, :]
    src[:, fw:] = src[:, fw - 1:fw]
    O.orc_frame_init_lowres(ptr(src), *[ptr(p, org) for p in planes], IP(fw + 2), IP(stride), lw, lh)
    for p in planes:
        O.orc_extend_pic_border(ptr(p, org), IP(stride), lw, lh, margin, margin)
    return planes, stride, org, lw, lh


def run_both(O, R, depth, rng, w, h, method, subme, lowres, smooth, merange, qp=30):
    mx = (1 << depth) - 1
    W, H, margin = 256, 192, 96
    lam = R.x265ref_lambda(qp)
    tab = mvcost_table(O, lam)
    if lowres:
        yy, xx = np.mgrid[0:H * 2, 0:W * 2]
        def img(shift):
            if smooth:
                v = 128 + 60 * np.sin((xx + 3 * shift) / 37.0) + 40 * np.cos((yy - 2 * shift) / 29.0) + rng.integers(-6, 7, xx.shape)
                return (np.clip(v, 0, 255).astype(np.int64) << (depth - 8)).astype(pixel_dtype(depth))
            return rng.integers(0, mx + 1, xx.shape).astype(pixel_dtype(depth))
        fplanes, stride, org, lw, lh = lowres_planes(O, depth, img(0), W * 2, H * 2, margin)
        rplanes, _, _, _, _ = lowres_planes(O, depth, img(2), W * 2, H * 2, margin)
        fenc = fplanes[0]; refs = rplanes
    else:
        fenc, stride, org = make_plane(rng, depth, W, H, margin, smooth=smooth)
        refb, _, _ = make_plane(rng, depth, W, H, margin, smooth=smooth)
        if smooth:
            # reference = shifted source + noise so the search has something to find
            sh = np.roll(np.roll(fenc, int(rng.integers(-9, 10)), axis=0), int(rng.integers(-9, 10)), axis=1)
            refb = np.clip(sh.astype(np.int64) + rng.integers(-3, 4, sh.shape), 0, mx).astype(fenc.dtype)
        refs = [refb, refb, refb, refb]
    bx = int(rng.integers(0, (W - w) // 4 + 1)) * 4; by = int(rng.integers(0, (H - h) // 4 + 1)) * 4
    offset = org + by * stride + bx
    # search window: +-merange around the predictor, clipped so all reads stay inside the margins
    qmvp = (int(rng.integers(-40, 41)), int(rng.integers(-40, 41)))
    lim = margin - 12
    mvmin = (max(-bx - lim, (qmvp[0] >> 2) - merange), max(-by - lim, (qmvp[1] >> 2) - merange))
    mvmax = (min(W - w - bx + lim, (qmvp[0] >> 2) + merange), min(H - h - by + lim, (qmvp[1] >> 2) + merange))
    ncand = 0 if lowres else int(rng.integers(0, 4))
    mvc = rng.integers(-60, 61, (max(ncand, 1), 2)).astype(np.int32)
    out_r = np.zeros(2, np.int32); out_o = np.zeros(2, np.int32)
    arr = (P * 4)(*[C.c_void_p(p.ctypes.data) for p in refs])
    R.x265ref_motion_estimate.argtypes = [P, IP, IP, P, IP, I, I, I, I, I, I, P, P, P, I, P, I, P]
    mn = np.array(mvmin, np.int32); mxv = np.array(mvmax, np.int32); mp = np.array(qmvp, np.int32)
    cr = R.x265ref_motion_estimate(ptr(fenc), stride, offset, arr, stride, lowres, w, h, method, subme, qp,
                                   ptr(mn), ptr(mxv), ptr(mp), ncand, ptr(mvc), merange, ptr(out_r))
    job = OrcMeJob()
    job.fenc = fenc.ctypes.data; job.fencStride = stride; job.offset = offset
    for i in range(4):
        job.ref[i] = refs[i].ctypes.data
    job.refStride = stride; job.lowres = lowres; job.pw = w; job.ph = h; job.method = method; job.subme = subme
    job.mvmin[0], job.mvmin[1] = mvmin; job.mvmax[0], job.mvmax[1] = mvmax; job.qmvp[0], job.qmvp[1] = qmvp
    job.numCand = ncand; job.mvc = mvc.ctypes.data; job.merange = merange
    job.mvcost = tab.ctypes.data + MVRANGE * 2
    O.orc_motion_estimate.argtypes = [C.POINTER(OrcMeJob), P]
    co = O.orc_motion_estimate(C.byref(job), ptr(out_o))
    return (cr, int(out_r[0]), int(out_r[1])), (co, int(out_o[0]), int(out_o[1]))


# jobs of tests/golden/me_chroma_*.npz (make_golden.py::gen_chroma): (method, w, h, subme)
CHROMA_CASES = [(m, w, h, sub) for m in (1, 3) for (w, h) in ((8, 8), (16, 16), (32, 16), (16, 32), (64, 64), (32, 24), (8, 32), (16, 12), (8, 4))
                for sub in (2, 3, 5)]


def chroma_case(depth, rng, w, h, smooth, merange, W=256, H=192, margin=96):
    """Planes and window of one 4:2:0 motionEstimate job: luma + Cb/Cr of source and reference (chroma planes at
    half resolution with half the margin, so a luma offset maps to chroma by halving its row and column)."""
    mx = (1 << depth) - 1
    fenc, stride, org = make_plane(rng, depth, W, H, margin, smooth=smooth)
    sy, sx = int(rng.integers(-9, 10)), int(rng.integers(-9, 10))

    def ref_of(src, dy, dx):
        if not smooth:
            return rng.integers(0, mx + 1, src.shape).astype(src.dtype)
        sh = np.roll(np.roll(src, dy, axis=0), dx, axis=1)
        return np.clip(sh.astype(np.int64) + rng.integers(-3, 4, sh.shape), 0, mx).astype(src.dtype)
    ref = ref_of(fenc, sy, sx)
    fc, rc = [], []
    for _ in range(2):
        c, cstride, corg = make_plane(rng, depth, W // 2, H // 2, margin // 2, smooth=smooth)
        fc.append(c); rc.append(ref_of(c, sy // 2, sx // 2))
    assert corg == (margin // 2) * cstride + margin // 2
    bx = int(rng.integers(0, (W - w) // 8 + 1)) * 8; by = int(rng.integers(0, (H - h) // 8 + 1)) * 8
    offset = org + by * stride + bx
    qmvp = (int(rng.integers(-40, 41)), int(rng.integers(-40, 41)))
    lim = margin - 12
    mvmin = (max(-bx - lim, (qmvp[0] >> 2) - merange), max(-by - lim, (qmvp[1] >> 2) - merange))
    mvmax = (min(W - w - bx + lim, (qmvp[0] >> 2) + merange), min(H - h - by + lim, (qmvp[1] >> 2) + merange))
    ncand = int(rng.integers(0, 4))
    mvc = rng.integers(-60, 61, (max(ncand, 1), 2)).astype(np.int32)
    return dict(fenc=fenc, ref=ref, stride=stride, fc=fc, rc=rc, cstride=cstride, offset=offset, qmvp=qmvp, mvmin=mvmin,
                mvmax=mvmax, ncand=ncand, mvc=mvc, w=w, h=h)


def orc_chroma_job(O, cs, method, subme, merange, tab):
    job = OrcMeJob()
    job.fenc = cs["fenc"].ctypes.data; job.fencStride = cs["stride"]; job.offset = cs["offset"]
    for i in range(4):
        job.ref[i] = cs["ref"].ctypes.data
    job.refStride = cs["stride"]; job.lowres = 0; job.pw = cs["w"]; job.ph = cs["h"]; job.method = method; job.subme = subme
    job.mvmin[0], job.mvmin[1] = cs["mvmin"]; job.mvmax[0], job.mvmax[1] = cs["mvmax"]; job.qmvp[0], job.qmvp[1] = cs["qmvp"]
    job.numCand = cs["ncand"]; job.mvc = cs["mvc"].ctypes.data; job.merange = merange
    job.mvcost = tab.ctypes.data + MVRANGE * 2
    job.chroma = 1; job.cstride = cs["cstride"]
    for i in range(2):
        job.fencC[i] = cs["fc"][i].ctypes.data; job.refC[i] = cs["rc"][i].ctypes.data
    return job


def run_both_chroma(O, R, depth, rng, w, h, method, subme, smooth, merange, qp=30):
    """One 4:2:0 job with the chroma-SATD term (motion.cpp:1601-1661) through the real MotionEstimate (Yuv variant of
    setSourcePU, bChroma = true) and through the oracle."""
    cs = chroma_case(depth, rng, w, h, smooth, merange)
    tab = mvcost_table(O, R.x265ref_lambda(qp))
    out_r = np.zeros(2, np.int32); out_o = np.zeros(2, np.int32)
    mn = np.array(cs["mvmin"], np.int32); mxv = np.array(cs["mvmax"], np.int32); mp = np.array(cs["qmvp"], np.int32)
    R.x265ref_motion_estimate_chroma.argtypes = [P, IP, IP, P, P, IP, P, IP, P, P, I, I, I, I, I, P, P, P, I, P, I, P]
    cr = R.x265ref_motion_estimate_chroma(ptr(cs["fenc"]), cs["stride"], cs["offset"], ptr(cs["fc"][0]), ptr(cs["fc"][1]), cs["cstride"],
                                          ptr(cs["ref"]), cs["stride"], ptr(cs["rc"][0]), ptr(cs["rc"][1]),
                                          w, h, method, subme, qp, ptr(mn), ptr(mxv), ptr(mp), cs["ncand"], ptr(cs["mvc"]), merange, ptr(out_r))
    job = orc_chroma_job(O, cs, method, subme, merange, tab)
    O.orc_motion_estimate.argtypes = [C.POINTER(OrcMeJob), P]
    co = O.orc_motion_estimate(C.byref(job), ptr(out_o))
    return (cr, int(out_r[0]), int(out_r[1])), (co, int(out_o[0]), int(out_o[1]))


def run_both_sea(O, R, depth, rng, w, h, subme, smooth, merange, qp=30, rec=lambda v: v):
    """X265_SEA (motion.cpp:1242-1395) through the real MotionEstimate with the 12 integral planes FrameFilter::computeMEIntegral
    would hand it (x265ref_build_integral: the real integral_init primitives) and through the oracle (orc_build_integral +
    method 4); also checks the two sets of planes against each other over the region the search can touch."""
    mx = (1 << depth) - 1
    W, H, margin = 256, 192, 96
    lam = R.x265ref_lambda(qp)
    tab = mvcost_table(O, lam)
    fenc, stride, org = make_plane(rng, depth, W, H, margin, smooth=smooth)
    refb, _, _ = make_plane(rng, depth, W, H, margin, smooth=smooth)
    if smooth:
        sh = np.roll(np.roll(fenc, int(rng.integers(-9, 10)), axis=0), int(rng.integers(-9, 10)), axis=1)
        refb = np.clip(sh.astype(np.int64) + rng.integers(-3, 4, sh.shape), 0, mx).astype(fenc.dtype)
    ipl_r = [np.zeros(refb.shape, np.uint32) for _ in range(12)]
    ipl_o = [np.zeros(refb.shape, np.uint32) for _ in range(12)]
    PA = P * 12
    arr_r = PA(*[p.ctypes.data + org * 4 for p in ipl_r]); arr_o = PA(*[p.ctypes.data + org * 4 for p in ipl_o])
    R.x265ref_build_integral.argtypes = [P, IP, I, C.POINTER(P)]; R.x265ref_build_integral.restype = None
    O.orc_build_integral.argtypes = [P, IP, I, C.POINTER(P)]; O.orc_build_integral.restype = None
    R.x265ref_build_integral(ptr(refb, org), stride, H // 64, arr_r)
    O.orc_build_integral(ptr(refb, org), stride, H // 64, arr_o)
    rows = slice(margin - 79, margin + H + 78)
    assert same(rec(np.stack([a[rows] for a in ipl_r])), np.stack([b[rows] for b in ipl_o]))
    bx = int(rng.integers(0, (W - w) // 4 + 1)) * 4; by = int(rng.integers(0, (H - h) // 4 + 1)) * 4
    offset = org + by * stride + bx
    qmvp = (int(rng.integers(-40, 41)), int(rng.integers(-40, 41)))
    lim = margin - 40
    mvmin = (max(-bx - lim, (qmvp[0] >> 2) - merange), max(-by - lim, (qmvp[1] >> 2) - merange))
    mvmax = (min(W - w - bx + lim, (qmvp[0] >> 2) + merange), min(H - h - by + lim, (qmvp[1] >> 2) + merange))
    ncand = int(rng.integers(0, 4))
    mvc = rng.integers(-60, 61, (max(ncand, 1), 2)).astype(np.int32)
    out_r = np.zeros(2, np.int32); out_o = np.zeros(2, np.int32)
    mn = np.array(mvmin, np.int32); mxv = np.array(mvmax, np.int32); mp = np.array(qmvp, np.int32)
    R.x265ref_motion_estimate_sea.argtypes = [P, IP, IP, P, IP, C.POINTER(P), I, I, I, I, P, P, P, I, P, I, P]
    cr = R.x265ref_motion_estimate_sea(ptr(fenc), stride, offset, ptr(refb), stride, arr_r, w, h, subme, qp,
                                       ptr(mn), ptr(mxv), ptr(mp), ncand, ptr(mvc), merange, ptr(out_r))
    job = OrcMeJob()
    job.fenc = fenc.ctypes.data; job.fencStride = stride; job.offset = offset
    for i in range(4):
        job.ref[i] = refb.ctypes.data
    job.refStride = stride; job.lowres = 0; job.pw = w; job.ph = h; job.method = 4; job.subme = subme
    job.mvmin[0], job.mvmin[1] = mvmin; job.mvmax[0], job.mvmax[1] = mvmax; job.qmvp[0], job.qmvp[1] = qmvp
    job.numCand = ncand; job.mvc = mvc.ctypes.data; job.merange = merange
    job.mvcost = tab.ctypes.data + MVRANGE * 2
    job.integral = C.cast(arr_o, C.c_void_p)
    O.orc_motion_estimate.argtypes = [C.POINTER(OrcMeJob), P]; O.orc_motion_estimate.restype = I
    co = O.orc_motion_estimate(C.byref(job), ptr(out_o))
    return (int(cr), int(out_r[0]), int(out_r[1])), (int(co), int(out_o[0]), int(out_o[1]))
