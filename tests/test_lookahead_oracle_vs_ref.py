"""Pins the lookahead restatement (oracle/oracle_lookahead.c: lowresIntraEstimate + estimateFrameCost /
estimateCUCost) against the REAL classes compiled from /root/reference (Lowres::init,
LookaheadTLD::lowresIntraEstimate, CostEstimateGroup::singleCost) through oracle/_ref.  CPU only."""
import ctypes as C

import numpy as np
import pytest

from common import load_oracle, ptr, P, I, IP, pixel_dtype, RefResults, same
from frame_helpers import gen_luma, MARGIN_X, MARGIN_Y
from lookahead_helpers import OracleLookahead, make_lowres

TRIPLES = [(0, 1, 1), (0, 2, 1), (0, 2, 2), (0, 3, 1), (0, 3, 2), (0, 3, 3), (1, 3, 2), (2, 3, 3)]


class RefLookahead:
    """The reference's Lookahead over `frames`; every result passes through `rec` (a RefResults replays stored ones)."""

    def __init__(self, R, frames, bframes=3, lslices=0, aq=0, chroma=None, rec=None):
        self.R = R
        self.rec = rec if rec is not None else (lambda v, whole=False: v)
        H, W = frames[0].shape
        self.keep = [np.ascontiguousarray(f) for f in frames]
        arr = (P * len(frames))(*[C.c_void_p(f.ctypes.data) for f in self.keep])
        R.x265ref_la_create.restype = P; R.x265ref_la_create.argtypes = [I, I, I, P, IP, I]
        R.x265ref_la_cost.restype = C.c_int64; R.x265ref_la_cost.argtypes = [P, I, I, I]
        R.x265ref_la_get.argtypes = [P, I, I, I, I, P]; R.x265ref_la_geometry.argtypes = [P, P]
        self.slices = None
        if aq:
            # adaptive quantisation on: real Frame objects, calcAdaptiveQuantFrame before lowresIntraEstimate
            cbs = [np.ascontiguousarray(c[0]) for c in chroma]; crs = [np.ascontiguousarray(c[1]) for c in chroma]
            self.keep += cbs + crs
            acb = (P * len(frames))(*[C.c_void_p(f.ctypes.data) for f in cbs]); acr = (P * len(frames))(*[C.c_void_p(f.ctypes.data) for f in crs])
            R.x265ref_la_create_aq.restype = P; R.x265ref_la_create_aq.argtypes = [I, I, I, P, P, P, IP, IP, I, I, I]
            self.h = R.x265ref_la_create_aq(W, H, len(frames), arr, acb, acr, W, W // 2, bframes, lslices, aq)
            if lslices:
                sl = np.zeros(2, np.int32); R.x265ref_la_slices.argtypes = [P, P]; R.x265ref_la_slices(self.h, ptr(sl))
                sl = self.rec(sl)
                self.slices = (int(sl[0]), int(sl[1])) if sl[0] > 1 else None
        elif lslices:
            R.x265ref_la_create_slices.restype = P; R.x265ref_la_create_slices.argtypes = [I, I, I, P, IP, I, I]
            self.h = R.x265ref_la_create_slices(W, H, len(frames), arr, W, bframes, lslices)
            sl = np.zeros(2, np.int32); R.x265ref_la_slices.argtypes = [P, P]; R.x265ref_la_slices(self.h, ptr(sl))
            sl = self.rec(sl)
            self.slices = (int(sl[0]), int(sl[1]))
        else:
            self.h = R.x265ref_la_create(W, H, len(frames), arr, W, bframes)
        g = np.zeros(7, np.int32); R.x265ref_la_geometry(self.h, ptr(g))
        g = self.rec(g)
        self.w8, self.h8, self.stride, self.lw, self.lh = [int(x) for x in g[:5]]
        self.ncu = self.w8 * self.h8

    def cost(self, p0, p1, b):
        return self.rec(int(self.R.x265ref_la_cost(self.h, p0, p1, b)))

    def get(self, frame, what, d0=0, d1=0, dtype=np.int32, n=None, view=None, whole=False):
        """Lookahead array `what` of `frame` (x265ref_la_get), `view` applied before it is compared or stored."""
        out = np.zeros(n if n is not None else self.ncu, dtype)
        assert self.R.x265ref_la_get(self.h, frame, what, d0, d1, ptr(out)) == 0
        return self.rec(view(out) if view else out, whole)


@pytest.mark.parametrize("depth", [8, 10])
@pytest.mark.parametrize("size,noise", [((416, 240), False), ((200, 136), True)])
def test_lookahead(depth, size, noise):
    rec = RefResults("lookahead_%d_%dx%d_%d" % (depth, size[0], size[1], int(noise)), depth)
    O = load_oracle(depth)
    W, H = size
    frames = [gen_luma(W, H, i, s1=17.0, s2=11.0, bits=depth, noise=noise) for i in range(4)]
    ref = RefLookahead(rec.R, frames, rec=rec)
    orc = OracleLookahead(O, frames, depth)
    assert (ref.w8, ref.h8, ref.stride) == (orc.w8, orc.h8, orc.stride)
    # lowres planes incl. margins (Lowres::init)
    rows = ref.lh + 2 * MARGIN_Y
    for k in range(4):
        vw = ref.lw + 2 * MARGIN_X
        pl = ref.get(1, 7, k, 0, pixel_dtype(depth), rows * ref.stride, view=lambda a: a.reshape(rows, ref.stride)[:, :vw])
        assert same(pl, orc.fr[1]["planes"][k][:, :vw]), "plane %d" % k
    for f in range(4):
        assert same(ref.get(f, 0), orc.fr[f]["intraCost"])
        assert same(ref.get(f, 1, dtype=np.uint8), orc.fr[f]["intraMode"])
        assert same(ref.get(f, 2, 0, 0, np.uint16), orc.fr[f]["lowresCosts"][(0, 0)])
        assert same(ref.get(f, 3, 0, 0, np.int32, ref.h8), orc.fr[f]["rowSatds"][(0, 0)])
    for (p0, p1, b) in TRIPLES:
        a, c = ref.cost(p0, p1, b), orc.cost(p0, p1, b)
        assert a == c, ((p0, p1, b), a, c)
        d0, d1 = b - p0, p1 - b
        assert same(ref.get(b, 2, d0, d1, np.uint16), orc.fr[b]["lowresCosts"][(d0, d1)]), (p0, p1, b)
        assert same(ref.get(b, 3, d0, d1, np.int32, ref.h8), orc.fr[b]["rowSatds"][(d0, d1)])
        assert same(ref.get(b, 4, 0, d0, np.int32, 2 * ref.ncu, view=lambda a: a.reshape(-1, 2)), orc.fr[b]["mvs"][(0, d0)])
        assert same(ref.get(b, 5, 0, d0), orc.fr[b]["mvcosts"][(0, d0)])
        if p1 > b:
            assert same(ref.get(b, 4, 1, d1, np.int32, 2 * ref.ncu, view=lambda a: a.reshape(-1, 2)), orc.fr[b]["mvs"][(1, d1)])
        st = ref.get(b, 6, d0, d1, np.int64, 3)
        assert (int(st[0]), int(st[1])) == orc.fr[b]["costEst"][(d0, d1)]
        assert int(st[2]) == orc.fr[b]["intraMbs"].get(d0, 0)
    rec.done()


@pytest.mark.parametrize("depth,lslices", [(8, 4), (8, 8), (10, 4)])
def test_lookahead_cooperative_slices(depth, lslices):
    """estimateFrameCost as presets medium / slow run it (param.cpp:173 lookaheadSlices 8, :492 slow 4): the cooperative-slice
    path (slicetype.cpp:3075-3112, 3143-3173) of the REAL Lookahead (a pool without running workers: the caller processes
    every slice) against the oracle's slice loop -- frame costs, per-CU costs, row sums and motion fields."""
    rec = RefResults("lookahead_cooperative_slices_%d_%d" % (depth, lslices), depth)
    O = load_oracle(depth)
    W, H = 1280, 720                                  # slices need a source height >= 720 (slicetype.cpp:1022-1026)
    frames = [gen_luma(W, H, i, bits=depth) for i in range(3)]
    ref = RefLookahead(rec.R, frames, lslices=lslices, rec=rec)
    assert ref.slices[0] > 1, ref.slices
    orc = OracleLookahead(O, frames, depth, slices=ref.slices)
    for (p0, p1, b) in [(0, 1, 1), (0, 2, 1), (0, 2, 2)]:
        a, c = ref.cost(p0, p1, b), orc.cost(p0, p1, b)
        d0, d1 = b - p0, p1 - b
        assert same(ref.get(b, 4, 0, d0, np.int32, 2 * ref.ncu, view=lambda a: a.reshape(-1, 2)), orc.fr[b]["mvs"][(0, d0)]), (p0, p1, b)
        assert same(ref.get(b, 2, d0, d1, np.uint16), orc.fr[b]["lowresCosts"][(d0, d1)]), (p0, p1, b)
        assert same(ref.get(b, 3, d0, d1, np.int32, ref.h8), orc.fr[b]["rowSatds"][(d0, d1)])
        assert a == c, ((p0, p1, b), a, c)
    rec.done()
    # and the slices change the result (otherwise the test would not see them): serial path on the same frames
    ser = OracleLookahead(O, frames, depth)
    assert any(ser.cost(*t) != orc.cost(*t) or not np.array_equal(ser.fr[t[2]]["mvs"][(0, t[2] - t[0])], orc.fr[t[2]]["mvs"][(0, t[2] - t[0])])
               for t in [(0, 1, 1), (0, 2, 2)])


def aq_lookahead(rec, depth, lslices):
    """The 1280x720 lookahead with adaptive quantisation (aqMode AUTO_VARIANCE) on the reference: the frames, the
    RefLookahead and Lowres::invQscaleFactor of each frame, which the oracle and the device take as input."""
    from frame_helpers import gen_chroma
    W, H = 1280, 720
    frames = [gen_luma(W, H, i, bits=depth) for i in range(3)]
    chroma = [(gen_chroma(W, H, i, 1, bits=depth), gen_chroma(W, H, i, 2, bits=depth)) for i in range(3)]
    ref = RefLookahead(rec.R, frames, lslices=lslices, aq=2, chroma=chroma, rec=rec)
    return frames, ref, [ref.get(i, 8, whole=True) for i in range(3)]


@pytest.mark.parametrize("depth,lslices", [(8, 0), (8, 8), (10, 4)])
def test_lookahead_with_adaptive_quant(depth, lslices):
    """The lookahead as preset medium runs it (aqMode AUTO_VARIANCE, param.cpp:268): Lowres::invQscaleFactor comes from the
    REAL calcAdaptiveQuantFrame (slicetype.cpp:444-694, real Frame objects with 4:2:0 chroma); with it as input the oracle's
    intra and frame-cost paths must reproduce costEstAq, the AQ-weighted row sums and the frame costs of the reference."""
    rec = RefResults("lookahead_aq_%d_%d" % (depth, lslices), depth)
    O = load_oracle(depth)
    frames, ref, invq = aq_lookahead(rec, depth, lslices)
    assert any((q != 256).any() for q in invq), "AQ produced no offsets: the test would not see invQscale"
    orc = OracleLookahead(O, frames, depth, slices=ref.slices, invq=invq)
    for f in range(3):
        assert same(ref.get(f, 0), orc.fr[f]["intraCost"])
        assert same(ref.get(f, 3, 0, 0, np.int32, ref.h8), orc.fr[f]["rowSatds"][(0, 0)])
        st = ref.get(f, 6, 0, 0, np.int64, 3)
        assert (int(st[0]), int(st[1])) == orc.fr[f]["costEst"][(0, 0)]
    for (p0, p1, b) in [(0, 1, 1), (0, 2, 1), (0, 2, 2)]:
        a, c = ref.cost(p0, p1, b), orc.cost(p0, p1, b)
        d0, d1 = b - p0, p1 - b
        assert a == c, ((p0, p1, b), a, c)
        assert same(ref.get(b, 3, d0, d1, np.int32, ref.h8), orc.fr[b]["rowSatds"][(d0, d1)])
        st = ref.get(b, 6, d0, d1, np.int64, 3)
        assert (int(st[0]), int(st[1])) == orc.fr[b]["costEst"][(d0, d1)], (p0, p1, b)
    rec.done()


AQ_TRIPLES = [(0, 1, 1), (0, 2, 1), (0, 2, 2)]


def aq_inputs(depth, lslices):
    """What the device test of the AQ lookahead takes from the reference: the frames, Lowres::invQscaleFactor of each
    frame and the frame costs of AQ_TRIPLES (tests/golden/ref/lookahead_aq_inputs_*.npz)."""
    rec = RefResults("lookahead_aq_inputs_%d_%d" % (depth, lslices), depth)
    frames, ref, invq = aq_lookahead(rec, depth, lslices)
    costs = [ref.cost(*t) for t in AQ_TRIPLES]
    rec.done()
    return frames, invq, costs


@pytest.mark.parametrize("depth,lslices", [(8, 8), (10, 0)])
def test_lookahead_aq_inputs(depth, lslices):
    """The reference results aq_inputs hands the device test: with that invQscaleFactor the oracle reproduces the frame costs."""
    from x265_b200.lookahead import coop_slices
    frames, invq, costs = aq_inputs(depth, lslices)
    assert any((q != 256).any() for q in invq)
    sl = coop_slices(frames[0].shape[0], lslices)
    orc = OracleLookahead(load_oracle(depth), frames, depth, slices=sl if sl[0] > 1 else None, invq=invq)
    assert [orc.cost(*t) for t in AQ_TRIPLES] == costs


def _wp_stats(img):
    """Lowres::wp_sum[0] / wp_ssd[0] as calcAdaptiveQuantFrame leaves them (slicetype.cpp:49-57, 462-480, 665-676):
    sum of the luma samples and sum of squares minus the rounded mean-square term."""
    a = img.astype(np.int64)
    s, q, n = int(a.sum()), int((a * a).sum()), a.size
    return s, q - (s * s + n // 2) // n


@pytest.mark.parametrize("depth", [8, 10])
@pytest.mark.parametrize("case", ["same", "fade", "fade2", "bright", "offset", "noise_fade"])
def test_lookahead_weights_analyse(depth, case):
    """LookaheadTLD::weightsAnalyse + weightCostLuma (slicetype.cpp:807-961): the decision and the 4 re-weighted lowres
    planes of the oracle against the real class, on fades that take every exit of the analysis."""
    rec = RefResults("lookahead_weights_%d_%s" % (depth, case), depth)
    R = rec.R
    O = load_oracle(depth)
    W, H = 416, 240
    mx = (1 << depth) - 1
    base = gen_luma(W, H, 0, s1=17.0, s2=11.0, bits=depth, noise=case.startswith("noise")).astype(np.float64)
    nxt = gen_luma(W, H, 1, s1=17.0, s2=11.0, bits=depth, noise=case.startswith("noise")).astype(np.float64)
    sc = 1 << (depth - 8)
    # NB the analysis estimates the offset from full-resolution sums over the LOWRES area (slicetype.cpp:892-893), i.e. 4x the
    # true mean difference, so only (nearly) pure scalings end up weighted; "offset" exercises the rejected path
    cur = {"same": nxt, "fade": nxt * 0.78, "fade2": nxt * 0.55 + 1 * sc, "bright": nxt * 1.07, "offset": nxt + 21 * sc,
           "noise_fade": nxt * 0.6}[case]
    frames = [base.astype(pixel_dtype(depth)), np.clip(np.rint(cur), 0, mx).astype(pixel_dtype(depth))]
    ref = RefLookahead(R, frames, rec=rec)
    rows = ref.lh + 2 * MARGIN_Y
    planesize = rows * ref.stride
    # the analysis reads the 4 lowres planes of both frames: the oracle's own (Lowres::init restated), equal to the
    # reference's over the picture and its margins, are the input of both sides' stored results
    vw = ref.lw + 2 * MARGIN_X
    bufs = [make_lowres(O, f, depth)[0] for f in frames]
    for f in range(2):
        for k in range(4):
            pl = ref.get(f, 7, k, 0, pixel_dtype(depth), planesize, view=lambda a: a.reshape(rows, ref.stride)[:, :vw])
            assert same(pl, bufs[f][k][:, :vw]), (f, k)
    intra = ref.get(1, 0, whole=True)
    stats = np.array(list(_wp_stats(frames[1])) + list(_wp_stats(frames[0])), np.uint64)
    out = np.zeros(2, np.int64)
    wref = np.zeros(4 * planesize, pixel_dtype(depth))
    R.x265ref_la_weights.argtypes = [P, I, I, P, P, P]
    got_r = rec(int(R.x265ref_la_weights(ref.h, 1, 0, ptr(stats), ptr(out), ptr(wref))))
    out, wref = rec(tuple(int(x) for x in out)), rec(wref)
    assert int(out[0]) == planesize and int(out[1]) == rows

    refarr = (P * 4)(*[C.c_void_p(b.ctypes.data) for b in bufs[0]])
    worc = np.zeros(4 * planesize, pixel_dtype(depth))
    wp = np.zeros(3, np.int32)
    O.orc_la_weights_analyse.argtypes = [P, P, P, IP, IP, I, I, IP, P, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, P]
    got_o = O.orc_la_weights_analyse(ptr(bufs[1][0]), refarr, ptr(worc), planesize, ref.stride, ref.lw, ref.lh,
                                     MARGIN_Y * ref.stride + MARGIN_X, ptr(intra),
                                     int(stats[0]), int(stats[1]), int(stats[2]), int(stats[3]), ptr(wp))
    assert got_o == got_r, (case, got_o, got_r)
    assert (got_r == 0) == (case in ("same", "offset", "noise_fade")), (case, got_r)   # noise: inter never beats intra, no gain
    if got_r:
        assert same(worc, wref), (case, wp.tolist())
        assert 0 <= wp[0] <= 127 and 0 <= wp[1] <= 7 and -128 <= wp[2] <= 127
    rec.done()
