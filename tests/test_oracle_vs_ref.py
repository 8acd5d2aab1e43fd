"""Pins the plain-C oracle (oracle/*.c) against the REAL reference C primitives compiled from
/root/reference (oracle/_ref/libx265ref{8,10}.so, built by oracle/Makefile.ref).

Mirrors the reference's own TestBench strategy (source/test/testbench.cpp:155-233): same inputs
through both tables, exact integer equality / memcmp, fixtures = random / all-min / all-max
(pixelharness.cpp:31-80, mbdstharness.cpp:61-82).  CPU only.
"""
import ctypes as C
import numpy as np
import pytest

import table_checks
from common import load_oracle, ref_fn, RefResults, same

DEPTHS = [8, 10]
KINDS = ["rand", "min", "max"]


def pinned(name, depth):
    """The reference's results of this test (tests/golden/ref/<name>.npz, see common.RefResults) and the oracle."""
    return RefResults(name, depth), load_oracle(depth)


def ref_getter(rec):
    """The reference C table as table_checks asks for it: whether an entry exists and every value a primitive returns
    pass through `rec` (output arrays through the checks' `ref_out`)."""
    def get(name, restype, argtypes, i=0, j=0, k=0):
        f = ref_fn(rec.R, name, restype, argtypes, i, j, k) if rec.recording else None
        if not rec(int(f is not None) if rec.recording else 0):
            return None
        if restype is None:
            return f if rec.recording else (lambda *args: None)
        return lambda *args: rec(int(f(*args)) if rec.recording else 0)
    return get


@pytest.mark.parametrize("depth", DEPTHS)
def test_constants(depth):
    rec, O = pinned("constants_%d" % depth, depth)
    for n in (4, 8, 16, 32):
        a = rec(np.ctypeslib.as_array(C.cast(rec.R.x265ref_dct_matrix(n), C.POINTER(C.c_int16)), (n * n,)).copy() if rec.recording else None)
        b = np.ctypeslib.as_array(C.cast(O.orc_dct_matrix(n), C.POINTER(C.c_int16)), (n * n,))
        assert same(a, b)
    rec.done()


@pytest.mark.parametrize("depth", DEPTHS)
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("cls", ["pixelcmp", "blockops", "interp", "transforms", "intra"])
def test_table(depth, kind, cls):
    rec, O = pinned("table_%s_%s_%d" % (cls, kind, depth), depth)
    getattr(table_checks, "check_" + cls)(ref_getter(rec), O, depth, kind, ref_out=rec)
    rec.done()


@pytest.mark.parametrize("depth", DEPTHS)
def test_ads(depth):
    # not covered by the reference TestBench (SURVEY 4); checked directly against pixel.cpp:121-165
    rec, O = pinned("ads_%d" % depth, depth)
    table_checks.check_ads(ref_getter(rec), O, depth, ref_out=rec)
    rec.done()


@pytest.mark.parametrize("depth", DEPTHS)
def test_integral(depth):
    # SEA integral planes: not in the four TestBench harness classes used above; checked directly (framefilter.cpp:39-143)
    rec, O = pinned("integral_%d" % depth, depth)
    table_checks.check_integral(ref_getter(rec), O, depth, ref_out=rec)
    rec.done()


def _me_job(O, R, depth, rng, w, h, method, subme, lowres, smooth, merange, qp=30):
    """Run the same motionEstimate job through the real MotionEstimate and the oracle."""
    from me_helpers import run_both
    return run_both(O, R, depth, rng, w, h, method, subme, lowres, smooth, merange, qp)


@pytest.mark.parametrize("depth", DEPTHS)
@pytest.mark.parametrize("method", [0, 1, 2, 3])
def test_motion_estimate(depth, method):
    rec, O = pinned("motion_estimate_%d_%d" % (depth, method), depth)
    R = rec.R
    rng = np.random.default_rng(7 + method)
    sizes = [(8, 8), (16, 16), (32, 32), (64, 64), (16, 8), (8, 16), (32, 16), (16, 32), (64, 32), (32, 64),
             (16, 12), (12, 16), (16, 4), (4, 16), (32, 24), (24, 32), (32, 8), (8, 32), (64, 48), (48, 64), (64, 16), (16, 64), (8, 4), (4, 8)]
    n = 0
    for (w, h) in sizes:
        for subme in (0, 1, 2, 3, 4, 5, 7):
            for smooth in (True, False):
                r, o = _me_job(O, R, depth, rng, w, h, method, subme, 0, smooth, 57 if method == 3 else 16)
                r = rec(r)
                assert r == o, (w, h, method, subme, smooth, r, o)
                n += 1
    assert n > 100
    rec.done()


@pytest.mark.parametrize("depth", DEPTHS)
def test_motion_estimate_umh_wide(depth):
    """X265_UMH_SEARCH (motion.cpp:946-1130) with the presets' search range: the adaptive range, the cross and the hexagon grid run
    many more iterations than with the range of 16 test_motion_estimate uses."""
    rec, O = pinned("motion_estimate_umh_wide_%d" % depth, depth)
    R = rec.R
    rng = np.random.default_rng(909)
    n = 0
    for (w, h) in [(8, 8), (16, 16), (32, 32), (64, 64), (16, 8), (8, 16), (32, 16), (16, 32), (64, 32), (32, 64), (24, 32), (16, 4), (4, 8), (12, 16), (64, 48), (8, 32)]:
        for subme in (0, 3):
            for smooth in (True, False):
                for rep in range(2):
                    r, o = _me_job(O, R, depth, rng, w, h, 2, subme, 0, smooth, 57)
                    r = rec(r)
                    assert r == o, (w, h, subme, smooth, r, o)
                    n += 1
    assert n == 128
    rec.done()


@pytest.mark.parametrize("depth", DEPTHS)
def test_motion_estimate_full_search(depth):
    """X265_FULL_SEARCH (motion.cpp:1397-1440): exhaustive scan of [mvmin, mvmax]; small search ranges keep it quick."""
    rec, O = pinned("motion_estimate_full_search_%d" % depth, depth)
    R = rec.R
    rng = np.random.default_rng(77)
    n = 0
    for (w, h) in [(8, 8), (16, 16), (32, 32), (64, 64), (16, 8), (8, 16), (32, 16), (24, 32), (16, 4), (4, 8), (12, 16), (64, 48)]:
        for subme in (0, 2, 3):
            for smooth in (True, False):
                r, o = _me_job(O, R, depth, rng, w, h, 5, subme, 0, smooth, int(rng.integers(3, 12)))
                r = rec(r)
                assert r == o, (w, h, subme, smooth, r, o)
                n += 1
    assert n == 72
    rec.done()


@pytest.mark.parametrize("depth", DEPTHS)
def test_motion_estimate_sea(depth):
    """X265_SEA (motion.cpp:1242-1395) restated literally -- partition-dependent integral plane / ADS variant / delta, the row cost
    p_cost_mvy[tmv.y] << 2, the width rounded up to 4 -- against the real MotionEstimate fed with integral planes built by the real
    integral_init primitives in FrameFilter::computeMEIntegral's order.  Every PU size."""
    from me_helpers import run_both_sea
    rec, O = pinned("motion_estimate_sea_%d" % depth, depth)
    R = rec.R
    rng = np.random.default_rng(404)
    sizes = [(8, 8), (16, 16), (32, 32), (64, 64), (16, 8), (8, 16), (32, 16), (16, 32), (64, 32), (32, 64),
             (16, 12), (12, 16), (16, 4), (4, 16), (32, 24), (24, 32), (32, 8), (8, 32), (64, 48), (48, 64), (64, 16), (16, 64), (8, 4), (4, 8)]
    n = 0
    for (w, h) in sizes:
        for subme in (0, 2):
            for smooth in (True, False):
                r, o = run_both_sea(O, R, depth, rng, w, h, subme, smooth, int(rng.integers(4, 17)), rec=rec)
                r = rec(r)
                assert r == o, (w, h, subme, smooth, r, o)
                n += 1
    assert n == len(sizes) * 4
    rec.done()


@pytest.mark.parametrize("depth", DEPTHS)
def test_motion_estimate_lowres(depth):
    rec, O = pinned("motion_estimate_lowres_%d" % depth, depth)
    R = rec.R
    rng = np.random.default_rng(17)
    for method in (0, 1, 3):
        for subme in (0, 1, 2, 5):
            for smooth in (True, False):
                for it in range(4):
                    r, o = _me_job(O, R, depth, rng, 8, 8, method, subme, 1, smooth, 16)
                    r = rec(r)
                    assert r == o, (method, subme, smooth, r, o)
    rec.done()


@pytest.mark.parametrize("depth", DEPTHS)
@pytest.mark.parametrize("method", [1, 3])
def test_motion_estimate_chroma_satd(depth, method):
    """subpelCompare's chroma term (motion.cpp:1601-1661; active for subme > 2 when the chroma block has a SATD,
    motion.cpp:204-212): every PU size whose chroma block is a multiple of 4x4, plus sizes / sub-pel levels where
    the term must stay off."""
    from me_helpers import run_both_chroma
    rec, O = pinned("motion_estimate_chroma_satd_%d_%d" % (depth, method), depth)
    R = rec.R
    rng = np.random.default_rng(31 + method)
    sizes = [(8, 8), (16, 16), (32, 32), (64, 64), (16, 8), (8, 16), (32, 16), (16, 32), (64, 32), (32, 64),
             (32, 24), (24, 32), (32, 8), (8, 32), (64, 48), (48, 64), (64, 16), (16, 64),
             (8, 4), (4, 8), (16, 12), (12, 16), (16, 4), (4, 16)]
    n = diff = 0
    for (w, h) in sizes:
        for subme in (2, 3, 4, 5, 7):
            for smooth in (True, False):
                r, o = run_both_chroma(O, R, depth, rng, w, h, method, subme, smooth, 57 if method == 3 else 16)
                r = rec(r)
                assert r == o, (w, h, method, subme, smooth, r, o)
                n += 1
    assert n == len(sizes) * 10
    rec.done()


@pytest.mark.parametrize("depth", DEPTHS)
@pytest.mark.parametrize("smooth", [True, False])
def test_pred_cost(depth, smooth):
    """AMVP candidate SAD (Search::selectMVP), merge candidate SATD + chroma SATD (mergeEstimation, uni and bi through
    Predict::motionCompensation) and the pixelavg_pp bidir estimate of predInterSearch: the oracle's restatement against the
    REAL Predict / MotionEstimate classes, every PU size, full / half / quarter-pel vectors in both components."""
    import pred_helpers as ph
    rec, O = pinned("pred_cost_%d_%d" % (depth, int(smooth)), depth)
    R = rec.R
    rng = np.random.default_rng(400 + depth + int(smooth))
    pl = ph.make_planes(depth, rng, smooth)
    n = 0
    for (w, h) in ph.LUMA_PUS:
        for kind in ("amvp", "merge_uni", "merge_bi", "bidir_pp"):
            for _ in range(3):
                jb = ph.random_job(pl, rng, w, h, kind)
                r, o = rec(ph.ref_cost(R, pl, jb)), ph.oracle_cost(O, pl, jb)
                assert r == o, (w, h, kind, jb["mvs"], r, o)
                n += 1
    assert n == len(ph.LUMA_PUS) * 12
    rec.done()
