"""Quarter-pel phase planes of the frame analyser (x265_b200/csrc/phase_planes.cuh, X265CU_ME_PHASEPLANES).

The pre-check and sub-pel launches of the motion search read their candidates from 15 precomputed phase planes per
reference instead of interpolating every candidate.  The planes must hold exactly the oracle's luma_hpp / luma_vpp /
luma_hvpp outputs over every position a search can read, and the analysis must not change at all.  The last test needs
no GPU: it checks the bound arithmetic (x265_b200/csrc/phase_planes.h, compiled here with g++ through
tests/phase_planes_capi.cpp) against the jobs and results of the CPU frame driver."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from common import load_oracle, ptr
from frame_helpers import Workload, cpu_analyse, lambda_for, make_field, MARGIN_X, MARGIN_Y
from me_helpers import mvcost_table

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def cu():
    import x265_b200
    return x265_b200.load()


def make_analyser(cu, wl, amp=0, chroma=False):
    import x265_b200
    p = wl.params
    an = x265_b200.Analyser(cu, wl.W, wl.H, depth=wl.depth, numRefs=p["numRefs"], method=p["method"], subme=p["subme"],
                            merange=p["merange"], rect=p["rect"], qp=p["qp"], lam=lambda_for(p["qp"], wl.depth), amp=amp)
    H, W = wl.H, wl.W
    if chroma:
        an.enable_chroma()
    mx, my = MARGIN_X // 2, MARGIN_Y // 2

    def inner(c):
        return np.ascontiguousarray(c[my:my + H // 2, mx:mx + W // 2])
    for r, ref in enumerate(wl.refs):
        an.set_ref(r, ref[MARGIN_Y:MARGIN_Y + H, MARGIN_X:MARGIN_X + W])
        if chroma:
            an.set_ref_chroma(r, inner(wl.refC[r][0]), inner(wl.refC[r][1]))
    if chroma:
        an.load_chroma(inner(wl.fencC[0]), inner(wl.fencC[1]))
    return an


def results(an):
    return dict(me_out=an.fetch("me_out").copy(), me_packed=np.array(an.me_packed), cu_sse=np.array(an.cu_sse),
                cu_numsig=np.array(an.cu_numsig), cu_ref=np.array(an.cu_ref), intra_cost=np.array(an.intra_cost))


def inner_fenc(wl):
    return np.ascontiguousarray(wl.fenc[MARGIN_Y:MARGIN_Y + wl.H, MARGIN_X:MARGIN_X + wl.W])


@pytest.mark.gpu
@pytest.mark.parametrize("depth", [8, 10])
@pytest.mark.parametrize("size", [(200, 136), (416, 240)])
@pytest.mark.parametrize("kind", ["rand", "max", "zero"])
def test_phase_planes_match_oracle(cu, depth, size, kind, monkeypatch):
    """Every phase plane equals the oracle's 8-tap interpolation (orc_interp_hpp / vpp / hvpp) of plane 0 at every position
    of the built region, which covers the picture and the margins the jobs reach.  All-max inputs exercise the clipping."""
    monkeypatch.setenv("X265CU_ME_PHASEPLANES", "1")
    W, H = size
    O = load_oracle(depth)
    wl = Workload(W, H, depth=depth, numRefs=2, method=3, subme=3, merange=57, rect=1, qp=30, noise=True)
    mx = (1 << depth) - 1
    rng = np.random.default_rng(11 + depth)
    for r in range(2):
        img = {"rand": rng.integers(0, mx + 1, (H, W)), "max": np.full((H, W), mx), "zero": np.zeros((H, W))}[kind]
        wl.refs[r][MARGIN_Y:MARGIN_Y + H, MARGIN_X:MARGIN_X + W] = img
    an = make_analyser(cu, wl)
    an.analyse(inner_fenc(wl), wl.field, stages=1)
    assert an.phase_planes_ms() > 0.0
    pad = 76
    for r in range(2):
        x0, x1, y0, y1 = an.phase_region(r)
        assert -pad <= x0 <= 0 and W <= x1 <= W + pad and -pad <= y0 <= 0 and H <= y1 <= H + pad, (x0, x1, y0, y1)
        assert x0 < -48 and y0 < -48, "the jobs of the left / top CTUs reach into the margins"
        src = an.fetch_phase_plane(r, 0)
        stride = src.shape[1]
        for phase in range(1, 16):
            xf, yf = phase & 3, phase >> 2
            got = an.fetch_phase_plane(r, phase)[MARGIN_Y + y0:MARGIN_Y + y1, MARGIN_X + x0:MARGIN_X + x1]
            want = np.zeros((y1 - y0, x1 - x0), an.dtype)
            for ty in range(0, y1 - y0, 64):
                for tx in range(0, x1 - x0, 64):
                    th, tw = min(64, y1 - y0 - ty), min(64, x1 - x0 - tx)
                    s = ptr(src, (MARGIN_Y + y0 + ty) * stride + MARGIN_X + x0 + tx)
                    d = np.zeros((th, tw), an.dtype)
                    if not yf:
                        O.orc_interp_hpp(s, stride, ptr(d), tw, xf, 8, tw, th)
                    elif not xf:
                        O.orc_interp_vpp(s, stride, ptr(d), tw, yf, 8, tw, th)
                    else:
                        O.orc_interp_hvpp(s, stride, ptr(d), tw, xf, yf, 8, tw, th)
                    want[ty:ty + th, tx:tx + tw] = d
            bad = np.argwhere(got != want)
            assert len(bad) == 0, (r, phase, len(bad), (bad[:4] + [y0, x0]).tolist())
    an.close()


@pytest.mark.gpu
@pytest.mark.timeout(600)
@pytest.mark.parametrize("size,depth,amp,chroma,noise", [
    ((1024, 576), 8, 0, False, False), ((1024, 576), 8, 0, True, True), ((1024, 576), 10, 1, True, False),
    ((1024, 576), 10, 1, False, True), ((1024, 576), 8, 1, True, True),
    ((200, 136), 8, 1, True, True), ((200, 136), 10, 0, True, False), ((200, 136), 8, 0, False, True), ((200, 136), 10, 1, False, False)])
def test_phase_plane_path_equals_interpolating_path(cu, size, depth, amp, chroma, noise, monkeypatch):
    """Analysis with the phase planes (X265CU_ME_PHASEPLANES=1) and with the interpolating kernels (=0) on the same frame:
    every motionEstimate result, CU SSE, coefficient count, best reference and intra cost identical."""
    W, H = size
    wl = Workload(W, H, depth=depth, numRefs=3, method=3, subme=3, merange=57, rect=1, qp=30, noise=noise, amp=amp, chroma=chroma)
    res = {}
    for mode in ("0", "1"):
        monkeypatch.setenv("X265CU_ME_PHASEPLANES", mode)
        an = make_analyser(cu, wl, amp=amp, chroma=chroma)
        an.analyse(inner_fenc(wl), wl.field)
        assert (an.phase_planes_ms() > 0.0) == (mode == "1")
        res[mode] = results(an)
        jobs = an.fetch("jobs")
        an.close()
    a, b = res["0"]["me_out"].reshape(-1, 4), res["1"]["me_out"].reshape(-1, 4)
    bad = np.nonzero((a[:, :3] != b[:, :3]).any(axis=1))[0]
    assert len(bad) == 0, (len(bad), len(a), jobs[bad[:4]].tolist(), a[bad[:4]].tolist(), b[bad[:4]].tolist())
    for k in res["0"]:
        assert np.array_equal(res["0"][k], res["1"][k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("depth", [8, 10])
def test_phase_planes_row_slices_and_reference_updates(cu, depth, monkeypatch):
    """Row slices (each builds only the band its jobs read) reproduce one full run, and after a reference changes (recon_to_ref
    + ref_updated, set_ref) a run equals a fresh analyser's on the new references: the planes are rebuilt every run."""
    monkeypatch.setenv("X265CU_ME_PHASEPLANES", "1")
    W, H = 200, 200                                   # 4 CTU rows, the last one 8 pixels high
    wl = Workload(W, H, depth=depth, numRefs=2, method=3, subme=3, merange=57, rect=1, qp=30, noise=True)
    fenc = inner_fenc(wl)
    full = make_analyser(cu, wl)
    full.analyse(fenc, wl.field)
    want = results(full)
    full.close()

    an = make_analyser(cu, wl)
    for r0, r1 in [(3, 4), (1, 3), (0, 1)]:
        an.analyse_rows(fenc, wl.field, r0, r1)
        box = an.phase_region(0)
        assert box[2] >= r0 * 64 - 80 and box[3] <= min(H, r1 * 64) + 80, (r0, r1, box)
    got = results(an)
    for k in ("me_packed", "cu_sse", "cu_numsig", "cu_ref", "intra_cost"):
        assert np.array_equal(got[k], want[k]), k

    # reference 1 <- the CU-16 reconstruction of this frame, reference 0 <- another picture
    an.recon_to_ref(2, 1, 0, an.ctu_rows)
    an.ref_updated(1)
    new1 = an.fetch_phase_plane(1, 0)[MARGIN_Y:MARGIN_Y + H, MARGIN_X:MARGIN_X + W].copy()
    new0 = np.ascontiguousarray(wl.fenc[MARGIN_Y:MARGIN_Y + H, MARGIN_X:MARGIN_X + W][::-1, :])
    an.set_ref(0, new0)
    an.analyse(fenc, wl.field)
    got = results(an)
    an.close()
    wl.refs[0][MARGIN_Y:MARGIN_Y + H, MARGIN_X:MARGIN_X + W] = new0
    wl.refs[1][MARGIN_Y:MARGIN_Y + H, MARGIN_X:MARGIN_X + W] = new1
    fresh = make_analyser(cu, wl)
    fresh.analyse(fenc, wl.field)
    want = results(fresh)
    fresh.close()
    for k in want:
        assert np.array_equal(got[k], want[k]), k


# ---------------- CPU: the bound arithmetic against the CPU frame driver's jobs ----------------

@pytest.fixture(scope="module")
def capi(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("pp") / "libpp.so")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-o", so, os.path.join(HERE, "phase_planes_capi.cpp")])
    L = C.CDLL(so)
    L.pp_pad.restype = C.c_int
    return L


@pytest.mark.parametrize("name,W,H,depth,refs,method,subme,amp", [
    ("c3", 3840, 128, 8, 4, 3, 3, 0),                 # the c3 / c4 geometries at reduced height
    ("c4", 3840, 128, 10, 5, 3, 4, 1),
    ("odd-hex", 200, 136, 8, 2, 1, 7, 1),             # HEX / DIA move x without a range check; subme 7 = the longest sub-pel walk
    ("odd-dia", 200, 136, 10, 2, 0, 7, 0)])
def test_job_boxes_cover_every_read(capi, name, W, H, depth, refs, method, subme, amp):
    """Over the jobs the CPU frame driver emits: (1) every job box lies in the region the analyser builds, whose 8-tap
    support stays inside the plane margins; (2) every pre-check candidate (the clipped MVP, its full-pel rounding, MV 0,
    the clipped neighbour candidates) reads inside its job's box; (3) so does the final vector of every search together
    with the sub-pel neighbours its last rounds compared (+-2 quarter-pels in x, y clipped to the range)."""
    O = load_oracle(depth)
    qp = 30
    wl = Workload(W, H, depth=depth, numRefs=refs, method=method, subme=subme, merange=57, rect=1, qp=qp, amp=amp)
    wl.field = make_field(W, H, refs, seed=3) * 4                # larger predictors: more searches clipped at the picture edge
    res = cpu_analyse(O, "orc_analyse_frame", wl, mvcost_table(O, lambda_for(qp, depth)), threads=8, stages=1)
    jobs, me = res["jobs"], res["me_out"]
    n = len(jobs)
    assert n > 0
    y, x = np.divmod(jobs["offset"].astype(np.int64), wl.stride)
    w, h = jobs["pw"].astype(np.int64), jobs["ph"].astype(np.int64)
    mn, mx = jobs["mvmin"].astype(np.int64), jobs["mvmax"].astype(np.int64)
    desc = np.stack([x, y, w, h, mn[:, 0], mn[:, 1], mx[:, 0], mx[:, 1]], axis=1).astype(np.int32)
    boxes = np.zeros((n, 4), np.int32)
    capi.pp_job_boxes(desc.ctypes.data_as(C.c_void_p), n, boxes.ctypes.data_as(C.c_void_p))
    reg = np.zeros(4, np.int32)
    capi.pp_region(W, H, reg.ctypes.data_as(C.c_void_p))
    pad = capi.pp_pad()
    assert list(reg) == [-pad, W + pad, -pad, H + pad]
    # (1) region inside the allocation with the filter support: 3 before, 4 after every position
    assert reg[0] - 3 >= -MARGIN_X and reg[2] - 3 >= -MARGIN_Y
    assert reg[1] - 1 + 4 < wl.stride - MARGIN_X and reg[3] - 1 + 4 < H + MARGIN_Y
    assert (boxes[:, 0] >= reg[0]).all() and (boxes[:, 1] <= reg[1]).all()
    assert (boxes[:, 2] >= reg[2]).all() and (boxes[:, 3] <= reg[3]).all()

    def inside(qx, qy, sel=None):
        bx, by = x + (qx >> 2), y + (qy >> 2)
        ok = (bx >= boxes[:, 0]) & (bx + w <= boxes[:, 1]) & (by >= boxes[:, 2]) & (by + h <= boxes[:, 3])
        return ok if sel is None else (ok | ~sel)

    # (2) pre-checks (motion.cpp:771-814)
    qmin, qmax = mn * 4, mx * 4
    pmv = np.clip(jobs["qmvp"].astype(np.int64), qmin, qmax)
    assert inside(pmv[:, 0], pmv[:, 1]).all()
    assert inside(((pmv[:, 0] + 2) >> 2) * 4, ((pmv[:, 1] + 2) >> 2) * 4).all()
    zero = np.zeros(n, np.int64)
    assert inside(zero, zero).all()
    for k in range(4):
        sel = jobs["numCand"] > k
        c = np.clip(jobs["mvc"][:, 2 * k:2 * k + 2].astype(np.int64), qmin, qmax)
        assert inside(c[:, 0], c[:, 1], sel).all(), k
    # (3) search results and their last sub-pel neighbours
    bx, by = me[:, 1].astype(np.int64), me[:, 2].astype(np.int64)
    for dx in (-2, -1, 0, 1, 2):
        for dy in (-2, -1, 0, 1, 2):
            qy = np.clip(by + dy, qmin[:, 1], qmax[:, 1])
            assert inside(bx + dx, qy).all(), (dx, dy)
